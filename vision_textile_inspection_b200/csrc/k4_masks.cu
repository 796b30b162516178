// K4 -- mask-coefficient x prototype contraction fused with sigmoid, box crop, 4x bilinear upsample, > 0.5 threshold
// AND the nearest-resize mask statistics of the measure stage, so full-resolution masks are never materialised.
//
// Replaces (SURVEY.md 8a U6, M2, M3, M4): ultralytics ops.process_mask / crop_mask / F.interpolate / gt_(0.5)
// (variant A), reached from measurement.py:208-210 and consumed at :74-75, and then
//   measurement.py:78-81   cv2.resize(mask, (w,h), INTER_NEAREST) > 0        -> per-axis multiplicity LUTs
//   measurement.py:160-185 union of fabric masks + lower envelope            -> atomicMax per letterbox column
//   (Utils/check_stitch_distance.py:238-251 upper envelope                   -> atomicMin)
//   measurement.py:304-314 cv2.moments m00/m10/m01 + occupied column range   -> exact int64 sums
// Oracle: oracle/ultra_ref.py process_mask (real torch ops) + oracle/measure_port.py; parity bar IoU >= 0.999.
//
// v4: the work is a flat list of UNITS written by K3, one per (kept detection, VTI_K4_UR x VTI_K4_UC block of
// interpolation cells inside the detection's crop window).  The box crop makes the contraction sparse -- cfg2 needs
// ~1 % of the dense N x 32 x ph x pw products -- so the kernel is organised around the crop, not around a dense GEMM:
// one warp per unit, grid-stride over the list, no block barriers, no shared-memory staging of the prototypes
// (each unit reads its (UR+1) x (UC+1) x 32 prototype corner values straight from global/L2, 32 independent
// coalesced loads per lane).  Per unit:
//   (1) one lane per corner pixel: 32-term contraction + sigmoid + crop                       -> per-warp s_c
//   (2) one lane per interpolation cell (the 4x4 output pixels between four prototype pixels).  A cell whose four
//       corners are all > 0.5 (+margin) is entirely set, all < 0.5 (-margin) entirely clear -- bilinear weights are a
//       convex combination -- and its contribution to m00/m10/m01, the column extent and the envelope is closed-form
//       from prefix sums of the multiplicity tables; only boundary cells evaluate their 16 pixels, and those are
//       shared out over the warp two cells at a time, one pixel per lane (the mask edge crosses a unit as a line, so
//       few lanes hold one).
//   (3) warp reduction (three REDUX on 32-bit per-unit sums), one set of 64-bit global atomics per unit.
// Optional bit-packed mask export: cells OR their bits into the (pre-zeroed) global mask words.
// Mask variant B (vti_params.mask_variant = 1, newer Ultralytics: SURVEY 8a U6) is the same kernel in another threshold
// domain (template parameter VB): the corner values are the raw logits (no sigmoid), cropped-out corners are 0, the
// threshold is > 0.0; K5 then drops the detections whose letterbox mask stayed empty (flag VTI_F_LB_MASK never set).
// Bound: the prototype read (128 B per prototype pixel touched); algorithmic bytes 128*ph*pw per frame.
#include <climits>
#include <cstdlib>

#include "vti_internal.h"

namespace {

constexpr int K4_THREADS = 256;
constexpr int NWARP = K4_THREADS / 32;
constexpr int UR = VTI_K4_UR, UC = VTI_K4_UC;
constexpr int SCW = UC + 1;                 // corner columns per unit
constexpr float MARGIN = 1e-5f;             // >> fp32 rounding of the lerp; cells within the margin are evaluated per pixel
constexpr float MARGIN_B = 1e-3f;           // variant B: logits (|values| up to ~30) instead of probabilities

struct K4Args {
    const float* proto;         // [B][32][ph][pw]
    vti_det* dets;              // [B][max_det]
    const float* det_coef;      // [B][max_det][32]
    const uint4* units;
    const int32_t* unit_count;
    AxisLut ly, lx;
    int32_t* env;               // [B][LW] frame-row envelope per letterbox column
    uint32_t* masks;            // optional [B][max_det][LH][LW/32]
    int LH, LW, ph, pw, max_det;
    int upper;                  // envelope mode
};

__global__ void k4_zero_masks_kernel(uint32_t* masks, const int32_t* counts, int max_det, size_t words_per_mask) {
    const int k = blockIdx.x, b = blockIdx.y;
    if (k >= counts[b]) return;
    uint4* p = reinterpret_cast<uint4*>(masks + ((size_t)b * max_det + k) * words_per_mask);
    const size_t n4 = words_per_mask / 4;
    for (size_t i = threadIdx.x; i < n4; i += blockDim.x) p[i] = make_uint4(0u, 0u, 0u, 0u);
}

// Phases 2 and 3 of a unit: classify the interpolation cells from the corner values `sc` (pitch SCW), accumulate the
// nearest-resize statistics, flush the unit's fabric envelope and reduce across the warp.
template <bool EXPORT, bool VB>
__device__ __forceinline__ void unit_cells(const K4Args& a, int b, int k, vti_det* __restrict__ det, bool fabric, int R0,
                                           int C0, int nr, int ncw, const float* sc, int* envw, int lane) {
    const int ex0 = 4 * C0 - 2;                            // first output column of the unit
    constexpr float THR = VB ? 0.0f : 0.5f, MRG = VB ? MARGIN_B : MARGIN;
    bool any = false;                                      // a letterbox pixel of this detection is set
    // (2) cells
    const int ncc = ncw - 1;
    const float inv_ncc = 1.0f / (float)ncc;
    // per-unit sums fit 32 bits (<= 1024 pixels x multiplicity^2 x frame size; vti_create refuses geometries that do not),
    // so the warp reduction is three REDUX instructions instead of thirty 64-bit shuffle-adds
    unsigned m00 = 0u, m10 = 0u, m01 = 0u;
    int cmin = INT_MAX, cmax = -1;
    uint32_t* __restrict__ mrow = EXPORT ? a.masks + ((size_t)b * a.max_det + k) * a.LH * (a.LW / 32) : nullptr;
    const int ncells = (nr - 1) * ncc;
    for (int i0 = 0; i0 < ncells; i0 += 32) {              // warp-uniform trip count: the boundary cells are shared out below
        const int i = i0 + lane;
        const int r = (int)(((float)i + 0.5f) * inv_ncc), c = i - r * ncc;
        // cell (R, C) covers output rows 4R-2 .. 4R+1 and cols 4C-2 .. 4C+1, clipped to the image
        const int cy_first = 4 * (R0 + r) - 2, cx_first = 4 * (C0 + c) - 2;
        const int ya = max(cy_first, 0), yb = min(cy_first + 3, a.LH - 1);
        const int xa = max(cx_first, 0), xb = min(cx_first + 3, a.LW - 1);
        const bool valid = i < ncells && ya <= yb && xa <= xb;
        float c00 = 0.0f, c01 = 0.0f, c10 = 0.0f, c11 = 0.0f;
        if (valid) {
            c00 = sc[r * SCW + c]; c01 = sc[r * SCW + c + 1];
            c10 = sc[(r + 1) * SCW + c]; c11 = sc[(r + 1) * SCW + c + 1];
        }
        const float vmin = fminf(fminf(c00, c01), fminf(c10, c11));
        const float vmax = fmaxf(fmaxf(c00, c01), fmaxf(c10, c11));
        const bool full = valid && vmin > THR + MRG;
        if (full) {
            any = true;
            // fully set: closed form from the prefix sums of the nearest-resize multiplicity tables
            const int f_cy = a.ly.pc[yb + 1] - a.ly.pc[ya], f_sy = a.ly.ps[yb + 1] - a.ly.ps[ya];
            const int f_cx = a.lx.pc[xb + 1] - a.lx.pc[xa], f_sx = a.lx.ps[xb + 1] - a.lx.ps[xa];
            m00 += f_cy * f_cx; m10 += f_cy * f_sx; m01 += f_sy * f_cx;
            if (f_cy > 0 && f_cx > 0) {
                cmin = min(cmin, a.lx.next_first[xa]); cmax = max(cmax, a.lx.prev_last[xb]);
                if (fabric) {
                    const int f_env = a.upper ? a.ly.next_first[ya] : a.ly.prev_last[yb];
                    for (int X = xa; X <= xb; ++X)
                        if (a.lx.cnt[X] > 0) {
                            if (a.upper) atomicMin(&envw[X - ex0], f_env);
                            else atomicMax(&envw[X - ex0], f_env);
                        }
                }
            }
            if (EXPORT) {
                const unsigned long long bits = ((1ull << (xb - xa + 1)) - 1ull) << (xa & 31);
                for (int Y = ya; Y <= yb; ++Y) {
                    uint32_t* wp = mrow + (size_t)Y * (a.LW / 32) + (xa >> 5);
                    atomicOr(wp, (unsigned)bits);
                    if ((unsigned)(bits >> 32)) atomicOr(wp + 1, (unsigned)(bits >> 32));
                }
            }
        }
        // Boundary cells evaluate their 16 pixels (torch upsample_bilinear2d, align_corners=False, scale 1/4).  Few lanes
        // of a warp hold one -- the mask edge crosses a unit as a line -- so the warp takes them two at a time, one
        // pixel per lane, instead of every holder looping over its 16 pixels with the other lanes idle.
        unsigned bm = __ballot_sync(0xffffffffu, valid && !full && vmax >= THR - MRG);
        while (bm) {
            const int s0 = __ffs(bm) - 1;
            bm &= bm - 1;
            const bool pair = bm != 0u;
            const int s1 = pair ? __ffs(bm) - 1 : s0;
            bm &= bm - 1;
            const int src = lane < 16 ? s0 : s1;
            const float q00 = __shfl_sync(0xffffffffu, c00, src), q01 = __shfl_sync(0xffffffffu, c01, src);
            const float q10 = __shfl_sync(0xffffffffu, c10, src), q11 = __shfl_sync(0xffffffffu, c11, src);
            const int rc = __shfl_sync(0xffffffffu, (r << 16) | c, src);
            const int py = (lane >> 2) & 3, px = lane & 3;
            const int Y = 4 * (R0 + (rc >> 16)) - 2 + py, X = 4 * (C0 + (rc & 0xFFFF)) - 2 + px;
            if ((lane < 16 || pair) && Y >= 0 && Y < a.LH && X >= 0 && X < a.LW) {
                const float ly1 = (float)(2 * py + 1) * 0.125f, lx1 = (float)(2 * px + 1) * 0.125f;
                const float top = (1.0f - lx1) * q00 + lx1 * q01;
                const float bot = (1.0f - lx1) * q10 + lx1 * q11;
                const float v = (1.0f - ly1) * top + ly1 * bot;
                if (v > THR) {
                    any = true;
                    const int cY = a.ly.cnt[Y], sY = a.ly.sum[Y], cX = a.lx.cnt[X];
                    m00 += cY * cX; m10 += cY * a.lx.sum[X]; m01 += sY * cX;
                    if (cY > 0 && cX > 0) {
                        cmin = min(cmin, a.lx.first[X]);
                        cmax = max(cmax, a.lx.last[X]);
                        if (fabric) {
                            if (a.upper) atomicMin(&envw[X - ex0], a.ly.first[Y]);
                            else atomicMax(&envw[X - ex0], a.ly.last[Y]);
                        }
                    }
                    if (EXPORT) atomicOr(mrow + (size_t)Y * (a.LW / 32) + (X >> 5), 1u << (X & 31));
                }
            }
        }
    }
    if (fabric) {                                       // one RED per touched column and unit
        __syncwarp();
        int32_t* __restrict__ env = a.env + (size_t)b * a.LW;
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
            const int ev = envw[lane + 32 * hh], X = ex0 + lane + 32 * hh;
            if (a.upper) { if (ev != INT_MAX) atomicMin(env + X, ev); }
            else { if (ev >= 0) atomicMax(env + X, ev); }
        }
    }
    // (3) warp reduction, one set of global atomics per unit
    if (__any_sync(0xffffffffu, any) && lane == 0) atomicOr(&det->flags, VTI_F_LB_MASK);
    m00 = __reduce_add_sync(0xffffffffu, m00);
    if (m00 > 0u) {
        m10 = __reduce_add_sync(0xffffffffu, m10);
        m01 = __reduce_add_sync(0xffffffffu, m01);
        cmin = __reduce_min_sync(0xffffffffu, cmin);
        cmax = __reduce_max_sync(0xffffffffu, cmax);
        if (lane == 0) {
            atomicAdd((unsigned long long*)&det->m00, (unsigned long long)m00);
            atomicAdd((unsigned long long*)&det->m10, (unsigned long long)m10);
            atomicAdd((unsigned long long*)&det->m01, (unsigned long long)m01);
            atomicMin(&det->col_min, cmin);
            atomicMax(&det->col_max, cmax);
        }
    }
}

template <bool EXPORT, bool VB>
__global__ void __launch_bounds__(K4_THREADS, 1024 / K4_THREADS) k4_units_kernel(const K4Args a) {
    __shared__ float s_c[NWARP][(UR + 1) * SCW];
    __shared__ __align__(16) float s_coef[NWARP][VTI_NM];   // registers go to the 32 in-flight prototype loads
    __shared__ int s_envw[NWARP][4 * UC];                   // fabric envelope of the unit's columns (one RED each)
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int total = *a.unit_count;
    const int nwarps = gridDim.x * NWARP;
    float* sc = s_c[warp];
    const size_t plane = (size_t)a.ph * a.pw;
    const unsigned long long plane_bytes = plane * sizeof(float);

    for (int u = blockIdx.x * NWARP + warp; u < total; u += nwarps) {
        const uint4 un = __ldg(a.units + u);
        const int b = (int)(un.x & 0x7FFFu), k = (int)(un.x >> 16), br = (int)(un.y & 0xFFFFu), bc = (int)(un.y >> 16);
        const bool fabric = (un.x & 0x8000u) != 0u;
        vti_det* __restrict__ det = a.dets + (size_t)b * a.max_det + k;
        VtiWindow w;                                        // the crop window travels in the unit record
        w.cx_lo = (int)(un.z & 0xFFFFu); w.cy_lo = (int)(un.z >> 16);
        w.cx_hi = (int)(un.w & 0xFFFFu); w.cy_hi = (int)(un.w >> 16);
        // cells of this unit (global cell coordinates) and their corner rectangle
        const int R0 = w.cy_lo + br * UR, R1 = min(R0 + UR - 1, w.cy_hi + 1);
        const int C0 = w.cx_lo + bc * UC, C1 = min(C0 + UC - 1, w.cx_hi + 1);
        const int nr = R1 - R0 + 2, ncw = C1 - C0 + 2;
        const float inv_ncw = 1.0f / (float)ncw;
        __syncwarp();
        s_coef[warp][lane] = __ldg(a.det_coef + ((size_t)b * a.max_det + k) * VTI_NM + lane);
        if (fabric) { s_envw[warp][lane] = a.upper ? INT_MAX : -1; s_envw[warp][lane + 32] = a.upper ? INT_MAX : -1; }
        const float* __restrict__ proto = a.proto + (size_t)b * VTI_NM * plane;
        __syncwarp();
        // (1) logits -> sigmoid -> crop over the corner rectangle (replicate-clamped at the plane border)
        for (int i = lane; i < nr * ncw; i += 32) {
            const int r = (int)(((float)i + 0.5f) * inv_ncw), c = i - r * ncw;
            const int py = min(max(R0 - 1 + r, 0), a.ph - 1), px = min(max(C0 - 1 + c, 0), a.pw - 1);
            float v = 0.0f;
            if (py >= w.cy_lo && py <= w.cy_hi && px >= w.cx_lo && px <= w.cx_hi) {
                // walk the 32 channel planes with one 64-bit add per load (the compiler's own q * plane indexing costs
                // a wide multiply + two LEAs per load)
                const char* src = reinterpret_cast<const char*>(proto + (size_t)py * a.pw + px);
                float pv[VTI_NM];
#pragma unroll
                for (int q = 0; q < VTI_NM; ++q) {
                    pv[q] = __ldg(reinterpret_cast<const float*>(src));
                    asm volatile("add.u64 %0, %0, %1;" : "+l"(src) : "l"(plane_bytes));
                }
                float acc = 0.0f;
#pragma unroll
                for (int q = 0; q < VTI_NM; q += 4) {
                    const float4 cf = *reinterpret_cast<const float4*>(&s_coef[warp][q]);
                    acc = fmaf(cf.x, pv[q], acc); acc = fmaf(cf.y, pv[q + 1], acc);
                    acc = fmaf(cf.z, pv[q + 2], acc); acc = fmaf(cf.w, pv[q + 3], acc);
                }
                v = VB ? acc : 1.0f / (1.0f + expf(-acc));
            }
            sc[r * SCW + c] = v;
        }
        __syncwarp();
        unit_cells<EXPORT, VB>(a, b, k, det, fabric, R0, C0, nr, ncw, sc, s_envw[warp], lane);
    }
}


// Host-buffer path: copy, per frame and channel, the union rectangle of the crop windows (the only prototype values the
// unit kernel reads) from device-mapped pinned host memory into the device prototype buffer.  Rows are widened to
// 16-byte boundaries for float4 accesses; blockIdx = (channel, frame), warps take rows.
__global__ void __launch_bounds__(256) k4_fetch_proto_kernel(const float* __restrict__ src, float* __restrict__ dst,
                                                             const int4* __restrict__ bbox, int ph, int pw) {
    const int q = blockIdx.x, b = blockIdx.y;
    const int4 bb = bbox[b];
    if (bb.z < bb.x || bb.w < bb.y) return;
    const int x0 = bb.x & ~3, x1 = min((bb.z + 4) & ~3, pw);               // [x0, x1) float4-aligned (pw % 4 == 0)
    const int n4 = (x1 - x0) >> 2;
    const size_t plane = (size_t)ph * pw, base = ((size_t)b * VTI_NM + q) * plane;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int y = bb.y + warp; y <= bb.w; y += 8) {
        const float4* s4 = reinterpret_cast<const float4*>(src + base + (size_t)y * pw + x0);
        float4* d4 = reinterpret_cast<float4*>(dst + base + (size_t)y * pw + x0);
        for (int i = lane; i < n4; i += 32) d4[i] = s4[i];
    }
}

}  // namespace

int vti_launch_k4(vti_handle* h, const float* proto, int B, vti_det* dets, const int32_t* counts, uint32_t* masks,
                  cudaStream_t s) {
    K4Args a;
    a.proto = proto;
    a.dets = dets;
    a.det_coef = h->d_det_coef;
    a.units = h->d_units;
    a.unit_count = h->d_cand_count + h->p.max_batch;
    a.ly = h->lutY; a.lx = h->lutX;
    a.env = h->d_env;
    a.masks = masks;
    a.LH = h->g.LH; a.LW = h->g.LW; a.ph = h->g.ph; a.pw = h->g.pw; a.max_det = h->p.max_det;
    a.upper = (h->p.variant == 1);
    if (masks) {
        const size_t wpm = (size_t)a.LH * (a.LW / 32);
        k4_zero_masks_kernel<<<dim3(a.max_det, B), 256, 0, s>>>(masks, counts, a.max_det, wpm);
        h->launches++;
    }
    // Alone, K4 is fastest with four 8-warp CTAs per SM (66 vs 88 us on cfg2), but those fill every register file and
    // K1 -- which runs beside it on the pre stream -- then waits for K4 to finish.  Two CTAs per SM leave half of each SM
    // to K1: the K1 || K2-K5 step is 2.3 % faster on cfg2 / cfg3.  When K1 has little to do (no remap, no resize: cfg4)
    // K4 is on the critical path and keeps the four.
    const bool vb = h->p.mask_variant == 1;
    const bool k1_heavy = h->p.undistort || h->p.frame_w != h->g.new_w || h->p.frame_h != h->g.new_h;
    const int grid = (k1_heavy ? 2 : 4) * h->num_sms;
    if (masks && vb) k4_units_kernel<true, true><<<grid, K4_THREADS, 0, s>>>(a);
    else if (masks) k4_units_kernel<true, false><<<grid, K4_THREADS, 0, s>>>(a);
    else if (vb) k4_units_kernel<false, true><<<grid, K4_THREADS, 0, s>>>(a);
    else k4_units_kernel<false, false><<<grid, K4_THREADS, 0, s>>>(a);
    h->launches++;
    VTI_CUDA(cudaGetLastError());
    return VTI_OK;
}

int vti_launch_fetch_proto(vti_handle* h, const float* host_proto_mapped, float* dev_proto, int B, cudaStream_t s) {
    if (h->g.pw % 4) {                                     // unaligned rows: plain copy of everything
        VTI_CUDA(cudaMemcpyAsync(dev_proto, host_proto_mapped, sizeof(float) * (size_t)B * VTI_NM * h->g.ph * h->g.pw,
                                 cudaMemcpyDefault, s));
        return VTI_OK;
    }
    k4_fetch_proto_kernel<<<dim3(VTI_NM, B), 256, 0, s>>>(host_proto_mapped, dev_proto, h->d_proto_bbox, h->g.ph, h->g.pw);
    h->launches++;
    VTI_CUDA(cudaGetLastError());
    return VTI_OK;
}

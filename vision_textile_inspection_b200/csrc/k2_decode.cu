// K2 -- YOLOv8 head tail: class sigmoid + confidence filter (warp ballot, warp-aggregated compaction) and, for the
// surviving anchors only, DFL softmax-expectation + dist2bbox + xywh->xyxy.
//
// Replaces (SURVEY.md 8a U3 + the prelude of U4): ultralytics Detect._inference / DFL.forward / dist2bbox and the
// `xc = amax(cls) > conf` selection of ops.non_max_suppression, reached from measurement.py:208-210.
// Spec: oracle/post_spec.py decode_spec / candidates_spec -- every float op below is the same single-rounded
// IEEE op in the same order (no FMA contraction), so boxes and scores are bit-identical to the spec.
//
// Two kernels:
//   k2_decode_kernel  4 anchors per thread (a warp covers 32 consecutive anchors of one level: coalesced 128-byte
//                     class-logit lines, all of a thread's loads in flight at once), class sigmoid + `> conf`, one
//                     atomicAdd per block to append the (score bits | ~anchor | class) keys.  The order inside the
//                     list is irrelevant: K3 sorts by the composite key, which reproduces torchvision's stable
//                     descending sort over ascending anchor order.
//   k2_box_kernel     DFL softmax expectation of the CANDIDATES only, over the flat per-frame lists: one lane per
//                     (candidate, box side), the four sides meet through shuffles.  (Fused into the classifying
//                     kernel, the block that owned a row of stitches decoded ~400 candidates alone.)
#include "vti_internal.h"

namespace {

constexpr int K2_THREADS = 256;
constexpr int K2_NA = 4;                    // anchors per thread
constexpr int K2_SPAN = K2_NA * K2_THREADS; // anchors per block

struct K2Args {
    const float* lvl[3];
    int lvl_h[3], lvl_w[3];
    int a_begin[4];            // anchor offset of each level, a_begin[3] = A
    int nc, A, cap, cap_pad;
    float conf;
    int32_t* cand_count;       // [B]
    unsigned long long* cand_key;   // [B][cap]
    float4* cand_box;          // [B][A]
};

__global__ void __launch_bounds__(K2_THREADS) k2_decode_kernel(const K2Args a) {
    __shared__ int s_cnt, s_base;
    __shared__ int s_idx[K2_SPAN];             // candidate -> index inside the level | cls << 24
    __shared__ float s_best[K2_SPAN];

    const int b = blockIdx.y, tid = threadIdx.x, lane = tid & 31;
    // blocks are laid out per level so that a warp never straddles two levels; a block covers K2_SPAN anchors
    int blk = blockIdx.x, l = 0;
#pragma unroll
    for (int i = 0; i < 2; ++i) {
        const int nblk = (a.a_begin[l + 1] - a.a_begin[l] + K2_SPAN - 1) / K2_SPAN;
        if (blk >= nblk) { blk -= nblk; ++l; }
    }
    const int plane = a.lvl_h[l] * a.lvl_w[l];
    const float* __restrict__ base = a.lvl[l] + (size_t)b * (64 + a.nc) * plane;
    if (tid == 0) s_cnt = 0;
    __syncthreads();

    // ---- phase 1: class sigmoid, confidence filter, block-local candidate list.  K2_NA anchors per thread with all
    //      their class logits in flight at once (the kernel is a chain of two memory latencies, not a bandwidth problem)
    if (a.nc <= 4) {
        float lg[K2_NA][4];
#pragma unroll
        for (int k = 0; k < K2_NA; ++k) {
            const int i = blk * K2_SPAN + k * K2_THREADS + tid;
#pragma unroll
            for (int c = 0; c < 4; ++c)
                lg[k][c] = (c < a.nc && i < plane) ? __ldg(base + (size_t)(64 + c) * plane + i) : -100.0f;
        }
#pragma unroll
        for (int k = 0; k < K2_NA; ++k) {
            const int i = blk * K2_SPAN + k * K2_THREADS + tid;
            float best = 0.0f;
            int cls = 0;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                if (c < a.nc) {
                    const float pr = vti_sigmoid_spec(lg[k][c]);
                    if (c == 0 || pr > best) { best = pr; cls = c; }     // first maximum wins, as torch.max
                }
            }
            const bool cand = (i < plane) && (best > a.conf);
            const unsigned m = __ballot_sync(0xffffffffu, cand);
            if (m != 0u) {
                int p0 = 0;
                if (lane == 0) p0 = atomicAdd(&s_cnt, __popc(m));
                p0 = __shfl_sync(0xffffffffu, p0, 0);
                if (cand) {
                    const int p = p0 + __popc(m & ((1u << lane) - 1u));
                    s_idx[p] = (int)((unsigned)i | ((unsigned)cls << 24));
                    s_best[p] = best;
                }
            }
        }
    } else {
        for (int k = 0; k < K2_NA; ++k) {
            const int i = blk * K2_SPAN + k * K2_THREADS + tid;
            float best = 0.0f;
            int cls = 0;
            if (i < plane)
                for (int c = 0; c < a.nc; ++c) {
                    const float pr = vti_sigmoid_spec(__ldg(base + (size_t)(64 + c) * plane + i));
                    if (c == 0 || pr > best) { best = pr; cls = c; }
                }
            const bool cand = (i < plane) && (best > a.conf);
            const unsigned m = __ballot_sync(0xffffffffu, cand);
            if (m != 0u) {
                int p0 = 0;
                if (lane == 0) p0 = atomicAdd(&s_cnt, __popc(m));
                p0 = __shfl_sync(0xffffffffu, p0, 0);
                if (cand) {
                    const int p = p0 + __popc(m & ((1u << lane) - 1u));
                    s_idx[p] = (int)((unsigned)i | ((unsigned)cls << 24));
                    s_best[p] = best;
                }
            }
        }
    }
    __syncthreads();
    const int n = s_cnt;
    if (n == 0) return;
    if (tid == 0) s_base = atomicAdd(a.cand_count + b, n);
    __syncthreads();
    // keys of this block's candidates (the order inside the list is irrelevant: K3 sorts)
    for (int c = tid; c < n; c += K2_THREADS) {
        const int slot = s_base + c;
        if (slot < a.cap) {
            const int anchor = a.a_begin[l] + (s_idx[c] & 0xFFFFFF);
            a.cand_key[(size_t)b * a.cap_pad + slot] = ((unsigned long long)__float_as_uint(s_best[c]) << 32) |
                                                        ((unsigned long long)(0xFFFFFFu - (unsigned)anchor) << 8) |
                                                        ((unsigned)s_idx[c] >> 24);     // unsigned: classes >= 128 must not sign-extend
        }
    }
}

// K2b -- DFL decode of the candidates only, over the flat per-frame candidate lists: one lane per (candidate, box
// side), so the 16-bin softmax expectations run on full warps and are spread over the whole grid.  (Fused into the
// classifying kernel, the block that owned a row of stitches decoded ~400 candidates alone: 37 us of one SM.)
__global__ void __launch_bounds__(K2_THREADS) k2_box_kernel(const K2Args a) {
    const int b = blockIdx.y, tid = threadIdx.x, lane = tid & 31;
    const int n = min(a.cand_count[b], a.cap);
    const unsigned long long* __restrict__ keys = a.cand_key + (size_t)b * a.cap_pad;
    for (int it0 = blockIdx.x * K2_THREADS; it0 < 4 * n; it0 += gridDim.x * K2_THREADS) {
        const int item = it0 + tid;
        const bool act = item < 4 * n;
        const int side = item & 3;
        int anchor = 0, l = 0;
        if (act) {
            anchor = 0xFFFFFF - (int)((keys[item >> 2] >> 8) & 0xFFFFFFull);
            l = (anchor >= a.a_begin[1]) + (anchor >= a.a_begin[2]);
        }
        const int plane = a.lvl_h[l] * a.lvl_w[l];
        const int ci = anchor - a.a_begin[l];
        const float* __restrict__ base = a.lvl[l] + (size_t)b * (64 + a.nc) * plane;
        float dside = 0.0f;
        if (act) {
            float v[16];
#pragma unroll
            for (int k = 0; k < 16; ++k) v[k] = __ldg(base + (size_t)(side * 16 + k) * plane + ci);
            float mx = v[0];
#pragma unroll
            for (int k = 1; k < 16; ++k) mx = fmaxf(mx, v[k]);
            float S = 0.0f;
#pragma unroll
            for (int k = 0; k < 16; ++k) {
                v[k] = vti_exp_spec(__fsub_rn(v[k], mx));
                S = __fadd_rn(S, v[k]);
            }
            float acc = 0.0f;
#pragma unroll
            for (int k = 0; k < 16; ++k) acc = __fadd_rn(acc, __fmul_rn((float)k, __fdiv_rn(v[k], S)));
            dside = acc;
        }
        // the four sides of a candidate sit in four consecutive lanes
        const int l0 = lane & ~3;
        const float d0 = __shfl_sync(0xffffffffu, dside, l0), d1 = __shfl_sync(0xffffffffu, dside, l0 + 1);
        const float d2 = __shfl_sync(0xffffffffu, dside, l0 + 2), d3 = __shfl_sync(0xffffffffu, dside, l0 + 3);
        if (act && side == 0) {
            const int gy = ci / a.lvl_w[l], gx = ci - gy * a.lvl_w[l];
            const float ax = __fadd_rn((float)gx, 0.5f), ay = __fadd_rn((float)gy, 0.5f);
            const float x1 = __fsub_rn(ax, d0), y1 = __fsub_rn(ay, d1);
            const float x2 = __fadd_rn(ax, d2), y2 = __fadd_rn(ay, d3);
            const float st = (float)(8 << l);
            const float cx = __fmul_rn(__fdiv_rn(__fadd_rn(x1, x2), 2.0f), st);
            const float cy = __fmul_rn(__fdiv_rn(__fadd_rn(y1, y2), 2.0f), st);
            const float w = __fmul_rn(__fsub_rn(x2, x1), st);
            const float hh = __fmul_rn(__fsub_rn(y2, y1), st);
            const float hw2 = __fdiv_rn(w, 2.0f), hh2 = __fdiv_rn(hh, 2.0f);
            a.cand_box[(size_t)b * a.A + anchor] =
                make_float4(__fsub_rn(cx, hw2), __fsub_rn(cy, hh2), __fadd_rn(cx, hw2), __fadd_rn(cy, hh2));
        }
    }
}

}  // namespace

int vti_launch_k2(vti_handle* h, const float* p3, const float* p4, const float* p5, int B, cudaStream_t s) {
    K2Args a;
    a.lvl[0] = p3; a.lvl[1] = p4; a.lvl[2] = p5;
    int off = 0, nblk = 0;
    for (int l = 0; l < 3; ++l) {
        a.lvl_h[l] = h->g.lvl_h[l];
        a.lvl_w[l] = h->g.lvl_w[l];
        a.a_begin[l] = off;
        off += a.lvl_h[l] * a.lvl_w[l];
        nblk += (a.lvl_h[l] * a.lvl_w[l] + K2_SPAN - 1) / K2_SPAN;
    }
    a.a_begin[3] = off;
    a.nc = h->p.nc; a.A = h->g.A; a.cap = h->g.max_candidates; a.cap_pad = vti_k3_cap_pad(a.cap);
    a.conf = h->p.conf;
    a.cand_count = h->d_cand_count;
    a.cand_key = h->d_cand_key;
    a.cand_box = h->d_cand_box;
    VTI_CUDA(cudaMemsetAsync(h->d_cand_count, 0, sizeof(int32_t) * (h->p.max_batch + 1), s));   // + K4 unit counter
    k2_decode_kernel<<<dim3(nblk, B), K2_THREADS, 0, s>>>(a);
    k2_box_kernel<<<dim3(16, B), K2_THREADS, 0, s>>>(a);      // 16 x 256 lanes = 1024 candidates per pass and frame; idle blocks exit
    h->launches += 2;
    VTI_CUDA(cudaGetLastError());
    return VTI_OK;
}

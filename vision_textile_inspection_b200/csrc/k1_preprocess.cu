// K1 -- fused [cv2.undistort] + Ultralytics LetterBox (cv2.resize INTER_LINEAR + 114 border) + HWC->CHW + /255.
//
// Replaces (SURVEY.md 8a U0-U2): cv2.undistort (north-star addition), ultralytics LetterBox.__call__ and
// BasePredictor.preprocess, reached from measurement.py:205-210.
// Spec: oracle/cv_fixed.py (bit-exact integer formulas, pinned against cv2 in tests/test_oracle_cv.py).
//
// One CTA produces a TY x TX tile of the letterboxed output for all three planes.  Pixels travel through shared
// memory as ONE 32-bit word each (B | G<<8 | R<<16), so a bilinear tap is a single LDS for all three channels.
//   stage   MODE_RAW   the raw-frame bounding box of the tile's remap taps (host-planned per tile) is copied with
//                      aligned 32-bit loads, 12 bytes -> 4 packed pixels -> one 128-bit shared store
//           MODE_PLAIN the tile's source footprint itself is staged that way (no undistort)
//           MODE_GATHER generic fallback: per-pixel byte gathers from global (>= 2x shrink, odd widths, huge warps)
//   remap   (undistort only) every footprint pixel = 4-tap fixed-point remap of the staged raw pixels with OpenCV's
//           5-bit fractions; B and R ride in one register (two 16-bit lanes), the two rows' G in another.  The
//           intermediate uint8 rounding of cv2.undistort is preserved -- a composed single bilinear sample is NOT
//           bit-exact.
//   resize  11-bit H pass + V pass of cv2.resize from shared memory, /255 through a 256-entry table (a true
//           division, not *1/255), warp-coalesced stores of the three fp32 planes; pad = 114/255.
// HBM traffic: frame read once (tile halos hit L2) + 12*LH*LW written once; the 4 B/px remap table is L2-resident
// across the batch.
#include <algorithm>
#include <vector>

#include "vti_internal.h"

namespace {

constexpr int TX = VTI_K1_TX;
constexpr int TY = VTI_K1_TY;
constexpr int K1_THREADS = 256;
constexpr int MAXROWS = 2 * TY + 2;
constexpr int MAXCOLS = 2 * TX + 2;
enum { MODE_PLAIN = 0, MODE_RAW = 1, MODE_GATHER = 2, MODE_FAST_PLAIN = 3, MODE_FAST_REMAP = 4 };

struct K1Args {
    const uint8_t* frames;
    float* out;
    const int32_t* tap_x_idx;   // [new_w]
    const int16_t* tap_x_a;     // [new_w][2]
    const int32_t* tap_y_i;     // [new_h][2]
    const int16_t* tap_y_b;     // [new_h][2]
    const int32_t* und_lut;     // [camera][h*w] (dy16 << 16) | (dx16 & 0xffff)
    const int4* tile_box;       // MODE_RAW: [camera] per tile (bx0, by0, bw, bh | interior << 30)
    int h, w, new_h, new_w, top, left, LH, LW;
    int area2x;                 // exact-2x shrink: OpenCV's INTER_AREA switch
    int flip;
    int pitch_u;                // words per row of the footprint buffer
    int rows_u;                 // rows of the footprint buffer
    int undistort;
    int n_cameras;
    const int32_t* camera;      // [B] camera id per frame, or null: camera 0 for every frame
};
// K1Args and K1FastArgs stay within 128 bytes: past that, nvcc compiles every K1 kernel differently, also those that
// read no camera.
static_assert(sizeof(K1Args) <= 128, "K1Args: parameter block over 128 bytes");

__device__ __forceinline__ unsigned pack_px(unsigned b0, unsigned b1, unsigned b2, int flip) {
    return flip ? (b2 | (b1 << 8) | (b0 << 16)) : (b0 | (b1 << 8) | (b2 << 16));
}

// Copy `npx` pixels (multiple of 4) starting at pixel x0 (multiple of 4) of one frame row into packed words.
// row must be 4-byte aligned (w % 4 == 0).  dst[i] receives pixel x0 + i for i in [keep_lo, keep_hi).
__device__ __forceinline__ void stage_row_packed(const uint8_t* __restrict__ row, int x0, int npx, unsigned* dst,
                                                 int keep_lo, int keep_hi, int lane, int flip) {
    const unsigned* __restrict__ src = reinterpret_cast<const unsigned*>(row + (size_t)x0 * 3);
    for (int g = lane; g < (npx >> 2); g += 32) {
        const unsigned w0 = __ldg(src + 3 * g), w1 = __ldg(src + 3 * g + 1), w2 = __ldg(src + 3 * g + 2);
        unsigned p0 = w0 & 0xFFFFFFu;
        unsigned p1 = __funnelshift_r(w0, w1, 24) & 0xFFFFFFu;
        unsigned p2 = __funnelshift_r(w1, w2, 16) & 0xFFFFFFu;
        unsigned p3 = w2 >> 8;
        if (flip) {
            p0 = __byte_perm(p0, 0, 0x3012); p1 = __byte_perm(p1, 0, 0x3012);
            p2 = __byte_perm(p2, 0, 0x3012); p3 = __byte_perm(p3, 0, 0x3012);
        }
        const int i = 4 * g;
        if (i >= keep_lo && i + 3 < keep_hi) {
            *reinterpret_cast<uint4*>(dst + i) = make_uint4(p0, p1, p2, p3);
        } else {
            if (i >= keep_lo && i < keep_hi) dst[i] = p0;
            if (i + 1 >= keep_lo && i + 1 < keep_hi) dst[i + 1] = p1;
            if (i + 2 >= keep_lo && i + 2 < keep_hi) dst[i + 2] = p2;
            if (i + 3 >= keep_lo && i + 3 < keep_hi) dst[i + 3] = p3;
        }
    }
}

// 4-tap fixed-point remap of packed pixels: returns the packed uint8 result of cv2.remap(INTER_LINEAR).
//   acc_c = (32-fy) * [(32-fx) p00 + fx p01] + fy * [(32-fx) p10 + fx p11];  out = (acc + 512) >> 10
// (== (sum(w15 * p) + 2^14) >> 15: every 15-bit OpenCV weight is exactly 32 * the 10-bit product weight)
__device__ __forceinline__ unsigned remap_packed(unsigned t00, unsigned t01, unsigned t10, unsigned t11, int fx, int fy) {
    const unsigned wx0 = 32 - fx, wy0 = 32 - fy;
    const unsigned br0 = (t00 & 0x00FF00FFu) * wx0 + (t01 & 0x00FF00FFu) * fx;       // B | R<<16, each <= 8160
    const unsigned br1 = (t10 & 0x00FF00FFu) * wx0 + (t11 & 0x00FF00FFu) * fx;
    const unsigned g01 = __byte_perm(t00, t10, 0x3531) * wx0 + __byte_perm(t01, t11, 0x3531) * fx;  // G0 | G1<<16
    const unsigned b = ((br0 & 0xFFFFu) * wy0 + (br1 & 0xFFFFu) * fy + 512u) >> 10;
    const unsigned r = ((br0 >> 16) * wy0 + (br1 >> 16) * fy + 512u) >> 10;
    const unsigned g = ((g01 & 0xFFFFu) * wy0 + (g01 >> 16) * fy + 512u) >> 10;
    return b | (g << 8) | (r << 16);
}

// Frame b takes the remap tables of camera a.camera[b] (null ids, or an id out of range: camera 0's).
template <int MODE>
__global__ void __launch_bounds__(K1_THREADS) k1_letterbox_kernel(const K1Args a) {
    extern __shared__ __align__(128) unsigned s_dyn[];     // [footprint rows][pitch_u] then the raw box (MODE_RAW)
    __shared__ float s_div[256];
    __shared__ int s_rowsrc[MAXROWS];
    __shared__ int s_colsrc[MAXCOLS + 4];
    __shared__ int4 s_rowtap[TY];

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int X0 = blockIdx.x * TX, Y0 = blockIdx.y * TY;
    const int b = blockIdx.z;
    const uint8_t* __restrict__ frame = a.frames + (size_t)b * a.h * a.w * 3;
    float* __restrict__ out = a.out + (size_t)b * 3 * a.LH * a.LW;
    unsigned* s_und = s_dyn;
    // the camera's first row in und_lut [camera][h][w]; an offset pointer instead takes MODE_RAW from 32 to 40 registers
    int cam_row = 0;
    const int4* tile_box = a.tile_box;
    if (MODE != MODE_PLAIN && a.camera) {
        const int cam = __ldg(a.camera + b);
        if ((unsigned)cam < (unsigned)a.n_cameras) {
            cam_row = cam * a.h;
            tile_box += (size_t)cam * gridDim.x * gridDim.y;
        }
    }

    s_div[tid] = __fdiv_rn((float)tid, 255.0f);

    const int ry_lo = max(Y0 - a.top, 0), ry_hi = min(Y0 + TY - 1 - a.top, a.new_h - 1);
    const int rx_lo = max(X0 - a.left, 0), rx_hi = min(X0 + TX - 1 - a.left, a.new_w - 1);
    const bool any = (ry_lo <= ry_hi) && (rx_lo <= rx_hi);
    int nrows = 0, ncols = 0, r_lo = 0, c_lo = 0;
    bool row_contig = true, col_contig = true;
    // MODE_PLAIN stages whole 4-pixel groups with 128-bit shared stores: its column origin is 4-aligned
    const bool vec_plain = (MODE == MODE_PLAIN) && ((a.w & 3) == 0);
    if (any) {
        r_lo = a.tap_y_i[2 * ry_lo];
        const int r_hi = a.tap_y_i[2 * ry_hi + 1];
        row_contig = (r_hi - r_lo + 1) <= MAXROWS;
        nrows = row_contig ? (r_hi - r_lo + 1) : 2 * (ry_hi - ry_lo + 1);
        c_lo = a.tap_x_idx[rx_lo];
        const int c_hi = min(a.tap_x_idx[rx_hi] + 1, a.w - 1);
        col_contig = (c_hi - c_lo + 1) <= MAXCOLS;
        if (col_contig && vec_plain) c_lo &= ~3;
        ncols = col_contig ? (c_hi - c_lo + 1) : 2 * (rx_hi - rx_lo + 1);
        for (int i = tid; i < nrows; i += K1_THREADS)
            s_rowsrc[i] = row_contig ? (r_lo + i) : a.tap_y_i[2 * ry_lo + i];
        for (int i = tid; i < ncols; i += K1_THREADS)
            s_colsrc[i] = col_contig ? (c_lo + i) : min(a.tap_x_idx[rx_lo + (i >> 1)] + (i & 1), a.w - 1);
        if (tid < TY) {
            const int ry = Y0 + tid - a.top;
            int4 t = make_int4(0, 0, 0, 0);
            if (ry >= 0 && ry < a.new_h) {
                t.x = row_contig ? (a.tap_y_i[2 * ry] - r_lo) : 2 * (ry - ry_lo);
                t.y = row_contig ? (a.tap_y_i[2 * ry + 1] - r_lo) : 2 * (ry - ry_lo) + 1;
                t.z = a.tap_y_b[2 * ry];
                t.w = a.tap_y_b[2 * ry + 1];
            }
            s_rowtap[tid] = t;
        }
    }
    __syncthreads();

    // ------------------------------------------------------------------------------------------------ stage
    if (any) {
        if (MODE == MODE_PLAIN) {
            if (col_contig && vec_plain) {
                const int npx = (ncols + 3) & ~3;          // c_lo is 4-aligned, w % 4 == 0: stays inside the row
                for (int r = warp; r < nrows; r += K1_THREADS / 32)
                    stage_row_packed(frame + (size_t)s_rowsrc[r] * a.w * 3, c_lo, npx, s_und + r * a.pitch_u, 0, npx,
                                     lane, a.flip);
            } else {
                for (int r = warp; r < nrows; r += K1_THREADS / 32) {
                    const uint8_t* __restrict__ row = frame + (size_t)s_rowsrc[r] * a.w * 3;
                    for (int c = lane; c < ncols; c += 32) {
                        const uint8_t* p = row + (size_t)s_colsrc[c] * 3;
                        s_und[r * a.pitch_u + c] = pack_px(__ldg(p), __ldg(p + 1), __ldg(p + 2), a.flip);
                    }
                }
            }
        } else if (MODE == MODE_RAW) {
            unsigned* s_raw = s_dyn + a.rows_u * a.pitch_u;
            const int4 box = tile_box[blockIdx.y * gridDim.x + blockIdx.x];
            const int bx0 = box.x, by0 = box.y, bw = box.z, bh = box.w & 0xFFFF;
            const bool interior = (box.w >> 30) & 1;
            for (int r = warp; r < bh; r += K1_THREADS / 32)
                stage_row_packed(frame + (size_t)(by0 + r) * a.w * 3, bx0, bw, s_raw + r * bw, 0, bw, lane, a.flip);
            __syncthreads();
            for (int r = warp; r < nrows; r += K1_THREADS / 32) {
                const int sy = s_rowsrc[r];
                const int32_t* __restrict__ lrow = a.und_lut + (size_t)(cam_row + sy) * a.w;
                for (int c = lane; c < ncols; c += 32) {
                    const int sx = c_lo + c;
                    const int lut = __ldg(lrow + sx);
                    const int ix = sx * 32 + (int)(short)(lut & 0xffff), iy = sy * 32 + (lut >> 16);
                    const int x = ix >> 5, y = iy >> 5;
                    const int idx = (y - by0) * bw + (x - bx0);
                    unsigned t00, t01, t10, t11;
                    if (interior) {
                        t00 = s_raw[idx]; t01 = s_raw[idx + 1]; t10 = s_raw[idx + bw]; t11 = s_raw[idx + bw + 1];
                    } else {
                        const bool x0 = (unsigned)x < (unsigned)a.w, x1 = (unsigned)(x + 1) < (unsigned)a.w;
                        const bool y0 = (unsigned)y < (unsigned)a.h, y1 = (unsigned)(y + 1) < (unsigned)a.h;
                        t00 = (y0 && x0) ? s_raw[idx] : 0u;
                        t01 = (y0 && x1) ? s_raw[idx + 1] : 0u;
                        t10 = (y1 && x0) ? s_raw[idx + bw] : 0u;
                        t11 = (y1 && x1) ? s_raw[idx + bw + 1] : 0u;
                    }
                    s_und[r * a.pitch_u + c] = remap_packed(t00, t01, t10, t11, ix & 31, iy & 31);
                }
            }
        } else {   // MODE_GATHER
            for (int r = warp; r < nrows; r += K1_THREADS / 32) {
                const int sy = s_rowsrc[r];
                for (int c = lane; c < ncols; c += 32) {
                    const int sx = s_colsrc[c];
                    const int lut = __ldg(a.und_lut + (size_t)(cam_row + sy) * a.w + sx);
                    const int ix = sx * 32 + (int)(short)(lut & 0xffff), iy = sy * 32 + (lut >> 16);
                    const int x = ix >> 5, y = iy >> 5;
                    const bool x0 = (unsigned)x < (unsigned)a.w, x1 = (unsigned)(x + 1) < (unsigned)a.w;
                    const bool y0 = (unsigned)y < (unsigned)a.h, y1 = (unsigned)(y + 1) < (unsigned)a.h;
                    const uint8_t* q0 = frame + ((size_t)y * a.w + x) * 3;
                    const uint8_t* q1 = q0 + (size_t)a.w * 3;
                    const unsigned t00 = (y0 && x0) ? pack_px(q0[0], q0[1], q0[2], a.flip) : 0u;
                    const unsigned t01 = (y0 && x1) ? pack_px(q0[3], q0[4], q0[5], a.flip) : 0u;
                    const unsigned t10 = (y1 && x0) ? pack_px(q1[0], q1[1], q1[2], a.flip) : 0u;
                    const unsigned t11 = (y1 && x1) ? pack_px(q1[3], q1[4], q1[5], a.flip) : 0u;
                    s_und[r * a.pitch_u + c] = remap_packed(t00, t01, t10, t11, ix & 31, iy & 31);
                }
            }
        }
    }
    __syncthreads();

    // ----------------------------------------------------------------------------------------------- resize
    // warp = (column group of 32, row group of 8); lane = output column => conflict-free LDS, coalesced STG
    const float pad = s_div[114];
    const int X = X0 + 32 * (warp & 3) + lane;
    if (X >= a.LW) return;
    const int rx = X - a.left;
    const bool xin = (rx >= 0) && (rx < a.new_w);
    int cs0 = 0, cs1 = 0;
    unsigned a0 = 0, a1 = 0;
    if (xin && any) {
        if (col_contig) {
            const int sx = a.tap_x_idx[rx];
            cs0 = sx - c_lo;
            cs1 = min(sx + 1, a.w - 1) - c_lo;
        } else {
            cs0 = 2 * (rx - rx_lo);
            cs1 = cs0 + 1;
        }
        a0 = (unsigned)a.tap_x_a[2 * rx];
        a1 = (unsigned)a.tap_x_a[2 * rx + 1];
    }
    const size_t plane = (size_t)a.LH * a.LW;
    const bool area = a.area2x != 0;
#pragma unroll 2
    for (int i = 0; i < TY / 2; ++i) {
        const int j = (warp >> 2) * (TY / 2) + i;
        const int Y = Y0 + j;
        if (Y >= a.LH) break;
        const int ry = Y - a.top;
        float v0 = pad, v1 = pad, v2 = pad;
        if (xin && ry >= 0 && ry < a.new_h) {
            const int4 rt = s_rowtap[j];
            const unsigned* row0 = s_und + rt.x * a.pitch_u;
            const unsigned* row1 = s_und + rt.y * a.pitch_u;
            const unsigned t00 = row0[cs0], t01 = row0[cs1], t10 = row1[cs0], t11 = row1[cs1];
            const unsigned b0 = (unsigned)rt.z, b1 = (unsigned)rt.w;
            unsigned q[3];
#pragma unroll
            for (int ch = 0; ch < 3; ++ch) {
                // all quantities are non-negative: unsigned shifts are single instructions
                const unsigned p00 = (t00 >> (8 * ch)) & 255u, p01 = (t01 >> (8 * ch)) & 255u;
                const unsigned p10 = (t10 >> (8 * ch)) & 255u, p11 = (t11 >> (8 * ch)) & 255u;
                if (area) {
                    q[ch] = (p00 + p01 + p10 + p11 + 2u) >> 2;
                } else {
                    const unsigned S0 = p00 * a0 + p01 * a1, S1 = p10 * a0 + p11 * a1;
                    q[ch] = min(((((b0 * (S0 >> 4)) >> 16) + ((b1 * (S1 >> 4)) >> 16) + 2u) >> 2), 255u);
                }
            }
            v0 = s_div[q[0]]; v1 = s_div[q[1]]; v2 = s_div[q[2]];
        }
        float* o = out + (size_t)Y * a.LW + X;
        o[0] = v0;
        o[plane] = v1;
        o[2 * plane] = v2;
    }
}


// ====================================================================================================================
// Fast path (v3): frame width % 4 == 0 and every tile's source footprint contiguous (shrink < 2x, or upscale).
//
// The ALU pipe (LOP3/SHF/PRMT, 0.5 warp-inst/clk/SMSP) bounded v2, so v3 is organised around instruction count:
//   * the remap table is PER TILE and pre-resolved on the host: entry = shared-memory byte offset of the 2x2 raw
//     neighbourhood | fy << 8 | fx.  Out-of-image taps point into a zero margin staged around the raw box, so the
//     inner loop has no bounds logic.  The table is read linearly (coalesced) and is L2-resident across the batch.
//   * remap math: per channel, PRMT builds (p_x | p_x+1 << 16) for both rows, two IMADs blend the rows for both
//     columns at once, one IDP.2A (dp2a) does the column blend + rounding constant: 2 PRMT + 2 IMAD + 1 IDP + 1 SHF.
//   * resize math: PRMT pairs the two horizontal taps of two channels, IDP.2A applies the 11-bit (a0, a1) taps;
//     the V pass multiplies by (b0, b1), PRMT extracts both >>16 at once and IDP.2A adds them with the +2.
// What was tried and rejected: DESIGN.md 5.
// ====================================================================================================================
constexpr int FTX = 64, FTY = 32;            // fast-path output tile
constexpr int FT_THREADS = 256;
constexpr int FT_MINB = 5;                   // __launch_bounds__ minimum resident CTAs per SM (caps registers at 48)
constexpr int FT_CHUNK = 2 * FT_THREADS;     // the remap loop handles 2 entries per thread and iteration (prefetched)
constexpr int FT_MAXROWS = 2 * FTY + 2, FT_MAXCOLS = 2 * FTX + 2;
constexpr int K1_RAWP = 112;                 // raw-box row pitch (words) baked into the remap kernel when no tile needs more

struct K1FastArgs {
    const uint8_t* frames;
    float* out;
    const int4* tile_hdr;       // [camera][tiles][2]: (bx0, by0, bw, bh), (r_lo, c_lo, nrows, ncols)
    const unsigned* lut;        // [camera][tiles][lut_stride] 4-byte entries, + one spare chunk   (REMAP only)
    const int32_t* tap_x_idx;   // [new_w]
    const int16_t* tap_x_a;     // [new_w][2]
    const int32_t* tap_y_i;     // [new_h][2]
    const int16_t* tap_y_b;     // [new_h][2]
    int h, w, new_h, new_w, top, left, LH, LW;
    int flip;
    int pitch_u;
    int n_cameras;              // (in a dropped field's slot: the fields keep their offsets, the one-camera kernels their code)
    int und_words;              // words reserved for the footprint buffer (multiple of FT_CHUNK, > its rows * pitch_u)
    int lut_stride;             // entries per tile (multiple of FT_CHUNK)
    int raw_pitch;              // words per row of the raw box in shared memory (the same for every tile and camera)
    const int32_t* camera;      // [B] camera id per frame   (MULTI only)
};
static_assert(sizeof(K1FastArgs) <= 128, "K1FastArgs: parameter block over 128 bytes (see K1Args)");

// Stage rows [y0, y0+nr) x 8-pixel groups [x0, x0 + 8*ng) of the frame as packed words (B | G<<8 | R<<16, byte 3 = 0);
// anything outside the image becomes 0 (the zero margin of cv2.remap's BORDER_CONSTANT).  x0 % 8 == 0, w % 8 == 0, so a
// group is 24 contiguous 8-byte-aligned bytes and never straddles the image edge.  Loads of STAGE_R rounds are issued
// back to back from clamped addresses (no branch between them) so that 3*STAGE_R 64-bit loads are in flight per
// thread; v3.1 waited on one group at a time and spent 40 % of its stall samples here.
constexpr int STAGE_R = 3;
__device__ __forceinline__ void stage_box(const uint8_t* __restrict__ frame, int h, int w, int x0, int y0, int ng, int nr,
                                          unsigned* dst, int tid, int flip, int pitch = 0) {
    const int total = ng * nr;
    const float inv_ng = 1.0f / (float)ng;
    // PRMT selectors: byte 4 (of the zero second operand) clears the top byte; the flipped variants reverse B and R
    const unsigned sel_lo = flip ? 0x4012u : 0x4210u;      // word already holds the pixel in bytes 0..2
    const unsigned sel_hi = flip ? 0x4123u : 0x4321u;      // pixel in bytes 1..3
    for (int base = tid; base < total; base += STAGE_R * FT_THREADS) {
        uint2 q[STAGE_R][3];
        bool ok[STAGE_R];
        int dofs[STAGE_R];
#pragma unroll
        for (int k = 0; k < STAGE_R; ++k) {
            const int i = base + k * FT_THREADS;
            // i / ng for i < 2^14, ng <= 2^7: (i + 0.5) / ng is never within 1/(2 ng) of an integer, far above fp32 error
            const int r = (int)(((float)i + 0.5f) * inv_ng);
            const int g = i - r * ng;
            const int y = y0 + r, x = x0 + 8 * g;
            dofs[k] = pitch ? r * pitch + 8 * g : 8 * i;   // rows at a fixed pitch (>= 8 ng) or packed
            ok[k] = (i < total) && ((unsigned)y < (unsigned)h) && ((unsigned)x < (unsigned)w);
            const unsigned off = ok[k] ? (unsigned)(y * w + x) * 3u : 0u;        // frames are < 2^31 bytes
            const uint2* __restrict__ src = reinterpret_cast<const uint2*>(frame + off);
            q[k][0] = __ldg(src); q[k][1] = __ldg(src + 1); q[k][2] = __ldg(src + 2);
        }
#pragma unroll
        for (int k = 0; k < STAGE_R; ++k) {
            const int i = base + k * FT_THREADS;
            if (i >= total) break;
            uint4 lo = make_uint4(0u, 0u, 0u, 0u), hi = lo;
            if (ok[k]) {
                const unsigned w0 = q[k][0].x, w1 = q[k][0].y, w2 = q[k][1].x, w3 = q[k][1].y, w4 = q[k][2].x, w5 = q[k][2].y;
                lo.x = __byte_perm(w0, 0u, sel_lo);
                lo.y = __byte_perm(__funnelshift_r(w0, w1, 24), 0u, sel_lo);
                lo.z = __byte_perm(__funnelshift_r(w1, w2, 16), 0u, sel_lo);
                lo.w = __byte_perm(w2, 0u, sel_hi);
                hi.x = __byte_perm(w3, 0u, sel_lo);
                hi.y = __byte_perm(__funnelshift_r(w3, w4, 24), 0u, sel_lo);
                hi.z = __byte_perm(__funnelshift_r(w4, w5, 16), 0u, sel_lo);
                hi.w = __byte_perm(w5, 0u, sel_hi);
            }
            uint4* d = reinterpret_cast<uint4*>(dst + dofs[k]);
            d[0] = lo; d[1] = hi;
        }
    }
}

// 32-bit shared-window addresses and ld.shared: the address of a tap is ONE integer add away from the per-thread
// base (generic pointers cost an extra instruction per load to re-add the window base).
__device__ __forceinline__ unsigned smem_addr(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
template <int OFF>
__device__ __forceinline__ unsigned lds32(unsigned addr) {
    unsigned v;
    asm volatile("ld.shared.u32 %0, [%1+%2];" : "=r"(v) : "r"(addr), "n"(OFF));
    return v;
}

// 4-byte entry (off16 | fy | fx) on shared-window addresses; RAWP_T > 0: second row at an immediate offset
template <int RAWP_T>
__device__ __forceinline__ unsigned remap_fast4(unsigned raw, unsigned e, unsigned bw4) {
    const unsigned p0 = raw + (e >> 16);
    const unsigned fx = e & 0xFFu, fy = __byte_perm(e, 0, 0x4441);
    unsigned t00 = lds32<0>(p0), t01 = lds32<4>(p0), t10, t11;
    if (RAWP_T > 0) { t10 = lds32<4 * RAWP_T>(p0); t11 = lds32<4 * RAWP_T + 4>(p0); }
    else { t10 = lds32<0>(p0 + bw4); t11 = lds32<4>(p0 + bw4); }
    const unsigned wy0 = fy * 0xFFFFFFFFu + 32u;               // 32 - fy, as a multiply-add (FMA pipe)
    const unsigned wxb = fx * 255u + 32u;                      // (32 - fx) | fx << 8
    const unsigned vB = __byte_perm(t00, t01, 0x3430) * wy0 + __byte_perm(t10, t11, 0x3430) * fy;
    const unsigned vG = __byte_perm(t00, t01, 0x3531) * wy0 + __byte_perm(t10, t11, 0x3531) * fy;
    const unsigned vR = __byte_perm(t00, t01, 0x3632) * wy0 + __byte_perm(t10, t11, 0x3632) * fy;
    const unsigned b = __dp2a_lo(vB, wxb, 512u) * 64u;
    const unsigned g = __dp2a_lo(vG, wxb, 512u) * 64u;
    const unsigned r = __dp2a_lo(vR, wxb, 512u) * 64u;
    return __byte_perm(__byte_perm(b, g, 0x7762), r, 0x7610);
}

// base[idx] = v with the address formed by ONE mad.wide (FMA pipe) -- the compiler's own 64-bit index arithmetic
// costs four ALU-pipe instructions per store, and the ALU pipe is what bounds this kernel.
__device__ __forceinline__ void store_at(float* base, int idx, float v) {
    asm volatile("{\n\t.reg .u64 a;\n\tmad.wide.s32 a, %1, 4, %0;\n\tst.global.f32 [a], %2;\n\t}"
                 :: "l"(base), "r"(idx), "f"(v) : "memory");
}

// float32(v) / 255.0f for q = 4 v + (0..3), v in 0..255, without a table: x = float(4 v) is exact, 1/1020 is split
// into c1 + c2 (c1 = RN(1/1020), c2 = RN(1/1020 - c1)), t = RN(x c2), y = RN(x c1 + t) (one FMA).  x c1 + x c2 differs
// from the quotient by < 2^-48 relative, far below the distance of any v / 255 to a rounding boundary: all 256 values
// were checked against numpy's float32 division with exact rational arithmetic (tools/check_div255.py), and
// tests/test_gpu_parity.py::test_k1_bit_exact compares the kernel's output with cv2 + torch bit for bit.
// K1 is bound by the L1 data pipe (shared-memory wavefronts), not by issue slots: 2 more instructions per value on the
// otherwise idle FP32 pipe replace one table LDS (1.34 wavefronts measured, values in a warp collide on banks).
__device__ __forceinline__ float div255_q(unsigned q) {
    const float x = __uint2float_rn(q & 0x3FCu);
    return __fmaf_rn(x, __uint_as_float(0x3a808081u), __fmul_rn(x, __uint_as_float(0xae7efeffu)));
}

// One output pixel (3 channels) of the exact-2x area average + /255.
__device__ __forceinline__ void area_px(const unsigned char* p0, const unsigned char* p1, unsigned a01, float& v0,
                                        float& v1, float& v2) {
    const unsigned t00 = *reinterpret_cast<const unsigned*>(p0), t01 = *reinterpret_cast<const unsigned*>(p0 + 4);
    const unsigned t10 = *reinterpret_cast<const unsigned*>(p1), t11 = *reinterpret_cast<const unsigned*>(p1 + 4);
    const unsigned bg0 = __byte_perm(t00, t01, 0x5140), rr0 = __byte_perm(t00, t01, 0x3362);
    const unsigned bg1 = __byte_perm(t10, t11, 0x5140), rr1 = __byte_perm(t10, t11, 0x3362);
    const unsigned S0b = __dp2a_lo(a01, bg0, 0u), S0g = __dp2a_hi(a01, bg0, 0u), S0r = __dp2a_lo(a01, rr0, 0u);
    // 4 * quantised value + (0..3)
    const unsigned qb = __dp2a_lo(a01, bg1, S0b + 2u), qg = __dp2a_hi(a01, bg1, S0g + 2u), qr = __dp2a_lo(a01, rr1, S0r + 2u);
    v0 = div255_q(qb);
    v1 = div255_q(qg);
    v2 = div255_q(qr);
}

// One plane store.  LW_T > 0: the row pitch is a compile-time constant, the address is base + immediate.
template <int LW_T>
__device__ __forceinline__ void store_px(float* base, int i, int oi, float v) {
    if (LW_T > 0) base[i * LW_T] = v;
    else store_at(base, oi, v);
}

// Resize of one thread's strip of RPT output rows (one column, three planes) with the H pass of shared source rows
// kept in registers.  Consecutive output rows of a shrink < 2x mostly share a source row (row i's lower tap row is
// row i + 1's upper one: 2 of 3 rows at 4/3), so its H pass is not reloaded and recomputed; the test is warp-uniform
// (the row taps are per tile row).  CHECK: the strip may hold letterbox padding rows (offset -2) or end early.
template <int LW_T, bool CHECK>
__device__ __forceinline__ void resize_strip(const int4* rowtap, unsigned col, unsigned a01, float* o0, float* o1,
                                             float* o2, int LW, int n_out, float pad) {
    constexpr int RPT = FTY / (FT_THREADS / FTX);
    unsigned pb = 0u, pg = 0u, pr = 0u;                    // (H pass >> 4) of the source row at byte offset `have`
    int have = -1, oi = 0;
#pragma unroll
    for (int i = 0; i < RPT; ++i, oi += LW) {
        const int4 rt = rowtap[i];
        if (CHECK) {
            if (i >= n_out) break;
            if (rt.x < 0) {
                store_px<LW_T>(o0, i, oi, pad); store_px<LW_T>(o1, i, oi, pad); store_px<LW_T>(o2, i, oi, pad);
                continue;
            }
        }
        if (rt.x != have) {
            const unsigned t0 = lds32<0>(col + rt.x), t1 = lds32<4>(col + rt.x);
            const unsigned bg = __byte_perm(t0, t1, 0x5140), rr = __byte_perm(t0, t1, 0x3362);
            pb = __dp2a_lo(a01, bg, 0u) >> 4; pg = __dp2a_hi(a01, bg, 0u) >> 4; pr = __dp2a_lo(a01, rr, 0u) >> 4;
        }
        const unsigned t0 = lds32<0>(col + rt.y), t1 = lds32<4>(col + rt.y);
        const unsigned bg = __byte_perm(t0, t1, 0x5140), rr = __byte_perm(t0, t1, 0x3362);
        const unsigned nb = __dp2a_lo(a01, bg, 0u) >> 4, ng = __dp2a_hi(a01, bg, 0u) >> 4, nr = __dp2a_lo(a01, rr, 0u) >> 4;
        const unsigned b0 = (unsigned)rt.z, b1 = (unsigned)rt.w;
        unsigned qb, qg, qr;
        // ((b0 (S0 >> 4)) >> 16) + ((b1 (S1 >> 4)) >> 16) + 2: PRMT takes both >> 16 at once, dp2a adds them.
        // The plan guarantees a0 + a1 <= 2049 and b0 + b1 <= 2049, so the sum is <= 1022: no saturation needed.
        qb = __dp2a_lo(__byte_perm(b0 * pb, b1 * nb, 0x7632), 0x0101u, 2u);
        qg = __dp2a_lo(__byte_perm(b0 * pg, b1 * ng, 0x7632), 0x0101u, 2u);
        qr = __dp2a_lo(__byte_perm(b0 * pr, b1 * nr, 0x7632), 0x0101u, 2u);
        store_px<LW_T>(o0, i, oi, div255_q(qb));
        store_px<LW_T>(o1, i, oi, div255_q(qg));
        store_px<LW_T>(o2, i, oi, div255_q(qr));
        pb = nb; pg = ng; pr = nr; have = rt.y;
    }
}

// The resize phase of one thread: RPT output rows of one column, three planes, written to o0 / o0 + plane / o0 + 2 plane
// with row pitch LW_T (compile time) or LW; `o0` is the thread's first output pixel.
template <bool AREA, int LW_T>
__device__ __forceinline__ void resize_phase(const K1FastArgs& a, float* __restrict__ o0, size_t plane, int LW, int X, int Y0,
                                             int j0, int nrows, int c_lo, const unsigned* s_und, const int4* s_rowtap) {
    const float pad = __uint_as_float(0x3ee4e4e5u);            // float32(114) / 255.0f, the LetterBox border
    constexpr int RPT = FTY / (FT_THREADS / FTX);          // rows per thread
    float* __restrict__ o1 = o0 + plane;
    float* __restrict__ o2 = o1 + plane;
    int oi = 0;
    const int rx = X - a.left;
    const int ry0 = Y0 + j0 - a.top;
    // rows of this thread's strip that exist in the letterboxed frame, then those that are resized image rows
    const int n_out = min(RPT, a.LH - (Y0 + j0));
    if (rx < 0 || rx >= a.new_w || nrows == 0 || ry0 + n_out <= 0 || ry0 >= a.new_h) {     // nothing but padding
#pragma unroll
        for (int i = 0; i < RPT; ++i, oi += LW) {
            if (i < n_out) { store_px<LW_T>(o0, i, oi, pad); store_px<LW_T>(o1, i, oi, pad); store_px<LW_T>(o2, i, oi, pad); }
        }
        return;
    }
    const int sx = a.tap_x_idx[rx];
    const unsigned a01 = (unsigned)(unsigned short)a.tap_x_a[2 * rx] | ((unsigned)(unsigned short)a.tap_x_a[2 * rx + 1] << 16);
    const unsigned char* col = reinterpret_cast<const unsigned char*>(s_und) + (sx - c_lo) * 4;   // taps at col, col + 4
    const bool full = (ry0 >= 0) && (ry0 + RPT <= a.new_h) && (n_out == RPT);      // warp-uniform
    if (AREA) {
        for (int i = 0; i < n_out; ++i, oi += LW) {
            const int4 rt = s_rowtap[j0 + i];
            float v0 = pad, v1 = pad, v2 = pad;
            if (rt.x >= 0) area_px(col + rt.x, col + rt.y, a01, v0, v1, v2);
            store_px<LW_T>(o0, i, oi, v0); store_px<LW_T>(o1, i, oi, v1); store_px<LW_T>(o2, i, oi, v2);
        }
    } else if (full) {
        resize_strip<LW_T, false>(s_rowtap + j0, smem_addr(col), a01, o0, o1, o2, LW, RPT, pad);
    } else {                                                // padding rows in the strip, or it ends at row LH
        resize_strip<LW_T, true>(s_rowtap + j0, smem_addr(col), a01, o0, o1, o2, LW, n_out, pad);
    }
}

// MULTI (REMAP only): frame b takes the headers and remap table of camera a.camera[b] (an id out of range: camera 0's).
// A test of a.camera at run time instead makes the one-camera remap kernel 0.3 % slower on cfg2 (DESIGN.md 3).
template <bool REMAP, bool AREA, int LW_T, int RAWP_T, bool MULTI>
__global__ void __launch_bounds__(FT_THREADS, FT_MINB) k1_fast_kernel(const K1FastArgs a) {
    extern __shared__ __align__(128) unsigned s_dyn[];     // s_und [und_words], then the raw box (REMAP)
    __shared__ int4 s_rowtap[FTY];                          // (byte offset row0, byte offset row1, b0, b1)

    const int tid = threadIdx.x;
    const int X0 = blockIdx.x * FTX, Y0 = blockIdx.y * FTY;
    const int b = blockIdx.z;
    const int tile = blockIdx.y * gridDim.x + blockIdx.x;
    const int LW = LW_T > 0 ? LW_T : a.LW;
    const uint8_t* __restrict__ frame = a.frames + (size_t)b * a.h * a.w * 3;
    float* __restrict__ out = a.out + (size_t)b * 3 * a.LH * LW;
    unsigned* s_und = s_dyn;
    const int4* tile_hdr = a.tile_hdr;
    const unsigned* lut_base = a.lut;
    if constexpr (MULTI) {
        const int cam = __ldg(a.camera + b);
        if ((unsigned)cam < (unsigned)a.n_cameras) {
            const size_t ntiles = (size_t)gridDim.x * gridDim.y;
            tile_hdr += 2 * ntiles * cam;
            lut_base += ntiles * a.lut_stride * cam;
        }
    }

    const int4 h0 = __ldg(tile_hdr + 2 * tile), h1 = __ldg(tile_hdr + 2 * tile + 1);
    const int r_lo = h1.x, c_lo = h1.y, nrows = h1.z;
    if (tid < FTY) {
        const int ry = Y0 + tid - a.top;
        int4 t = make_int4(-2, -2, 0, 0);                   // padding row (never equal to a real row offset)
        if (ry >= 0 && ry < a.new_h && nrows > 0) {
            t.x = (a.tap_y_i[2 * ry] - r_lo) * a.pitch_u * 4;
            t.y = (a.tap_y_i[2 * ry + 1] - r_lo) * a.pitch_u * 4;
            t.z = a.tap_y_b[2 * ry];
            t.w = a.tap_y_b[2 * ry + 1];
        }
        s_rowtap[tid] = t;
    }


    // ------------------------------------------------------------------------------------------- stage (+ remap)
    if (nrows > 0) {
        if (!REMAP) {
            stage_box(frame, a.h, a.w, c_lo, r_lo, a.pitch_u >> 3, nrows, s_und, tid, a.flip);
        } else {
            unsigned* s_raw = s_dyn + a.und_words;
            stage_box(frame, a.h, a.w, h0.x, h0.y, h0.z >> 3, h0.w, s_raw, tid, a.flip, a.raw_pitch);
            __syncthreads();
            unsigned* dst = s_und + tid;
            const int total = nrows * a.pitch_u;
            const int n_it = total / FT_CHUNK;                 // whole chunks; table and buffer are padded
            const int rem = total - n_it * FT_CHUNK;
            const unsigned raw8 = smem_addr(s_raw);
            const unsigned bw4 = (unsigned)a.raw_pitch * 4u;
            const unsigned* __restrict__ lut = lut_base + (size_t)tile * a.lut_stride + tid;
            unsigned e0 = __ldg(lut), e1 = __ldg(lut + FT_THREADS);
            for (int it = 0; it < n_it; ++it, dst += FT_CHUNK) {
                lut += FT_CHUNK;                               // next entries in flight while these are computed
                const unsigned n0 = __ldg(lut), n1 = __ldg(lut + FT_THREADS);   // (the table has one spare chunk)
                dst[0] = remap_fast4<RAWP_T>(raw8, e0, bw4);
                dst[FT_THREADS] = remap_fast4<RAWP_T>(raw8, e1, bw4);
                e0 = n0; e1 = n1;
            }
            // tail of the footprint: only the warps that still have cells (a 44 x 87 footprint leaves 244 of 512)
            if (tid < rem) dst[0] = remap_fast4<RAWP_T>(raw8, e0, bw4);
            if (tid + FT_THREADS < rem) dst[FT_THREADS] = remap_fast4<RAWP_T>(raw8, e1, bw4);
        }
    }
    __syncthreads();

    // ----------------------------------------------------------------------------------------------- resize
    const int X = X0 + (tid & (FTX - 1));
    constexpr int RPT = FTY / (FT_THREADS / FTX);          // rows per thread
    const int j0 = (tid / FTX) * RPT;
    if (X >= LW) return;
    resize_phase<AREA, LW_T>(a, out + (size_t)(Y0 + j0) * LW + X, (size_t)a.LH * LW, LW, X, Y0, j0, nrows, c_lo, s_und, s_rowtap);
}

}  // namespace

// ---------------------------------------------------------------------------------------------------- host plan
// Mirrors the kernel's per-tile footprint logic to size the shared buffers and, with undistort on, to find the
// raw-frame bounding box of every tile's remap taps.
// Fast-path plan: per-tile headers and (undistort) the per-tile pre-resolved remap table, per camera.  The footprints
// come from the resize taps alone and are the same for every camera; the raw boxes and the remap entries are per camera,
// at one raw-box pitch common to all cameras.  Returns false when the geometry is not eligible for every camera (the
// generic kernel below takes over).
static bool k1_fast_plan(vti_handle* h, const std::vector<int32_t>& xi, const std::vector<int32_t>& yi,
                         const std::vector<int16_t>& xa, const std::vector<int16_t>& yb,
                         const std::vector<int32_t>* und_ix, const std::vector<int32_t>* und_iy,
                         std::vector<int4>& hdr, std::vector<unsigned>& lut, int& pitch_u, int& rows_u, size_t& raw_words,
                         int& lut_stride, int& raw_pitch) {
    const vti_geometry& g = h->g;
    const int fw = h->p.frame_w, fh = h->p.frame_h;
    if (fw & 7) return false;
    if (h->resize_mode == 1) {
        // no-saturation guarantee of resize_strip, and the unconditional read of column sx + 1
        for (int d = 0; d < g.new_w; ++d) {
            if (xa[2 * d] < 0 || xa[2 * d + 1] < 0 || xa[2 * d] + xa[2 * d + 1] > 2049) return false;
            if (xi[d] + 1 > fw - 1 && xa[2 * d + 1] != 0) return false;
        }
        for (int d = 0; d < g.new_h; ++d)
            if (yb[2 * d] < 0 || yb[2 * d + 1] < 0 || yb[2 * d] + yb[2 * d + 1] > 2049) return false;
    }
    const int ntx = (g.LW + FTX - 1) / FTX, nty = (g.LH + FTY - 1) / FTY;
    hdr.assign((size_t)ntx * nty * 2, make_int4(0, 0, 0, 0));
    pitch_u = 8; rows_u = 1; raw_words = 0;
    // pass 1: footprints
    for (int ty = 0; ty < nty; ++ty)
        for (int tx = 0; tx < ntx; ++tx) {
            const int X0 = tx * FTX, Y0 = ty * FTY;
            const int ry_lo = std::max(Y0 - g.top, 0), ry_hi = std::min(Y0 + FTY - 1 - g.top, g.new_h - 1);
            const int rx_lo = std::max(X0 - g.left, 0), rx_hi = std::min(X0 + FTX - 1 - g.left, g.new_w - 1);
            if (ry_lo > ry_hi || rx_lo > rx_hi) continue;                     // pure padding tile: nrows = 0
            int r_lo = INT32_MAX, r_hi = -1, c_lo = INT32_MAX, c_hi = -1;
            for (int ry = ry_lo; ry <= ry_hi; ++ry) {
                r_lo = std::min(r_lo, std::min(yi[2 * ry], yi[2 * ry + 1]));
                r_hi = std::max(r_hi, std::max(yi[2 * ry], yi[2 * ry + 1]));
            }
            for (int rx = rx_lo; rx <= rx_hi; ++rx) {
                c_lo = std::min(c_lo, xi[rx]);
                c_hi = std::max(c_hi, std::min(xi[rx] + 1, fw - 1));
            }
            if (!und_ix) c_lo &= ~7;                               // only the direct staging needs 8-pixel groups
            const int nrows = r_hi - r_lo + 1, ncols = c_hi - c_lo + 1;
            if (nrows > FT_MAXROWS || ncols > FT_MAXCOLS + 8) return false;
            rows_u = std::max(rows_u, nrows);
            pitch_u = std::max(pitch_u, und_ix ? ncols : ((ncols + 7) & ~7));   // remapped footprints pack tightly
            hdr[2 * ((size_t)ty * ntx + tx) + 1] = make_int4(r_lo, c_lo, nrows, ncols);
        }

    lut_stride = (rows_u * pitch_u + FT_CHUNK - 1) / FT_CHUNK * FT_CHUNK;
    raw_pitch = 0;
    if (!und_ix) return true;
    // pass 2: (1) every camera's raw boxes, (2) one raw-box pitch and height for all of them, (3) every camera's remap
    // entries at that pitch (entry 0 = offset 0, weights 0: a valid cell for the padded tail)
    const size_t ntiles = (size_t)ntx * nty, npx = (size_t)fh * fw;
    const int ncam = h->n_cameras;
    auto clampx = [&](int x) { return x < -1 ? -2 : (x > fw - 1 ? fw : x); };
    auto clampy = [&](int y) { return y < -1 ? -2 : (y > fh - 1 ? fh : y); };
    int bh_max = 0;
    std::vector<int4> boxes((size_t)ncam * ntiles, make_int4(0, 0, 0, 0));
    for (int cam = 0; cam < ncam; ++cam) {
        const int32_t* ux = und_ix->data() + cam * npx;
        const int32_t* uy = und_iy->data() + cam * npx;
        for (size_t t = 0; t < ntiles; ++t) {
            const int4 f = hdr[2 * t + 1];
            const int r_lo = f.x, c_lo = f.y, nrows = f.z;
            if (nrows == 0) continue;
            const int c_end = std::min(c_lo + pitch_u, fw);        // remap every staged column that exists
            int minx = INT32_MAX, miny = INT32_MAX, maxx = INT32_MIN, maxy = INT32_MIN;
            for (int sy = r_lo; sy < r_lo + nrows; ++sy)
                for (int sx = c_lo; sx < c_end; ++sx) {
                    const size_t i = (size_t)sy * fw + sx;
                    const int x = clampx(ux[i] >> 5), y = clampy(uy[i] >> 5);
                    minx = std::min(minx, x); maxx = std::max(maxx, x);
                    miny = std::min(miny, y); maxy = std::max(maxy, y);
                }
            const int bx0 = (minx >= 0) ? (minx & ~7) : -8;
            const int bx1 = (maxx + 2 + 7) & ~7;                    // exclusive, covers x + 1
            const int bw = bx1 - bx0, by0 = miny, bh = maxy + 2 - miny;
            if ((size_t)bw * bh > 16384) return false;              // 16-bit byte offsets
            raw_pitch = std::max(raw_pitch, bw);
            bh_max = std::max(bh_max, bh);
            boxes[cam * ntiles + t] = make_int4(bx0, by0, bw, bh);
        }
    }
    {                                                               // every tile's raw box at ONE pitch
        if (raw_pitch <= K1_RAWP) raw_pitch = K1_RAWP;              // the pitch the kernel has as an immediate
        if ((size_t)raw_pitch * bh_max > 16384) return false;
        raw_words = (size_t)raw_pitch * bh_max;                     // every tile's box at the one pitch
    }
    const std::vector<int4> foot(hdr);
    hdr.assign((size_t)ncam * ntiles * 2, make_int4(0, 0, 0, 0));
    lut.assign((size_t)ncam * ntiles * lut_stride + FT_CHUNK, 0u);  // + one spare chunk: the loop prefetches
    for (int cam = 0; cam < ncam; ++cam)
    for (size_t t = 0; t < ntiles; ++t) {
        const int4 f = foot[2 * t + 1], bx = boxes[cam * ntiles + t];
        hdr[2 * (cam * ntiles + t)] = bx;
        hdr[2 * (cam * ntiles + t) + 1] = f;
        const int r_lo = f.x, c_lo = f.y, nrows = f.z;
        if (nrows == 0) continue;
        const int bx0 = bx.x, by0 = bx.y, bw = raw_pitch;
        const int32_t* ux = und_ix->data() + cam * npx;
        const int32_t* uy = und_iy->data() + cam * npx;
        unsigned* L = lut.data() + (cam * ntiles + t) * lut_stride;
        for (int r = 0; r < nrows; ++r)
            for (int c = 0; c < pitch_u; ++c) {
                const int sy = r_lo + r, sx = c_lo + c;
                unsigned off = 0u, fx = 0u, fy = 0u;                // columns past the frame: any valid cell
                if (sx < fw) {
                    const size_t i = (size_t)sy * fw + sx;
                    const int ix = ux[i], iy = uy[i];
                    const int x = clampx(ix >> 5), y = clampy(iy >> 5);
                    off = (unsigned)(((y - by0) * bw + (x - bx0)) * 4);
                    fx = (unsigned)(ix & 31); fy = (unsigned)(iy & 31);
                }
                const size_t e = (size_t)r * pitch_u + c;
                L[e] = (off << 16) | (fy << 8) | fx;
            }
    }
    return true;
}

// The one place that names every instantiation of the fast kernel: launch == 0 raises each one's dynamic
// shared-memory limit (plan time), launch == 1 launches the one that matches the handle.
template <bool REMAP, bool AREA, int LW_T, int RAWP_T, bool MULTI>
static int k1_fast_one(const K1FastArgs* f, int launch, const dim3* grid, size_t smem, cudaStream_t s) {
    if (!launch) return vti_raise_dyn_smem((const void*)k1_fast_kernel<REMAP, AREA, LW_T, RAWP_T, MULTI>, smem);
    k1_fast_kernel<REMAP, AREA, LW_T, RAWP_T, MULTI><<<*grid, FT_THREADS, smem, s>>>(*f);
    return VTI_OK;
}
template <bool AREA, int LW_T, int RAWP_T>
static int k1_fast_remap(bool multi, const K1FastArgs* f, int launch, const dim3* grid, size_t smem, cudaStream_t s) {
    int rc = VTI_OK;
    if (!launch || !multi) if ((rc = k1_fast_one<true, AREA, LW_T, RAWP_T, false>(f, launch, grid, smem, s))) return rc;
    if (!launch || multi) rc = k1_fast_one<true, AREA, LW_T, RAWP_T, true>(f, launch, grid, smem, s);
    return rc;
}
template <int LW_T>
static int k1_fast_lw(bool remap, bool area, int rawp, bool multi, const K1FastArgs* f, int launch, const dim3* grid,
                      size_t smem, cudaStream_t s) {
    int rc = VTI_OK;
    const bool fixed = rawp == K1_RAWP;
    if (!launch || (remap && area && fixed)) if ((rc = k1_fast_remap<true, LW_T, K1_RAWP>(multi, f, launch, grid, smem, s))) return rc;
    if (!launch || (remap && !area && fixed)) if ((rc = k1_fast_remap<false, LW_T, K1_RAWP>(multi, f, launch, grid, smem, s))) return rc;
    if (!launch || (remap && area && !fixed)) if ((rc = k1_fast_remap<true, LW_T, 0>(multi, f, launch, grid, smem, s))) return rc;
    if (!launch || (remap && !area && !fixed)) if ((rc = k1_fast_remap<false, LW_T, 0>(multi, f, launch, grid, smem, s))) return rc;
    if (!launch || (!remap && area)) if ((rc = k1_fast_one<false, true, LW_T, 0, false>(f, launch, grid, smem, s))) return rc;
    if (!launch || (!remap && !area)) if ((rc = k1_fast_one<false, false, LW_T, 0, false>(f, launch, grid, smem, s))) return rc;
    return rc;
}
// multi: the per-frame camera form (remap only; without undistort K1 does not depend on the camera)
static int k1_fast_dispatch(vti_handle* h, const K1FastArgs* f, int launch, const dim3* grid, size_t smem,
                            cudaStream_t s = nullptr, bool multi = false) {
    const bool remap = h->k1_mode == MODE_FAST_REMAP, area = h->resize_mode == 2;
    const int LW = h->g.LW, rawp = h->k1_raw_pitch;
    int rc = VTI_OK;
    // imgsz 960 and 640 letterboxes (every BASELINE config) get the output row pitch as a compile-time constant: the
    // plane stores take immediate offsets
    if (!launch || LW == 960) if ((rc = k1_fast_lw<960>(remap, area, rawp, multi, f, launch, grid, smem, s))) return rc;
    if (!launch || LW == 640) if ((rc = k1_fast_lw<640>(remap, area, rawp, multi, f, launch, grid, smem, s))) return rc;
    if (!launch || (LW != 960 && LW != 640)) rc = k1_fast_lw<0>(remap, area, rawp, multi, f, launch, grid, smem, s);
    return rc;
}

int vti_k1_plan(vti_handle* h, const std::vector<int32_t>& xi, const std::vector<int32_t>& yi,
                const std::vector<int16_t>& xa, const std::vector<int16_t>& yb,
                const std::vector<int32_t>* und_ix, const std::vector<int32_t>* und_iy,
                const std::vector<int32_t>* und_packed) {
    const vti_geometry& g = h->g;
    const int fw = h->p.frame_w, fh = h->p.frame_h;
    const int ntx = (g.LW + TX - 1) / TX, nty = (g.LH + TY - 1) / TY;
    const int ncam = h->n_cameras;
    const size_t npx = (size_t)fh * fw, ntiles = (size_t)ntx * nty;
    {
        std::vector<int4> hdr;
        std::vector<unsigned> lut;
        int pitch_u = 0, rows_u = 0, lut_stride = 0, raw_pitch = 0;
        size_t raw_words = 0;
        if (k1_fast_plan(h, xi, yi, xa, yb, und_ix, und_iy, hdr, lut, pitch_u, rows_u, raw_words, lut_stride, raw_pitch)) {
            const int und_words = (rows_u * pitch_u + 4 + FT_CHUNK - 1) / FT_CHUNK * FT_CHUNK;
            // The measured configuration: the region past the footprint buffer is at least one output tile (3 x FTY x
            // FTX floats, 24 KB), so the plain path (no raw box) asks for these 24 KB too.  This sets how many K1 CTAs
            // share an SM with the post kernels (DESIGN.md 5a); dropping it is a change to measure on its own.
            raw_words = std::max(raw_words, (size_t)3 * FTY * FTX);
            size_t smem = ((size_t)und_words + raw_words) * 4;
            // Leave room on every SM for the post kernels that run beside K1 (two streams): at most 4 resident K1 CTAs.
            // Measured: 5 CTAs/SM make K1 alone 5 % faster and the whole pre || post step 8 % slower.
            if (und_ix) smem = std::max(smem, (size_t)(46 * 1024 + 512));     // (measured with the remap path)
            if (smem <= 110 * 1024) {
                h->k1_mode = und_ix ? MODE_FAST_REMAP : MODE_FAST_PLAIN;
                h->k1_pitch_u = pitch_u; h->k1_smem = smem;
                h->k1_und_words = und_words; h->k1_lut_stride = lut_stride; h->k1_raw_pitch = raw_pitch;
                int rc;
                if ((rc = vti_upload(h, &h->d_k1_tiles, hdr)) || (und_ix && (rc = vti_upload(h, &h->d_k1_lut, lut)))) return rc;
                return k1_fast_dispatch(h, nullptr, 0, nullptr, smem);          // raises the shared-memory limits only
            }
        }
    }
    int ncols_max = 4, nrows_max = 1;
    bool all_contig = true;
    std::vector<int4> boxes(ncam * ntiles, make_int4(0, 0, 0, 0));
    size_t raw_max = 0;
    for (int ty = 0; ty < nty; ++ty)
        for (int tx = 0; tx < ntx; ++tx) {
            const int X0 = tx * TX, Y0 = ty * TY;
            const int ry_lo = std::max(Y0 - g.top, 0), ry_hi = std::min(Y0 + TY - 1 - g.top, g.new_h - 1);
            const int rx_lo = std::max(X0 - g.left, 0), rx_hi = std::min(X0 + TX - 1 - g.left, g.new_w - 1);
            if (ry_lo > ry_hi || rx_lo > rx_hi) continue;
            const int r_lo = yi[2 * ry_lo], r_hi = yi[2 * ry_hi + 1];
            const bool rc = (r_hi - r_lo + 1) <= MAXROWS;
            const int nrows = rc ? (r_hi - r_lo + 1) : 2 * (ry_hi - ry_lo + 1);
            const int c_lo = xi[rx_lo], c_hi = std::min(xi[rx_hi] + 1, fw - 1);
            const bool cc = (c_hi - c_lo + 1) <= MAXCOLS;
            const int ncols = (cc ? (c_hi - c_lo + 1) : 2 * (rx_hi - rx_lo + 1)) + 6;   // + 4-alignment slack
            nrows_max = std::max(nrows_max, nrows);
            ncols_max = std::max(ncols_max, ncols);
            all_contig = all_contig && rc && cc;
            if (und_ix && rc && cc) {
                for (int cam = 0; cam < ncam; ++cam) {
                    const int32_t* ux = und_ix->data() + cam * npx;
                    const int32_t* uy = und_iy->data() + cam * npx;
                    int minx = INT32_MAX, miny = INT32_MAX, maxx = -1, maxy = -1;
                    bool interior = true;
                    for (int sy = r_lo; sy <= r_hi; ++sy)
                        for (int sx = c_lo; sx <= c_hi; ++sx) {
                            const size_t i = (size_t)sy * fw + sx;
                            const int x = ux[i] >> 5, y = uy[i] >> 5;
                            for (int dy = 0; dy < 2; ++dy)
                                for (int dx = 0; dx < 2; ++dx) {
                                    const int xx = x + dx, yy = y + dy;
                                    if (xx < 0 || xx >= fw || yy < 0 || yy >= fh) { interior = false; continue; }
                                    minx = std::min(minx, xx); maxx = std::max(maxx, xx);
                                    miny = std::min(miny, yy); maxy = std::max(maxy, yy);
                                }
                        }
                    int4 bx = make_int4(0, 0, 4, 0);
                    if (maxx >= 0) {
                        bx.x = minx & ~3;
                        bx.z = std::min(((maxx + 1 + 3) & ~3), (fw + 3) & ~3) - bx.x;
                        bx.y = miny;
                        bx.w = maxy - miny + 1;
                    }
                    raw_max = std::max(raw_max, (size_t)bx.z * (bx.w & 0xFFFF));
                    if (bx.w > 0xFFFF) all_contig = false;
                    bx.w |= interior ? (1 << 30) : 0;
                    boxes[cam * ntiles + (size_t)ty * ntx + tx] = bx;
                }
            }
        }
    h->k1_pitch_u = (ncols_max + 3) & ~3;
    h->k1_rows_u = nrows_max;
    const size_t und_bytes = (size_t)nrows_max * h->k1_pitch_u * 4;
    h->k1_mode = MODE_PLAIN;
    h->k1_smem = und_bytes;
    if (h->p.undistort) {
        if (const int rc = vti_upload(h, &h->d_und_lut, *und_packed)) return rc;
        const size_t tot = und_bytes + raw_max * 4;
        if (all_contig && (fw & 3) == 0 && tot <= 160 * 1024) {
            h->k1_mode = MODE_RAW;
            h->k1_smem = tot;
            if (const int rc = vti_upload(h, &h->d_k1_tiles, boxes)) return rc;
        } else {
            h->k1_mode = MODE_GATHER;
        }
    }
    if (h->k1_mode == MODE_RAW) return vti_raise_dyn_smem((const void*)k1_letterbox_kernel<MODE_RAW>, h->k1_smem);
    if (h->k1_mode == MODE_GATHER) return vti_raise_dyn_smem((const void*)k1_letterbox_kernel<MODE_GATHER>, h->k1_smem);
    return vti_raise_dyn_smem((const void*)k1_letterbox_kernel<MODE_PLAIN>, h->k1_smem);
}

// camera: per-frame ids (device) or null.  Only the remap depends on the camera, and a one-camera handle has one set of
// tables for every id, so ids reach the kernels only for undistort with more than one camera: the fast path then runs
// its per-frame camera form, and the generic kernel reads ids only when they are not null.
int vti_launch_k1(vti_handle* h, const uint8_t* frames, int B, float* net_in, const int32_t* camera, cudaStream_t s) {
    const bool multi = camera && h->p.undistort && h->n_cameras > 1;
    if (h->k1_mode == MODE_FAST_PLAIN || h->k1_mode == MODE_FAST_REMAP) {
        if ((reinterpret_cast<uintptr_t>(frames) & 7) || (reinterpret_cast<uintptr_t>(net_in) & 3)) {
            vti_set_error("vti_preprocess: frames must be 8-byte aligned and net_in 4-byte aligned (64-bit staging loads)");
            return VTI_EINVAL;
        }
        K1FastArgs f;
        f.frames = frames; f.out = net_in;
        f.tile_hdr = h->d_k1_tiles; f.lut = h->d_k1_lut;
        f.tap_x_idx = h->d_tap_x_idx; f.tap_x_a = h->d_tap_x_a; f.tap_y_i = h->d_tap_y_i; f.tap_y_b = h->d_tap_y_b;
        f.h = h->p.frame_h; f.w = h->p.frame_w; f.new_h = h->g.new_h; f.new_w = h->g.new_w;
        f.top = h->g.top; f.left = h->g.left; f.LH = h->g.LH; f.LW = h->g.LW;
        f.flip = h->p.channel_flip;
        f.pitch_u = h->k1_pitch_u;
        f.und_words = h->k1_und_words; f.lut_stride = h->k1_lut_stride;
        f.raw_pitch = h->k1_raw_pitch;
        f.camera = camera; f.n_cameras = h->n_cameras;
        dim3 grid((f.LW + FTX - 1) / FTX, (f.LH + FTY - 1) / FTY, B);
        int rc = k1_fast_dispatch(h, &f, 1, &grid, h->k1_smem, s, multi);
        if (rc) return rc;
        h->launches++;
        VTI_CUDA(cudaGetLastError());
        return VTI_OK;
    }
    K1Args a;
    a.frames = frames;
    a.out = net_in;
    a.tap_x_idx = h->d_tap_x_idx;
    a.tap_x_a = h->d_tap_x_a;
    a.tap_y_i = h->d_tap_y_i;
    a.tap_y_b = h->d_tap_y_b;
    a.und_lut = h->d_und_lut;
    a.tile_box = h->d_k1_tiles;
    a.h = h->p.frame_h; a.w = h->p.frame_w;
    a.new_h = h->g.new_h; a.new_w = h->g.new_w;
    a.top = h->g.top; a.left = h->g.left;
    a.LH = h->g.LH; a.LW = h->g.LW;
    a.area2x = (h->resize_mode == 2);
    a.flip = h->p.channel_flip;
    a.pitch_u = h->k1_pitch_u;
    a.rows_u = h->k1_rows_u;
    a.undistort = h->p.undistort;
    a.camera = multi ? camera : nullptr; a.n_cameras = h->n_cameras;
    dim3 grid((a.LW + TX - 1) / TX, (a.LH + TY - 1) / TY, B);
    if (h->k1_mode == MODE_RAW)
        k1_letterbox_kernel<MODE_RAW><<<grid, K1_THREADS, h->k1_smem, s>>>(a);
    else if (h->k1_mode == MODE_GATHER)
        k1_letterbox_kernel<MODE_GATHER><<<grid, K1_THREADS, h->k1_smem, s>>>(a);
    else
        k1_letterbox_kernel<MODE_PLAIN><<<grid, K1_THREADS, h->k1_smem, s>>>(a);
    h->launches++;
    VTI_CUDA(cudaGetLastError());
    return VTI_OK;
}

// K3 -- class-offset greedy NMS with torchvision.ops.nms semantics, block-wide, one CTA per frame, followed by the
// scale_boxes / clip / int() / ROI epilogue and the coefficient gather for the kept detections.
//
// Replaces (SURVEY.md 8a U4, U5, U7 and the box half of M1): ops.non_max_suppression + torchvision.ops.nms +
// ops.scale_boxes (reached from measurement.py:208-210) and measurement.py:251-260.
// Spec: oracle/post_spec.py nms_spec / scale_boxes_spec (bit-identical: same fp32 op order, no FMA, IoU compared
// against the threshold in double exactly like the C++ kernel's `ovr > iou_threshold`).
//
//   1. bitonic sort of the 64-bit keys (score bits | ~anchor | cls), descending
//      == stable descending score sort over ascending anchor order.  Up to 1024 candidates sort in registers; more
//      candidates are cut into descending score buckets of <= 1024 by a histogram of the score bits and each bucket
//      is compacted + sorted only if the sweep still has room below max_det (lazy sort)
//   2. greedy sweep in chunks of 64 sorted candidates:
//        a. every (candidate, already-kept box) pair is tested in parallel           -> suppressed-by-earlier bits
//        b. the 64x64 intra-chunk IoU bitmask is built with one ballot per row half  -> row masks
//        c. one warp resolves the chunk in rounds (all candidates no live earlier one suppresses are kept at once;
//           the transposed bitmask tells who those are) -> keep bits
//      stops as soon as max_det boxes are kept ( == torchvision nms followed by [:max_det] )
//   3. epilogue: un-letterbox + clip, int() truncation, ROI test on the truncated centre, class routing flags,
//      gather of the 32 mask coefficients of each kept anchor into a compact [max_det][32] block for K4.
#include <climits>
#include <cmath>
#include <cstring>

#include "vti_internal.h"

namespace {

constexpr int K3_THREADS = 1024;
constexpr int CHUNK = 64;
constexpr int MAX_DET_CAP = 1024;
constexpr int HIST_BINS = 2048;     // score bins of the lazy bucket sort
constexpr int KEYS_SMEM = 2048;     // sort buffer in shared memory (a score bucket holds <= 1024 keys unless one bin is oversized)

struct K3Args {
    const int32_t* cand_count;
    unsigned long long* cand_key;
    const float4* cand_box;
    const float* coef;          // [B][32][A]
    vti_det* dets;              // [B][max_det]
    int32_t* counts;            // [B]
    float* det_coef;            // [B][max_det][32]
    int32_t* env;               // [B][LW]
    int32_t* flags;             // [B] : bit0 overflow, bits 8.. = n_cand
    int cap, cap_pad, A, max_det, LW;
    double iou;                 // torchvision: (double)ovr > iou
    double iou_mid;             // midpoint of the two float32 neighbours that straddle iou (see iou_gt)
    int iou_tie_up;             // a quotient exactly at the midpoint rounds up (to even) -> suppressed
    unsigned hist_lo;           // score bits of the confidence threshold (every candidate score is above it)
    int hist_shift;             // (score bits - hist_lo) >> hist_shift < HIST_BINS for scores <= 1
    float gain, padx, pady, fw, fh;
    int roi_active, rx1, ry1, rx2, ry2;
    int stitch_id, fabric_id;
    int env_init;
    int ph, pw, all_dets, units_per_det;
    int32_t* unit_count;        // one counter for the whole batch
    uint4* units;
    int4* proto_bbox;           // [B] union of the crop windows K4 will read (x_lo, y_lo, x_hi, y_hi), empty = (1, 1, 0, 0)
};

// torchvision's test is `float32(inter / uni) > iou` with iou a double.  Let T be the smallest float32 above iou and
// P its predecessor: RN(inter / uni) >= T  <=>  inter / uni > (P + T) / 2, or == with the tie rounding to T (T's
// mantissa even).  (P + T) / 2 has 25 significant bits, uni 24: the product is exact in double, so the comparison
// below decides exactly what the division would, without the division (it was 21 % of this kernel's instructions).
__device__ __forceinline__ bool iou_gt(const float4 a, float aarea, const float4 b, float barea, const K3Args& k) {
    const float xx1 = fmaxf(a.x, b.x), yy1 = fmaxf(a.y, b.y);
    const float xx2 = fminf(a.z, b.z), yy2 = fminf(a.w, b.w);
    const float w = fmaxf(0.0f, __fsub_rn(xx2, xx1));
    const float h = fmaxf(0.0f, __fsub_rn(yy2, yy1));
    // disjoint boxes (the common case: most candidates are nowhere near most kept boxes): 0 / uni > iou is false for
    // every iou >= 0, and NaN (uni == 0) compares false as well
    if (!(w > 0.0f && h > 0.0f) && k.iou >= 0.0) return false;
    const float inter = __fmul_rn(w, h);
    const float uni = __fsub_rn(__fadd_rn(aarea, barea), inter);
    if (uni > 0.0f && uni < 3.0e38f) {
        const double lhs = (double)inter, rhs = __dmul_rn(k.iou_mid, (double)uni);
        return k.iou_tie_up ? (lhs >= rhs) : (lhs > rhs);
    }
    return (double)__fdiv_rn(inter, uni) > k.iou;          // degenerate boxes: the literal formula (NaN -> false)
}

// Bitonic sort (descending) of m keys: in registers + shuffles when there is at most one key per thread, in the
// buffer `keys` (shared or global) otherwise.  `src` is where the unsorted keys are; the result is in keys[0..m_pad).
__device__ __forceinline__ void sort_desc(unsigned long long* keys, const unsigned long long* src, int m, int tid,
                                          unsigned long long* s_keys) {
    int m_pad = 64;
    while (m_pad < m) m_pad <<= 1;
    if (m_pad <= K3_THREADS) {
        // one key per thread in a register; partners closer than a warp come through shuffles, no barrier
        unsigned long long key = (tid < m) ? src[tid] : 0ull;
        __syncthreads();                                   // src may be s_keys itself
        for (int k = 2; k <= m_pad; k <<= 1) {
            for (int j = k >> 1; j > 0; j >>= 1) {
                unsigned long long other;
                if (j >= 32) {
                    s_keys[tid] = key;
                    __syncthreads();
                    other = s_keys[tid ^ j];
                    __syncthreads();
                } else {
                    other = __shfl_xor_sync(0xffffffffu, key, j);
                }
                const bool keep_max = (((tid & k) == 0) == ((tid & j) == 0));
                key = keep_max ? (key > other ? key : other) : (key < other ? key : other);
            }
        }
        s_keys[tid] = key;
        __syncthreads();
    } else {
        for (int i = tid; i < m_pad; i += K3_THREADS) {
            if (keys != src) keys[i] = (i < m) ? src[i] : 0ull;
            else if (i >= m) keys[i] = 0ull;
        }
        __syncthreads();
        for (int k = 2; k <= m_pad; k <<= 1) {
            for (int j = k >> 1; j > 0; j >>= 1) {
                for (int i = tid; i < m_pad; i += K3_THREADS) {
                    const int p = i ^ j;
                    if (p > i) {
                        const unsigned long long x = keys[i], y = keys[p];
                        const bool desc = (i & k) == 0;
                        if (desc ? (x < y) : (x > y)) { keys[i] = y; keys[p] = x; }
                    }
                }
                __syncthreads();
            }
        }
    }
}

__global__ void __launch_bounds__(K3_THREADS, 1) k3_nms_kernel(const K3Args a) {
    extern __shared__ __align__(16) unsigned long long s_keys[];   // KEYS_SMEM entries
    __shared__ float4 s_kbox[MAX_DET_CAP];      // kept boxes (class offset applied)
    __shared__ float s_karea[MAX_DET_CAP];
    __shared__ unsigned long long s_kkey[MAX_DET_CAP];   // key of each kept box
    __shared__ float4 s_cbox[CHUNK];
    __shared__ float s_carea[CHUNK];
    __shared__ int s_sup[CHUNK];
    __shared__ unsigned long long s_row[CHUNK];
    __shared__ unsigned long long s_col[CHUNK];   // transpose of s_row: bit j of s_col[k] = candidate j (< k) suppresses k
    __shared__ int s_nk, s_m, s_lo_bin;
    __shared__ int s_upre[MAX_DET_CAP + 1];     // exclusive prefix of K4 work units per kept detection
    __shared__ int s_ubase;
    __shared__ int s_bb[4];
    __shared__ int s_hist[HIST_BINS];           // candidates per score bin (lazy bucket sort)

    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int n = a.cand_count[b];
    const bool overflow = n > a.cap;
    n = min(n, a.cap);

    unsigned long long* gkeys = a.cand_key + (size_t)b * a.cap_pad;
    for (int i = tid; i < a.LW; i += K3_THREADS) a.env[(size_t)b * a.LW + i] = a.env_init;
    if (tid == 0) s_nk = 0;

    // ---- 1 + 2. sort and greedy sweep.  Up to one key per thread: one sort of everything.  More candidates (low
    // confidence thresholds, thousands per frame): LAZY score buckets -- a histogram of the score bits cuts the
    // candidates into descending score ranges of <= 1024 each; a range is compacted, sorted and swept only when the
    // ranges above it left room below max_det, so the tail of low scores is usually never sorted at all.  (Equal
    // scores share a bin, hence a bucket: the order inside a bucket is the exact (score, anchor) order.)
    const bool bucketed = n > K3_THREADS;
    if (bucketed) {
        for (int i = tid; i < HIST_BINS; i += K3_THREADS) s_hist[i] = 0;
        __syncthreads();
        for (int i = tid; i < n; i += K3_THREADS) {
            const unsigned sb = (unsigned)(gkeys[i] >> 32);
            atomicAdd(&s_hist[min((int)((sb - a.hist_lo) >> a.hist_shift), HIST_BINS - 1)], 1);
        }
    }
    __syncthreads();
    const float4* __restrict__ gbox = a.cand_box + (size_t)b * a.A;
    int nk = 0, hi_bin = HIST_BINS - 1;
    bool last = !bucketed;
    for (;;) {
        int m = n;
        unsigned long long* keys = s_keys;
        if (!bucketed) {
            sort_desc(s_keys, gkeys, n, tid, s_keys);
        } else {
            // next bucket: bins [lo_bin, hi_bin] holding <= K3_THREADS candidates (at least one bin)
            if (warp == 0) {
                int acc = 0, top = hi_bin, taken = 0;
                bool stop = false;
                while (!stop && top >= 0) {
                    const int bin = top - lane;
                    int c = bin >= 0 ? s_hist[bin] : 0, pre = c;
#pragma unroll
                    for (int o = 1; o < 32; o <<= 1) {
                        const int v = __shfl_up_sync(0xffffffffu, pre, o);
                        if (lane >= o) pre += v;
                    }
                    const unsigned fit = __ballot_sync(0xffffffffu, bin >= 0 && acc + pre <= K3_THREADS);
                    int cnt = (fit == 0xffffffffu) ? 32 : (__ffs(~fit) - 1);   // leading lanes (bins) that still fit
                    if (cnt == 0 && taken == 0) cnt = 1;                       // a single oversized bin still forms a bucket
                    const int got = __shfl_sync(0xffffffffu, pre, max(cnt, 1) - 1);
                    if (cnt > 0) { acc += got; taken += cnt; top -= cnt; }
                    stop = cnt < 32;
                }
                if (lane == 0) { s_lo_bin = top + 1; s_m = 0; }
            }
            __syncthreads();
            const int lo_bin = s_lo_bin;
            for (int i = tid; i < n; i += K3_THREADS) {
                const unsigned long long key = gkeys[i];
                const int bin = min((int)(((unsigned)(key >> 32) - a.hist_lo) >> a.hist_shift), HIST_BINS - 1);
                if (bin >= lo_bin && bin <= hi_bin) {
                    const int pos = atomicAdd(&s_m, 1);
                    if (pos < KEYS_SMEM) s_keys[pos] = key;
                }
            }
            __syncthreads();
            m = s_m;
            last = lo_bin <= 0;
            hi_bin = lo_bin - 1;
            if (m > KEYS_SMEM) {
                // a pathological score distribution (thousands of candidates in one bin): sort everything at once in
                // the global buffer and start over
                m = n; keys = gkeys; nk = 0; last = true;
                __syncthreads();
                if (tid == 0) s_nk = 0;
            }
            if (m > 0) sort_desc(keys, keys, m, tid, s_keys);
            __syncthreads();
        }
        // ---- greedy sweep over this bucket's sorted keys, 64 at a time
        for (int c0 = 0; c0 < m && nk < a.max_det; c0 += CHUNK) {
            if (tid < CHUNK) {
                const int i = c0 + tid;
                float4 bx = make_float4(0.f, 0.f, 0.f, 0.f);
                float ar = 0.f;
                if (i < m) {
                    const unsigned long long key = keys[i];
                    const int anchor = 0xFFFFFF - (int)((key >> 8) & 0xFFFFFFull);
                    const float off = __fmul_rn((float)(int)(key & 0xFFull), 7680.0f);
                    const float4 r = gbox[anchor];
                    bx = make_float4(__fadd_rn(r.x, off), __fadd_rn(r.y, off), __fadd_rn(r.z, off), __fadd_rn(r.w, off));
                    ar = __fmul_rn(__fsub_rn(bx.z, bx.x), __fsub_rn(bx.w, bx.y));
                }
                s_cbox[tid] = bx;
                s_carea[tid] = ar;
                s_sup[tid] = (i < m) ? 0 : 1;
                s_col[tid] = 0ull;
            }
            __syncthreads();
            // a. against every box kept so far
            {
                const int j = tid & (CHUNK - 1);
                const float4 cb = s_cbox[j];
                const float ca = s_carea[j];
                bool sup = false;
                for (int k = tid >> 6; k < nk; k += K3_THREADS / CHUNK) sup |= iou_gt(s_kbox[k], s_karea[k], cb, ca, a);
                if (sup) s_sup[j] = 1;
            }
            // b. intra-chunk rows: warp w builds rows w and w+32; bit k of row j = IoU(j,k) > thr, k > j only
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                const int j = warp + 32 * half;
                const float4 jb = s_cbox[j];
                const float ja = s_carea[j];
                const bool lo = (lane > j) && iou_gt(jb, ja, s_cbox[lane], s_carea[lane], a);
                const bool hi = (lane + 32 > j) && iou_gt(jb, ja, s_cbox[lane + 32], s_carea[lane + 32], a);
                const unsigned mlo = __ballot_sync(0xffffffffu, lo), mhi = __ballot_sync(0xffffffffu, hi);
                if (lane == 0) s_row[j] = (unsigned long long)mlo | ((unsigned long long)mhi << 32);
                // (suppressing pairs are sparse: a handful of shared atomics per chunk)
                if (lo) atomicOr(&s_col[lane], 1ull << j);
                if (hi) atomicOr(&s_col[lane + 32], 1ull << j);
            }
            __syncthreads();
            // c. resolve on one warp
            if (warp == 0) {
                const unsigned slo = __ballot_sync(0xffffffffu, s_sup[lane] != 0);
                const unsigned shi = __ballot_sync(0xffffffffu, s_sup[lane + 32] != 0);
                unsigned long long removed = (unsigned long long)slo | ((unsigned long long)shi << 32);
                unsigned long long keep = 0ull;
                int room = a.max_det - nk;
                // Greedy resolve in ROUNDS instead of one dependent step per kept box: a live candidate that no LIVE
                // earlier candidate suppresses is kept whatever happens to the others (whoever could suppress it is
                // already dead), so all such candidates are kept at once, their rows retire more candidates, and the
                // next round looks again.  The number of rounds is the depth of the suppression chains inside the chunk
                // (2-4), not the number of boxes kept (20-30 in the stress scenes: 31 % of this kernel's time as a
                // serial chain of dependent shared-memory loads).  Identical result to the sequential scan.
                {
                    const unsigned long long rowA = s_row[lane], rowB = s_row[lane + 32];
                    const unsigned long long colA = s_col[lane], colB = s_col[lane + 32];
                    unsigned long long rem = removed, kp = 0ull;
                    for (;;) {
                        const unsigned long long alive = ~rem;
                        const bool fa = ((alive >> lane) & 1ull) && (colA & alive) == 0ull;
                        const bool fb = ((alive >> (lane + 32)) & 1ull) && (colB & alive) == 0ull;
                        const unsigned long long fr = (unsigned long long)__ballot_sync(0xffffffffu, fa) |
                                                      ((unsigned long long)__ballot_sync(0xffffffffu, fb) << 32);
                        if (fr == 0ull) break;
                        const unsigned long long mine = (fa ? rowA : 0ull) | (fb ? rowB : 0ull);
                        const unsigned lo32 = __reduce_or_sync(0xffffffffu, (unsigned)mine);
                        const unsigned hi32 = __reduce_or_sync(0xffffffffu, (unsigned)(mine >> 32));
                        kp |= fr;
                        rem |= fr | (unsigned long long)lo32 | ((unsigned long long)hi32 << 32);
                    }
                    if (__popcll(kp) <= room) {
                        keep = kp;
                    } else {
                        // max_det is reached inside this chunk: the FIRST `room` kept boxes in score order are wanted, and
                        // the rounds do not find them in order -- the sequential scan decides (last chunk of a frame only)
                        unsigned long long alive = ~removed;
                        while (alive != 0ull && room > 0) {
                            const int i = __ffsll((long long)alive) - 1;
                            keep |= (1ull << i);
                            removed |= s_row[i] | (1ull << i);
                            alive = ~removed & (i == 63 ? 0ull : (~0ull << (i + 1)));
                            --room;
                        }
                    }
                }
#pragma unroll
                for (int half = 0; half < 2; ++half) {
                    const int i = lane + 32 * half;
                    if ((keep >> i) & 1ull) {
                        const int pos = nk + __popcll(keep & ((1ull << i) - 1ull));
                        s_kbox[pos] = s_cbox[i];
                        s_karea[pos] = s_carea[i];
                        s_kkey[pos] = keys[c0 + i];
                    }
                }
                if (lane == 0) s_nk = nk + __popcll(keep);
            }
            __syncthreads();
            nk = s_nk;
        }
        if (last || nk >= a.max_det) break;
    }

    // ---- 3. epilogue
    vti_det* __restrict__ dets = a.dets + (size_t)b * a.max_det;
    int4* s_win = reinterpret_cast<int4*>(s_kbox);        // the sweep is over: s_kbox is reused for the crop windows
    unsigned* s_kflags = reinterpret_cast<unsigned*>(s_karea);   // ... and s_karea for the routing flags
    int nu = 0;                                            // K4 work units of this thread's detection
    __syncthreads();
    if (tid < nk) {
        const unsigned long long key = s_kkey[tid];
        const int anchor = 0xFFFFFF - (int)((key >> 8) & 0xFFFFFFull);
        const int cls = (int)(key & 0xFFull);
        const float4 r = gbox[anchor];
        vti_det d;
        d.box_lb[0] = r.x; d.box_lb[1] = r.y; d.box_lb[2] = r.z; d.box_lb[3] = r.w;
        const float fx1 = fminf(fmaxf(__fdiv_rn(__fsub_rn(r.x, a.padx), a.gain), 0.0f), a.fw);
        const float fy1 = fminf(fmaxf(__fdiv_rn(__fsub_rn(r.y, a.pady), a.gain), 0.0f), a.fh);
        const float fx2 = fminf(fmaxf(__fdiv_rn(__fsub_rn(r.z, a.padx), a.gain), 0.0f), a.fw);
        const float fy2 = fminf(fmaxf(__fdiv_rn(__fsub_rn(r.w, a.pady), a.gain), 0.0f), a.fh);
        d.box_frame[0] = fx1; d.box_frame[1] = fy1; d.box_frame[2] = fx2; d.box_frame[3] = fy2;
        const int x1 = (int)fx1, y1 = (int)fy1, x2 = (int)fx2, y2 = (int)fy2;
        d.box_int[0] = x1; d.box_int[1] = y1; d.box_int[2] = x2; d.box_int[3] = y2;
        d.conf = __uint_as_float((unsigned)(key >> 32));
        d.cls = cls;
        d.anchor = anchor;
        unsigned f = 0;
        bool in_roi = true;
        if (a.roi_active) {
            const int sx = x1 + x2, sy = y1 + y2;    // 0.5*(x1+x2) in [rx1, rx2]  <=>  x1+x2 in [2 rx1, 2 rx2]
            in_roi = (2 * a.rx1 <= sx) && (sx <= 2 * a.rx2) && (2 * a.ry1 <= sy) && (sy <= 2 * a.ry2);
        }
        if (in_roi) f |= VTI_F_IN_ROI;
        if (cls == a.stitch_id) f |= VTI_F_STITCH;
        else if (cls == a.fabric_id) f |= VTI_F_FABRIC;
        d.flags = f;
        d.m00 = 0; d.m10 = 0; d.m01 = 0;
        d.col_min = INT_MAX; d.col_max = -1;
        const double qnan = __longlong_as_double(0x7ff8000000000000LL);
        d.cx = qnan; d.cy = qnan; d.left_px = qnan; d.right_px = qnan;
        d.width_mm = qnan; d.edge_y = qnan; d.dist_mm = qnan; d.area_mm2 = qnan;
        dets[tid] = d;
        const bool wanted = a.all_dets || ((f & VTI_F_IN_ROI) && (f & (VTI_F_STITCH | VTI_F_FABRIC)));
        const VtiWindow w = vti_det_window(d.box_lb, a.ph, a.pw);
        s_win[tid] = make_int4(w.cx_lo, w.cx_hi, w.cy_lo, w.cy_hi);
        s_kflags[tid] = f;
        if (wanted && !w.empty)
            nu = ((w.cy_hi - w.cy_lo + 2 + VTI_K4_UR - 1) / VTI_K4_UR) * ((w.cx_hi - w.cx_lo + 2 + VTI_K4_UC - 1) / VTI_K4_UC);
    }
    // ---- K4 work units: one per (kept detection, VTI_K4_UR x VTI_K4_UC block of interpolation cells)
    {
        // block-wide exclusive scan (1024 threads = 32 warps)
        int incl = nu;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += v;
        }
        __shared__ int s_wsum[32];
        if (lane == 31) s_wsum[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            int ws = s_wsum[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int v = __shfl_up_sync(0xffffffffu, ws, o);
                if (lane >= o) ws += v;
            }
            s_wsum[lane] = ws;
        }
        __syncthreads();
        const int excl = incl - nu + (warp ? s_wsum[warp - 1] : 0);
        if (tid <= nk) s_upre[tid] = excl;                 // s_upre[nk] = total (nu = 0 there)
        const int total = s_wsum[31];
        if (tid == 0) { s_ubase = total ? atomicAdd(a.unit_count, total) : 0; s_bb[0] = INT_MAX; s_bb[1] = INT_MAX; s_bb[2] = -1; s_bb[3] = -1; }
        __syncthreads();
        if (tid < nk && nu > 0) {                          // union of the windows that have work units
            const int4 w = s_win[tid];
            atomicMin(&s_bb[0], w.x); atomicMin(&s_bb[1], w.z); atomicMax(&s_bb[2], w.y); atomicMax(&s_bb[3], w.w);
        }
        __syncthreads();
        if (tid == 0) a.proto_bbox[b] = s_bb[2] >= 0 ? make_int4(s_bb[0], s_bb[1], s_bb[2], s_bb[3]) : make_int4(1, 1, 0, 0);
        uint4* __restrict__ units = a.units + s_ubase;
        for (int i = tid; i < total; i += K3_THREADS) {
            int lo = 0, hi = nk - 1;                       // last detection with s_upre[k] <= i
            while (lo < hi) {
                const int mid = (lo + hi + 1) >> 1;
                if (s_upre[mid] <= i) lo = mid; else hi = mid - 1;
            }
            const int k = lo, local = i - s_upre[k];
            const int4 w = s_win[k];
            const int nb = (w.y - w.x + 2 + VTI_K4_UC - 1) / VTI_K4_UC;
            const int br = local / nb, bc = local - br * nb;
            const unsigned fabric = ((s_kflags[k] & VTI_F_FABRIC) && (s_kflags[k] & VTI_F_IN_ROI)) ? 0x8000u : 0u;
            units[i] = make_uint4((unsigned)b | fabric | ((unsigned)k << 16), (unsigned)br | ((unsigned)bc << 16),
                                  (unsigned)w.x | ((unsigned)w.z << 16), (unsigned)w.y | ((unsigned)w.w << 16));
        }
    }
    // coefficient gather: [32][A] strided -> compact [nk][32]
    const float* __restrict__ coef = a.coef + (size_t)b * VTI_NM * a.A;
    float* __restrict__ dc = a.det_coef + (size_t)b * a.max_det * VTI_NM;
    for (int i = tid; i < nk * VTI_NM; i += K3_THREADS) {
        const int k = i >> 5, c = i & 31;
        const unsigned long long key = s_kkey[k];
        const int anchor = 0xFFFFFF - (int)((key >> 8) & 0xFFFFFFull);
        dc[i] = __ldg(coef + (size_t)c * a.A + anchor);
    }
    if (tid == 0) {
        a.counts[b] = nk;
        a.flags[b] = (overflow ? 1 : 0) | (n << 8);
    }
}

}  // namespace

size_t vti_k3_smem_bytes(int) { return (size_t)KEYS_SMEM * sizeof(unsigned long long); }

int vti_k3_cap_pad(int cap) {
    int n_pad = 64;
    while (n_pad < cap) n_pad <<= 1;
    return n_pad;
}

int vti_k3_prepare(int cap) {
    return vti_raise_dyn_smem((const void*)k3_nms_kernel, vti_k3_smem_bytes(cap));
}

int vti_launch_k3(vti_handle* h, const float* coef, int B, vti_det* dets, int32_t* counts, int all_dets, cudaStream_t s) {
    K3Args a;
    a.cand_count = h->d_cand_count;
    a.cand_key = h->d_cand_key;
    a.cand_box = h->d_cand_box;
    a.coef = coef;
    a.dets = dets;
    a.counts = counts;
    a.det_coef = h->d_det_coef;
    a.env = h->d_env;
    a.flags = h->d_flags;
    a.cap = h->g.max_candidates; a.cap_pad = vti_k3_cap_pad(a.cap); a.A = h->g.A; a.max_det = h->p.max_det; a.LW = h->g.LW;
    a.iou = (h->p.iou_threshold != 0.0) ? h->p.iou_threshold : (double)h->p.iou;
    {
        float T = (float)a.iou;                                   // smallest float32 strictly above the threshold
        if (!((double)T > a.iou)) T = nextafterf(T, INFINITY);
        const float P = nextafterf(T, -INFINITY);
        a.iou_mid = ((double)P + (double)T) * 0.5;
        unsigned bits;
        memcpy(&bits, &T, sizeof(bits));
        a.iou_tie_up = (bits & 1u) == 0u;
    }
    const int fh = h->p.frame_h, fw = h->p.frame_w, LH = h->g.LH, LW = h->g.LW;
    // ops.scale_boxes: gain/pad are Python doubles, the tensor math is float32 (oracle/post_spec.py scale_boxes_spec)
    const double g1 = (double)LH / fh, g2 = (double)LW / fw;
    const double gain = g1 < g2 ? g1 : g2;
    a.gain = (float)gain;
    a.padx = (float)nearbyint((LW - fw * gain) / 2 - 0.1);
    a.pady = (float)nearbyint((LH - fh * gain) / 2 - 0.1);
    a.fw = (float)fw; a.fh = (float)fh;
    a.roi_active = h->roi.active; a.rx1 = h->roi.x1; a.ry1 = h->roi.y1; a.rx2 = h->roi.x2; a.ry2 = h->roi.y2;
    a.stitch_id = h->p.stitch_id; a.fabric_id = h->p.fabric_id;
    {
        const float c = h->p.conf > 0.0f ? h->p.conf : 0.0f, one = 1.0f;
        unsigned cb, ob;
        memcpy(&cb, &c, 4); memcpy(&ob, &one, 4);
        a.hist_lo = cb;
        a.hist_shift = 0;
        while (((ob - cb) >> a.hist_shift) >= (unsigned)HIST_BINS) ++a.hist_shift;
    }
    a.env_init = (h->p.variant == 1) ? INT_MAX : -1;
    a.ph = h->g.ph; a.pw = h->g.pw; a.all_dets = all_dets; a.units_per_det = h->units_per_det;
    a.unit_count = h->d_cand_count + h->p.max_batch;
    a.units = h->d_units;
    a.proto_bbox = h->d_proto_bbox;
    k3_nms_kernel<<<B, K3_THREADS, vti_k3_smem_bytes(h->g.max_candidates), s>>>(a);
    h->launches++;
    VTI_CUDA(cudaGetLastError());
    return VTI_OK;
}

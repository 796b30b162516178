// K5 -- the measure stage on the per-detection statistics K4 produced: routing, frame-resolution envelope, centroids,
// column extent, 1-D k-means row selection, envelope-proximity filter and the fp64 pixel -> millimetre projection.
//
// Replaces (SURVEY.md 8a M1, M3-M8; all fp64, exactly the reference's decisions):
//   measurement.py:44-65    compute_camera_plane / pixel_to_world_using_camera_plane
//                                           (cv2.undistortPoints == exactly 5 fixed-point iterations, (u-cx)*(1/fx))
//   measurement.py:88-113   kmeans_1d_two_clusters (labels NOT updated on break)
//   measurement.py:280-289, 302-330, 343-356, 390-430, 440-472
//   variant 1: Utils/check_stitch_distance.py:143-171 (labels updated on break), :331-334 (bbox-filled
//              fabric fallback), :349 (upper envelope), :442-443 (0 < d < 150), :489-507 (widths of final stitches only)
// Spec / oracle: oracle/measure_port.py (pinned against the verbatim reference through tests/golden/).
//
// One CTA per frame.  Per-stitch work is thread-parallel; the order-dependent pieces (k-means, numpy's pairwise
// summation order for np.mean, ordered list building) run on warp 0 so that results follow the reference's
// floating-point evaluation order.  The kernel is a latency chain, so the chain is kept short: while warp 0 iterates
// the k-means, warps 1..7 compute EVERY stitch's width, envelope-proximity decision and edge distance speculatively
// (pure functions of the stitch and the envelope) and the per-detection areas; the selection then only picks from
// what is already there.  Shared memory is sized by max_det (14 KB at 200), so that a K5 CTA fits beside K1's.
// Compiled with --fmad=false: numpy / OpenCV do not fuse multiply-adds.
// The 8-frame temporal median (measurement.py:474-484) is frame-ordered state and stays on the host.
#include <climits>
#include <vector>

#include "vti_internal.h"

namespace {

constexpr int K5_THREADS = 256;

struct Camera {
    double fx, fy, cx, cy, ifx, ify;
    double k1, k2, p1, p2, k3;
    double R[9], t[3], n[3], d_c;
};

struct K5Args {
    vti_det* dets;
    const int32_t* counts;
    const int32_t* env;        // [B][LW]
    int32_t* env_frame;        // [B][w]
    const int32_t* xmap;       // [w]
    const int32_t* flags;
    vti_frame_result* res;
    Camera cam;
    int max_det, LW, w, h;
    int variant, min_stitches, max_px, nb;
    int mask_variant;
    int cap;                   // entries per shared array: max_det rounded up to 8
    const Camera* cams;        // [n_cameras] (multi-camera kernel)
    const int32_t* camera;     // [B] camera id per frame (multi-camera kernel)
    int n_cameras;
};

// measurement.py:44-48 for one calibration.  undistort: the image was already undistorted by K1, so points are
// measured with dist = 0.  One function for the handle's own camera and for every camera of the device array, so that
// camera 0 of a multi-camera handle projects bit for bit like a one-camera handle.
Camera camera_of(const double K[9], const double dist[5], const double R[9], const double t[3], int undistort) {
    Camera c;
    c.fx = K[0]; c.fy = K[4]; c.cx = K[2]; c.cy = K[5];
    c.ifx = 1.0 / c.fx; c.ify = 1.0 / c.fy;
    const bool lens = !undistort;
    c.k1 = lens ? dist[0] : 0.0; c.k2 = lens ? dist[1] : 0.0;
    c.p1 = lens ? dist[2] : 0.0; c.p2 = lens ? dist[3] : 0.0; c.k3 = lens ? dist[4] : 0.0;
    for (int i = 0; i < 9; ++i) c.R[i] = R[i];
    for (int i = 0; i < 3; ++i) c.t[i] = t[i];
    c.n[0] = R[2]; c.n[1] = R[5]; c.n[2] = R[8];                 // n_c = R[:, 2]   (measurement.py:46)
    c.d_c = -(c.n[0] * t[0] + c.n[1] * t[1] + c.n[2] * t[2]);     // measurement.py:47
    return c;
}

__device__ __forceinline__ bool pixel_to_world(const Camera& c, double u, double v, double out[3]) {
    const double x0 = (u - c.cx) * c.ifx, y0 = (v - c.cy) * c.ify;
    double x = x0, y = y0;
#pragma unroll 1
    for (int it = 0; it < 5; ++it) {
        const double r2 = x * x + y * y;
        const double icd = 1.0 / (1.0 + ((c.k3 * r2 + c.k2) * r2 + c.k1) * r2);
        const double dx = 2.0 * c.p1 * x * y + c.p2 * (r2 + 2.0 * x * x);
        const double dy = c.p1 * (r2 + 2.0 * y * y) + 2.0 * c.p2 * x * y;
        x = (x0 - dx) * icd;
        y = (y0 - dy) * icd;
    }
    const double den = c.n[0] * x + c.n[1] * y + c.n[2];
    if (fabs(den) < 1e-9) return false;
    const double s = -c.d_c / den;
    const double v0 = s * x - c.t[0], v1 = s * y - c.t[1], v2 = s - c.t[2];
    out[0] = c.R[0] * v0 + c.R[3] * v1 + c.R[6] * v2;
    out[1] = c.R[1] * v0 + c.R[4] * v1 + c.R[7] * v2;
    out[2] = c.R[2] * v0 + c.R[5] * v1 + c.R[8] * v2;
    return true;
}

__device__ __forceinline__ bool dist_mm(const Camera& c, double u0, double v0, double u1, double v1, double* mm) {
    double a[3], b[3];
    if (!pixel_to_world(c, u0, v0, a) || !pixel_to_world(c, u1, v1, b)) return false;
    const double d0 = b[0] - a[0], d1 = b[1] - a[1], d2 = b[2] - a[2];
    *mm = sqrt(d0 * d0 + d1 * d1 + d2 * d2) * 1000.0;
    return true;
}

// np.add.reduce on one warp, same association order as numpy's pairwise_sum (add.reduce on a contiguous float64
// vector): the 8 partial sums r[j] of a <= 128-element block live in lanes 0..7, are combined as
// ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)), the tail is added sequentially, and longer vectors split at n/2 rounded down to a
// multiple of 8.  Every lane returns the sum.  (Warp-uniform control flow.)  The <= 128 block -- every vector of the
// configured scenes -- is inlined into the kernel (shared-memory loads, several in flight, no call frame: as a plain
// recursive function it took 80 % of warp 0's time); longer vectors take the recursive path.
__device__ __forceinline__ double np_block_warp(const double* a, int n, int lane) {      // n <= 128
    if (n < 8) {
        double r = 0.0;
        for (int i = 0; i < n; ++i) r += a[i];
        return r;
    }
    const int nb = n & ~7;
    double r = 0.0;
    if (lane < 8) {
        r = a[lane];
        int i = 8 + lane;
        for (; i + 24 < nb; i += 32) {                     // four loads in flight; the adds keep numpy's order
            const double x0 = a[i], x1 = a[i + 8], x2 = a[i + 16], x3 = a[i + 24];
            r += x0; r += x1; r += x2; r += x3;
        }
        for (; i < nb; i += 8) r += a[i];
    }
    r += __shfl_down_sync(0xffffffffu, r, 1);
    r += __shfl_down_sync(0xffffffffu, r, 2);
    r += __shfl_down_sync(0xffffffffu, r, 4);
    r = __shfl_sync(0xffffffffu, r, 0);
    double t[7];
#pragma unroll
    for (int k = 0; k < 7; ++k) t[k] = (nb + k < n) ? a[nb + k] : 0.0;
#pragma unroll
    for (int k = 0; k < 7; ++k)
        if (nb + k < n) r += t[k];
    return r;
}

__device__ __noinline__ double np_sum_warp_long(const double* a, int n, int lane) {
    if (n <= 128) return np_block_warp(a, n, lane);
    int n2 = n / 2;
    n2 -= n2 % 8;
    return np_sum_warp_long(a, n2, lane) + np_sum_warp_long(a + n2, n - n2, lane);
}

__device__ __forceinline__ double np_sum_warp(const double* a, int n, int lane) {
    return n <= 128 ? np_block_warp(a, n, lane) : np_sum_warp_long(a, n, lane);
}

// Two independent vectors at once (the two k-means clusters, distance and width averages): the same operations in the
// same order per vector, the two dependency chains interleaved.  Both n <= 128.
__device__ __forceinline__ void np_block_warp2(const double* a0, int n0, const double* a1, int n1, int lane, double& s0, double& s1) {
    const int nb0 = n0 & ~7, nb1 = n1 & ~7;
    double r0 = 0.0, r1 = 0.0;
    if (lane < 8) {
        if (nb0) r0 = a0[lane];
        if (nb1) r1 = a1[lane];
        const int nbm = max(nb0, nb1);
        for (int i = 8 + lane; i < nbm; i += 8) {
            if (i < nb0) r0 += a0[i];
            if (i < nb1) r1 += a1[i];
        }
    }
#pragma unroll
    for (int o = 1; o < 8; o <<= 1) {
        r0 += __shfl_down_sync(0xffffffffu, r0, o);
        r1 += __shfl_down_sync(0xffffffffu, r1, o);
    }
    r0 = __shfl_sync(0xffffffffu, r0, 0);
    r1 = __shfl_sync(0xffffffffu, r1, 0);
    double t0[7], t1[7];
#pragma unroll
    for (int k = 0; k < 7; ++k) {
        t0[k] = (nb0 + k < n0) ? a0[nb0 + k] : 0.0;
        t1[k] = (nb1 + k < n1) ? a1[nb1 + k] : 0.0;
    }
#pragma unroll
    for (int k = 0; k < 7; ++k) {
        if (nb0 + k < n0) r0 += t0[k];
        if (nb1 + k < n1) r1 += t1[k];
    }
    s0 = r0; s1 = r1;
}

__device__ __forceinline__ void np_sum_warp2(const double* a0, int n0, const double* a1, int n1, int lane, double& s0, double& s1) {
    if (n0 <= 128 && n1 <= 128) { np_block_warp2(a0, n0, a1, n1, lane, s0, s1); return; }
    s0 = np_sum_warp(a0, n0, lane);
    s1 = np_sum_warp(a1, n1, lane);
}

// dst0 <- the src[i] with flag[i] == 0, dst1 <- those with flag[i] == 1 (i in [0, n), order preserved): both clusters in one pass
__device__ __forceinline__ void compact2_warp(const double* src, const unsigned char* flag, int n, double* dst0, double* dst1,
                                              int& m0, int& m1, int lane) {
    m0 = 0; m1 = 0;
    const unsigned lt = (1u << lane) - 1u;
    for (int base = 0; base < n; base += 32) {
        const int i = base + lane;
        const int f = (i < n) ? (int)flag[i] : 2;
        const double v = (i < n) ? src[i] : 0.0;
        const unsigned k0 = __ballot_sync(0xffffffffu, f == 0), k1 = __ballot_sync(0xffffffffu, f == 1);
        if (f == 0) dst0[m0 + __popc(k0 & lt)] = v;
        else if (f == 1) dst1[m1 + __popc(k1 & lt)] = v;
        m0 += __popc(k0); m1 += __popc(k1);
    }
    __syncwarp();
}

// dst[0..m) = src[i] for the i in [0, n) with flag[i] == want, order preserved; returns m (one warp).
__device__ __forceinline__ int compact_warp(const double* src, const unsigned char* flag, int want, int n, double* dst, int lane) {
    int m = 0;
    for (int base = 0; base < n; base += 32) {
        const int i = base + lane;
        const bool p = (i < n) && (flag[i] == want);
        const unsigned msk = __ballot_sync(0xffffffffu, p);
        if (p) dst[m + __popc(msk & ((1u << lane) - 1u))] = src[i];
        m += __popc(msk);
    }
    __syncwarp();
    return m;
}

// median of the valid envelope rows at columns clip(cx_int + dx, 0, w-1), dx in [-nb, nb]; false if none valid
__device__ __forceinline__ bool env_median(const int32_t* envf, int w, int cx_int, int nb, double* med) {
    int v[16];
    int m = 0;
    for (int dx = -nb; dx <= nb; ++dx) {
        const int x = min(max(cx_int + dx, 0), w - 1);
        const int e = envf[x];
        if (e >= 0) {
            int j = m++;
            while (j > 0 && v[j - 1] > e) { v[j] = v[j - 1]; --j; }
            v[j] = e;
        }
    }
    if (m == 0) return false;
    *med = (m & 1) ? (double)v[m >> 1] : ((double)v[(m >> 1) - 1] + (double)v[m >> 1]) / 2.0;
    return true;
}

// Area of every bitmap on the fabric plane (north-star "area"; spec: oracle/measure_port.py defect_area_mm2): m00 pixels x
// the plane area of one pixel at the centroid, |dP/du x dP/dv| by central differences.  The four projections of a
// detection run on four neighbouring lanes.  Called by whole warps: thread t of nt (both multiples of 32 apart).
__device__ void areas(const Camera& cam, vti_det* __restrict__ dets, int n, int t, int nt, int lane) {
    for (int base = 0; base < 4 * n; base += nt) {                   // warp-uniform trip count (shuffles below)
        const int q4 = base + t, k = q4 >> 2, j = q4 & 3;
        double p[3] = {0.0, 0.0, 0.0};
        bool ok = false;
        long long m00 = 0;
        if (k < n) {
            m00 = dets[k].m00;
            if (m00 > 0) {
                const double cx = (double)dets[k].m10 / (double)m00, cy = (double)dets[k].m01 / (double)m00;
                ok = pixel_to_world(cam, cx + (j == 0 ? -0.5 : (j == 1 ? 0.5 : 0.0)), cy + (j == 2 ? -0.5 : (j == 3 ? 0.5 : 0.0)), p);
            }
        }
        const int l0 = lane & ~3;
        double q[4][3];
#pragma unroll
        for (int jj = 0; jj < 4; ++jj)
#pragma unroll
            for (int c = 0; c < 3; ++c) q[jj][c] = __shfl_sync(0xffffffffu, p[c], l0 + jj);
        const unsigned okm = __ballot_sync(0xffffffffu, ok);
        if (k < n && j == 0 && m00 > 0 && ((okm >> l0) & 0xFu) == 0xFu) {
            const double ux = q[1][0] - q[0][0], uy = q[1][1] - q[0][1], uz = q[1][2] - q[0][2];
            const double vx = q[3][0] - q[2][0], vy = q[3][1] - q[2][1], vz = q[3][2] - q[2][2];
            const double c0 = uy * vz - uz * vy, c1 = uz * vx - ux * vz, c2 = ux * vy - uy * vx;
            dets[k].area_mm2 = (double)m00 * sqrt(c0 * c0 + c1 * c1 + c2 * c2) * 1e6;
        }
    }
}

// MULTI: frame b is measured with camera a.camera[b] of a.cams (an id out of range: VTI_ST_BAD_CAMERA, nothing measured)
template <bool MULTI>
__global__ void __launch_bounds__(K5_THREADS, 4) k5_measure_kernel(const K5Args a) {
    // everything warp 0 walks sequentially lives in shared memory (global round trips were 70 % of v1's time); the
    // arrays hold a.cap = max_det (rounded up to 8) entries each
    extern __shared__ __align__(16) unsigned char s_raw[];
    const int N = a.cap;
    double* s_cy = reinterpret_cast<double*>(s_raw);
    double* s_tmp = s_cy + N;
    double* s_w = s_tmp + N;              // per stitch: width_mm (NaN = none)
    double* s_d = s_w + N;                // per final entry: dist_mm (NaN = none)
    double* s_med = s_d + N;              // per stitch (speculative): envelope median at the stitch's column
    double* s_dsp = s_med + N;            // per stitch (speculative): dist_mm (NaN = none)
    double* s_wsp = s_dsp + N;            // per stitch (speculative, variant 1): width_mm (NaN = none)
    unsigned* s_flags = reinterpret_cast<unsigned*>(s_wsp + N);   // per detection
    short* s_st = reinterpret_cast<short*>(s_flags + N);          // stitch list -> det index
    short* s_sel = s_st + N;                                      // selected -> stitch index
    short* s_fin = s_sel + N;
    unsigned char* s_lab = reinterpret_cast<unsigned char*>(s_fin + N);
    unsigned char* s_new = s_lab + N;
    unsigned char* s_pass = s_new + N;    // per stitch (speculative): passes the envelope-proximity filter
    unsigned char* s_mok = s_pass + N;    // per stitch (speculative): the envelope median exists
    __shared__ int s_ns, s_nsel, s_nfin, s_nfab, s_ndrop;
    __shared__ long long s_envsum;
    __shared__ int s_envcnt;

    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31;
    const int n = a.counts[b];
    vti_det* __restrict__ dets = a.dets + (size_t)b * a.max_det;
    int32_t* __restrict__ envf = a.env_frame + (size_t)b * a.w;
    const double qnan = __longlong_as_double(0x7ff8000000000000LL);
    int cam_id = 0;
    if (MULTI) {
        cam_id = a.camera[b];
        if ((unsigned)cam_id >= (unsigned)a.n_cameras) {
            for (int x = tid; x < a.w; x += K5_THREADS) envf[x] = -1;    // no envelope for the overlay to draw
            if (tid == 0) {
                vti_frame_result r;
                r.status = VTI_ST_BAD_CAMERA | ((a.flags[b] & 1) ? VTI_ST_OVERFLOW : 0);
                r.n_det = n;
                r.n_cand = a.flags[b] >> 8;
                r.n_stitch = 0; r.n_fabric = 0; r.n_dist = 0; r.n_width = 0; r.env_valid = 0;
                r.avg_dist = qnan; r.avg_width = qnan; r.env_mean = qnan;
                a.res[b] = r;
            }
            return;
        }
    }
    const Camera& cam = MULTI ? a.cams[cam_id] : a.cam;

    if (tid == 0) { s_envsum = 0; s_envcnt = 0; s_nfab = 0; s_ns = 0; s_ndrop = 0; }
    __syncthreads();
    // ---- finalize K4's statistics, frame-resolution envelope
    for (int k = tid; k < n; k += K5_THREADS) {
        unsigned f = dets[k].flags;
        const long long m00 = dets[k].m00;
        if (a.mask_variant == 1 && !(f & VTI_F_LB_MASK)) {
            // newer Ultralytics (construct_result): `keep = masks.amax((-2, -1)) > 0` removes the detection
            f |= VTI_F_DROPPED;
            atomicAdd(&s_ndrop, 1);
        }
        if (m00 > 0) {
            f |= VTI_F_HAS_MASK;
        } else {
            dets[k].col_min = -1; dets[k].col_max = -1;
        }
        dets[k].flags = f;
        s_flags[k] = f;
    }
    const int* __restrict__ env = a.env + (size_t)b * a.LW;
    // envelope at frame columns (variant 1 keeps INT_MAX = none for now).  Two dependent global loads per column: four
    // columns per thread are in flight at once, and the valid-row sum is taken from the registers (variant 0)
    long long esum = 0;
    int ecnt = 0;
    for (int x0 = tid; x0 < a.w; x0 += 4 * K5_THREADS) {
        int xi[4], e[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) { const int x = x0 + q * K5_THREADS; xi[q] = x < a.w ? __ldg(a.xmap + x) : 0; }
#pragma unroll
        for (int q = 0; q < 4; ++q) e[q] = env[xi[q]];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int x = x0 + q * K5_THREADS;
            if (x < a.w) {
                envf[x] = e[q];
                if (e[q] >= 0 && e[q] != INT_MAX) { esum += e[q]; ++ecnt; }
            }
        }
    }
    __syncthreads();
    if (a.variant == 1) {
        // mask-less fabric detection -> filled bbox rectangle (check_stitch_distance.py:331-334), upper envelope
        for (int k = 0; k < n; ++k) {
            const unsigned f = s_flags[k];
            if (!(f & VTI_F_FABRIC) || (f & VTI_F_HAS_MASK) || (f & VTI_F_DROPPED)) continue;
            const int x1 = max(min(dets[k].box_int[0], dets[k].box_int[2]), 0);
            const int x2 = min(max(dets[k].box_int[0], dets[k].box_int[2]), a.w - 1);
            const int y1 = max(min(dets[k].box_int[1], dets[k].box_int[3]), 0);
            const int y2 = min(max(dets[k].box_int[1], dets[k].box_int[3]), a.h - 1);
            if (y1 > y2) continue;
            for (int x = x1 + tid; x <= x2; x += K5_THREADS) envf[x] = min(envf[x], y1);
            __syncthreads();               // uniform: n and the flags are the same for every thread
        }
        __syncthreads();
        esum = 0; ecnt = 0;                // the fallback may have changed columns: sum what is there now
        for (int x = tid; x < a.w; x += K5_THREADS) {
            int e = envf[x];
            if (e == INT_MAX) { e = -1; envf[x] = -1; }
            if (e >= 0) { esum += e; ++ecnt; }
        }
        __syncthreads();
    }
    {
        for (int o = 16; o > 0; o >>= 1) {
            esum += __shfl_xor_sync(0xffffffffu, esum, o);
            ecnt += __shfl_xor_sync(0xffffffffu, ecnt, o);
        }
        if (lane == 0 && ecnt > 0) {
            atomicAdd((unsigned long long*)&s_envsum, (unsigned long long)esum);
            atomicAdd(&s_envcnt, ecnt);
        }
    }
    // ---- routing (measurement.py:249-272): ordered stitch list, one warp, ballot compaction
    if (tid < 32) {
        int ns = 0, nf = 0;
        for (int base = 0; base < n; base += 32) {
            const int k = base + lane;
            const unsigned f = k < n ? s_flags[k] : 0u;
            const bool roi = (f & VTI_F_IN_ROI) && !(f & VTI_F_DROPPED);
            const bool st = roi && (f & VTI_F_STITCH);
            const bool fb = roi && !(f & VTI_F_STITCH) && (f & VTI_F_FABRIC) && ((f & VTI_F_HAS_MASK) || a.variant == 1);
            const unsigned ms = __ballot_sync(0xffffffffu, st), mf = __ballot_sync(0xffffffffu, fb);
            if (st) s_st[ns + __popc(ms & ((1u << lane) - 1u))] = (short)k;
            ns += __popc(ms);
            nf += __popc(mf);
        }
        if (lane == 0) { s_ns = ns; s_nfab = nf; }
    }
    __syncthreads();
    const int ns = s_ns;
    vti_frame_result r;
    r.status = VTI_ST_OK;
    r.n_det = n - s_ndrop;
    r.n_cand = a.flags[b] >> 8;
    r.n_stitch = ns;
    r.n_fabric = s_nfab;
    r.n_dist = 0; r.n_width = 0;
    r.env_valid = s_envcnt;
    r.avg_dist = qnan; r.avg_width = qnan;
    r.env_mean = s_envcnt > 0 ? (double)s_envsum / (double)s_envcnt : qnan;
    const int ovf = (a.flags[b] & 1) ? VTI_ST_OVERFLOW : 0;
    if (s_envcnt == 0 || ns == 0) {
        if (tid == 0) {
            r.status = (s_envcnt == 0 ? VTI_ST_NO_FABRIC : VTI_ST_NO_STITCH) | ovf;
            a.res[b] = r;
        }
        areas(cam, dets, n, tid, K5_THREADS, lane);
        return;
    }

    // ---- per-stitch centroid / extent (measurement.py:302-330)
    for (int i = tid; i < ns; i += K5_THREADS) {
        vti_det& d = dets[s_st[i]];
        double cx, cy, left, right;
        const int x1 = d.box_int[0], y1 = d.box_int[1], x2 = d.box_int[2], y2 = d.box_int[3];
        const long long m00 = d.m00;
        if (m00 > 0) {
            cx = (double)d.m10 / (double)m00;
            cy = (double)d.m01 / (double)m00;
            left = (double)d.col_min;
            right = (double)d.col_max;
        } else {
            cx = (double)(x1 + x2) / 2.0;
            cy = (double)(y1 + y2) / 2.0;
            left = (double)x1;
            right = (double)x2;
        }
        d.cx = cx; d.cy = cy; d.left_px = left; d.right_px = right;
        s_cy[i] = cy;
        s_w[i] = qnan;
    }
    __syncthreads();

    // ---- row selection (measurement.py:390-406): warp 0, lanes cooperate, numpy's evaluation order is kept
    if (tid < 32) {
        int nsel = 0;
        if (ns >= 2) {
            double c0 = 1e300, c1 = -1e300;
            for (int i = lane; i < ns; i += 32) { c0 = fmin(c0, s_cy[i]); c1 = fmax(c1, s_cy[i]); }
            for (int o = 16; o > 0; o >>= 1) {
                c0 = fmin(c0, __shfl_xor_sync(0xffffffffu, c0, o));
                c1 = fmax(c1, __shfl_xor_sync(0xffffffffu, c1, o));
            }
            for (int i = lane; i < ns; i += 32) s_lab[i] = 0;
            __syncwarp();
            bool lab_means = false;                          // (lm0, lm1) are the means of the groups s_lab describes
            double lm0 = 0.0, lm1 = 0.0;
            for (int it = 0; it < 10; ++it) {
                int ones = 0;
                for (int base = 0; base < ns; base += 32) {
                    const int i = base + lane;
                    const bool nw = (i < ns) && (fabs(s_cy[i] - c1) < fabs(s_cy[i] - c0));
                    if (i < ns) s_new[i] = nw;
                    ones += __popc(__ballot_sync(0xffffffffu, nw));
                }
                __syncwarp();
                bool stop = (ones == 0 || ones == ns);
                double n0 = 0.0, n1 = 0.0;
                bool means = false;                          // (n0, n1) are the cluster means of s_new
                if (!stop) {
                    int m0, m1;
                    double t0, t1;
                    compact2_warp(s_cy, s_new, ns, s_tmp, s_d, m0, m1, lane);      // s_d is free until the final list exists
                    np_sum_warp2(s_tmp, m0, s_d, m1, lane, t0, t1);
                    __syncwarp();
                    n0 = t0 / (double)m0; n1 = t1 / (double)m1;
                    means = true;
                    stop = (n0 == c0 && n1 == c1);
                }
                if (!stop || a.variant == 1) {               // the reference's break leaves the labels stale (variant 0)
                    for (int i = lane; i < ns; i += 32) s_lab[i] = s_new[i];
                    lab_means = means; lm0 = n0; lm1 = n1;
                }
                __syncwarp();
                if (stop) break;
                c0 = n0; c1 = n1;
            }
            int chosen = 0;
            {
                // means of the two label groups: the k-means has them already whenever the labels are those of an
                // iteration that computed its means (the usual exit); otherwise (first-iteration exits) compute them
                const double fm = (double)s_envsum / (double)s_envcnt;
                double m0 = 1e9, m1 = 1e9;
                if (lab_means) {
                    m0 = lm0; m1 = lm1;
                } else {
                    int c_0, c_1;
                    double t0, t1;
                    compact2_warp(s_cy, s_lab, ns, s_tmp, s_d, c_0, c_1, lane);
                    np_sum_warp2(s_tmp, c_0, s_d, c_1, lane, t0, t1);
                    __syncwarp();
                    if (c_0 > 0) m0 = t0 / (double)c_0;
                    if (c_1 > 0) m1 = t1 / (double)c_1;
                }
                chosen = (fabs(m0 - fm) < fabs(m1 - fm)) ? 0 : 1;
            }
            for (int base = 0; base < ns; base += 32) {
                const int i = base + lane;
                const bool p = (i < ns) && (s_lab[i] == chosen);
                const unsigned msk = __ballot_sync(0xffffffffu, p);
                if (p) s_sel[nsel + __popc(msk & ((1u << lane) - 1u))] = (short)i;
                nsel += __popc(msk);
            }
        } else {
            for (int i = lane; i < ns; i += 32) s_sel[i] = (short)i;
            nsel = ns;
        }
        if (lane == 0) s_nsel = nsel;
    } else {
        // ---- warps 1..7, while warp 0 selects the row: everything that is a pure function of one stitch and the envelope,
        //      for EVERY stitch -- width (measurement.py:343-356), envelope-proximity decision (:409-430), edge distance
        //      (:440-459) [+ variant 1's width of a final stitch] -- and the per-detection areas
        const int t0 = tid - 32, NT = K5_THREADS - 32;
        for (int i = t0; i < ns; i += NT) {
            vti_det& d = dets[s_st[i]];
            const double cx = d.cx, cy = d.cy, left = d.left_px, right = d.right_px;
            double med, mm;
            if (a.variant == 0) {
                if (dist_mm(cam, left, cy, right, cy, &mm)) { d.width_mm = mm; s_w[i] = mm; }
            }
            bool ok = false;
            if (env_median(envf, a.w, (int)rint(cx), a.nb, &med)) {
                const double env_y = (double)(int)rint(med);
                const double dd = cy - env_y;
                ok = (a.variant == 0) ? (fabs(dd) < (double)a.max_px) : (dd > 0.0 && dd < (double)a.max_px);
            }
            s_pass[i] = ok;
            const int cx_int = min(max((int)rint(cx), 0), a.w - 1);
            const bool mok = env_median(envf, a.w, cx_int, a.nb, &med);
            s_mok[i] = mok;
            s_med[i] = mok ? med : qnan;
            s_dsp[i] = (mok && dist_mm(cam, cx, cy, cx, med, &mm)) ? mm : qnan;
            if (a.variant == 1) {
                double wv = qnan;
                if (dist_mm(cam, left, cy, right, cy, &mm)) wv = mm;
                else if (dist_mm(cam, cx, cy, cx + 10.0, cy, &mm)) wv = ((right - left) / 10.0) * mm;
                s_wsp[i] = wv;
            }
        }
        areas(cam, dets, n, t0, NT, lane);
    }
    __syncthreads();
    const int nsel = s_nsel;

    // ---- envelope-proximity filter (measurement.py:409-430): the decisions are there, warp 0 builds the ordered list
    if (tid < 32) {
        int nf = 0;
        for (int base = 0; base < nsel; base += 32) {
            const int j = base + lane;
            const bool p = (j < nsel) && s_pass[s_sel[j]];
            const unsigned msk = __ballot_sync(0xffffffffu, p);
            if (p) s_fin[nf + __popc(msk & ((1u << lane) - 1u))] = s_sel[j];
            nf += __popc(msk);
        }
        if (nf == 0) { for (int j = lane; j < nsel; j += 32) s_fin[j] = s_sel[j]; nf = nsel; }
        if (lane == 0) s_nfin = nf;
    }
    __syncthreads();
    const int nfin = s_nfin;

    // ---- edge distances (measurement.py:440-459) [+ widths of the final stitches, variant 1]: picked from what warps
    //      1..7 computed for every stitch
    for (int j = tid; j < nfin; j += K5_THREADS) {
        const int i = s_fin[j];
        vti_det& d = dets[s_st[i]];
        const double dv = s_dsp[i];
        s_d[j] = dv;
        if (s_mok[i]) {
            d.edge_y = s_med[i];
            if (dv == dv) d.dist_mm = dv;
        }
        if (a.variant == 1) {
            const double wv = s_wsp[i];
            if (wv == wv) { d.width_mm = wv; s_w[i] = wv; }
        }
    }
    __syncthreads();
    // ---- record flags: one writer per detection
    for (int j = tid; j < nsel; j += K5_THREADS) s_flags[s_st[s_sel[j]]] |= VTI_F_SELECTED;
    __syncthreads();
    for (int j = tid; j < nfin; j += K5_THREADS) {
        unsigned f = VTI_F_FINAL;
        if (s_d[j] == s_d[j]) f |= VTI_F_HAS_DIST;
        s_flags[s_st[s_fin[j]]] |= f;
    }
    __syncthreads();
    for (int i = tid; i < ns; i += K5_THREADS) {
        unsigned f = s_flags[s_st[i]];
        if (s_w[i] == s_w[i]) f |= VTI_F_HAS_WIDTH;
        dets[s_st[i]].flags = f;
    }

    // ---- averages (measurement.py:469-472), numpy summation order, warp 0
    __syncthreads();
    if (tid < 32) {
        // s_new / s_lab mark the valid entries so that compact_warp can gather them in order; the two sums run interleaved
        for (int j = lane; j < nfin; j += 32) s_new[j] = (s_d[j] == s_d[j]);
        const double* wsrc = s_w;
        int wn = ns;
        if (a.variant == 0) {
            for (int i = lane; i < ns; i += 32) s_lab[i] = (s_w[i] == s_w[i]);
        } else {
            for (int j = lane; j < nfin; j += 32) { const double wv = s_w[s_fin[j]]; s_cy[j] = wv; s_lab[j] = (wv == wv); }
            wsrc = s_cy; wn = nfin;
        }
        __syncwarp();
        const int md = compact_warp(s_d, s_new, 1, nfin, s_tmp, lane);
        const int mw = compact_warp(wsrc, s_lab, 1, wn, s_dsp, lane);          // s_dsp is free once the final list is written
        double sd, sw;
        np_sum_warp2(s_tmp, md, s_dsp, mw, lane, sd, sw);
        r.n_dist = md;
        if (md >= a.min_stitches) r.avg_dist = sd / (double)md;
        r.n_width = mw;
        if (mw >= a.min_stitches) r.avg_width = sw / (double)mw;
        r.status = VTI_ST_OK | ovf;
        if (lane == 0) a.res[b] = r;
    }
}

}  // namespace

// 7 double, 1 unsigned, 3 short and 4 byte arrays of max_det (rounded up to 8) entries
size_t vti_k5_smem_bytes(int max_det) { return (size_t)((max_det + 7) & ~7) * (7 * 8 + 4 + 3 * 2 + 4); }

int vti_k5_prepare(int max_det) {
    int rc = vti_raise_dyn_smem((const void*)k5_measure_kernel<false>, vti_k5_smem_bytes(max_det));
    if (!rc) rc = vti_raise_dyn_smem((const void*)k5_measure_kernel<true>, vti_k5_smem_bytes(max_det));
    return rc;
}

int vti_k5_cameras(vti_handle* h, const vti_camera* cams, int n) {
    std::vector<Camera> c(n);
    for (int i = 0; i < n; ++i) c[i] = camera_of(cams[i].K, cams[i].dist, cams[i].R, cams[i].t, h->p.undistort);
    Camera* d = nullptr;
    const int rc = vti_upload(h, &d, c);
    h->d_k5_cams = d;
    return rc;
}

int vti_launch_k5(vti_handle* h, int B, vti_det* dets, const int32_t* counts, vti_frame_result* res, const int32_t* camera,
                  cudaStream_t s) {
    K5Args a;
    a.dets = dets;
    a.counts = counts;
    a.env = h->d_env;
    a.env_frame = h->d_env_frame;
    a.xmap = h->d_xmap;
    a.flags = h->d_flags;
    a.res = res;
    const vti_params& p = h->p;
    a.cam = camera_of(p.K, p.dist, p.R, p.t, p.undistort);
    a.max_det = p.max_det; a.LW = h->g.LW; a.w = p.frame_w; a.h = p.frame_h;
    a.variant = p.variant; a.min_stitches = p.min_stitches; a.max_px = p.max_px_distance; a.nb = p.neighborhood;
    a.mask_variant = p.mask_variant;
    a.cap = (p.max_det + 7) & ~7;
    a.cams = static_cast<const Camera*>(h->d_k5_cams);
    a.camera = camera;
    a.n_cameras = h->n_cameras;
    if (camera)
        k5_measure_kernel<true><<<B, K5_THREADS, vti_k5_smem_bytes(p.max_det), s>>>(a);
    else
        k5_measure_kernel<false><<<B, K5_THREADS, vti_k5_smem_bytes(p.max_det), s>>>(a);
    h->launches++;
    VTI_CUDA(cudaGetLastError());
    return VTI_OK;
}

// C-ABI glue of libvti.so: host-side planning (letterbox geometry, cv2 resize taps, undistort map, nearest-resize
// multiplicity tables), handle lifetime, stage entry points.  See include/vti.h for the contract.
//
// Planning mirrors oracle/cv_fixed.py (bit-exact vs OpenCV) and ultralytics LetterBox geometry (SURVEY.md 8a U0/U1/M2);
// tests/test_abi_cpu.py checks these host functions against the oracle without a GPU.
#include <algorithm>
#include <cfloat>
#include <climits>
#include <cmath>
#include <cstdlib>
#include <initializer_list>
#include <map>
#include <mutex>
#include <utility>

#include "vti_internal.h"

static thread_local std::string g_err;
void vti_set_error(const std::string& s) { g_err = s; }

// cudaFuncAttributeMaxDynamicSharedMemorySize belongs to the kernel FUNCTION (per device), not to a handle: a later
// handle with a smaller need must not lower it under an earlier handle that still launches with more.  Only raise.
int vti_raise_dyn_smem(const void* func, size_t bytes) {
    static std::mutex mu;
    static std::map<std::pair<int, const void*>, size_t> cur;
    int dev = 0;
    VTI_CUDA(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lock(mu);
    size_t& have = cur[std::make_pair(dev, func)];
    if (bytes > have) {
        VTI_CUDA(cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
        have = bytes;
    }
    return VTI_OK;
}

extern "C" const char* vti_last_error(void) { return g_err.c_str(); }
extern "C" int vti_abi_version(void) { return 1; }

// Python round(): half to even on a double
static inline int py_round(double x) { return (int)nearbyint(x); }

extern "C" int vti_plan_geometry(int frame_h, int frame_w, int imgsz, int stride, int max_det, int max_candidates,
                                 vti_geometry* g) {
    if (!g || frame_h <= 0 || frame_w <= 0 || imgsz <= 0 || stride <= 0 || (stride % 32) != 0) {
        vti_set_error("vti_plan_geometry: bad argument (stride must be a multiple of 32)");
        return VTI_EINVAL;
    }
    const double r = std::fmin((double)imgsz / frame_h, (double)imgsz / frame_w);
    g->new_w = py_round(frame_w * r);
    g->new_h = py_round(frame_h * r);
    double dw = (double)(((imgsz - g->new_w) % stride + stride) % stride) / 2.0;
    double dh = (double)(((imgsz - g->new_h) % stride + stride) % stride) / 2.0;
    g->top = py_round(dh - 0.1); g->bottom = py_round(dh + 0.1);
    g->left = py_round(dw - 0.1); g->right = py_round(dw + 0.1);
    g->LH = g->new_h + g->top + g->bottom;
    g->LW = g->new_w + g->left + g->right;
    if (g->LH % 32 || g->LW % 32) {
        vti_set_error("vti_plan_geometry: letterboxed size is not a multiple of 32");
        return VTI_EINVAL;
    }
    g->ph = g->LH / 4; g->pw = g->LW / 4;
    g->A = 0;
    for (int l = 0; l < 3; ++l) {
        g->lvl_h[l] = g->LH / (8 << l);
        g->lvl_w[l] = g->LW / (8 << l);
        g->A += g->lvl_h[l] * g->lvl_w[l];
    }
    g->mask_words = g->LW / 32;
    int cap = max_candidates > 0 ? max_candidates : VTI_CAND_CAP_DEFAULT;
    if (cap > g->A) cap = g->A;
    if (cap > VTI_CAND_CAP_MAX) cap = VTI_CAND_CAP_MAX;
    g->max_candidates = cap;
    g->max_det = max_det;
    return VTI_OK;
}

// cv2.resize INTER_LINEAR coefficient tables (oracle/cv_fixed.py linear_taps_x / linear_taps_y)
static void taps_core(int sn, int dn, int d, int* s_out, float* f_out) {
    const double scale = 1.0 / ((double)dn / (double)sn);
    float f = (float)((d + 0.5) * scale - 0.5);
    const int s = (int)std::floor(f);
    f -= (float)s;
    *s_out = s;
    *f_out = f;
}

extern "C" int vti_plan_resize_taps_x(int sn, int dn, int32_t* idx, int16_t* a0, int16_t* a1) {
    for (int d = 0; d < dn; ++d) {
        int s; float f;
        taps_core(sn, dn, d, &s, &f);
        if (s < 0) { s = 0; f = 0.f; }
        if (s >= sn - 1) { s = sn - 1; f = 0.f; }
        idx[d] = s;
        a0[d] = (int16_t)lrintf((1.f - f) * 2048.f);
        a1[d] = (int16_t)lrintf(f * 2048.f);
    }
    return VTI_OK;
}

extern "C" int vti_plan_resize_taps_y(int sn, int dn, int32_t* i0, int32_t* i1, int16_t* b0, int16_t* b1) {
    for (int d = 0; d < dn; ++d) {
        int s; float f;
        taps_core(sn, dn, d, &s, &f);
        i0[d] = s < 0 ? 0 : (s > sn - 1 ? sn - 1 : s);
        i1[d] = s + 1 < 0 ? 0 : (s + 1 > sn - 1 ? sn - 1 : s + 1);
        b0[d] = (int16_t)lrintf((1.f - f) * 2048.f);
        b1[d] = (int16_t)lrintf(f * 2048.f);
    }
    return VTI_OK;
}

extern "C" int vti_plan_undistort_map(const double K[9], const double dist[5], int h, int w, int32_t* ix, int32_t* iy) {
    const double fx = K[0], fy = K[4], cx = K[2], cy = K[5];
    const double k1 = dist[0], k2 = dist[1], p1 = dist[2], p2 = dist[3], k3 = dist[4];
    for (int v = 0; v < h; ++v) {
        const double y = ((double)v - cy) / fy;
        for (int u = 0; u < w; ++u) {
            const double x = ((double)u - cx) / fx;
            const double x2 = x * x, y2 = y * y;
            const double r2 = x2 + y2;
            const double _2xy = 2.0 * x * y;
            const double kr = 1.0 + ((k3 * r2 + k2) * r2 + k1) * r2;
            const double xd = x * kr + p1 * _2xy + p2 * (r2 + 2.0 * x2);
            const double yd = y * kr + p1 * (r2 + 2.0 * y2) + p2 * _2xy;
            const double mx = fx * xd + cx, my = fy * yd + cy;
            ix[(size_t)v * w + u] = (int32_t)nearbyint(mx * 32.0);
            iy[(size_t)v * w + u] = (int32_t)nearbyint(my * 32.0);
        }
    }
    return VTI_OK;
}

extern "C" int vti_plan_nearest_map(int dst_n, int src_n, int32_t* map) {
    const double ifx = 1.0 / ((double)dst_n / (double)src_n);
    for (int d = 0; d < dst_n; ++d) {
        int s = (int)std::floor(d * ifx);
        map[d] = s < src_n - 1 ? s : src_n - 1;
    }
    return VTI_OK;
}

// ---------------------------------------------------------------------------------------------------------------
static int build_axis_lut(vti_handle* h, int frame_n, int lb_n, AxisLut* lut, int32_t** d_map) {
    std::vector<int32_t> map(frame_n), cnt(lb_n, 0), sum(lb_n, 0), first(lb_n, INT_MAX), last(lb_n, -1);
    vti_plan_nearest_map(frame_n, lb_n, map.data());
    for (int d = 0; d < frame_n; ++d) {
        const int s = map[d];
        cnt[s]++;
        sum[s] += d;
        if (d < first[s]) first[s] = d;
        if (d > last[s]) last[s] = d;
    }
    std::vector<int32_t> pc(lb_n + 1, 0), ps(lb_n + 1, 0), prev_last(lb_n, -1), next_first(lb_n, INT_MAX);
    for (int i = 0; i < lb_n; ++i) {
        pc[i + 1] = pc[i] + cnt[i];
        ps[i + 1] = ps[i] + sum[i];
        prev_last[i] = std::max(i ? prev_last[i - 1] : -1, last[i]);
    }
    for (int i = lb_n - 1; i >= 0; --i) next_first[i] = std::min(i + 1 < lb_n ? next_first[i + 1] : INT_MAX, first[i]);
    int rc;
    if ((rc = vti_upload(h, &lut->cnt, cnt)) || (rc = vti_upload(h, &lut->sum, sum)) || (rc = vti_upload(h, &lut->first, first)) ||
        (rc = vti_upload(h, &lut->last, last)) || (rc = vti_upload(h, &lut->pc, pc)) || (rc = vti_upload(h, &lut->ps, ps)) ||
        (rc = vti_upload(h, &lut->prev_last, prev_last)) || (rc = vti_upload(h, &lut->next_first, next_first))) return rc;
    if (d_map) return vti_upload(h, d_map, map);
    return VTI_OK;
}

static int create_events(cudaEvent_t* ev, int n, unsigned flags) {
    for (int i = 0; i < n; ++i) VTI_CUDA(cudaEventCreateWithFlags(&ev[i], flags));
    return VTI_OK;
}

static void destroy_events(cudaEvent_t* ev, int n) {
    for (int i = 0; i < n; ++i)
        if (ev[i]) { cudaEventDestroy(ev[i]); ev[i] = nullptr; }
}

// frees the handle's allocations past the first `keep`, and the streams and events of the host-buffer path
static void release_from(vti_handle* h, size_t keep) {
    for (size_t i = keep; i < h->allocs.size(); ++i) cudaFree(h->allocs[i]);
    h->allocs.resize(keep);
    if (h->own_stream) cudaStreamDestroy(h->own_stream);
    if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
    h->own_stream = h->copy_stream = nullptr;
    destroy_events(h->chunk_ev, 4);
}

extern "C" void vti_destroy(vti_handle* h) {
    if (!h) return;
    int caller = h->device;
    cudaGetDevice(&caller);
    cudaSetDevice(h->device);
    release_from(h, 0);
    destroy_events(h->ev, 8);
    if (caller != h->device) cudaSetDevice(caller);
    delete h;
}

// vti_create_multi after the argument checks; on failure the caller destroys the partial handle
static int init_handle(vti_handle* h, const vti_params* params, int n_cameras, const vti_camera* cams) {
    VTI_CUDA(cudaGetDevice(&h->device));
    VTI_CUDA(cudaDeviceGetAttribute(&h->num_sms, cudaDevAttrMultiProcessorCount, h->device));
    h->p = *params;
    std::copy(cams[0].K, cams[0].K + 9, h->p.K);               // camera 0 is the handle's own calibration
    std::copy(cams[0].dist, cams[0].dist + 5, h->p.dist);
    std::copy(cams[0].R, cams[0].R + 9, h->p.R);
    std::copy(cams[0].t, cams[0].t + 3, h->p.t);
    h->n_cameras = n_cameras;
    const vti_params* p = &h->p;
    int rc = vti_plan_geometry(p->frame_h, p->frame_w, p->imgsz, p->stride, p->max_det, p->max_candidates, &h->g);
    if (rc) return rc;
    {
        // K4 accumulates a work unit's moments (<= 1024 letterbox pixels, each standing for up to my x mx frame pixels
        // at coordinates < max(h, w)) in 32 bits before its 64-bit atomics
        const unsigned long long my = (p->frame_h + h->g.LH - 1) / h->g.LH + 1, mx = (p->frame_w + h->g.LW - 1) / h->g.LW + 1;
        if (1024ull * my * mx * (unsigned long long)std::max(p->frame_h, p->frame_w) >= (1ull << 31)) {
            vti_set_error("vti_create: frame too large for the imgsz (mask moments would overflow a work unit's 32-bit sums)");
            return VTI_EINVAL;
        }
    }
    const vti_geometry& g = h->g;
    const int fh = p->frame_h, fw = p->frame_w;
    if (p->variant == 0 && p->roi_enabled) {                // measurement.py:220-238
        const int x_min = std::clamp(p->roi_x_min, 0, fw - 1), x_max = std::clamp(p->roi_x_max, 0, fw - 1);
        const int y_min = std::clamp(p->roi_y_min, 0, fh - 1), y_max = std::clamp(p->roi_y_max, 0, fh - 1);
        if (x_min < x_max && y_min < y_max) h->roi = VtiRoi{1, x_min, y_min, x_max, y_max};
    }

    // ---- K1 tables
    std::vector<int32_t> xi(g.new_w), yi(2 * (size_t)g.new_h);
    std::vector<int16_t> xa(2 * (size_t)g.new_w), yb(2 * (size_t)g.new_h);
    if (fw == 2 * g.new_w && fh == 2 * g.new_h) {
        h->resize_mode = 2;                                  // OpenCV's silent INTER_AREA switch
        for (int d = 0; d < g.new_w; ++d) { xi[d] = 2 * d; xa[2 * d] = 1; xa[2 * d + 1] = 1; }
        for (int d = 0; d < g.new_h; ++d) { yi[2 * d] = 2 * d; yi[2 * d + 1] = 2 * d + 1; yb[2 * d] = 1; yb[2 * d + 1] = 1; }
    } else {
        h->resize_mode = 1;
        std::vector<int32_t> i0(g.new_h), i1(g.new_h);
        std::vector<int16_t> a0(g.new_w), a1(g.new_w), b0(g.new_h), b1(g.new_h);
        if (fw == g.new_w && fh == g.new_h) {                // LetterBox skips cv2.resize: identity taps
            for (int d = 0; d < g.new_w; ++d) { xi[d] = d; a0[d] = 2048; a1[d] = 0; }
            for (int d = 0; d < g.new_h; ++d) { i0[d] = d; i1[d] = d; b0[d] = 2048; b1[d] = 0; }
        } else {
            vti_plan_resize_taps_x(fw, g.new_w, xi.data(), a0.data(), a1.data());
            vti_plan_resize_taps_y(fh, g.new_h, i0.data(), i1.data(), b0.data(), b1.data());
        }
        for (int d = 0; d < g.new_w; ++d) { xa[2 * d] = a0[d]; xa[2 * d + 1] = a1[d]; }
        for (int d = 0; d < g.new_h; ++d) { yi[2 * d] = i0[d]; yi[2 * d + 1] = i1[d]; yb[2 * d] = b0[d]; yb[2 * d + 1] = b1[d]; }
    }
    if ((rc = vti_upload(h, &h->d_tap_x_idx, xi)) || (rc = vti_upload(h, &h->d_tap_x_a, xa)) ||
        (rc = vti_upload(h, &h->d_tap_y_i, yi)) || (rc = vti_upload(h, &h->d_tap_y_b, yb))) return rc;
    {
        // every camera's cv2.undistort source map, [camera][fh * fw] (1/32 px), and its packed displacements
        std::vector<int32_t> ix, iy, packed;
        if (p->undistort) {
            const size_t npx = (size_t)fh * fw;
            ix.resize(n_cameras * npx); iy.resize(n_cameras * npx); packed.resize(n_cameras * npx);
            for (int c = 0; c < n_cameras; ++c) {
                int32_t* cx = ix.data() + c * npx;
                int32_t* cy = iy.data() + c * npx;
                vti_plan_undistort_map(cams[c].K, cams[c].dist, fh, fw, cx, cy);
                for (int v = 0; v < fh; ++v)
                    for (int u = 0; u < fw; ++u) {
                        const size_t i = (size_t)v * fw + u;
                        const int dx = cx[i] - 32 * u, dy = cy[i] - 32 * v;
                        if (dx < -32768 || dx > 32767 || dy < -32768 || dy > 32767) {
                            vti_set_error(n_cameras == 1 ? std::string("vti_create: lens displacement exceeds +-1024 px, unsupported")
                                                         : "vti_create_multi: lens displacement of camera " + std::to_string(c) +
                                                               " exceeds +-1024 px, unsupported");
                            return VTI_EINVAL;
                        }
                        packed[c * npx + i] = (int32_t)(((uint32_t)(uint16_t)(int16_t)dy << 16) | (uint32_t)(uint16_t)(int16_t)dx);
                    }
            }
        }
        if ((rc = vti_k1_plan(h, xi, yi, xa, yb, p->undistort ? &ix : nullptr, p->undistort ? &iy : nullptr,
                              p->undistort ? &packed : nullptr)))
            return rc;
    }
    if ((rc = vti_k5_cameras(h, cams, n_cameras))) return rc;
    // ---- measurement tables
    if ((rc = build_axis_lut(h, fh, g.LH, &h->lutY, nullptr)) || (rc = build_axis_lut(h, fw, g.LW, &h->lutX, &h->d_xmap)))
        return rc;
    // ---- post scratch
    const size_t B = p->max_batch;
    auto alloc = [&](auto** ptr, size_t bytes) { if (!rc) rc = vti_alloc(h, ptr, bytes); };
    alloc(&h->d_cand_count, sizeof(int32_t) * (B + 1));
    alloc(&h->d_cand_key, sizeof(unsigned long long) * B * vti_k3_cap_pad(g.max_candidates));
    alloc(&h->d_cand_box, sizeof(float4) * B * g.A);
    alloc(&h->d_det_coef, sizeof(float) * B * p->max_det * VTI_NM);
    alloc(&h->d_env, sizeof(int32_t) * B * g.LW);
    alloc(&h->d_env_frame, sizeof(int32_t) * B * fw);
    alloc(&h->d_flags, sizeof(int32_t) * B);
    for (int l = 0; l < 3; ++l) h->head_floats[l] = (size_t)(64 + p->nc) * g.lvl_h[l] * g.lvl_w[l];
    h->head_floats[3] = (size_t)VTI_NM * g.A;
    h->head_floats[4] = (size_t)VTI_NM * g.ph * g.pw;
    h->units_per_det = ((g.ph + 1 + VTI_K4_UR - 1) / VTI_K4_UR) * ((g.pw + 1 + VTI_K4_UC - 1) / VTI_K4_UC);
    alloc(&h->d_units, sizeof(uint4) * B * p->max_det * h->units_per_det);
    alloc(&h->d_proto_bbox, sizeof(int4) * B);
    if (rc) return rc;
    if ((rc = vti_k3_prepare(g.max_candidates)) || (rc = vti_k5_prepare(p->max_det))) return rc;
    return VTI_OK;
}

// the checks of vti_params that need no device
static int check_params(const vti_params* p) {
    if (p->struct_size != (int32_t)sizeof(vti_params)) {
        vti_set_error("vti_create: vti_params.struct_size mismatch (ABI)");
        return VTI_EINVAL;
    }
    // nc: K2 packs the class into the top byte of a candidate key; max_batch: K3 packs the frame index into 15 bits
    if (p->nc < 1 || p->nc > 255 || p->max_det < 1 || p->max_det > 1024 || p->max_batch < 1 || p->max_batch > 32767 ||
        p->neighborhood < 0 || p->neighborhood > 7 || (p->variant != 0 && p->variant != 1) ||
        (p->mask_variant != 0 && p->mask_variant != 1)) {
        vti_set_error("vti_create: parameter out of range (nc 1..255, max_det 1..1024, max_batch 1..32767, "
                      "neighborhood 0..7, variant 0/1, mask_variant 0/1)");
        return VTI_EINVAL;
    }
    return VTI_OK;
}

// after the argument checks of both create calls
static int create_checked(const vti_params* p, int n_cameras, const vti_camera* cams, vti_handle** out) {
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        vti_set_error("vti_create: no CUDA device -- this library has no CPU fallback");
        return VTI_ENODEV;
    }
    vti_handle* h = new vti_handle();
    const int rc = init_handle(h, p, n_cameras, cams);
    if (rc) { vti_destroy(h); return rc; }
    *out = h;
    return VTI_OK;
}

extern "C" int vti_create(const vti_params* p, vti_handle** out) {
    if (!p || !out) { vti_set_error("vti_create: null argument"); return VTI_EINVAL; }
    *out = nullptr;
    int rc = check_params(p);
    if (rc) return rc;
    vti_camera cam{};                                          // the one camera: p's own calibration
    cam.struct_size = (int32_t)sizeof(vti_camera);
    std::copy(p->K, p->K + 9, cam.K);
    std::copy(p->dist, p->dist + 5, cam.dist);
    std::copy(p->R, p->R + 9, cam.R);
    std::copy(p->t, p->t + 3, cam.t);
    return create_checked(p, 1, &cam, out);
}

extern "C" int vti_create_multi(const vti_params* p, int n_cameras, const vti_camera* cameras, vti_handle** out) {
    if (!p || !cameras || !out) { vti_set_error("vti_create_multi: null argument"); return VTI_EINVAL; }
    *out = nullptr;
    int rc = check_params(p);
    if (rc) return rc;
    if (n_cameras < 1 || n_cameras > VTI_MAX_CAMERAS) {
        vti_set_error("vti_create_multi: n_cameras must be 1.." + std::to_string(VTI_MAX_CAMERAS));
        return VTI_EINVAL;
    }
    for (int c = 0; c < n_cameras; ++c)
        if (cameras[c].struct_size != (int32_t)sizeof(vti_camera)) {
            vti_set_error("vti_create_multi: cameras[" + std::to_string(c) + "].struct_size mismatch (ABI)");
            return VTI_EINVAL;
        }
    return create_checked(p, n_cameras, cameras, out);
}

extern "C" int vti_camera_count(const vti_handle* h) { return h ? h->n_cameras : VTI_EINVAL; }

extern "C" int vti_get_geometry(const vti_handle* h, vti_geometry* out) {
    if (!h || !out) return VTI_EINVAL;
    *out = h->g;
    return VTI_OK;
}

extern "C" int64_t vti_launch_count(const vti_handle* h) { return h ? h->launches : 0; }

static inline void mark(vti_handle* h, int i, cudaStream_t s) {
    if (!h->profiling) return;
    if (cudaEventRecord(h->ev[i], s) == cudaSuccess) h->ev_set[i] = true;
}

extern "C" int vti_set_profiling(vti_handle* h, int on) {
    if (!h) return VTI_EINVAL;
    if (on && !h->ev[0]) {
        const int rc = create_events(h->ev, 8, cudaEventDefault);
        if (rc) { destroy_events(h->ev, 8); return rc; }      // all or none: a retry starts clean
    }
    h->profiling = on ? 1 : 0;
    for (int i = 0; i < 8; ++i) h->ev_set[i] = false;
    return VTI_OK;
}

extern "C" int vti_get_stage_ms(vti_handle* h, float ms[5]) {
    if (!h || !ms) return VTI_EINVAL;
    const int a[5] = {0, 2, 3, 4, 6}, b[5] = {1, 3, 4, 5, 7};
    for (int k = 0; k < 5; ++k) {
        ms[k] = -1.0f;
        if (h->ev[0] && h->ev_set[a[k]] && h->ev_set[b[k]]) {
            VTI_CUDA(cudaEventSynchronize(h->ev[b[k]]));
            VTI_CUDA(cudaEventElapsedTime(&ms[k], h->ev[a[k]], h->ev[b[k]]));
        }
    }
    return VTI_OK;
}

static int check_batch(const vti_handle* h, int B) {
    if (!h || B < 1 || B > h->p.max_batch) {
        vti_set_error("batch size out of range for this handle (max_batch)");
        return VTI_EINVAL;
    }
    return VTI_OK;
}

struct Aligned { const char* name; const void* ptr; unsigned bytes; };

// VTI_EINVAL naming the first buffer not aligned to the width its kernels read it with (null passes)
static int check_aligned(const char* fn, std::initializer_list<Aligned> bufs) {
    for (const Aligned& b : bufs)
        if (reinterpret_cast<uintptr_t>(b.ptr) % b.bytes) {
            vti_set_error(std::string(fn) + ": " + b.name + " must be " + std::to_string(b.bytes) + "-byte aligned");
            return VTI_EINVAL;
        }
    return VTI_OK;
}

extern "C" int vti_preprocess_multi(vti_handle* h, const uint8_t* frames, const int32_t* camera, int B, float* net_in,
                                    void* stream) {
    int rc = check_batch(h, B);
    if (rc) return rc;
    if (!frames || !net_in) { vti_set_error("vti_preprocess: null buffer"); return VTI_EINVAL; }
    if ((rc = check_aligned("vti_preprocess_multi", {{"camera", camera, 4}}))) return rc;
    mark(h, 0, (cudaStream_t)stream);
    rc = vti_launch_k1(h, frames, B, net_in, camera, (cudaStream_t)stream);
    mark(h, 1, (cudaStream_t)stream);
    return rc;
}

extern "C" int vti_preprocess(vti_handle* h, const uint8_t* frames, int B, float* net_in, void* stream) {
    return vti_preprocess_multi(h, frames, nullptr, B, net_in, stream);
}

// K2 -> K3 -> K4 [-> K5], the one post chain of vti_postprocess (so of vti_post_measure) and of every chunk of
// vti_process_host.  head: p3, p4, p5, coef, proto.  fetch_into: the prototypes are device-mapped host memory, fetched
// after K3 (which sizes the rectangle K4 reads) into fetch_into.  results: K5 too, with the frames' camera ids (device,
// or null).  timed: record the stage events.
static int post_chain(vti_handle* h, const float* const head[5], float* fetch_into, int B, vti_det* dets, int32_t* counts,
                      uint32_t* masks, vti_frame_result* results, const int32_t* camera, bool timed, cudaStream_t s) {
    auto stage = [&](int i) { if (timed) mark(h, i, s); };
    // K3 and K4 evaluate the masks of every kept detection, not only of the routed stitch / fabric ones, when masks are
    // exported and for mask variant B: it removes every detection whose mask is empty (newer Ultralytics,
    // construct_result), routed or not.
    const int all_dets = masks != nullptr || h->p.mask_variant == 1;
    int rc;
    stage(2);
    if ((rc = vti_launch_k2(h, head[0], head[1], head[2], B, s))) return rc;
    stage(3);
    if ((rc = vti_launch_k3(h, head[3], B, dets, counts, all_dets, s))) return rc;
    stage(4);
    if (fetch_into && (rc = vti_launch_fetch_proto(h, head[4], fetch_into, B, s))) return rc;
    if ((rc = vti_launch_k4(h, fetch_into ? fetch_into : head[4], B, dets, counts, masks, s))) return rc;
    stage(5);
    return results ? vti_launch_k5(h, B, dets, counts, results, camera, s) : VTI_OK;
}

extern "C" int vti_postprocess(vti_handle* h, const float* p3, const float* p4, const float* p5, const float* coef,
                               const float* proto, int B, vti_det* dets, int32_t* counts, uint32_t* masks,
                               void* stream) {
    int rc = check_batch(h, B);
    if (rc) return rc;
    if (!p3 || !p4 || !p5 || !coef || !proto || !dets || !counts) { vti_set_error("vti_postprocess: null buffer"); return VTI_EINVAL; }
    if ((rc = check_aligned("vti_postprocess", {{"dets", dets, 8}, {"counts", counts, 4}, {"p3", p3, 4}, {"p4", p4, 4}, {"p5", p5, 4},
                                                {"coef", coef, 4}, {"proto", proto, 4}, {"masks", masks, 16}}))) return rc;
    const float* head[5] = {p3, p4, p5, coef, proto};
    return post_chain(h, head, nullptr, B, dets, counts, masks, nullptr, nullptr, true, (cudaStream_t)stream);
}

extern "C" int vti_measure_multi(vti_handle* h, int B, const int32_t* camera, vti_det* dets, const int32_t* counts,
                                 vti_frame_result* results, void* stream) {
    int rc = check_batch(h, B);
    if (rc) return rc;
    if (!dets || !counts || !results) { vti_set_error("vti_measure: null buffer"); return VTI_EINVAL; }
    if ((rc = check_aligned("vti_measure", {{"dets", dets, 8}, {"results", results, 8}, {"counts", counts, 4},
                                            {"camera", camera, 4}}))) return rc;
    mark(h, 6, (cudaStream_t)stream);
    rc = vti_launch_k5(h, B, dets, counts, results, camera, (cudaStream_t)stream);
    mark(h, 7, (cudaStream_t)stream);
    return rc;
}

extern "C" int vti_measure(vti_handle* h, int B, vti_det* dets, const int32_t* counts, vti_frame_result* results,
                           void* stream) {
    return vti_measure_multi(h, B, nullptr, dets, counts, results, stream);
}

extern "C" int vti_post_measure_multi(vti_handle* h, const float* p3, const float* p4, const float* p5, const float* coef,
                                      const float* proto, int B, const int32_t* camera, vti_det* dets, int32_t* counts,
                                      uint32_t* masks, vti_frame_result* results, void* stream) {
    int rc = vti_postprocess(h, p3, p4, p5, coef, proto, B, dets, counts, masks, stream);
    if (rc) return rc;
    return vti_measure_multi(h, B, camera, dets, counts, results, stream);
}

extern "C" int vti_post_measure(vti_handle* h, const float* p3, const float* p4, const float* p5, const float* coef,
                                const float* proto, int B, vti_det* dets, int32_t* counts, uint32_t* masks,
                                vti_frame_result* results, void* stream) {
    return vti_post_measure_multi(h, p3, p4, p5, coef, proto, B, nullptr, dets, counts, masks, results, stream);
}

// The host-buffer path's streams, events and buffers, made by its first call
static int create_staging(vti_handle* h) {
    const size_t B = h->p.max_batch;
    VTI_CUDA(cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking));
    VTI_CUDA(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
    int rc = create_events(h->chunk_ev, 4, cudaEventDisableTiming);
    auto alloc = [&](auto** ptr, size_t bytes) { if (!rc) rc = vti_alloc(h, ptr, bytes); };
    alloc(&h->d_frames, B * h->p.frame_h * h->p.frame_w * 3);
    alloc(&h->d_net_in, sizeof(float) * B * 3 * h->g.LH * h->g.LW);
    for (int t = 0; t < 5; ++t) alloc(&h->d_head[t], sizeof(float) * B * h->head_floats[t]);
    alloc(&h->d_dets, sizeof(vti_det) * B * h->p.max_det);
    alloc(&h->d_counts, sizeof(int32_t) * B);
    alloc(&h->d_results, sizeof(vti_frame_result) * B);
    alloc(&h->d_camera, sizeof(int32_t) * B);
    if (!rc) h->staged_batch = B;
    return rc;
}

extern "C" int vti_ingest_yuyv(vti_handle* h, const uint8_t* yuyv, int B, uint8_t* frames, void* stream) {
    int rc = check_batch(h, B);
    if (rc) return rc;
    if (!yuyv || !frames) { vti_set_error("vti_ingest_yuyv: null buffer"); return VTI_EINVAL; }
    if (h->p.frame_w & 1) { vti_set_error("vti_ingest_yuyv: packed 4:2:2 needs an even frame width"); return VTI_EINVAL; }
    if ((rc = check_aligned("vti_ingest_yuyv", {{"the YUYV buffer", yuyv, 4}}))) return rc;
    return vti_launch_k0_yuyv(h, yuyv, B, frames, (cudaStream_t)stream);
}

// The device alias of a pinned, device-mapped host buffer, or null: pageable memory, or VTI_NO_ZERO_COPY set (read on
// every call, so that one handle can time both paths).
static const float* mapped_alias(const float* host) {
    cudaPointerAttributes at;
    if (getenv("VTI_NO_ZERO_COPY")) return nullptr;
    if (cudaPointerGetAttributes(&at, host) != cudaSuccess) { cudaGetLastError(); return nullptr; }   // old drivers: pageable
    return at.type == cudaMemoryTypeHost ? static_cast<const float*>(at.devicePointer) : nullptr;
}

// fmt 0: BGR frames (3 bytes per pixel); 1: camera-native YUYV (2 bytes per pixel, converted by K0 on the device).
// camera: HOST camera ids, or null (camera 0 throughout)
static int process_host_impl(vti_handle* h, const uint8_t* frames, int fmt, const float* p3, const float* p4, const float* p5,
                             const float* coef, const float* proto, int B, const int32_t* camera, float* net_in,
                             vti_det* dets, int32_t* counts, vti_frame_result* results) {
    int rc = check_batch(h, B);
    if (rc) return rc;
    if (!frames || !p3 || !p4 || !p5 || !coef || !proto || !dets || !counts || !results) {
        vti_set_error("vti_process_host: null buffer");
        return VTI_EINVAL;
    }
    for (int b = 0; camera && b < B; ++b)
        if (camera[b] < 0 || camera[b] >= h->n_cameras) {
            vti_set_error("vti_process_host_multi: camera id " + std::to_string(camera[b]) + " of frame " + std::to_string(b) +
                          " is outside [0, " + std::to_string(h->n_cameras) + ")");
            return VTI_EINVAL;
        }
    if (fmt == 1 && (h->p.frame_w & 1)) { vti_set_error("vti_process_host_yuyv: packed 4:2:2 needs an even frame width"); return VTI_EINVAL; }
    const size_t keep = h->allocs.size();                  // all or nothing: a call after a failure starts clean
    if (!h->staged_batch && (rc = create_staging(h))) { release_from(h, keep); return rc; }
    if (fmt == 1 && !h->d_yuyv && (rc = vti_alloc(h, &h->d_yuyv, (size_t)h->p.max_batch * h->p.frame_h * h->p.frame_w * 2)))
        return rc;
    cudaStream_t s = h->own_stream, cs = h->copy_stream;
    // The batch goes through in up to 4 chunks: chunk i+1's host->device copies (copy stream) run under chunk i's
    // kernels and device->host record copies (compute stream), so the call costs the PCIe time of its inputs plus
    // one chunk of compute.
    const int nchunk = B < 4 ? 1 : 4;
    const size_t fsz = (size_t)h->p.frame_h * h->p.frame_w * 3, nsz = (size_t)3 * h->g.LH * h->g.LW;
    const size_t ysz = (size_t)h->p.frame_h * h->p.frame_w * 2;
    const size_t* hsz = h->head_floats;
    // Head tensors that sit in PINNED (device-mapped) host memory are not copied: K2 reads only the class planes and the
    // 64 box logits of each candidate, K3 only the coefficient rows of the kept detections -- a few hundred KB of the
    // 4.2 MB per frame -- so those kernels read them in place over PCIe (zero copy) and the DMA engine moves only the
    // frames and the prototypes.  Pinned prototypes are not DMA-copied either: the post chain fetches, per frame, only
    // the union rectangle of the crop windows (all that K4 ever touches).  Pageable buffers are copied whole.
    const float* host[5] = {p3, p4, p5, coef, proto};
    const float* mapped[5];
    for (int t = 0; t < 5; ++t) mapped[t] = mapped_alias(host[t]);
    for (int c = 0; c < nchunk; ++c) {
        const int b0 = (int)((long long)B * c / nchunk), b1 = (int)((long long)B * (c + 1) / nchunk), nb = b1 - b0;
        if (nb <= 0) continue;
        if (fmt == 1) VTI_CUDA(cudaMemcpyAsync(h->d_yuyv + b0 * ysz, frames + b0 * ysz, nb * ysz, cudaMemcpyHostToDevice, cs));
        else VTI_CUDA(cudaMemcpyAsync(h->d_frames + b0 * fsz, frames + b0 * fsz, nb * fsz, cudaMemcpyHostToDevice, cs));
        const int32_t* cam = camera ? h->d_camera + b0 : nullptr;
        if (camera) VTI_CUDA(cudaMemcpyAsync(h->d_camera + b0, camera + b0, sizeof(int32_t) * nb, cudaMemcpyHostToDevice, cs));
        const float* head[5];
        for (int t = 0; t < 5; ++t) {
            head[t] = (mapped[t] ? mapped[t] : h->d_head[t]) + b0 * hsz[t];
            if (!mapped[t])
                VTI_CUDA(cudaMemcpyAsync(h->d_head[t] + b0 * hsz[t], host[t] + b0 * hsz[t], sizeof(float) * nb * hsz[t],
                                         cudaMemcpyHostToDevice, cs));
        }
        VTI_CUDA(cudaEventRecord(h->chunk_ev[c], cs));
        VTI_CUDA(cudaStreamWaitEvent(s, h->chunk_ev[c], 0));
        vti_det* cd = h->d_dets + (size_t)b0 * h->p.max_det;
        if (fmt == 1 && (rc = vti_launch_k0_yuyv(h, h->d_yuyv + b0 * ysz, nb, h->d_frames + b0 * fsz, s))) return rc;
        if ((rc = vti_launch_k1(h, h->d_frames + b0 * fsz, nb, h->d_net_in + b0 * nsz, cam, s))) return rc;
        if ((rc = post_chain(h, head, mapped[4] ? h->d_head[4] + b0 * hsz[4] : nullptr, nb, cd, h->d_counts + b0, nullptr,
                             h->d_results + b0, cam, false, s)))
            return rc;
        if (net_in)
            VTI_CUDA(cudaMemcpyAsync(net_in + b0 * nsz, h->d_net_in + b0 * nsz, sizeof(float) * nb * nsz, cudaMemcpyDeviceToHost, s));
        VTI_CUDA(cudaMemcpyAsync(dets + (size_t)b0 * h->p.max_det, cd, sizeof(vti_det) * nb * h->p.max_det, cudaMemcpyDeviceToHost, s));
        VTI_CUDA(cudaMemcpyAsync(counts + b0, h->d_counts + b0, sizeof(int32_t) * nb, cudaMemcpyDeviceToHost, s));
        VTI_CUDA(cudaMemcpyAsync(results + b0, h->d_results + b0, sizeof(vti_frame_result) * nb, cudaMemcpyDeviceToHost, s));
    }
    VTI_CUDA(cudaStreamSynchronize(s));
    return VTI_OK;
}

extern "C" int vti_process_host(vti_handle* h, const uint8_t* frames, const float* p3, const float* p4, const float* p5,
                                const float* coef, const float* proto, int B, float* net_in, vti_det* dets,
                                int32_t* counts, vti_frame_result* results) {
    return process_host_impl(h, frames, 0, p3, p4, p5, coef, proto, B, nullptr, net_in, dets, counts, results);
}

extern "C" int vti_process_host_multi(vti_handle* h, const uint8_t* frames, const float* p3, const float* p4, const float* p5,
                                      const float* coef, const float* proto, int B, const int32_t* camera, float* net_in,
                                      vti_det* dets, int32_t* counts, vti_frame_result* results) {
    return process_host_impl(h, frames, 0, p3, p4, p5, coef, proto, B, camera, net_in, dets, counts, results);
}

extern "C" int vti_process_host_yuyv(vti_handle* h, const uint8_t* yuyv, const float* p3, const float* p4, const float* p5,
                                     const float* coef, const float* proto, int B, float* net_in, vti_det* dets,
                                     int32_t* counts, vti_frame_result* results) {
    return process_host_impl(h, yuyv, 1, p3, p4, p5, coef, proto, B, nullptr, net_in, dets, counts, results);
}

extern "C" int vti_process_host_yuyv_multi(vti_handle* h, const uint8_t* yuyv, const float* p3, const float* p4,
                                           const float* p5, const float* coef, const float* proto, int B,
                                           const int32_t* camera, float* net_in, vti_det* dets, int32_t* counts,
                                           vti_frame_result* results) {
    return process_host_impl(h, yuyv, 1, p3, p4, p5, coef, proto, B, camera, net_in, dets, counts, results);
}

// Internal declarations shared by the kernels and the C-ABI glue of libvti.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "../../include/vti.h"

static_assert(sizeof(vti_det) == 160, "vti_det must stay 160 bytes");
static_assert(sizeof(vti_params) == 320, "vti_params must stay 320 bytes (struct_size of existing callers)");
static_assert(sizeof(vti_camera) == 216, "vti_camera is 216 bytes");

#define VTI_CAND_CAP_MAX 32768      /* hard ceiling of the per-frame candidate list */
#define VTI_CAND_CAP_DEFAULT 30000  /* Ultralytics' max_nms: with A <= 30000 anchors the list can never overflow */
#define VTI_K1_TX 128        // K1 output tile
#define VTI_K1_TY 16
#define VTI_K4_UR 4          // K4 work unit: interpolation cells per unit, rows x cols
#define VTI_K4_UC 16

// Per-axis letterbox-pixel -> frame-pixel multiplicity tables of cv2.resize(INTER_NEAREST) (measurement.py:78-79).
// A letterbox row Y is hit by cnt[Y] frame rows whose indices sum to sum[Y]; first/last are the extreme frame rows.
struct AxisLut {
    int32_t* cnt;
    int32_t* sum;
    int32_t* first;   // INT_MAX when cnt == 0
    int32_t* last;    // -1 when cnt == 0
    int32_t* pc;      // [n+1] prefix sums of cnt
    int32_t* ps;      // [n+1] prefix sums of sum
    int32_t* prev_last;   // max last[] over entries <= i (-1 if none)
    int32_t* next_first;  // min first[] over entries >= i (INT_MAX if none)
};

// The ROI rectangle of measurement.py:220-238 clamped to the frame; active only for variant 0 with a non-empty clamp.
struct VtiRoi { int active, x1, y1, x2, y2; };

// Value-initialised (`new vti_handle()`): every pointer and count starts at zero.
struct vti_handle {
    vti_params p;
    vti_geometry g;
    int device;
    int num_sms;
    int64_t launches;
    VtiRoi roi;
    int n_cameras;                                 // calibrations of the handle (camera 0 is also in p)
    std::vector<void*> allocs;                     // every device allocation of the handle (vti_alloc)

    // ---- K1 tables (device)
    int32_t* d_tap_x_idx;  int16_t* d_tap_x_a;    // [new_w], [new_w*2]
    int32_t* d_tap_y_i;    int16_t* d_tap_y_b;    // [new_h*2], [new_h*2]
    int32_t* d_und_lut;                            // [camera][frame_h*frame_w] packed (dy16<<16 | dx16), generic remap only
    int resize_mode;                               // 1 bilinear (incl. identity taps), 2 exact-2x area
    int k1_mode, k1_pitch_u, k1_rows_u;            // staging mode + shared footprint buffer shape (k1 plan)
    size_t k1_smem;
    int k1_und_words, k1_lut_stride;               // fast path: footprint buffer words, table entries per tile
    int k1_raw_pitch;                              // fast remap path: words per row of the staged raw box
    int4* d_k1_tiles;                              // [camera] per-tile headers (fast path) / raw bounding boxes (MODE_RAW)
    unsigned* d_k1_lut;                            // [camera] per-tile pre-resolved remap entries (fast path, undistort)
    // ---- measurement tables (device)
    AxisLut lutY, lutX;                            // [LH], [LW]
    int32_t* d_xmap;                               // [frame_w] frame col -> letterbox col
    // ---- post scratch (device), sized for max_batch
    int32_t* d_cand_count;                         // [max_batch + 1]; the last entry counts K4 work units
    unsigned long long* d_cand_key;                // [B][cap]
    float4* d_cand_box;                            // [B][A]   xyxy by anchor
    float* d_det_coef;                             // [B][max_det][32]
    int32_t* d_env;                                // [B][LW]  envelope in frame rows at letterbox columns
    int32_t* d_env_frame;                          // [B][frame_w]
    int32_t* d_flags;                              // [B] overflow etc.
    uint4* d_units;                                // K4 work units: (frame | fabric << 15 | det << 16, block row | block col << 16,
                                                   //                 cx_lo | cy_lo << 16, cx_hi | cy_hi << 16)
    int units_per_det;                             // capacity per detection slot
    int4* d_proto_bbox;                            // [B] union of the crop windows of a frame (prototype pixels K4 reads)
    void* d_k5_cams;                               // [n_cameras] K5's per-camera projection constants
    // ---- host-buffer path
    cudaStream_t own_stream, copy_stream;
    cudaEvent_t chunk_ev[4];
    uint8_t* d_yuyv;                               // camera-native staging (vti_process_host_yuyv), allocated on first use
    uint8_t* d_frames; float* d_net_in; float* d_head[5];     // head: p3, p4, p5, coef, proto
    size_t head_floats[5];                         // floats per frame of each head tensor
    vti_det* d_dets; int32_t* d_counts; vti_frame_result* d_results;
    int32_t* d_camera;                             // [max_batch] the camera ids of vti_process_host[_yuyv]_multi
    size_t staged_batch;
    // ---- optional per-kernel event timing
    int profiling;
    cudaEvent_t ev[8];       // K1: 0,1   K2: 2,3   K3: 3,4   K4: 4,5   K5: 6,7
    bool ev_set[8];
};

void vti_set_error(const std::string& s);
#define VTI_CUDA(expr)                                                                             \
    do {                                                                                           \
        cudaError_t _e = (expr);                                                                   \
        if (_e != cudaSuccess) {                                                                   \
            vti_set_error(std::string(#expr) + ": " + cudaGetErrorString(_e));                     \
            return VTI_ECUDA;                                                                      \
        }                                                                                          \
    } while (0)

// Every device allocation of a handle goes through here: the handle records it, and vti_destroy frees the record.
template <typename T>
int vti_alloc(vti_handle* h, T** dptr, size_t bytes) {
    void* p = nullptr;
    if (const cudaError_t e = cudaMalloc(&p, bytes)) {
        cudaGetLastError();                        // not sticky: clear it, or the next launch check would report it
        vti_set_error(std::string("cudaMalloc: ") + cudaGetErrorString(e));
        return VTI_ENOMEM;
    }
    h->allocs.push_back(p);
    *dptr = static_cast<T*>(p);
    return VTI_OK;
}
template <typename T>
int vti_upload(vti_handle* h, T** dptr, const std::vector<T>& v) {
    if (const int rc = vti_alloc(h, dptr, sizeof(T) * (v.empty() ? 1 : v.size()))) return rc;
    if (!v.empty()) VTI_CUDA(cudaMemcpy(*dptr, v.data(), sizeof(T) * v.size(), cudaMemcpyHostToDevice));
    return VTI_OK;
}

// raises (never lowers) a kernel function's dynamic shared-memory limit on the current device
int vti_raise_dyn_smem(const void* func, size_t bytes);
// create-time preparation of the post kernels (dynamic shared-memory limits) and K3's padded candidate list length
int vti_k3_prepare(int cap);
int vti_k3_cap_pad(int cap);
int vti_k5_prepare(int max_det);
// uploads K5's projection constants of every camera of the handle (h->d_k5_cams)
int vti_k5_cameras(vti_handle* h, const vti_camera* cams, int n);
// K1 plan.  With undistort on, und_ix / und_iy hold the cv2.undistort source maps of every camera ([camera][h*w], 1/32
// px) and und_packed their packed displacements ([camera][h*w], uploaded only if the generic kernel runs).
int vti_k1_plan(vti_handle* h, const std::vector<int32_t>& xi, const std::vector<int32_t>& yi,
                const std::vector<int16_t>& xa, const std::vector<int16_t>& yb,
                const std::vector<int32_t>* und_ix, const std::vector<int32_t>* und_iy,
                const std::vector<int32_t>* und_packed);
// kernel launchers (each returns VTI_OK / VTI_ECUDA).  camera: device ids per frame, or null (camera 0 throughout)
int vti_launch_k0_yuyv(vti_handle* h, const uint8_t* yuyv, int B, uint8_t* frames, cudaStream_t s);
int vti_launch_k1(vti_handle* h, const uint8_t* frames, int B, float* net_in, const int32_t* camera, cudaStream_t s);
int vti_launch_k2(vti_handle* h, const float* p3, const float* p4, const float* p5, int B, cudaStream_t s);
int vti_launch_k3(vti_handle* h, const float* coef, int B, vti_det* dets, int32_t* counts, int all_dets, cudaStream_t s);
int vti_launch_k4(vti_handle* h, const float* proto, int B, vti_det* dets, const int32_t* counts, uint32_t* masks,
                  cudaStream_t s);
int vti_launch_k5(vti_handle* h, int B, vti_det* dets, const int32_t* counts, vti_frame_result* res, const int32_t* camera,
                  cudaStream_t s);
// copies, per frame, the prototype rectangle K4 will read (all 32 channels) from device-mapped host memory
int vti_launch_fetch_proto(vti_handle* h, const float* host_proto_mapped, float* dev_proto, int B, cudaStream_t s);

#ifdef __CUDACC__
// Where a detection's mask can be non-zero.  crop_mask keeps prototype pixel (Y, X) iff X >= x1/4 && X < x2/4 &&
// Y >= y1/4 && Y < y2/4 (float compares on integer grid coordinates); the bilinear upsample spreads a kept pixel over
// the interpolation cells around it.  Cell (R, C) = the 4x4 output pixels between prototype rows R-1, R and columns
// C-1, C (rows 4R-2 .. 4R+1): the non-zero cells of a detection are R in [cy_lo, cy_hi+1], C in [cx_lo, cx_hi+1].
struct VtiWindow {
    int cx_lo, cx_hi, cy_lo, cy_hi;   // cropped prototype window (inclusive)
    bool empty;
};
__device__ __forceinline__ VtiWindow vti_det_window(const float* box, int ph, int pw) {
    const float dx1 = box[0] * 0.25f, dy1 = box[1] * 0.25f, dx2 = box[2] * 0.25f, dy2 = box[3] * 0.25f;
    VtiWindow w;
    w.cx_lo = max((int)ceilf(dx1), 0);
    w.cy_lo = max((int)ceilf(dy1), 0);
    w.cx_hi = min((int)ceilf(dx2) - 1, pw - 1);
    w.cy_hi = min((int)ceilf(dy2) - 1, ph - 1);
    w.empty = (w.cx_lo > w.cx_hi) || (w.cy_lo > w.cy_hi) || !(dx1 == dx1) || !(dx2 == dx2) || !(dy1 == dy1) || !(dy2 == dy2);
    return w;
}
// ---- bit-reproducible float32 exp / sigmoid: mirrors oracle/post_spec.py exp_spec / sigmoid_spec op for op.
__device__ __forceinline__ float vti_exp_spec(float x) {
    x = fminf(fmaxf(x, -86.0f), 88.0f);
    const float n = rintf(__fmul_rn(x, 1.4426950408889634f));
    float r = __fsub_rn(x, __fmul_rn(n, 0.693359375f));
    r = __fsub_rn(r, __fmul_rn(n, -2.12194440e-4f));
    float p = 1.0f / 5040.0f;
    p = __fadd_rn(__fmul_rn(p, r), 1.0f / 720.0f);
    p = __fadd_rn(__fmul_rn(p, r), 1.0f / 120.0f);
    p = __fadd_rn(__fmul_rn(p, r), 1.0f / 24.0f);
    p = __fadd_rn(__fmul_rn(p, r), 1.0f / 6.0f);
    p = __fadd_rn(__fmul_rn(p, r), 0.5f);
    p = __fadd_rn(__fmul_rn(p, r), 1.0f);
    p = __fadd_rn(__fmul_rn(p, r), 1.0f);
    return __fmul_rn(p, __int_as_float(((int)n + 127) << 23));
}
__device__ __forceinline__ float vti_sigmoid_spec(float x) {
    return __fdiv_rn(1.0f, __fadd_rn(1.0f, vti_exp_spec(-x)));
}
#endif

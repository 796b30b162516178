/*
 * vti.h -- C ABI of libvti.so, the B200-native per-frame inspection hot path.
 *
 * Drop-in boundary (SURVEY.md 8b).  The reference is pure Python and has no FFI of its own; the calls this
 * library replaces are
 *
 *   outer:  StitchMeasurementApp.process_frame(frame)            measurement.py:188  (main.py:211)
 *   inner:  self.model.predict(rgb, conf, iou, max_det, imgsz)   measurement.py:208-210
 *           (config 3: Utils/check_stitch_distance.py:281, :286)
 *
 * and the binding a maintainer adds is a ctypes stub (INTEGRATION.md; ours is vision_textile_inspection_b200/_lib.py).
 * Plain pointers and sizes only: no torch / Python types.  Device pointers are raw CUDA device addresses, `stream`
 * is a cudaStream_t passed as void* (0 = legacy default stream).  Every entry point returns 0 or a negative
 * VTI_E* code; vti_last_error() gives the message.  No call allocates in steady state: vti_create sizes every
 * scratch buffer for `max_batch` frames.
 *
 * Stages (kernels in vision_textile_inspection_b200/csrc/):
 *   vti_preprocess   K1  fused [cv2.undistort] + LetterBox resize/pad + HWC->CHW + /255      (SURVEY 8a U0-U2)
 *   vti_postprocess  K2  DFL decode + class sigmoid + confidence filter + compaction          (U3, U4 prelude)
 *                    K3  class-offset greedy NMS (torchvision semantics) + scale_boxes        (U4, U5, U7)
 *                    K4  coef x proto contraction + sigmoid + crop + 4x bilinear + >0.5,
 *                        fused with the nearest-resize mask statistics of measurement.py      (U6, M2-M4)
 *   vti_measure      K5  ROI routing, envelope, centroids, k-means row pick, pixel->mm         (M1, M3-M8)
 *   vti_annotate     K6  overlay rasterisation (+ vti_encode_jpeg: nvJPEG), off the hot path   (8f rank 3)
 */
#ifndef VTI_H_
#define VTI_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VTI_OK 0
#define VTI_EINVAL (-1)   /* bad argument / unsupported geometry */
#define VTI_ECUDA (-2)    /* CUDA runtime error (message in vti_last_error) */
#define VTI_ENOMEM (-3)
#define VTI_ENODEV (-4)   /* no CUDA device: the product path has no CPU fallback */

#define VTI_NM 32          /* mask coefficients / prototype channels */
#define VTI_REG_MAX 16     /* DFL bins */

/* det.flags */
#define VTI_F_IN_ROI 1u      /* passed measurement.py:253-260 (always set when ROI is off) */
#define VTI_F_STITCH 2u
#define VTI_F_FABRIC 4u
#define VTI_F_HAS_MASK 8u    /* frame-resolution bitmap non-empty (measurement.py:81) */
#define VTI_F_SELECTED 16u   /* k-means row selection (measurement.py:390-406) */
#define VTI_F_FINAL 32u      /* envelope-proximity filter (measurement.py:409-430) */
#define VTI_F_HAS_WIDTH 64u
#define VTI_F_HAS_DIST 128u
#define VTI_F_LB_MASK 256u   /* the letterbox-resolution mask (Results.masks.data) has at least one pixel set */
#define VTI_F_DROPPED 512u   /* mask_variant 1 only: empty mask, removed by Ultralytics' construct_result (not routed,
                                not counted in vti_frame_result.n_det; hosts skip these records) */

/* frame_result.status */
#define VTI_ST_OK 0
#define VTI_ST_NO_FABRIC 2   /* 'Fabric not detected'   measurement.py:281-287 */
#define VTI_ST_NO_STITCH 3   /* 'No stitches detected'  measurement.py:332-337 */
#define VTI_ST_OVERFLOW 0x100 /* OR-ed in: more NMS candidates than max_candidates (results truncated) */
#define VTI_ST_BAD_CAMERA 0x200 /* OR-ed in: the frame's camera id was outside [0, n_cameras) (nothing routed or measured) */

#define VTI_MAX_CAMERAS 256   /* cameras of one handle (vti_create_multi) */

typedef struct vti_handle vti_handle;

typedef struct vti_params {
    int32_t struct_size;          /* = sizeof(vti_params), ABI check */
    int32_t frame_h, frame_w;     /* camera frame, rows x cols */
    int32_t imgsz, stride;        /* predict(imgsz=...), model stride (32) */
    int32_t nc;                   /* classes (2: stitch, fabric) */
    int32_t max_det;              /* predict(max_det=...)  <= 1024 */
    int32_t max_batch;            /* frames per call upper bound */
    int32_t variant;              /* 0 = measurement.py semantics, 1 = Utils/check_stitch_distance.py semantics */
    int32_t undistort;            /* 1 = K1 remaps the image like cv2.undistort(K, dist); measure then uses dist = 0 */
    int32_t channel_flip;         /* 0: net plane c = frame channel c (reference: BGR->RGB->flip back); 1: reversed */
    int32_t stitch_id, fabric_id; /* config.py:69-70 */
    int32_t roi_enabled, roi_x_min, roi_x_max, roi_y_min, roi_y_max; /* config.py:91-95 (variant 0 only) */
    int32_t min_stitches;         /* config.py:79 */
    int32_t max_px_distance;      /* config.py:81 (150 in check_stitch_distance.py:38) */
    int32_t neighborhood;         /* config.py:82 */
    int32_t max_candidates;       /* per-frame NMS candidate capacity, 0 = min(A, 30000) (Ultralytics' max_nms: no
                                     overflow is possible below 30000 anchors); more confidence-passing anchors than the
                                     capacity raise VTI_ST_OVERFLOW (which of them are kept is then unspecified) */
    float conf, iou;              /* predict(conf=..., iou=...) */
    double K[9];                  /* camera_matrix, row major, for frame_w x frame_h */
    double dist[5];               /* k1 k2 p1 p2 k3 */
    double R[9];                  /* Rodrigues(rvec), row major */
    double t[3];                  /* tvec, metres */
    double iou_threshold;         /* predict(iou=...) as the DOUBLE torchvision.ops.nms compares against
                                     (`ovr > iou_threshold`, ovr float32); 0 = use (double)iou */
    int32_t mask_variant;         /* SURVEY 8a U6.  0 = "A" (Ultralytics <= 8.0.x, the north-star wording):
                                     sigmoid -> crop -> bilinear x4 -> > 0.5.  1 = "B" (newer releases): no sigmoid,
                                     crop, bilinear x4, > 0.0, and detections whose mask is empty are dropped */
} vti_params;

/* One camera's calibration on a multi-camera handle (vti_create_multi).  216 bytes. */
typedef struct vti_camera {
    int32_t struct_size;          /* = sizeof(vti_camera), ABI check */
    int32_t reserved;             /* 0 */
    double K[9], dist[5], R[9], t[3];   /* same meaning as in vti_params */
} vti_camera;

typedef struct vti_geometry {
    int32_t new_h, new_w;         /* resized (unpadded) size */
    int32_t top, bottom, left, right;
    int32_t LH, LW;               /* letterboxed net input */
    int32_t ph, pw;               /* prototype plane = LH/4 x LW/4 */
    int32_t lvl_h[3], lvl_w[3];   /* strides 8, 16, 32 */
    int32_t A;                    /* anchors */
    int32_t mask_words;           /* uint32 words per exported mask row = LW/32 */
    int32_t max_candidates;
    int32_t max_det;
} vti_geometry;

/* One kept detection ("defect record", SURVEY 8e).  160 bytes, fixed stride, gatherable across GPUs. */
typedef struct vti_det {
    float box_lb[4];              /* xyxy, letterbox px, unclipped (what process_mask crops with) */
    float box_frame[4];           /* xyxy, frame px, clipped (Results.boxes.xyxy) */
    int32_t box_int[4];           /* int() truncation, measurement.py:251 */
    float conf;
    int32_t cls;
    int32_t anchor;               /* NMS keep index = anchor index in Ultralytics order */
    uint32_t flags;
    int64_t m00, m10, m01;        /* raw moments of the frame-resolution bitmap (cv2.moments), exact */
    int32_t col_min, col_max;     /* occupied frame columns (measurement.py:311-314), -1 if none */
    double cx, cy;                /* stitch centroid (or bbox fallback) */
    double left_px, right_px;
    double width_mm;              /* NaN if not computed */
    double edge_y;                /* median envelope row near cx */
    double dist_mm;               /* NaN if not computed */
    double area_mm2;              /* area of the frame-resolution bitmap on the fabric plane: m00 x the area of one
                                     pixel at the centroid, |dP/du x dP/dv| by central differences of the
                                     pixel -> world projection (north-star "area"; the reference has no such
                                     output, oracle/measure_port.py defect_area_mm2 is the spec).  NaN if no mask */
} vti_det;

typedef struct vti_frame_result {
    int32_t status;
    int32_t n_det, n_cand;        /* n_det: kept detections (minus VTI_F_DROPPED ones); n_cand: confidence-passing anchors */
    int32_t n_stitch, n_fabric;   /* routed stitch boxes / fabric masks after the ROI filter */
    int32_t n_dist, n_width;      /* len(per_dists), len(all_widths) */
    int32_t env_valid;            /* frame columns with fabric */
    double avg_dist, avg_width;   /* pre-median averages, NaN = None (measurement.py:471-472) */
    double env_mean;              /* mean envelope row over valid columns */
} vti_frame_result;

const char* vti_last_error(void);
int vti_abi_version(void);

/* Host-only planning helpers (no GPU needed; used by vti_create and by the CPU tests). */
int vti_plan_geometry(int frame_h, int frame_w, int imgsz, int stride, int max_det, int max_candidates,
                      vti_geometry* out);
/* cv2.resize INTER_LINEAR taps.  x: idx[dn], a0[dn], a1[dn];  y: i0[dn], i1[dn], b0[dn], b1[dn] (11-bit). */
int vti_plan_resize_taps_x(int sn, int dn, int32_t* idx, int16_t* a0, int16_t* a1);
int vti_plan_resize_taps_y(int sn, int dn, int32_t* i0, int32_t* i1, int16_t* b0, int16_t* b1);
/* cv2.undistort source map in 1/32 px, (h*w) entries each. */
int vti_plan_undistort_map(const double K[9], const double dist[5], int h, int w, int32_t* ix, int32_t* iy);
/* cv2.resize INTER_NEAREST index map: src index for every dst index. */
int vti_plan_nearest_map(int dst_n, int src_n, int32_t* map);

int vti_create(const vti_params* p, vti_handle** out);
void vti_destroy(vti_handle* h);
int vti_get_geometry(const vti_handle* h, vti_geometry* out);

/* K1.  frames: device, B x frame_h x frame_w x 3 uint8.  net_in: device, B x 3 x LH x LW float32. */
int vti_preprocess(vti_handle* h, const uint8_t* frames, int B, float* net_in, void* stream);

/* K2+K3+K4.  Raw head tensors, device float32, contiguous NCHW:
 *   p3/p4/p5 : B x (64+nc) x Hl x Wl   (box channel = side*16+bin, then nc class logits)
 *   coef     : B x 32 x A              proto: B x 32 x ph x pw
 * Outputs (device): dets B x max_det, counts B, masks (optional, may be NULL) B x max_det x LH x (LW/32) uint32
 * bit-packed letterbox-resolution masks (bit i of word j = pixel 32j+i), rows of unused slots are not written. */
int vti_postprocess(vti_handle* h, const float* p3, const float* p4, const float* p5, const float* coef,
                    const float* proto, int B, vti_det* dets, int32_t* counts, uint32_t* masks, void* stream);

/* K5.  Completes the per-defect records in place and writes one vti_frame_result per frame. */
int vti_measure(vti_handle* h, int B, vti_det* dets, const int32_t* counts, vti_frame_result* results, void* stream);

/* vti_postprocess + vti_measure. */
int vti_post_measure(vti_handle* h, const float* p3, const float* p4, const float* p5, const float* coef,
                     const float* proto, int B, vti_det* dets, int32_t* counts, uint32_t* masks,
                     vti_frame_result* results, void* stream);

/* End-to-end with HOST buffers: K1..K5 over the batch in up to 4 pipelined chunks (copies of chunk i+1 under the
 * kernels of chunk i), D2H of net_in (optional, may be NULL), records, counts and frame results; returns after
 * everything has landed.  Pageable buffers are copied whole.  PINNED (device-mapped) head tensors are NOT copied:
 * K2 reads the class planes and the 64 box logits of each candidate in place over PCIe, K3 the coefficient rows of
 * the kept detections, and a fetch kernel brings only the union rectangle of the crop windows of the prototypes --
 * the path moves what it reads (the frames always travel by DMA). */
int vti_process_host(vti_handle* h, const uint8_t* frames, const float* p3, const float* p4, const float* p5,
                     const float* coef, const float* proto, int B, float* net_in, vti_det* dets, int32_t* counts,
                     vti_frame_result* results);

/* K6 (SURVEY 8f rank 3, off the hot path) -- the annotated overlay of measurement.py:230-236, 268-272, 292-296, 358-368,
 * 460-462 rasterised on the GPU.  Call after vti_measure / vti_post_measure of the SAME batch on the same handle (the
 * fabric envelope of that call is read).  frames / annotated: device, B x frame_h x frame_w x 3 uint8 BGR; annotated
 * receives a copy of the frames with the ROI rectangle, detection boxes, envelope polyline, stitch width markers and
 * edge-distance lines drawn in the reference's colours and order. */
int vti_annotate(vti_handle* h, const uint8_t* frames, int B, const vti_det* dets, const int32_t* counts,
                 uint8_t* annotated, void* stream);
/* One text line (5 x 7 bitmap font, `scale` pixels per dot) into frame `frame` of an annotated batch: measurement.py:500-504
 * (cv2.putText there). */
int vti_draw_text(vti_handle* h, uint8_t* annotated, int frame, int x, int y, const char* text, int scale, int b, int g,
                  int r, void* stream);
/* K0 -- camera-native frame ingest (SURVEY 8f rank 2).  The reference opens its camera without a FOURCC
 * (measurement.py:22-38), so OpenCV's V4L2 backend negotiates packed YUV 4:2:2 ("YUYV"/"YUY2", 2 bytes per pixel) and
 * converts every frame to BGR on the CPU inside cap.read() (main.py:188).  vti_ingest_yuyv does that conversion on the
 * device, bit-exact against cv2.cvtColor(.., COLOR_YUV2BGR_YUY2): yuyv = B x frame_h x frame_w x 2 bytes (device,
 * 4-byte aligned, frame_w even) -> frames = B x frame_h x frame_w x 3 BGR (device), ready for vti_preprocess. */
int vti_ingest_yuyv(vti_handle* h, const uint8_t* yuyv, int B, uint8_t* frames, void* stream);
/* vti_process_host with the frames as the camera delivered them (HOST YUYV bytes): 2/3 of the BGR bytes cross PCIe,
 * K0 converts in front of K1.  Everything else as vti_process_host. */
int vti_process_host_yuyv(vti_handle* h, const uint8_t* yuyv, const float* p3, const float* p4, const float* p5,
                          const float* coef, const float* proto, int B, float* net_in, vti_det* dets, int32_t* counts,
                          vti_frame_result* results);

/* nvJPEG encode of ONE device frame (frame_h x frame_w x 3 BGR) -- main.py:314's cv2.imwrite(.., annotated).  quality
 * 1..100 (0 = 95, cv2's default), 4:2:0.  Returns the number of bytes written to the HOST buffer `out`, or VTI_E*. */
long long vti_encode_jpeg(vti_handle* h, const uint8_t* image, int quality, uint8_t* out, long long capacity, void* stream);

/* Compressed frame ingest (SURVEY 8f rank 2): nvJPEG decode of ONE JPEG (HOST bytes, e.g. a camera's MJPEG frame that
 * cv2.VideoCapture would decode on the CPU, main.py:188) into a DEVICE frame buffer (frame_h x frame_w x 3 BGR) that
 * vti_preprocess reads.  Asynchronous on `stream`. */
int vti_decode_jpeg(vti_handle* h, const uint8_t* jpeg, long long nbytes, uint8_t* frame, void* stream);

/* The batched form: n JPEG streams (HOST bytes) -> n consecutive device frames, through nvjpegDecodeBatched.  The first
 * call picks the best nvJPEG backend that accepts the streams -- the NVJPG hardware engines, GPU-assisted Huffman, the
 * default hybrid (CPU Huffman) -- and vti_jpeg_backend() names it ("nvjpeg-hardware" | "nvjpeg-gpu-hybrid" |
 * "nvjpeg-hybrid" | "none").  Replaces the per-frame CPU decode inside cv2.VideoCapture.read (main.py:188). */
int vti_decode_jpeg_batch(vti_handle* h, const uint8_t* const* jpegs, const long long* nbytes, int n, uint8_t* frames,
                          void* stream);
const char* vti_jpeg_backend(void);

/* ---- Several cameras of one frame size behind one handle.
 * vti_create_multi: like vti_create, with the calibration of camera c taken from cameras[c] (p->K / dist / R / t are
 * ignored).  n_cameras is 1..VTI_MAX_CAMERAS and every struct_size must match; both are checked before the device, so a
 * machine without a GPU still reports VTI_EINVAL for bad arguments.  cameras[0] becomes the handle's own calibration:
 * every entry point without a camera argument (vti_preprocess, vti_measure, vti_post_measure, vti_process_host[_yuyv],
 * vti_annotate) treats each frame as camera 0.  vti_create(p) is vti_create_multi(p, 1, {p's calibration}).  Every
 * per-camera table is built at create; steady state still allocates nothing.  Only K1 (the undistort remap) and K5
 * (the pixel -> world projection) depend on the camera; vti_postprocess and vti_annotate take no camera ids.
 *
 * `camera`: one int32 camera id per frame -- a DEVICE array for the stream entry points, read by the kernels when they
 * run (a captured CUDA graph follows the buffer's current contents), a HOST array for the two host-buffer entry points.
 * NULL means camera 0 for every frame.  A device id outside [0, n_cameras) is never used as an index: K1 undistorts
 * that frame with camera 0's tables (its net_in is unspecified), and K5 ORs VTI_ST_BAD_CAMERA into its status, leaves
 * its records as K4 left them and routes and measures nothing (n_stitch = n_fabric = n_dist = n_width = env_valid = 0,
 * NaN averages).  The host entry points check their ids before any work and return VTI_EINVAL. */
int vti_create_multi(const vti_params* p, int n_cameras, const vti_camera* cameras, vti_handle** out);
int vti_camera_count(const vti_handle* h);
int vti_preprocess_multi(vti_handle* h, const uint8_t* frames, const int32_t* camera, int B, float* net_in, void* stream);
int vti_measure_multi(vti_handle* h, int B, const int32_t* camera, vti_det* dets, const int32_t* counts,
                      vti_frame_result* results, void* stream);
int vti_post_measure_multi(vti_handle* h, const float* p3, const float* p4, const float* p5, const float* coef,
                           const float* proto, int B, const int32_t* camera, vti_det* dets, int32_t* counts,
                           uint32_t* masks, vti_frame_result* results, void* stream);
int vti_process_host_multi(vti_handle* h, const uint8_t* frames, const float* p3, const float* p4, const float* p5,
                           const float* coef, const float* proto, int B, const int32_t* camera, float* net_in,
                           vti_det* dets, int32_t* counts, vti_frame_result* results);
int vti_process_host_yuyv_multi(vti_handle* h, const uint8_t* yuyv, const float* p3, const float* p4, const float* p5,
                                const float* coef, const float* proto, int B, const int32_t* camera, float* net_in,
                                vti_det* dets, int32_t* counts, vti_frame_result* results);

/* Number of kernel launches issued by this handle since creation (bench.py's gpu_launches). */
int64_t vti_launch_count(const vti_handle* h);

/* Per-kernel timing with CUDA events recorded on the caller's stream around each kernel (off by default).
 * vti_get_stage_ms synchronises on the events of the most recent vti_preprocess / vti_postprocess / vti_measure
 * calls and returns their durations in ms: ms[0..4] = K1, K2, K3, K4, K5 (-1 where no event pair was recorded). */
int vti_set_profiling(vti_handle* h, int on);
int vti_get_stage_ms(vti_handle* h, float ms[5]);

#ifdef __cplusplus
}
#endif
#endif /* VTI_H_ */

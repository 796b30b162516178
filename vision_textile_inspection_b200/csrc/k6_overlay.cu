// K6 -- annotated overlay rasterised on the GPU + JPEG encode with nvJPEG (SURVEY.md 8f rank 3).
//
// Replaces the drawing calls of measurement.py (they have no effect on the numbers; main.py:302-314 saves
// the annotated frame as a JPEG for every inspected frame):
//   :230-236  ROI rectangle                       cv2.rectangle(.., ROI_BORDER_COLOR, 2)
//   :268-272  per-detection boxes                 stitch (255,255,0) thickness 1, fabric (255,0,255) thickness 2
//   :292-296  fabric envelope polyline            cv2.polylines(.., (255,128,0), 2)
//   :358-368  per-stitch width markers            circles r = 3 at (left, cy), (right, cy), (cx, cy) + the line between
//   :460-462  per-measured-stitch edge distance   line (cx, edge_y) - (cx, cy), circle r = 2 at the edge point
//   :500-504  the two text lines                  (5 x 7 bitmap font here; the reference uses Hershey Simplex)
// Rectangles, circles and the axis-aligned lines reproduce cv2's pixel sets exactly (tests/test_overlay.py compares with
// cv2 itself); the thick envelope polyline stamps cv2's radius-1 brush along each segment (>= 95 % of cv2's pixels).
// Mask contours (:496-499) need the frame-resolution bitmaps the fused path never builds and are not drawn.
// Layers are separate launches in the reference's drawing order, so overlapping primitives resolve the same way.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <algorithm>
#include <string>
#include <thread>
#include <vector>

#include <nvjpeg.h>

#include "vti_internal.h"

namespace {

struct K6Args {
    uint8_t* img;               // [B][h][w][3] BGR, already a copy of the frames
    const vti_det* dets;        // [B][max_det]
    const int32_t* counts;
    const int32_t* env_frame;   // [B][w]   (-1 = no fabric in that column)
    int h, w, max_det;
    int roi_active, rx1, ry1, rx2, ry2;
};

__device__ __forceinline__ void put(const K6Args& a, int b, int x, int y, uchar3 c) {
    if ((unsigned)x < (unsigned)a.w && (unsigned)y < (unsigned)a.h) {
        uint8_t* p = a.img + (((size_t)b * a.h + y) * a.w + x) * 3;
        p[0] = c.x; p[1] = c.y; p[2] = c.z;
    }
}

// cv2.rectangle((x1,y1),(x2,y2), color, t): t = 1 the four edges; t = 2 three-pixel-wide bars without the four outermost
// corner pixels (OpenCV draws thick lines as polygons with round caps).
__device__ void rect(const K6Args& a, int b, int x1, int y1, int x2, int y2, int t, uchar3 c, int tid, int nthr) {
    if (x1 > x2) { const int s = x1; x1 = x2; x2 = s; }
    if (y1 > y2) { const int s = y1; y1 = y2; y2 = s; }
    const int r = t >= 2 ? 1 : 0;
    const int W = x2 - x1 + 1 + 2 * r, H = y2 - y1 + 1 + 2 * r;
    for (int i = tid; i < W * (2 * r + 1); i += nthr) {          // top and bottom bars
        const int dx = i % W, dy = i / W - r;
        const bool corner = r && (dx == 0 || dx == W - 1);
        if (!(corner && dy == -r)) put(a, b, x1 - r + dx, y1 + dy, c);
        if (!(corner && dy == r)) put(a, b, x1 - r + dx, y2 + dy, c);
    }
    for (int i = tid; i < H * (2 * r + 1); i += nthr) {          // left and right bars
        const int dy = i % H, dx = i / H - r;
        const bool corner = r && (dy == 0 || dy == H - 1);
        if (!(corner && dx == -r)) put(a, b, x1 + dx, y1 - r + dy, c);
        if (!(corner && dx == r)) put(a, b, x2 + dx, y1 - r + dy, c);
    }
}

// cv2.circle(.., radius, color, -1) for the two radii the reference uses: half-widths of the rows dy = -r .. r.
// Thread-parallel over the (2r+1)^2 bounding square.
__device__ void disc(const K6Args& a, int b, int cx, int cy, int r, uchar3 c, int tid, int nthr) {
    const int hw3[7] = {0, 2, 2, 3, 2, 2, 0}, hw2[5] = {0, 1, 2, 1, 0};
    const int side = 2 * r + 1;
    for (int i = tid; i < side * side; i += nthr) {
        const int dy = i / side - r, dx = i % side - r;
        const int hw = r == 3 ? hw3[dy + 3] : hw2[dy + 2];
        if (abs(dx) <= hw) put(a, b, cx + dx, cy + dy, c);
    }
}

__device__ __forceinline__ int iround(double v) { return (int)rint(v); }      // Python round(): half to even

__global__ void k6_boxes_kernel(const K6Args a, int layer) {
    const int b = blockIdx.y, k = blockIdx.x;
    if (layer == 0) {                                            // the ROI rectangle goes first
        if (k == 0 && a.roi_active) rect(a, b, a.rx1, a.ry1, a.rx2, a.ry2, 2, make_uchar3(144, 238, 144), threadIdx.x, blockDim.x);
        return;
    }
    if (k >= a.counts[b]) return;
    const vti_det& d = a.dets[(size_t)b * a.max_det + k];
    if (!(d.flags & VTI_F_IN_ROI) || (d.flags & VTI_F_DROPPED)) return;
    // boxes of one class share a colour, so their mutual overlaps need no ordering; fabric boxes go first (the reference
    // draws in detection order: where a fabric box crosses a stitch box detected before it the two orders differ)
    if (layer == 1) {
        if (d.flags & VTI_F_FABRIC) rect(a, b, d.box_int[0], d.box_int[1], d.box_int[2], d.box_int[3], 2, make_uchar3(255, 0, 255), threadIdx.x, blockDim.x);
    } else if (d.flags & VTI_F_STITCH) {
        rect(a, b, d.box_int[0], d.box_int[1], d.box_int[2], d.box_int[3], 1, make_uchar3(255, 255, 0), threadIdx.x, blockDim.x);
    }
}

// envelope polyline, thickness 2: every segment (x, env[x]) - (x+1, env[x+1]) between consecutive fabric columns, a radius-1
// brush stamped on each pixel of the segment (the segment between columns that are not adjacent is the straight line cv2
// draws between the two points, walked in x)
__global__ void k6_envelope_kernel(const K6Args a) {
    const int b = blockIdx.y;
    const int32_t* env = a.env_frame + (size_t)b * a.w;
    const uchar3 c = make_uchar3(255, 128, 0);
    for (int x = blockIdx.x * blockDim.x + threadIdx.x; x < a.w; x += gridDim.x * blockDim.x) {
        const int y0 = env[x];
        if (y0 < 0) continue;
        int xn = x + 1;
        while (xn < a.w && env[xn] < 0) ++xn;                    // next fabric column
        const int y1 = xn < a.w ? env[xn] : y0, x1 = xn < a.w ? xn : x;
        const int steps = max(abs(y1 - y0), x1 - x);
        for (int s = 0; s <= steps; ++s) {
            const int px = x + (steps ? iround((double)(x1 - x) * s / steps) : 0);
            const int py = y0 + (steps ? iround((double)(y1 - y0) * s / steps) : 0);
            put(a, b, px, py, c); put(a, b, px - 1, py, c); put(a, b, px + 1, py, c); put(a, b, px, py - 1, c); put(a, b, px, py + 1, c);
        }
    }
}

// Stitch markers.  The reference draws stitch after stitch, so where the markers of two stitches overlap the LATER stitch
// wins: one CTA per frame walks the detections in order, its threads share the pixels of each primitive, a barrier
// separates primitives of different colours.
__global__ void k6_markers_kernel(const K6Args a, int layer) {
    const int b = blockIdx.x, tid = threadIdx.x, nthr = blockDim.x;
    const int n = a.counts[b];
    for (int k = 0; k < n; ++k) {
        const vti_det& d = a.dets[(size_t)b * a.max_det + k];
        if (!(d.flags & VTI_F_STITCH) || !(d.flags & VTI_F_IN_ROI) || (d.flags & VTI_F_DROPPED) || !(d.cx == d.cx)) continue;
        const int cy = iround(d.cy), cx = iround(d.cx);
        if (layer == 0) {                                        // measurement.py:358-363
            const int xl = iround(d.left_px), xr = iround(d.right_px);
            disc(a, b, xl, cy, 3, make_uchar3(200, 200, 0), tid, nthr);
            disc(a, b, xr, cy, 3, make_uchar3(200, 200, 0), tid, nthr);
            for (int x = min(xl, xr) + tid; x <= max(xl, xr); x += nthr) put(a, b, x, cy, make_uchar3(200, 200, 0));
            __syncthreads();
            disc(a, b, cx, cy, 3, make_uchar3(200, 0, 0), tid, nthr);
            __syncthreads();
        } else if (d.flags & VTI_F_HAS_DIST) {                   // measurement.py:460-462
            const int ey = iround(d.edge_y);
            for (int y = min(ey, cy) + tid; y <= max(ey, cy); y += nthr) put(a, b, cx, y, make_uchar3(0, 255, 0));
            __syncthreads();
            disc(a, b, cx, ey, 2, make_uchar3(255, 0, 255), tid, nthr);
            __syncthreads();
        }
    }
}

// 5 x 7 bitmap font, ASCII 32..126, one byte per column, bit 0 = top row (the classic public-domain glcd font)
__constant__ unsigned char c_font[95 * 5] = {
    0x00,0x00,0x00,0x00,0x00, 0x00,0x00,0x5F,0x00,0x00, 0x00,0x07,0x00,0x07,0x00, 0x14,0x7F,0x14,0x7F,0x14, 0x24,0x2A,0x7F,0x2A,0x12,
    0x23,0x13,0x08,0x64,0x62, 0x36,0x49,0x55,0x22,0x50, 0x00,0x05,0x03,0x00,0x00, 0x00,0x1C,0x22,0x41,0x00, 0x00,0x41,0x22,0x1C,0x00,
    0x14,0x08,0x3E,0x08,0x14, 0x08,0x08,0x3E,0x08,0x08, 0x00,0x50,0x30,0x00,0x00, 0x08,0x08,0x08,0x08,0x08, 0x00,0x60,0x60,0x00,0x00,
    0x20,0x10,0x08,0x04,0x02, 0x3E,0x51,0x49,0x45,0x3E, 0x00,0x42,0x7F,0x40,0x00, 0x42,0x61,0x51,0x49,0x46, 0x21,0x41,0x45,0x4B,0x31,
    0x18,0x14,0x12,0x7F,0x10, 0x27,0x45,0x45,0x45,0x39, 0x3C,0x4A,0x49,0x49,0x30, 0x01,0x71,0x09,0x05,0x03, 0x36,0x49,0x49,0x49,0x36,
    0x06,0x49,0x49,0x29,0x1E, 0x00,0x36,0x36,0x00,0x00, 0x00,0x56,0x36,0x00,0x00, 0x08,0x14,0x22,0x41,0x00, 0x14,0x14,0x14,0x14,0x14,
    0x00,0x41,0x22,0x14,0x08, 0x02,0x01,0x51,0x09,0x06, 0x32,0x49,0x79,0x41,0x3E, 0x7E,0x11,0x11,0x11,0x7E, 0x7F,0x49,0x49,0x49,0x36,
    0x3E,0x41,0x41,0x41,0x22, 0x7F,0x41,0x41,0x22,0x1C, 0x7F,0x49,0x49,0x49,0x41, 0x7F,0x09,0x09,0x09,0x01, 0x3E,0x41,0x49,0x49,0x7A,
    0x7F,0x08,0x08,0x08,0x7F, 0x00,0x41,0x7F,0x41,0x00, 0x20,0x40,0x41,0x3F,0x01, 0x7F,0x08,0x14,0x22,0x41, 0x7F,0x40,0x40,0x40,0x40,
    0x7F,0x02,0x0C,0x02,0x7F, 0x7F,0x04,0x08,0x10,0x7F, 0x3E,0x41,0x41,0x41,0x3E, 0x7F,0x09,0x09,0x09,0x06, 0x3E,0x41,0x51,0x21,0x5E,
    0x7F,0x09,0x19,0x29,0x46, 0x46,0x49,0x49,0x49,0x31, 0x01,0x01,0x7F,0x01,0x01, 0x3F,0x40,0x40,0x40,0x3F, 0x1F,0x20,0x40,0x20,0x1F,
    0x3F,0x40,0x38,0x40,0x3F, 0x63,0x14,0x08,0x14,0x63, 0x07,0x08,0x70,0x08,0x07, 0x61,0x51,0x49,0x45,0x43, 0x00,0x7F,0x41,0x41,0x00,
    0x02,0x04,0x08,0x10,0x20, 0x00,0x41,0x41,0x7F,0x00, 0x04,0x02,0x01,0x02,0x04, 0x40,0x40,0x40,0x40,0x40, 0x00,0x01,0x02,0x04,0x00,
    0x20,0x54,0x54,0x54,0x78, 0x7F,0x48,0x44,0x44,0x38, 0x38,0x44,0x44,0x44,0x20, 0x38,0x44,0x44,0x48,0x7F, 0x38,0x54,0x54,0x54,0x18,
    0x08,0x7E,0x09,0x01,0x02, 0x0C,0x52,0x52,0x52,0x3E, 0x7F,0x08,0x04,0x04,0x78, 0x00,0x44,0x7D,0x40,0x00, 0x20,0x40,0x44,0x3D,0x00,
    0x7F,0x10,0x28,0x44,0x00, 0x00,0x41,0x7F,0x40,0x00, 0x7C,0x04,0x18,0x04,0x78, 0x7C,0x08,0x04,0x04,0x78, 0x38,0x44,0x44,0x44,0x38,
    0x7C,0x14,0x14,0x14,0x08, 0x08,0x14,0x14,0x18,0x7C, 0x7C,0x08,0x04,0x04,0x08, 0x48,0x54,0x54,0x54,0x20, 0x04,0x3F,0x44,0x40,0x20,
    0x3C,0x40,0x40,0x20,0x7C, 0x1C,0x20,0x40,0x20,0x1C, 0x3C,0x40,0x30,0x40,0x3C, 0x44,0x28,0x10,0x28,0x44, 0x0C,0x50,0x50,0x50,0x3C,
    0x44,0x64,0x54,0x4C,0x44, 0x00,0x08,0x36,0x41,0x00, 0x00,0x00,0x7F,0x00,0x00, 0x00,0x41,0x36,0x08,0x00, 0x10,0x08,0x08,0x10,0x08,
};

struct K6Text {
    char s[160];
    int n, x, y, scale;         // (x, y) = top-left corner of the first glyph
    unsigned char b, g, r;
};

__global__ void k6_text_kernel(uint8_t* img, int h, int w, int frame, const K6Text t) {
    const int per = 6 * 7 * t.scale * t.scale;                   // 5 columns + 1 gap, 7 rows, scale^2 pixels each
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < t.n * per; i += gridDim.x * blockDim.x) {
        const int ch = i / per, r = i - ch * per;
        const int py = r / (6 * t.scale), px = r - py * 6 * t.scale;
        const int col = px / t.scale, row = py / t.scale;
        const int code = (int)(unsigned char)t.s[ch] - 32;
        if (col >= 5 || code < 0 || code >= 95) continue;
        if (!((c_font[code * 5 + col] >> row) & 1)) continue;
        const int X = t.x + ch * 6 * t.scale + px, Y = t.y + py;
        if ((unsigned)X < (unsigned)w && (unsigned)Y < (unsigned)h) {
            uint8_t* p = img + (((size_t)frame * h + Y) * w + X) * 3;
            p[0] = t.b; p[1] = t.g; p[2] = t.r;
        }
    }
}

// ---- nvJPEG (one encoder per process, guarded; annotation is off the hot path)
struct Jpeg {
    nvjpegHandle_t handle = nullptr;
    nvjpegEncoderState_t state = nullptr;
    nvjpegEncoderParams_t params = nullptr;
    nvjpegJpegState_t dec = nullptr;
    std::mutex mu;
    bool ok = false, dec_ok = false;
};
Jpeg g_jpeg;

}  // namespace

extern "C" int vti_annotate(vti_handle* h, const uint8_t* frames, int B, const vti_det* dets, const int32_t* counts,
                            uint8_t* annotated, void* stream) {
    if (!h || !frames || !dets || !counts || !annotated) { vti_set_error("vti_annotate: null argument"); return VTI_EINVAL; }
    if (B < 1 || B > h->p.max_batch) { vti_set_error("vti_annotate: batch size out of range"); return VTI_EINVAL; }
    cudaStream_t s = (cudaStream_t)stream;
    const int fh = h->p.frame_h, fw = h->p.frame_w;
    VTI_CUDA(cudaMemcpyAsync(annotated, frames, (size_t)B * fh * fw * 3, cudaMemcpyDeviceToDevice, s));
    K6Args a;
    a.img = annotated; a.dets = dets; a.counts = counts; a.env_frame = h->d_env_frame;
    a.h = fh; a.w = fw; a.max_det = h->p.max_det;
    a.roi_active = h->roi.active; a.rx1 = h->roi.x1; a.ry1 = h->roi.y1; a.rx2 = h->roi.x2; a.ry2 = h->roi.y2;
    const dim3 gdet(a.max_det, B);
    k6_boxes_kernel<<<dim3(1, B), 128, 0, s>>>(a, 0);            // ROI
    k6_boxes_kernel<<<gdet, 128, 0, s>>>(a, 1);                  // fabric boxes
    k6_boxes_kernel<<<gdet, 128, 0, s>>>(a, 2);                  // stitch boxes
    k6_envelope_kernel<<<dim3((fw + 255) / 256, B), 256, 0, s>>>(a);
    k6_markers_kernel<<<B, 64, 0, s>>>(a, 0);
    k6_markers_kernel<<<B, 64, 0, s>>>(a, 1);
    h->launches += 6;
    VTI_CUDA(cudaGetLastError());
    return VTI_OK;
}

extern "C" int vti_draw_text(vti_handle* h, uint8_t* annotated, int frame, int x, int y, const char* text, int scale,
                             int b, int g, int r, void* stream) {
    if (!h || !annotated || !text || frame < 0 || scale < 1 || scale > 8) { vti_set_error("vti_draw_text: bad argument"); return VTI_EINVAL; }
    K6Text t;
    std::memset(&t, 0, sizeof(t));
    t.n = (int)std::strlen(text);
    if (t.n > (int)sizeof(t.s) - 1) t.n = (int)sizeof(t.s) - 1;
    std::memcpy(t.s, text, t.n);
    t.x = x; t.y = y; t.scale = scale; t.b = (unsigned char)b; t.g = (unsigned char)g; t.r = (unsigned char)r;
    if (t.n == 0) return VTI_OK;
    k6_text_kernel<<<(t.n * 42 * scale * scale + 255) / 256, 256, 0, (cudaStream_t)stream>>>(annotated, h->p.frame_h, h->p.frame_w, frame, t);
    h->launches++;
    VTI_CUDA(cudaGetLastError());
    return VTI_OK;
}

// JPEG-encodes ONE annotated frame (device, h x w x 3 BGR interleaved) with nvJPEG: returns the number of bytes written
// to `out` (host), or a negative VTI_E* code; `capacity` too small -> VTI_EINVAL with the needed size in the message.
extern "C" long long vti_encode_jpeg(vti_handle* h, const uint8_t* image, int quality, uint8_t* out, long long capacity,
                                      void* stream) {
    if (!h || !image || !out) { vti_set_error("vti_encode_jpeg: null argument"); return VTI_EINVAL; }
    std::lock_guard<std::mutex> lock(g_jpeg.mu);
    cudaStream_t s = (cudaStream_t)stream;
    if (!g_jpeg.ok) {
        if ((!g_jpeg.handle && nvjpegCreateSimple(&g_jpeg.handle) != NVJPEG_STATUS_SUCCESS) ||
            nvjpegEncoderStateCreate(g_jpeg.handle, &g_jpeg.state, s) != NVJPEG_STATUS_SUCCESS ||
            nvjpegEncoderParamsCreate(g_jpeg.handle, &g_jpeg.params, s) != NVJPEG_STATUS_SUCCESS) {
            vti_set_error("vti_encode_jpeg: nvJPEG initialisation failed");
            return VTI_ECUDA;
        }
        g_jpeg.ok = true;
    }
    nvjpegEncoderParamsSetQuality(g_jpeg.params, quality < 1 ? 95 : (quality > 100 ? 100 : quality), s);   // cv2.imwrite default 95
    nvjpegEncoderParamsSetSamplingFactors(g_jpeg.params, NVJPEG_CSS_420, s);                               // cv2's default subsampling
    nvjpegEncoderParamsSetOptimizedHuffman(g_jpeg.params, 0, s);
    nvjpegImage_t src;
    std::memset(&src, 0, sizeof(src));
    src.channel[0] = const_cast<unsigned char*>(image);
    src.pitch[0] = (size_t)h->p.frame_w * 3;
    if (nvjpegEncodeImage(g_jpeg.handle, g_jpeg.state, g_jpeg.params, &src, NVJPEG_INPUT_BGRI, h->p.frame_w, h->p.frame_h, s) !=
        NVJPEG_STATUS_SUCCESS) {
        vti_set_error("vti_encode_jpeg: nvjpegEncodeImage failed");
        return VTI_ECUDA;
    }
    size_t len = 0;
    if (nvjpegEncodeRetrieveBitstream(g_jpeg.handle, g_jpeg.state, nullptr, &len, s) != NVJPEG_STATUS_SUCCESS) {
        vti_set_error("vti_encode_jpeg: nvjpegEncodeRetrieveBitstream (size) failed");
        return VTI_ECUDA;
    }
    if ((long long)len > capacity) {
        vti_set_error("vti_encode_jpeg: output buffer too small (" + std::to_string(len) + " bytes needed)");
        return VTI_EINVAL;
    }
    if (nvjpegEncodeRetrieveBitstream(g_jpeg.handle, g_jpeg.state, out, &len, s) != NVJPEG_STATUS_SUCCESS) {
        vti_set_error("vti_encode_jpeg: nvjpegEncodeRetrieveBitstream failed");
        return VTI_ECUDA;
    }
    VTI_CUDA(cudaStreamSynchronize(s));
    return (long long)len;
}

// Frame ingest from a compressed camera stream (SURVEY.md 8f rank 2): the camera of the reference delivers MJPEG
// (cv2.VideoCapture, main.py:188 decodes it on the CPU before process_frame sees the array).  Decodes ONE
// baseline JPEG (host bytes) with nvJPEG straight into the device frame buffer K1 reads (frame_h x frame_w x 3 BGR), so
// that the frame crosses PCIe compressed.  The image must have the handle's frame size.
extern "C" int vti_decode_jpeg(vti_handle* h, const uint8_t* jpeg, long long nbytes, uint8_t* frame, void* stream) {
    if (!h || !jpeg || nbytes <= 0 || !frame) { vti_set_error("vti_decode_jpeg: bad argument"); return VTI_EINVAL; }
    std::lock_guard<std::mutex> lock(g_jpeg.mu);
    cudaStream_t s = (cudaStream_t)stream;
    if (!g_jpeg.handle && nvjpegCreateSimple(&g_jpeg.handle) != NVJPEG_STATUS_SUCCESS) {
        vti_set_error("vti_decode_jpeg: nvJPEG initialisation failed");
        return VTI_ECUDA;
    }
    if (!g_jpeg.dec_ok) {
        if (nvjpegJpegStateCreate(g_jpeg.handle, &g_jpeg.dec) != NVJPEG_STATUS_SUCCESS) {
            vti_set_error("vti_decode_jpeg: nvjpegJpegStateCreate failed");
            return VTI_ECUDA;
        }
        g_jpeg.dec_ok = true;
    }
    int nc = 0, widths[NVJPEG_MAX_COMPONENT], heights[NVJPEG_MAX_COMPONENT];
    nvjpegChromaSubsampling_t css;
    if (nvjpegGetImageInfo(g_jpeg.handle, jpeg, (size_t)nbytes, &nc, &css, widths, heights) != NVJPEG_STATUS_SUCCESS) {
        vti_set_error("vti_decode_jpeg: not a JPEG stream nvJPEG can parse");
        return VTI_EINVAL;
    }
    if (widths[0] != h->p.frame_w || heights[0] != h->p.frame_h) {
        vti_set_error("vti_decode_jpeg: image is " + std::to_string(widths[0]) + "x" + std::to_string(heights[0]) +
                      ", the handle was created for " + std::to_string(h->p.frame_w) + "x" + std::to_string(h->p.frame_h));
        return VTI_EINVAL;
    }
    nvjpegImage_t dst;
    std::memset(&dst, 0, sizeof(dst));
    dst.channel[0] = frame;
    dst.pitch[0] = (size_t)h->p.frame_w * 3;
    if (nvjpegDecode(g_jpeg.handle, g_jpeg.dec, jpeg, (size_t)nbytes, NVJPEG_OUTPUT_BGRI, &dst, s) != NVJPEG_STATUS_SUCCESS) {
        vti_set_error("vti_decode_jpeg: nvjpegDecode failed");
        return VTI_ECUDA;
    }
    return VTI_OK;
}

// ---- batched ingest: the batch through nvjpegDecodeBatched, split over a few host threads ("lanes").  nvJPEG's batched
// decoder does its bitstream parsing and Huffman-table set-up on the calling thread, so one call per batch leaves the
// GPU waiting on one host core; each lane owns its nvJPEG handle, state and stream and takes a contiguous slice of the
// batch, and the caller's stream waits on every lane's event.  Backends are tried once per process, best first: the NVJPG
// hardware engines (Huffman + IDCT off the SMs), GPU-assisted Huffman, then the default hybrid (CPU Huffman).
// `vti_jpeg_backend()` names the one that decoded the last batch.
namespace {
constexpr int JB_MAX_LANES = 8;
struct JpegLane {
    nvjpegHandle_t handle = nullptr;
    nvjpegJpegState_t state = nullptr;
    cudaStream_t stream = nullptr;
    cudaEvent_t done = nullptr;
    int backend = -1, batch = 0, device = -1;
    bool on_device(int dev) {                      // stream + event live as long as the process (or until the device changes)
        if (device == dev) return true;
        release();
        if (stream) { cudaStreamDestroy(stream); stream = nullptr; }
        if (done) { cudaEventDestroy(done); done = nullptr; }
        device = -1;
        if (cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking) != cudaSuccess) return false;
        if (cudaEventCreateWithFlags(&done, cudaEventDisableTiming) != cudaSuccess) return false;
        device = dev;
        return true;
    }
    void release() {
        if (state) { nvjpegJpegStateDestroy(state); state = nullptr; }
        if (handle) { nvjpegDestroy(handle); handle = nullptr; }
        batch = 0;
        backend = -1;
    }
    bool open(int idx) {
        release();
        if (nvjpegCreateEx(kBackendsOf(idx), nullptr, nullptr, NVJPEG_FLAGS_DEFAULT, &handle) != NVJPEG_STATUS_SUCCESS) {
            handle = nullptr;
            return false;
        }
        if (nvjpegJpegStateCreate(handle, &state) != NVJPEG_STATUS_SUCCESS) {
            state = nullptr;
            release();
            return false;
        }
        backend = idx;
        return true;
    }
    static nvjpegBackend_t kBackendsOf(int idx) {
        return idx == 0 ? NVJPEG_BACKEND_HARDWARE : (idx == 1 ? NVJPEG_BACKEND_GPU_HYBRID : NVJPEG_BACKEND_DEFAULT);
    }
};
struct JpegBatch {
    JpegLane lane[JB_MAX_LANES];
    nvjpegHandle_t probe = nullptr;    // header parsing only
    int backend = -1;       // backend index of the last successful batch, -1 = none yet
    std::mutex mu;
};
JpegBatch g_jb;
const char* const kBackendNames[3] = {"nvjpeg-hardware", "nvjpeg-gpu-hybrid", "nvjpeg-hybrid"};

// one lane decodes images [i0, i1) with backend `idx`; false = this backend cannot take them
bool jb_lane_decode(JpegLane& L, int idx, int device, const uint8_t* const* jpegs, const size_t* len, nvjpegImage_t* dst, int i0,
                    int i1) {
    if (L.backend != idx && !L.open(idx)) return false;
    const int n = i1 - i0;
    if (L.batch != n) {
        if (nvjpegDecodeBatchedInitialize(L.handle, L.state, n, 1, NVJPEG_OUTPUT_BGRI) != NVJPEG_STATUS_SUCCESS) {
            L.release();
            return false;
        }
        L.batch = n;
    }
    if (nvjpegDecodeBatched(L.handle, L.state, (const unsigned char* const*)(jpegs + i0), len + i0, dst + i0, L.stream) !=
        NVJPEG_STATUS_SUCCESS) {
        L.release();
        return false;
    }
    return cudaEventRecord(L.done, L.stream) == cudaSuccess;
}
}  // namespace

extern "C" const char* vti_jpeg_backend(void) {
    std::lock_guard<std::mutex> lock(g_jb.mu);
    return g_jb.backend < 0 ? "none" : kBackendNames[g_jb.backend];
}

extern "C" int vti_decode_jpeg_batch(vti_handle* h, const uint8_t* const* jpegs, const long long* nbytes, int n, uint8_t* frames,
                                     void* stream) {
    if (!h || !jpegs || !nbytes || !frames || n <= 0 || n > h->p.max_batch) {
        vti_set_error("vti_decode_jpeg_batch: bad argument (1 <= n <= max_batch)");
        return VTI_EINVAL;
    }
    std::lock_guard<std::mutex> lock(g_jb.mu);
    cudaStream_t s = (cudaStream_t)stream;
    int device = 0;
    VTI_CUDA(cudaGetDevice(&device));
    const size_t frame_bytes = (size_t)h->p.frame_h * h->p.frame_w * 3;
    std::vector<size_t> len(n);
    std::vector<nvjpegImage_t> dst(n);
    for (int i = 0; i < n; ++i) {
        if (!jpegs[i] || nbytes[i] <= 0) { vti_set_error("vti_decode_jpeg_batch: empty stream in the batch"); return VTI_EINVAL; }
        len[i] = (size_t)nbytes[i];
        std::memset(&dst[i], 0, sizeof(nvjpegImage_t));
        dst[i].channel[0] = frames + (size_t)i * frame_bytes;
        dst[i].pitch[0] = (size_t)h->p.frame_w * 3;
    }
    // geometry check on every stream header (nvjpegGetImageInfo only parses the markers)
    {
        if (!g_jb.probe && nvjpegCreateSimple(&g_jb.probe) != NVJPEG_STATUS_SUCCESS) {
            g_jb.probe = nullptr;
            vti_set_error("vti_decode_jpeg_batch: nvJPEG initialisation failed");
            return VTI_ECUDA;
        }
        nvjpegHandle_t probe = g_jb.probe;
        for (int i = 0; i < n; ++i) {
            int nc = 0, widths[NVJPEG_MAX_COMPONENT], heights[NVJPEG_MAX_COMPONENT];
            nvjpegChromaSubsampling_t css;
            if (nvjpegGetImageInfo(probe, jpegs[i], len[i], &nc, &css, widths, heights) != NVJPEG_STATUS_SUCCESS) {
                vti_set_error("vti_decode_jpeg_batch: stream " + std::to_string(i) + " is not a JPEG nvJPEG can parse");
                return VTI_EINVAL;
            }
            if (widths[0] != h->p.frame_w || heights[0] != h->p.frame_h) {
                vti_set_error("vti_decode_jpeg_batch: image " + std::to_string(i) + " is " + std::to_string(widths[0]) + "x" +
                              std::to_string(heights[0]) + ", the handle was created for " + std::to_string(h->p.frame_w) + "x" +
                              std::to_string(h->p.frame_h));
                return VTI_EINVAL;
            }
        }
    }
    const char* force = std::getenv("VTI_JPEG_BACKEND");      // "hardware" | "gpu" | "hybrid": measurement aid
    int first = 0;
    if (force) first = !std::strcmp(force, "gpu") ? 1 : (!std::strcmp(force, "hybrid") ? 2 : 0);
    const char* lanes_env = std::getenv("VTI_JPEG_LANES");
    int lanes = lanes_env ? std::atoi(lanes_env) : 8;      // measured on the 16-core B200 host: 1 / 2 / 4 / 8 lanes = 1.31 / 0.69 / 1.18 / 1.79 k frames/s
    lanes = std::max(1, std::min(std::min(lanes, JB_MAX_LANES), n / 4 > 0 ? n / 4 : 1));      // at least 4 images per lane
    // the decoded frames must not overtake work already queued on the caller's stream that still reads the buffer
    cudaEvent_t ready;
    VTI_CUDA(cudaEventCreateWithFlags(&ready, cudaEventDisableTiming));
    VTI_CUDA(cudaEventRecord(ready, s));
    for (int idx = g_jb.backend >= first ? g_jb.backend : first; idx < 3; ++idx) {
        bool ok[JB_MAX_LANES];
        std::vector<std::thread> th;
        for (int l = 0; l < lanes; ++l) {
            const int i0 = (int)((long long)n * l / lanes), i1 = (int)((long long)n * (l + 1) / lanes);
            auto work = [&, l, i0, i1]() {
                ok[l] = false;
                if (cudaSetDevice(device) != cudaSuccess || !g_jb.lane[l].on_device(device)) return;
                if (cudaStreamWaitEvent(g_jb.lane[l].stream, ready, 0) != cudaSuccess) return;
                ok[l] = jb_lane_decode(g_jb.lane[l], idx, device, jpegs, len.data(), dst.data(), i0, i1);
            };
            if (lanes == 1) work(); else th.emplace_back(work);
        }
        for (auto& t : th) t.join();
        bool all = true;
        for (int l = 0; l < lanes; ++l) all = all && ok[l];
        if (all) {
            for (int l = 0; l < lanes; ++l) VTI_CUDA(cudaStreamWaitEvent(s, g_jb.lane[l].done, 0));
            cudaEventDestroy(ready);
            g_jb.backend = idx;
            return VTI_OK;
        }
        for (int l = 0; l < lanes; ++l) {              // a lane that did start must finish before the buffers are reused
            if (g_jb.lane[l].stream) cudaStreamSynchronize(g_jb.lane[l].stream);
            g_jb.lane[l].release();
        }
        cudaGetLastError();
    }
    cudaEventDestroy(ready);
    g_jb.backend = -1;
    vti_set_error("vti_decode_jpeg_batch: no nvJPEG backend decoded the batch");
    return VTI_ECUDA;
}

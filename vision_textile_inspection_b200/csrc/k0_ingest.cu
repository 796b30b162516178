// K0 -- camera-native frame ingest: packed YUV 4:2:2 (YUYV / "YUY2", 2 bytes per pixel) -> BGR u8, bit-exact against
// cv2.cvtColor(.., COLOR_YUV2BGR_YUY2).
//
// Replaces (SURVEY.md 8f rank 2): the colour conversion inside cv2.VideoCapture.read() -- main.py:188
// `ret, frame = measurement_app.cap.read()`; the reference opens the camera without a FOURCC
// (measurement.py:22-38), so OpenCV's V4L2 backend negotiates YUYV before MJPEG and converts every frame
// to BGR on the CPU before process_frame sees it.  Here the frame crosses PCIe as the camera delivered it (2/3 of the
// BGR bytes) and is converted on the device, in front of K1.
// Spec: oracle/cv_fixed.py yuyv_to_bgr (OpenCV's ITU-R BT.601 fixed-point form, 20 fractional bits):
//   y' = max(0, Y - 16) * 1220542;  u = U - 128;  v = V - 128
//   B = sat8((y' + 2116026 u + 2^19) >> 20)
//   G = sat8((y' -  409993 u - 852492 v + 2^19) >> 20)
//   R = sat8((y' + 1673527 v + 2^19) >> 20)
// Bound: HBM, 2 bytes read + 3 bytes written per pixel.
#include <algorithm>

#include "vti_internal.h"

namespace {

constexpr int K0_THREADS = 256;
constexpr int CY = 1220542, CUB = 2116026, CUG = -409993, CVG = -852492, CVR = 1673527, SHIFT = 20;

__device__ __forceinline__ unsigned sat8(int v) { return (unsigned)min(max(v, 0), 255); }

// the three colour terms of a chroma pair, shared by its two pixels
struct Chroma { int b, g, r; };
__device__ __forceinline__ Chroma chroma(unsigned U, unsigned V) {
    const int u = (int)U - 128, v = (int)V - 128;
    Chroma c;
    c.b = (1 << (SHIFT - 1)) + CUB * u;
    c.g = (1 << (SHIFT - 1)) + CVG * v + CUG * u;
    c.r = (1 << (SHIFT - 1)) + CVR * v;
    return c;
}
// one pixel -> B | G << 8 | R << 16
__device__ __forceinline__ unsigned pixel(unsigned Y, const Chroma& c) {
    const int y = max(0, (int)Y - 16) * CY;
    return sat8((y + c.b) >> SHIFT) | (sat8((y + c.g) >> SHIFT) << 8) | (sat8((y + c.r) >> SHIFT) << 16);
}

// 4 pixels per thread: one 8-byte load (Y0 U0 Y1 V0 Y2 U1 Y3 V1), three 4-byte stores (12 BGR bytes)
__global__ void __launch_bounds__(K0_THREADS) k0_yuyv4_kernel(const uint2* __restrict__ src, unsigned* __restrict__ dst, size_t nquads) {
    for (size_t i = (size_t)blockIdx.x * K0_THREADS + threadIdx.x; i < nquads; i += (size_t)gridDim.x * K0_THREADS) {
        const uint2 q = __ldg(src + i);
        const Chroma c0 = chroma((q.x >> 8) & 255u, q.x >> 24), c1 = chroma((q.y >> 8) & 255u, q.y >> 24);
        const unsigned p0 = pixel(q.x & 255u, c0), p1 = pixel((q.x >> 16) & 255u, c0);
        const unsigned p2 = pixel(q.y & 255u, c1), p3 = pixel((q.y >> 16) & 255u, c1);
        unsigned* o = dst + 3 * i;
        o[0] = p0 | (p1 << 24);
        o[1] = (p1 >> 8) | (p2 << 16);
        o[2] = (p2 >> 16) | (p3 << 8);
    }
}

// 2 pixels per thread (any even width): one 4-byte load, six byte stores
__global__ void __launch_bounds__(K0_THREADS) k0_yuyv2_kernel(const unsigned* __restrict__ src, uint8_t* __restrict__ dst, size_t npairs) {
    for (size_t i = (size_t)blockIdx.x * K0_THREADS + threadIdx.x; i < npairs; i += (size_t)gridDim.x * K0_THREADS) {
        const unsigned q = __ldg(src + i);
        const Chroma c = chroma((q >> 8) & 255u, q >> 24);
        const unsigned p0 = pixel(q & 255u, c), p1 = pixel((q >> 16) & 255u, c);
        uint8_t* o = dst + 6 * i;
        o[0] = (uint8_t)p0; o[1] = (uint8_t)(p0 >> 8); o[2] = (uint8_t)(p0 >> 16);
        o[3] = (uint8_t)p1; o[4] = (uint8_t)(p1 >> 8); o[5] = (uint8_t)(p1 >> 16);
    }
}

}  // namespace

int vti_launch_k0_yuyv(vti_handle* h, const uint8_t* yuyv, int B, uint8_t* frames, cudaStream_t s) {
    const size_t npx = (size_t)B * h->p.frame_h * h->p.frame_w;
    const bool quad = (npx % 4 == 0) && ((reinterpret_cast<uintptr_t>(yuyv) & 7) == 0) && ((reinterpret_cast<uintptr_t>(frames) & 3) == 0);
    const size_t items = quad ? npx / 4 : npx / 2;
    const size_t want = (items + K0_THREADS - 1) / K0_THREADS;
    const int grid = (int)std::min<size_t>(want, (size_t)h->num_sms * 8 * 4);      // 8 resident CTAs per SM, 4 waves at most: grid-stride beyond
    if (grid <= 0) return VTI_OK;
    if (quad) k0_yuyv4_kernel<<<grid, K0_THREADS, 0, s>>>(reinterpret_cast<const uint2*>(yuyv), reinterpret_cast<unsigned*>(frames), items);
    else k0_yuyv2_kernel<<<grid, K0_THREADS, 0, s>>>(reinterpret_cast<const unsigned*>(yuyv), frames, items);
    h->launches += 1;
    VTI_CUDA(cudaGetLastError());
    return VTI_OK;
}

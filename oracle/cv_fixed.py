"""TEST INFRASTRUCTURE ONLY -- numpy restatement of the OpenCV fixed-point image ops on the hot path.

This file is part of the CPU oracle.  Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
--impl reference legs may import it.  The product (vision_textile_inspection_b200) never does.

What is restated (SURVEY.md section 8a rows U0/U1/M2; the arithmetic lives in OpenCV, which the reference
pins as opencv-contrib-python==4.11.0.86 in requirements.txt:2 and reaches through
ultralytics LetterBox (measurement.py:208-210) and cv2.resize(INTER_NEAREST) (measurement.py:78-79)):

  * cv2.resize(..., INTER_LINEAR) on uint8: 11-bit coefficients, H pass then V pass
  * cv2.resize(..., INTER_NEAREST): index map
  * cv2.undistort: double-precision forward distortion map, 5 fractional bits, 15-bit bilinear weights

Every function here is pinned against the real cv2 in tests/test_oracle_cv.py (bit-exact), so this file is the
*kernel specification* for the CUDA path: integer formulas only, no library call.
"""
from __future__ import annotations

import numpy as np

INTER_RESIZE_COEF_BITS = 11
INTER_RESIZE_COEF_SCALE = 1 << INTER_RESIZE_COEF_BITS
INTER_BITS = 5
INTER_TAB_SIZE = 1 << INTER_BITS
INTER_REMAP_COEF_BITS = 15


def py_round(x: float) -> int:
    """Python round(): half to even (ultralytics uses the builtin on floats)."""
    return int(round(x))


def letterbox_geometry(h: int, w: int, imgsz: int = 960, stride: int = 32):
    """Ultralytics LetterBox(auto=True, scaleup=True, center=True) geometry [upstream; SURVEY 8a U1].

    Returns dict(new_w, new_h, top, bottom, left, right, LH, LW).
    """
    r = min(imgsz / h, imgsz / w)
    new_w, new_h = py_round(w * r), py_round(h * r)
    dw, dh = imgsz - new_w, imgsz - new_h
    dw, dh = dw % stride, dh % stride
    dw /= 2
    dh /= 2
    top, bottom = py_round(dh - 0.1), py_round(dh + 0.1)
    left, right = py_round(dw - 0.1), py_round(dw + 0.1)
    return dict(new_w=new_w, new_h=new_h, top=top, bottom=bottom, left=left, right=right,
                LH=new_h + top + bottom, LW=new_w + left + right)


def linear_taps_x(sn: int, dn: int):
    """Horizontal taps of cv2.resize INTER_LINEAR: (idx, a0, a1); index AND fraction clamp at borders."""
    scale = 1.0 / (dn / sn)
    d = np.arange(dn, dtype=np.float64)
    f = ((d + 0.5) * scale - 0.5).astype(np.float32)
    s = np.floor(f).astype(np.int64)
    f = (f - s.astype(np.float32)).astype(np.float32)
    lo = s < 0
    f[lo] = 0.0
    s[lo] = 0
    hi = s >= sn - 1
    f[hi] = 0.0
    s[hi] = sn - 1
    a0 = np.rint((np.float32(1.0) - f) * np.float32(INTER_RESIZE_COEF_SCALE)).astype(np.int32)
    a1 = np.rint(f * np.float32(INTER_RESIZE_COEF_SCALE)).astype(np.int32)
    return s.astype(np.int32), a0, a1


def linear_taps_y(sn: int, dn: int):
    """Vertical taps: (idx0, idx1, b0, b1); only the two row indices clamp, the fraction is kept."""
    scale = 1.0 / (dn / sn)
    d = np.arange(dn, dtype=np.float64)
    f = ((d + 0.5) * scale - 0.5).astype(np.float32)
    s = np.floor(f).astype(np.int64)
    f = (f - s.astype(np.float32)).astype(np.float32)
    i0 = np.clip(s, 0, sn - 1).astype(np.int32)
    i1 = np.clip(s + 1, 0, sn - 1).astype(np.int32)
    b0 = np.rint((np.float32(1.0) - f) * np.float32(INTER_RESIZE_COEF_SCALE)).astype(np.int32)
    b1 = np.rint(f * np.float32(INTER_RESIZE_COEF_SCALE)).astype(np.int32)
    return i0, i1, b0, b1


def resize_linear_u8(img: np.ndarray, dw: int, dh: int) -> np.ndarray:
    """Bit-exact cv2.resize(img, (dw, dh), interpolation=cv2.INTER_LINEAR) for uint8 HxWxC."""
    sh, sw = img.shape[:2]
    if (sw, sh) == (dw, dh):
        return img.copy()
    src = img.astype(np.int32)
    if sw == 2 * dw and sh == 2 * dh:
        # OpenCV silently switches an exact 2x INTER_LINEAR shrink to the INTER_AREA fast path
        s = src[0::2, 0::2] + src[0::2, 1::2] + src[1::2, 0::2] + src[1::2, 1::2]
        return ((s + 2) >> 2).astype(np.uint8)
    ix, a0, a1 = linear_taps_x(sw, dw)
    iy0, iy1, b0, b1 = linear_taps_y(sh, dh)
    ix1 = np.minimum(ix + 1, sw - 1)
    a0 = a0.reshape(1, -1, 1)
    a1 = a1.reshape(1, -1, 1)
    hrow = src[:, ix] * a0 + src[:, ix1] * a1          # (sh, dw, C) int32, scale 2^11
    s0 = hrow[iy0] >> 4
    s1 = hrow[iy1] >> 4
    b0 = b0.reshape(-1, 1, 1)
    b1 = b1.reshape(-1, 1, 1)
    out = (((b0 * s0) >> 16) + ((b1 * s1) >> 16) + 2) >> 2
    return np.clip(out, 0, 255).astype(np.uint8)


def nearest_map(dst_n: int, src_n: int) -> np.ndarray:
    """cv2.resize INTER_NEAREST source index per destination index (measurement.py:78-79 path).

    Note the double reciprocal: OpenCV computes ifx = 1/(dst/src) and floor(d*ifx)."""
    ifx = 1.0 / (dst_n / src_n)
    d = np.arange(dst_n, dtype=np.float64)
    return np.minimum(np.floor(d * ifx).astype(np.int64), src_n - 1).astype(np.int32)


def undistort_map_fixed(K: np.ndarray, dist: np.ndarray, h: int, w: int):
    """cv2.undistort(frame, K, dist) source map in 1/32 px: (ix, iy) int32 arrays of shape (h, w).

    Follows initUndistortRectifyMap with R=I, newCameraMatrix=K (double precision), then
    rint(map * 32) (saturate_cast<int> = round half to even)."""
    K = np.asarray(K, np.float64)
    k1, k2, p1, p2, k3 = [float(v) for v in np.asarray(dist, np.float64).ravel()[:5]]
    fx, fy, cx, cy = K[0, 0], K[1, 1], K[0, 2], K[1, 2]
    u = np.arange(w, dtype=np.float64)[None, :]
    v = np.arange(h, dtype=np.float64)[:, None]
    x = (u - cx) / fx + 0.0 * v
    y = (v - cy) / fy + 0.0 * u
    x2, y2 = x * x, y * y
    r2 = x2 + y2
    _2xy = 2.0 * x * y
    kr = 1.0 + ((k3 * r2 + k2) * r2 + k1) * r2
    xd = x * kr + p1 * _2xy + p2 * (r2 + 2.0 * x2)
    yd = y * kr + p1 * (r2 + 2.0 * y2) + p2 * _2xy
    mx = fx * xd + cx
    my = fy * yd + cy
    ix = np.rint(mx * INTER_TAB_SIZE).astype(np.int64)
    iy = np.rint(my * INTER_TAB_SIZE).astype(np.int64)
    return ix.astype(np.int32), iy.astype(np.int32)


def remap_bilinear_u8(img: np.ndarray, ix: np.ndarray, iy: np.ndarray) -> np.ndarray:
    """cv2.remap(INTER_LINEAR, BORDER_CONSTANT=0) with the fixed-point maps above; bit-exact for uint8."""
    sh, sw = img.shape[:2]
    sx = ix >> INTER_BITS
    sy = iy >> INTER_BITS
    fx = (ix & (INTER_TAB_SIZE - 1)).astype(np.int64)
    fy = (iy & (INTER_TAB_SIZE - 1)).astype(np.int64)
    # weights at scale 2^15: (32-fx)(32-fy)*32 etc. -- exact integers, always sum to 32768
    w00 = (INTER_TAB_SIZE - fx) * (INTER_TAB_SIZE - fy) * 32
    w01 = fx * (INTER_TAB_SIZE - fy) * 32
    w10 = (INTER_TAB_SIZE - fx) * fy * 32
    w11 = fx * fy * 32
    src = img.astype(np.int64)

    def tap(yy, xx):
        ok = (yy >= 0) & (yy < sh) & (xx >= 0) & (xx < sw)
        v = src[np.clip(yy, 0, sh - 1), np.clip(xx, 0, sw - 1)]
        return v * ok[..., None]

    acc = (tap(sy, sx) * w00[..., None] + tap(sy, sx + 1) * w01[..., None]
           + tap(sy + 1, sx) * w10[..., None] + tap(sy + 1, sx + 1) * w11[..., None])
    out = (acc + (1 << (INTER_REMAP_COEF_BITS - 1))) >> INTER_REMAP_COEF_BITS
    return np.clip(out, 0, 255).astype(np.uint8)


def undistort_u8(img: np.ndarray, K, dist) -> np.ndarray:
    h, w = img.shape[:2]
    ix, iy = undistort_map_fixed(K, dist, h, w)
    return remap_bilinear_u8(img, ix, iy)


def scale_K(K, w: int, h: int, calib_w: int = 1280, calib_h: int = 960) -> np.ndarray:
    """Intrinsics for a frame size other than the calibration size (SURVEY 7 'Frame sizes != calibration size')."""
    S = np.diag([w / calib_w, h / calib_h, 1.0])
    return S @ np.asarray(K, np.float64)


# ---- camera-native ingest: packed YUV 4:2:2 -> BGR (OpenCV modules/imgproc/src/color_yuv.simd.hpp, YUV422toRGB8Invoker /
# uvToRGBuv / yRGBuvToRGBA with the ITU-R BT.601 constants below; what cv2.VideoCapture.read() applies to a YUYV camera
# stream before main.py:188 hands the frame to process_frame).  Pinned in tests/test_oracle_cv.py against
# cv2.cvtColor(.., COLOR_YUV2BGR_YUY2) over every (Y, U, V) triple.
ITUR_BT_601_CY, ITUR_BT_601_CUB, ITUR_BT_601_CUG = 1220542, 2116026, -409993
ITUR_BT_601_CVG, ITUR_BT_601_CVR, ITUR_BT_601_SHIFT = -852492, 1673527, 20


def yuyv_to_bgr(yuyv: np.ndarray) -> np.ndarray:
    """(h, w, 2) uint8 packed Y0 U Y1 V -> (h, w, 3) uint8 BGR, bit-exact cv2.cvtColor(yuyv, cv2.COLOR_YUV2BGR_YUY2)."""
    assert yuyv.dtype == np.uint8 and yuyv.ndim == 3 and yuyv.shape[2] == 2 and yuyv.shape[1] % 2 == 0
    y = yuyv[:, :, 0].astype(np.int64)
    u = np.repeat(yuyv[:, 0::2, 1].astype(np.int64), 2, axis=1) - 128
    v = np.repeat(yuyv[:, 1::2, 1].astype(np.int64), 2, axis=1) - 128
    half = 1 << (ITUR_BT_601_SHIFT - 1)
    yy = np.maximum(0, y - 16) * ITUR_BT_601_CY
    b = (yy + half + ITUR_BT_601_CUB * u) >> ITUR_BT_601_SHIFT
    g = (yy + half + ITUR_BT_601_CVG * v + ITUR_BT_601_CUG * u) >> ITUR_BT_601_SHIFT
    r = (yy + half + ITUR_BT_601_CVR * v) >> ITUR_BT_601_SHIFT
    return np.clip(np.stack([b, g, r], -1), 0, 255).astype(np.uint8)

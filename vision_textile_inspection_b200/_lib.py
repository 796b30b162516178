"""ctypes binding of libvti.so (include/vti.h).  No fallback: if the library is missing it is built with nvcc, and if
that fails the import of the product path fails loudly."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("VTI_LIB", os.path.join(HERE, "libvti.so"))

VTI_NM = 32
F_IN_ROI, F_STITCH, F_FABRIC, F_HAS_MASK, F_SELECTED, F_FINAL, F_HAS_WIDTH, F_HAS_DIST = 1, 2, 4, 8, 16, 32, 64, 128
F_LB_MASK, F_DROPPED = 256, 512
ST_OK, ST_NO_FABRIC, ST_NO_STITCH, ST_OVERFLOW = 0, 2, 3, 0x100
ST_BAD_CAMERA = 0x200
MAX_CAMERAS = 256


class VtiParams(C.Structure):
    _fields_ = [
        ("struct_size", C.c_int32), ("frame_h", C.c_int32), ("frame_w", C.c_int32), ("imgsz", C.c_int32),
        ("stride", C.c_int32), ("nc", C.c_int32), ("max_det", C.c_int32), ("max_batch", C.c_int32),
        ("variant", C.c_int32), ("undistort", C.c_int32), ("channel_flip", C.c_int32), ("stitch_id", C.c_int32),
        ("fabric_id", C.c_int32), ("roi_enabled", C.c_int32), ("roi_x_min", C.c_int32), ("roi_x_max", C.c_int32),
        ("roi_y_min", C.c_int32), ("roi_y_max", C.c_int32), ("min_stitches", C.c_int32),
        ("max_px_distance", C.c_int32), ("neighborhood", C.c_int32), ("max_candidates", C.c_int32),
        ("conf", C.c_float), ("iou", C.c_float),
        ("K", C.c_double * 9), ("dist", C.c_double * 5), ("R", C.c_double * 9), ("t", C.c_double * 3),
        ("iou_threshold", C.c_double), ("mask_variant", C.c_int32),
    ]


class VtiCamera(C.Structure):
    _fields_ = [
        ("struct_size", C.c_int32), ("reserved", C.c_int32),
        ("K", C.c_double * 9), ("dist", C.c_double * 5), ("R", C.c_double * 9), ("t", C.c_double * 3),
    ]


class VtiGeometry(C.Structure):
    _fields_ = [
        ("new_h", C.c_int32), ("new_w", C.c_int32), ("top", C.c_int32), ("bottom", C.c_int32), ("left", C.c_int32),
        ("right", C.c_int32), ("LH", C.c_int32), ("LW", C.c_int32), ("ph", C.c_int32), ("pw", C.c_int32),
        ("lvl_h", C.c_int32 * 3), ("lvl_w", C.c_int32 * 3), ("A", C.c_int32), ("mask_words", C.c_int32),
        ("max_candidates", C.c_int32), ("max_det", C.c_int32),
    ]


# numpy mirrors of vti_det (160 B) and vti_frame_result (56 B)
DET_DTYPE = np.dtype([
    ("box_lb", "<f4", 4), ("box_frame", "<f4", 4), ("box_int", "<i4", 4), ("conf", "<f4"), ("cls", "<i4"),
    ("anchor", "<i4"), ("flags", "<u4"), ("m00", "<i8"), ("m10", "<i8"), ("m01", "<i8"), ("col_min", "<i4"),
    ("col_max", "<i4"), ("cx", "<f8"), ("cy", "<f8"), ("left_px", "<f8"), ("right_px", "<f8"), ("width_mm", "<f8"),
    ("edge_y", "<f8"), ("dist_mm", "<f8"), ("area_mm2", "<f8"),
])
RESULT_DTYPE = np.dtype([
    ("status", "<i4"), ("n_det", "<i4"), ("n_cand", "<i4"), ("n_stitch", "<i4"), ("n_fabric", "<i4"),
    ("n_dist", "<i4"), ("n_width", "<i4"), ("env_valid", "<i4"), ("avg_dist", "<f8"), ("avg_width", "<f8"),
    ("env_mean", "<f8"),
])
assert DET_DTYPE.itemsize == 160 and RESULT_DTYPE.itemsize == 56

EXPORTS = [
    "vti_last_error", "vti_abi_version", "vti_plan_geometry", "vti_plan_resize_taps_x", "vti_plan_resize_taps_y",
    "vti_plan_undistort_map", "vti_plan_nearest_map", "vti_create", "vti_destroy", "vti_get_geometry",
    "vti_preprocess", "vti_postprocess", "vti_measure", "vti_post_measure", "vti_process_host", "vti_launch_count",
    "vti_set_profiling", "vti_get_stage_ms", "vti_annotate", "vti_draw_text", "vti_encode_jpeg", "vti_decode_jpeg",
    "vti_decode_jpeg_batch", "vti_jpeg_backend", "vti_ingest_yuyv", "vti_process_host_yuyv",
    "vti_create_multi", "vti_camera_count", "vti_preprocess_multi", "vti_measure_multi", "vti_post_measure_multi",
    "vti_process_host_multi", "vti_process_host_yuyv_multi",
]

_lib = None


def load():
    """dlopen libvti.so (building it first if the sources are newer).  Raises if it cannot be had."""
    global _lib
    if _lib is not None:
        return _lib
    from . import build
    if not os.environ.get("VTI_NO_BUILD") and build.needs_build():   # (VTI_NO_BUILD: tuning sweeps load prebuilt variants)
        build.build_lib()
    lib = C.CDLL(LIB_PATH)
    vp, i32, i64 = C.c_void_p, C.c_int, C.c_int64
    lib.vti_last_error.restype = C.c_char_p
    lib.vti_abi_version.restype = i32
    lib.vti_plan_geometry.argtypes = [i32, i32, i32, i32, i32, i32, C.POINTER(VtiGeometry)]
    lib.vti_plan_resize_taps_x.argtypes = [i32, i32, vp, vp, vp]
    lib.vti_plan_resize_taps_y.argtypes = [i32, i32, vp, vp, vp, vp]
    lib.vti_plan_undistort_map.argtypes = [vp, vp, i32, i32, vp, vp]
    lib.vti_plan_nearest_map.argtypes = [i32, i32, vp]
    lib.vti_create.argtypes = [C.POINTER(VtiParams), C.POINTER(vp)]
    lib.vti_destroy.argtypes = [vp]
    lib.vti_destroy.restype = None
    lib.vti_get_geometry.argtypes = [vp, C.POINTER(VtiGeometry)]
    lib.vti_preprocess.argtypes = [vp, vp, i32, vp, vp]
    lib.vti_postprocess.argtypes = [vp, vp, vp, vp, vp, vp, i32, vp, vp, vp, vp]
    lib.vti_measure.argtypes = [vp, i32, vp, vp, vp, vp]
    lib.vti_post_measure.argtypes = [vp, vp, vp, vp, vp, vp, i32, vp, vp, vp, vp, vp]
    lib.vti_process_host.argtypes = [vp, vp, vp, vp, vp, vp, vp, i32, vp, vp, vp, vp]
    lib.vti_process_host_yuyv.argtypes = [vp, vp, vp, vp, vp, vp, vp, i32, vp, vp, vp, vp]
    lib.vti_ingest_yuyv.argtypes = [vp, vp, i32, vp, vp]
    lib.vti_launch_count.argtypes = [vp]
    lib.vti_launch_count.restype = i64
    lib.vti_set_profiling.argtypes = [vp, i32]
    lib.vti_get_stage_ms.argtypes = [vp, vp]
    lib.vti_annotate.argtypes = [vp, vp, i32, vp, vp, vp, vp]
    lib.vti_draw_text.argtypes = [vp, vp, i32, i32, i32, C.c_char_p, i32, i32, i32, i32, vp]
    lib.vti_encode_jpeg.argtypes = [vp, vp, i32, vp, i64, vp]
    lib.vti_encode_jpeg.restype = i64
    lib.vti_decode_jpeg.argtypes = [vp, C.c_char_p, i64, vp, vp]
    lib.vti_decode_jpeg_batch.argtypes = [vp, C.POINTER(C.c_char_p), C.POINTER(i64), i32, vp, vp]
    lib.vti_jpeg_backend.argtypes = []
    lib.vti_jpeg_backend.restype = C.c_char_p
    lib.vti_create_multi.argtypes = [C.POINTER(VtiParams), i32, C.POINTER(VtiCamera), C.POINTER(vp)]
    lib.vti_camera_count.argtypes = [vp]
    lib.vti_preprocess_multi.argtypes = [vp, vp, vp, i32, vp, vp]
    lib.vti_measure_multi.argtypes = [vp, i32, vp, vp, vp, vp, vp]
    lib.vti_post_measure_multi.argtypes = [vp, vp, vp, vp, vp, vp, i32, vp, vp, vp, vp, vp, vp]
    lib.vti_process_host_multi.argtypes = [vp, vp, vp, vp, vp, vp, vp, i32, vp, vp, vp, vp, vp]
    lib.vti_process_host_yuyv_multi.argtypes = [vp, vp, vp, vp, vp, vp, vp, i32, vp, vp, vp, vp, vp]
    for name in EXPORTS:
        getattr(lib, name)
    _lib = lib
    return lib


class VtiError(RuntimeError):
    pass


def check(rc: int, what: str):
    if rc != 0:
        raise VtiError(f"{what} failed ({rc}): {load().vti_last_error().decode()}")


def plan_geometry(frame_h, frame_w, imgsz, stride=32, max_det=200, max_candidates=0) -> VtiGeometry:
    g = VtiGeometry()
    check(load().vti_plan_geometry(frame_h, frame_w, imgsz, stride, max_det, max_candidates, C.byref(g)),
          "vti_plan_geometry")
    return g

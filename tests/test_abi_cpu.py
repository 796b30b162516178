"""No-GPU checks of the C-ABI library: it loads, exports every symbol include/vti.h declares, its host-side planning
(letterbox geometry, cv2 resize taps, undistort map, nearest maps) equals the oracle, and it refuses to run
without a CUDA device instead of falling back."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

from oracle import cv_fixed
from vision_textile_inspection_b200 import _lib, synth
from vision_textile_inspection_b200.engine import EngineConfig, InspectionEngine

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_exports_match_header():
    lib = _lib.load()
    hdr = open(os.path.join(ROOT, "include", "vti.h")).read()
    declared = set(re.findall(r"\b(vti_[a-z0-9_]+)\s*\(", hdr))
    assert declared == set(_lib.EXPORTS)
    for name in declared:
        assert getattr(lib, name) is not None
    assert lib.vti_abi_version() == 1


def test_struct_sizes_match_header():
    # 22 int32 + conf, iou + K, dist, R, t, iou_threshold doubles + mask_variant; the last 4 bytes are padding (the
    # struct is 8-byte aligned), so callers built when a second int32 followed mask_variant pass the same struct_size
    assert C.sizeof(_lib.VtiParams) == 22 * 4 + 2 * 4 + (9 + 5 + 9 + 3 + 1) * 8 + 4 + 4
    assert _lib.DET_DTYPE.itemsize == 160


@pytest.mark.parametrize("h,w,S", [(640, 640, 960), (960, 1280, 960), (720, 1280, 960), (1080, 1920, 640),
                                   (2160, 3840, 960), (1080, 1920, 960), (123, 457, 960), (640, 640, 640)])
def test_plan_geometry_and_taps(h, w, S):
    g = _lib.plan_geometry(h, w, S)
    o = cv_fixed.letterbox_geometry(h, w, S)
    assert (g.new_w, g.new_h, g.top, g.bottom, g.left, g.right, g.LH, g.LW) == (
        o["new_w"], o["new_h"], o["top"], o["bottom"], o["left"], o["right"], o["LH"], o["LW"])
    assert g.A == sum((g.LH // s) * (g.LW // s) for s in (8, 16, 32))
    lib = _lib.load()
    for sn, dn in ((w, g.new_w), (h, g.new_h)):
        idx = np.zeros(dn, np.int32); a0 = np.zeros(dn, np.int16); a1 = np.zeros(dn, np.int16)
        lib.vti_plan_resize_taps_x(sn, dn, idx.ctypes.data, a0.ctypes.data, a1.ctypes.data)
        ri, ra0, ra1 = cv_fixed.linear_taps_x(sn, dn)
        assert np.array_equal(idx, ri) and np.array_equal(a0, ra0) and np.array_equal(a1, ra1)
        i0 = np.zeros(dn, np.int32); i1 = np.zeros(dn, np.int32); b0 = np.zeros(dn, np.int16); b1 = np.zeros(dn, np.int16)
        lib.vti_plan_resize_taps_y(sn, dn, i0.ctypes.data, i1.ctypes.data, b0.ctypes.data, b1.ctypes.data)
        r0, r1, rb0, rb1 = cv_fixed.linear_taps_y(sn, dn)
        assert np.array_equal(i0, r0) and np.array_equal(i1, r1) and np.array_equal(b0, rb0) and np.array_equal(b1, rb1)
    for dst, src in ((h, g.LH), (w, g.LW)):
        m = np.zeros(dst, np.int32)
        lib.vti_plan_nearest_map(dst, src, m.ctypes.data)
        assert np.array_equal(m, cv_fixed.nearest_map(dst, src))


@pytest.mark.parametrize("h,w", [(960, 1280), (720, 1280), (1080, 1920)])
def test_plan_undistort_map_equals_opencv_spec(h, w, calib):
    K = cv_fixed.scale_K(np.array(calib["camera_matrix"]), w, h)
    dist = np.array(calib["dist_coeffs"], np.float64)
    ix = np.zeros((h, w), np.int32); iy = np.zeros((h, w), np.int32)
    Kc = np.ascontiguousarray(K.reshape(9))
    _lib.load().vti_plan_undistort_map(Kc.ctypes.data, dist.ctypes.data, h, w, ix.ctypes.data, iy.ctypes.data)
    rx, ry = cv_fixed.undistort_map_fixed(K, dist, h, w)          # pinned bit-exact vs cv2.undistort elsewhere
    assert np.array_equal(ix, rx) and np.array_equal(iy, ry)


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_no_cpu_fallback():
    cfg = synth.CONFIGS["cfg2"]
    with pytest.raises(_lib.VtiError):
        InspectionEngine(EngineConfig.for_workload(cfg, max_batch=1))
    p = EngineConfig.for_workload(cfg, max_batch=1).to_params()
    h = C.c_void_p()
    rc = _lib.load().vti_create(C.byref(p), C.byref(h))
    assert rc == -4 and b"no CPU fallback" in _lib.load().vti_last_error()


def test_bad_params_rejected():
    p = EngineConfig.for_workload(synth.CONFIGS["cfg2"], max_batch=1).to_params()
    p.struct_size = 12
    h = C.c_void_p()
    assert _lib.load().vti_create(C.byref(p), C.byref(h)) == -1

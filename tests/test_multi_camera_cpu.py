"""The multi-camera C ABI without a GPU: the vti_camera layout, the exports, the argument checks of vti_create_multi
(made before the device check) and the conversion of EngineConfig.cameras."""
import ctypes as C
import json

import numpy as np
import pytest

import helpers
from vision_textile_inspection_b200 import _lib
from vision_textile_inspection_b200 import app as A
from vision_textile_inspection_b200 import synth
from vision_textile_inspection_b200.engine import EngineConfig

NEW_SYMBOLS = ["vti_create_multi", "vti_camera_count", "vti_preprocess_multi", "vti_measure_multi",
               "vti_post_measure_multi", "vti_process_host_multi", "vti_process_host_yuyv_multi"]


def test_camera_struct_layout():
    assert C.sizeof(_lib.VtiCamera) == 216
    off = {name: getattr(_lib.VtiCamera, name).offset for name, _ in _lib.VtiCamera._fields_}
    assert off == {"struct_size": 0, "reserved": 4, "K": 8, "dist": 80, "R": 120, "t": 192}
    assert _lib.ST_BAD_CAMERA == 0x200 and _lib.MAX_CAMERAS == 256


def test_new_symbols_are_exported():
    lib = _lib.load()
    for name in NEW_SYMBOLS:
        assert name in _lib.EXPORTS
        assert getattr(lib, name) is not None
    assert lib.vti_camera_count(None) == -1


def cameras(n, struct_size=None):
    arr = (_lib.VtiCamera * n)()
    calib = helpers.load_calib()
    for c in arr:
        c.struct_size = C.sizeof(_lib.VtiCamera) if struct_size is None else struct_size
        c.K[:] = np.asarray(calib["camera_matrix"], np.float64).reshape(9).tolist()
        c.dist[:] = calib["dist_coeffs"]
        c.R[:] = np.eye(3).reshape(9).tolist()
        c.t[:] = [0.0, 0.0, 0.5]
    return arr


def params():
    return EngineConfig.for_workload(synth.CONFIGS["cfg2"], helpers.load_calib(), max_batch=4).to_params()


@pytest.mark.parametrize("n", [0, 257, -1])
def test_create_multi_rejects_a_camera_count_out_of_range(n):
    lib, h = _lib.load(), C.c_void_p()
    assert lib.vti_create_multi(C.byref(params()), n, cameras(1), C.byref(h)) == -1
    assert b"n_cameras" in lib.vti_last_error()
    assert not h.value


def test_create_multi_rejects_null_and_wrong_struct_size():
    lib, h = _lib.load(), C.c_void_p()
    assert lib.vti_create_multi(C.byref(params()), 2, None, C.byref(h)) == -1
    bad = cameras(3)
    bad[2].struct_size = 200
    assert lib.vti_create_multi(C.byref(params()), 3, bad, C.byref(h)) == -1
    assert b"cameras[2].struct_size" in lib.vti_last_error()
    p = params()
    p.struct_size = 16
    assert lib.vti_create_multi(C.byref(p), 1, cameras(1), C.byref(h)) == -1


@pytest.mark.skipif(_lib.load() and __import__("torch").cuda.is_available(), reason="checks the no-GPU behaviour")
def test_create_multi_with_valid_arguments_reports_no_device():
    lib, h = _lib.load(), C.c_void_p()
    assert lib.vti_create_multi(C.byref(params()), 256, cameras(256), C.byref(h)) == -4
    assert lib.vti_create_multi(C.byref(params()), 1, cameras(1), C.byref(h)) == -4


def test_engine_config_cameras_convert_to_vti_camera():
    calib = helpers.load_calib()
    K = np.asarray(calib["camera_matrix"], np.float64)
    cams = [dict(K=K, dist=np.array(calib["dist_coeffs"] + [0.0, 0.0]), R=np.eye(3), t=[0.1, 0.2, 0.3]),
            dict(K=K * 2, dist=[0.1, -0.2], R=np.diag([1.0, -1.0, -1.0]), t=np.array([[0.0], [0.0], [1.0]]))]
    ec = EngineConfig(frame_h=720, frame_w=1280, K=K, dist=np.zeros(5), R=np.eye(3), t=np.zeros(3), cameras=cams)
    arr = ec.to_cameras()
    assert len(arr) == 2 and all(c.struct_size == 216 and c.reserved == 0 for c in arr)
    assert list(arr[0].K) == K.reshape(9).tolist() and list(arr[1].K) == (2 * K).reshape(9).tolist()
    assert list(arr[0].dist) == list(calib["dist_coeffs"])
    assert list(arr[1].dist) == [0.1, -0.2, 0.0, 0.0, 0.0]
    assert list(arr[1].R) == [1.0, 0, 0, 0, -1.0, 0, 0, 0, -1.0] and list(arr[1].t) == [0.0, 0.0, 1.0]
    cams[1]["dist"] = [0.1, 0, 0, 0, 0, 0.5]                 # a rational-model term: not implemented, never dropped
    with pytest.raises(ValueError, match=r"cameras\[1\]\.dist"):
        ec.to_cameras()


def test_multi_camera_app_raises_like_the_reference(tmp_path):
    c = helpers.load_calib()
    cp, ep = tmp_path / "calib.json", tmp_path / "extr.json"
    cp.write_text(json.dumps({"camera_matrix": c["camera_matrix"], "dist_coeffs": c["dist_coeffs"]}))
    ep.write_text(json.dumps(c["extrinsics"]))
    with pytest.raises(FileNotFoundError, match="Calibration file missing"):
        A.MultiCameraApp([(str(cp), str(ep)), (str(tmp_path / "nope.json"), str(ep))], "best_Model.pt")
    with pytest.raises(FileNotFoundError, match="Extrinsics file missing"):
        A.MultiCameraApp([(str(cp), str(tmp_path / "nope.json"))], "best_Model.pt")
    with pytest.raises(ValueError):
        A.MultiCameraApp([], "best_Model.pt")

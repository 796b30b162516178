"""TEST INFRASTRUCTURE ONLY -- loads the reference's own measure-stage modules VERBATIM.

Source: a checkout of the reference application (github.com/RishWijewardhena/vision-textile-inspection), placed or
linked at oracle/_ref/ (git-ignored) or named by the environment variable VTI_REFERENCE_DIR, which takes precedence.
It is not part of this repository: without it the tests that run the reference live skip, and the committed goldens
stand for it.  Used by
oracle/gen_golden.py to produce tests/golden/*.json, by tests/test_oracle_measure.py to pin oracle/measure_port.py
against the reference itself, by tests/test_app.py to run the reference's own process_frame with the B200 predictor
plugged in (INTEGRATION.md 2), and by bench.py's CPU arm (kind "reference").  The modules are imported where they lie.

Recipe (SURVEY.md 8c): stub `ultralytics` (measurement.py:9) and `serial` (config.py:7 -> hardware_utils.py:1), set
dummy DB_* variables (config.py:132-133 raises without them), then build StitchMeasurementApp with __new__ so that
neither the camera nor YOLO is opened (measurement.py:145-147).
"""
from __future__ import annotations

import contextlib
import importlib
import io
import os
import sys
import types
from collections import deque

import numpy as np

REF = os.path.abspath(os.environ.get("VTI_REFERENCE_DIR") or os.path.join(os.path.dirname(__file__), "_ref"))


def available() -> bool:
    return os.path.isfile(os.path.join(REF, "measurement.py"))


def _stubs():
    if "ultralytics" not in sys.modules:
        m = types.ModuleType("ultralytics")
        m.YOLO = lambda *a, **k: None
        sys.modules["ultralytics"] = m
    if "serial" not in sys.modules:
        s = types.ModuleType("serial")
        st = types.ModuleType("serial.tools")
        lp = types.ModuleType("serial.tools.list_ports")
        lp.comports = lambda: []
        s.tools, st.list_ports = st, lp
        s.Serial = object
        s.SerialException = Exception
        sys.modules.update({"serial": s, "serial.tools": st, "serial.tools.list_ports": lp})
    for k in ("DB_HOST", "DB_USER", "DB_PASSWORD", "DB_DATABASE", "DB_NAME", "DB_TABLE", "DB_PORT"):
        os.environ.setdefault(k, "3306" if k == "DB_PORT" else "oracle")


def load(variant: int):
    """variant 0 -> <REF>/measurement.py, 1 -> <REF>/Utils/check_stitch_distance.py."""
    _stubs()
    path = REF if variant == 0 else os.path.join(REF, "Utils")
    if path not in sys.path:
        sys.path.insert(0, path)
    if REF not in sys.path:
        sys.path.insert(0, REF)
    with contextlib.redirect_stdout(io.StringIO()), contextlib.redirect_stderr(io.StringIO()):
        mod = importlib.import_module("measurement" if variant == 0 else "check_stitch_distance")
    mod.LOG_DEBUG = False
    return mod


class _FakeModel:
    def __init__(self, result):
        self.result = result

    def predict(self, *a, **k):
        return [self.result]


def make_app(variant: int, K, dist, R, t, roi=None, result=None):
    mod = load(variant)
    app = mod.StitchMeasurementApp.__new__(mod.StitchMeasurementApp)
    app.K = np.asarray(K, np.float64).reshape(3, 3)
    app.dist = np.asarray(dist, np.float64).ravel()
    app.R = np.asarray(R, np.float64).reshape(3, 3)
    app.t = np.asarray(t, np.float64).reshape(3)
    app.n_c, app.d_c = mod.compute_camera_plane(app.R, app.t)
    app.frame_buf_dist = deque(maxlen=8)
    app.frame_buf_width = deque(maxlen=8)
    app.min_stitches, app.stitch_id, app.fabric_id = 3, 0, 1
    app.running = True
    app.model = _FakeModel(result)
    if variant == 0 and roi is not None:
        mod.ROI_ENABLED, mod.ROI_X_MIN, mod.ROI_X_MAX, mod.ROI_Y_MIN, mod.ROI_Y_MAX = roi
    return mod, app


def run_frame(app, frame, result):
    app.model.result = result
    with contextlib.redirect_stdout(io.StringIO()):
        return app.process_frame(frame)

"""The drop-in host boundary (vision_textile_inspection_b200/app.py) against the reference's contract (SURVEY 8b):
constructor errors, the process_frame dict, error paths, and -- on the GPU -- the VERBATIM reference's frame sequence
(tests/golden/scenes.json, written by oracle/gen_golden.py through measurement.py)."""
import json
import os

import numpy as np
import pytest
import torch

import helpers
from vision_textile_inspection_b200 import app as A
from vision_textile_inspection_b200 import synth

G = os.path.join(os.path.dirname(__file__), "golden")


def write_calibration(tmp_path, extr="extrinsics"):
    c = helpers.load_calib()
    cp, ep = tmp_path / "camera_calibration.json", tmp_path / "extrinsics.json"
    cp.write_text(json.dumps({"camera_matrix": c["camera_matrix"], "dist_coeffs": c["dist_coeffs"]}))
    ep.write_text(json.dumps(c[extr]))
    return str(cp), str(ep)


def test_constructor_raises_like_the_reference(tmp_path):
    cp, ep = write_calibration(tmp_path)
    with pytest.raises(FileNotFoundError, match="Calibration file missing"):
        A.StitchMeasurementApp(str(tmp_path / "nope.json"), ep, "best_Model.pt", camera_index=None)
    with pytest.raises(FileNotFoundError, match="Extrinsics file missing"):
        A.StitchMeasurementApp(cp, str(tmp_path / "nope.json"), "best_Model.pt", camera_index=None)


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_no_cpu_fallback(tmp_path):
    from vision_textile_inspection_b200 import _lib
    cp, ep = write_calibration(tmp_path)
    with pytest.raises(_lib.VtiError):
        A.StitchMeasurementApp(cp, ep, "best_Model.pt", camera_index=None, backbone=lambda x: None)


def test_reference_defaults_are_mirrored():
    assert (A.CONF_THRESH, A.IOU_THRESH, A.MAX_DETECTIONS) == (0.20, 0.25, 200)          # config.py:71-73
    assert (A.FRAME_BUFFER, A.MIN_STITCHES, A.MAX_PX_DISTANCE, A.ENVELOPE_NEIGHBORHOOD) == (8, 3, 250, 3)
    assert A.ROI_DEFAULT == (1, 10, 1270, 300, 760)                                       # config.py:91-95


class PlantedBackbone:
    """Stands in for the PyTorch YOLOv8-seg backbone: returns the planted raw head tensors of the queued seeds."""

    def __init__(self, cfg):
        self.cfg, self.queue = cfg, []

    def __call__(self, net_in):
        B = net_in.shape[0]
        heads = [synth.planted_head(self.cfg, self.queue.pop(0)) for _ in range(B)]
        dev = net_in.device
        lv = [torch.from_numpy(np.stack([h["levels"][l] for h in heads])).to(dev) for l in range(3)]
        return (*lv, torch.from_numpy(np.stack([h["coef"] for h in heads])).to(dev),
                torch.from_numpy(np.stack([h["proto"] for h in heads])).to(dev))


@pytest.mark.gpu
def test_process_frame_reproduces_the_verbatim_reference_sequence(tmp_path):
    seq = json.load(open(os.path.join(G, "scenes.json")))["sequence"]
    cfg = synth.CONFIGS[seq["config"]]
    cp, ep = write_calibration(tmp_path)
    bb = PlantedBackbone(cfg)
    app = A.StitchMeasurementApp(cp, ep, "best_Model.pt", camera_index=None, calib_w=cfg.frame_w, calib_h=cfg.frame_h,
                                 backbone=bb, roi=cfg.roi(), imgsz=cfg.imgsz)
    assert app.cap is None and np.allclose(app.n_c, [0.2283871182499797, 0.7296665720553019, 0.6445355054940998])
    for fr in seq["frames"]:
        bb.queue.append(fr["seed"])
        frame = synth.fabric_frame(cfg, fr["seed"])
        before = frame.copy()
        annotated, m = app.process_frame(frame)
        assert np.array_equal(frame, before) and annotated is not frame and annotated.shape == frame.shape
        assert set(m) >= {"edge_distance_mm", "stitch_width_mm", "stitch_count", "timestamp"}
        assert m["stitch_count"] == fr["stitch_count"]
        assert m.get("error") == fr.get("error"), m
        for key in ("edge_distance_mm", "stitch_width_mm"):
            if fr[key] is None:
                assert m[key] is None, (key, m)
            else:
                assert m[key] is not None and abs(m[key] - fr[key]) <= 1e-3 * fr[key], (key, m, fr)    # bar: 0.1 %
    assert list(app.frame_buf_dist) == pytest.approx(seq["frames"][-1]["buf_dist"], rel=1e-3)


@pytest.mark.gpu
def test_process_frame_takes_camera_native_yuyv_frames(tmp_path):
    """SURVEY 8f rank 2: the frame as the V4L2 camera delivers it (packed YUYV) -- K0 converts on the device; the
    annotated frame is cv2's BGR decode of the same bytes, the network input is what K1 makes of that decode."""
    import cv2
    cfg = synth.CONFIGS["cfg2"]
    cp, ep = write_calibration(tmp_path)
    seen = []

    class Spy(PlantedBackbone):
        def __call__(self, net_in):
            seen.append(net_in.clone())
            return super().__call__(net_in)
    bb = Spy(cfg)
    app = A.StitchMeasurementApp(cp, ep, "best_Model.pt", camera_index=None, calib_w=cfg.frame_w, calib_h=cfg.frame_h,
                                 backbone=bb, roi=cfg.roi(), imgsz=cfg.imgsz, annotate=False)
    yuyv = synth.bgr_to_yuyv(synth.fabric_frame(cfg, 2003))
    bgr = cv2.cvtColor(yuyv, cv2.COLOR_YUV2BGR_YUY2)
    bb.queue += [2003, 2003]
    a1, m1 = app.process_frame(yuyv)
    a2, m2 = app.process_frame(bgr)
    assert np.array_equal(a1, bgr) and np.array_equal(a2, bgr)
    assert torch.equal(seen[0], seen[1])
    assert m1["stitch_count"] == m2["stitch_count"] > 0 and "error" not in m1


@pytest.mark.gpu
def test_process_frame_error_paths_never_raise(tmp_path):
    cfg = synth.CONFIGS["native"]
    cp, ep = write_calibration(tmp_path)

    def broken(net_in):
        raise RuntimeError("backbone exploded")
    app = A.StitchMeasurementApp(cp, ep, "best_Model.pt", camera_index=None, backbone=broken, roi=cfg.roi())
    frame = synth.fabric_frame(cfg, 3)
    annotated, m = app.process_frame(frame)
    assert m["error"] == "Model inference failed" and m["edge_distance_mm"] is None and m["stitch_count"] == 0
    assert np.array_equal(annotated, frame)

    def empty(net_in):                                       # no detections at all -> 'Fabric not detected'
        B, dev = net_in.shape[0], net_in.device
        lv = [torch.full((B, 64 + cfg.nc, cfg.LH // s, cfg.LW // s), -20.0, device=dev) for s in (8, 16, 32)]
        return (*lv, torch.zeros((B, 32, cfg.anchors), device=dev),
                torch.zeros((B, 32, cfg.LH // 4, cfg.LW // 4), device=dev))
    app2 = A.StitchMeasurementApp(cp, ep, "best_Model.pt", camera_index=None, backbone=empty, roi=cfg.roi())
    _, m2 = app2.process_frame(frame)
    assert m2["error"] == "Fabric not detected" and m2["stitch_count"] == 0


@pytest.mark.gpu
def test_predict_inner_boundary_matches_oracle():
    """B200Predictor.predict(rgb, conf=, iou=, max_det=, imgsz=) -> r.boxes.cls / r.boxes.xyxy / r.masks.data."""
    from oracle import cv_fixed, ultra_ref
    cfg = synth.CONFIGS["native"]
    calib = helpers.load_calib()
    K = cv_fixed.scale_K(np.array(calib["camera_matrix"]), cfg.frame_w, cfg.frame_h)
    bb = PlantedBackbone(cfg)
    seen = {}

    def spy(net_in):
        seen["net_in"] = net_in.clone()
        return bb(net_in)
    pred = A.B200Predictor(spy, K, calib["dist_coeffs"])
    seed = 1
    bb.queue.append(seed)
    bgr = synth.fabric_frame(cfg, seed)
    rgb = bgr[..., ::-1].copy()                               # measurement.py:205 hands predict() an RGB array
    r = pred.predict(rgb, verbose=False, conf=cfg.conf, iou=cfg.iou, max_det=cfg.max_det, imgsz=cfg.imgsz)[0]
    # the network input equals Ultralytics' letterbox of the RGB array with its channel flip
    ref_in = ultra_ref.preprocess([rgb], cfg.imgsz, flip_channels=True).numpy()
    assert np.array_equal(seen["net_in"].cpu().numpy(), ref_in)
    hd = synth.planted_head(cfg, seed)
    ref = ultra_ref.postprocess([l[None] for l in hd["levels"]], hd["coef"][None], hd["proto"][None],
                                (cfg.frame_h, cfg.frame_w), cfg.conf, cfg.iou, cfg.max_det, cfg.nc, return_soft=True)[0]
    assert np.array_equal(r.boxes.cls.numpy(), ref.boxes.cls.numpy())
    assert np.abs(r.boxes.xyxy.numpy() - ref.boxes.xyxy.numpy()).max() <= 1e-3
    got, exp = r.masks.data.numpy() > 0, ref.masks.data.numpy() > 0
    assert got.shape == exp.shape
    soft = ref.soft.numpy()
    for k in range(got.shape[0]):
        diff = np.logical_xor(got[k], exp[k])
        if diff.any():      # only where torch's own value sits on the threshold to within float rounding
            assert np.abs(soft[k][diff] - 0.5).max() <= 1e-5
        if exp[k].sum() >= 1000:
            assert np.logical_and(got[k], exp[k]).sum() / np.logical_or(got[k], exp[k]).sum() >= 0.999
        else:
            assert diff.sum() <= 1


@pytest.mark.gpu
def test_verbatim_reference_process_frame_with_b200_predictor_plugged_in():
    """INTEGRATION.md 2, the zero-edit drop-in: the reference's OWN process_frame (measurement.py:188-511, run where it
    lies: oracle/_ref/ or VTI_REFERENCE_DIR) with `app.model` replaced by
    B200Predictor -- letterbox, decode, NMS and masks on the GPU, the reference's measure stage on those results --
    must return what it returned with the CPU Ultralytics restatement when the goldens were written."""
    from oracle import cv_fixed, measure_port, ref_verbatim
    if not ref_verbatim.available():
        pytest.skip("needs a checkout of the reference at oracle/_ref/ or VTI_REFERENCE_DIR")
    g = json.load(open(os.path.join(G, "scenes.json")))
    calib = helpers.load_calib()
    cfg = synth.CONFIGS["native"]
    K = cv_fixed.scale_K(np.array(calib["camera_matrix"]), cfg.frame_w, cfg.frame_h)
    ex = calib[cfg.extrinsics]
    R, t = measure_port.rodrigues(ex["rvec"]), np.array(ex["tvec"], np.float64)
    bb = PlantedBackbone(cfg)
    mod, app = ref_verbatim.make_app(0, K, calib["dist_coeffs"], R, t, roi=cfg.roi())
    assert (mod.CONF_THRESH, mod.IOU_THRESH, mod.MAX_DETECTIONS) == (cfg.conf, cfg.iou, cfg.max_det)
    # the reference hands predict() an RGB array and Ultralytics flips it back: channel_flip=1 is B200Predictor's default
    app.model = A.B200Predictor(bb, K, calib["dist_coeffs"], R, t, nc=cfg.nc)
    frames = [fr for fr in g["sequence"]["frames"]]
    for fr in frames:
        bb.queue.append(fr["seed"])
        frame = synth.fabric_frame(cfg, fr["seed"])
        with __import__("contextlib").redirect_stdout(__import__("io").StringIO()):
            annotated, m = app.process_frame(frame)
        assert annotated.shape == frame.shape
        assert m["stitch_count"] == fr["stitch_count"] and m.get("error") == fr.get("error"), (m, fr)
        for key in ("edge_distance_mm", "stitch_width_mm"):
            if fr[key] is None:
                assert m[key] is None
            else:
                assert abs(m[key] - fr[key]) <= 1e-3 * fr[key], (key, m[key], fr[key])             # bar: 0.1 %
    assert list(app.frame_buf_dist) == pytest.approx(frames[-1]["buf_dist"], rel=1e-3)


@pytest.mark.gpu
def test_config3_outer_app_returns_the_reference_info_text(tmp_path):
    """Utils/check_stitch_distance.py:281-553 returns (annotated, info_text); goldens from the verbatim module."""
    g = json.load(open(os.path.join(G, "scenes.json")))
    scenes = [s for s in g["scenes"] if s["config"] == "cfg3"]
    assert scenes
    cfg = synth.CONFIGS["cfg3"]
    calib = helpers.load_calib()
    # cfg3 uses the second extrinsics file of the reference (camera_extrinsics.json)
    cp = tmp_path / "camera_calibration.json"
    ep = tmp_path / "camera_extrinsics.json"
    from oracle import cv_fixed
    K = cv_fixed.scale_K(np.array(calib["camera_matrix"]), cfg.frame_w, cfg.frame_h)
    cp.write_text(json.dumps({"camera_matrix": K.tolist(), "dist_coeffs": [calib["dist_coeffs"]]}))
    ep.write_text(json.dumps(calib[cfg.extrinsics]))
    for s in scenes:
        bb = PlantedBackbone(cfg)
        app = A.CheckStitchDistanceApp(str(cp), str(ep), "single_needle_model.pt", camera_index=None,
                                       calib_w=cfg.frame_w, calib_h=cfg.frame_h, backbone=bb, conf=cfg.conf, iou=cfg.iou,
                                       max_det=cfg.max_det)
        bb.queue.append(s["seed"])
        frame = synth.fabric_frame(cfg, s["seed"])
        annotated, text = app.process_frame(frame)
        assert isinstance(text, str) and annotated.shape == frame.shape and annotated is not frame
        assert text == s["info_text"], (text, s["info_text"])

    def broken(net_in):
        raise RuntimeError("boom")
    app = A.CheckStitchDistanceApp(str(cp), str(ep), "x.pt", camera_index=None, backbone=broken)
    assert app.process_frame(synth.fabric_frame(cfg, 1))[1] == "Model error"


@pytest.mark.gpu
def test_whole_frame_as_one_cuda_graph_with_standin_backbone(tmp_path):
    """SURVEY 8f rank 1: K1 -> backbone -> K2..K5 captured as ONE CUDA graph; the head writes into the buffers K2 reads
    (no copy in between); replays are bit-identical and equal the eager path on the same frames."""
    from vision_textile_inspection_b200.backbone import make_standin_backbone
    cfg = synth.CONFIGS["native"]
    cp, ep = write_calibration(tmp_path)
    torch.backends.cudnn.benchmark = False
    bb = make_standin_backbone(nc=cfg.nc, scale="n", device="cuda", seed=3)
    frames = np.stack([synth.fabric_frame(cfg, 40 + i) for i in range(2)])
    outs = []
    for graph in (False, True, True):
        app = A.StitchMeasurementApp(cp, ep, "best_Model.pt", camera_index=None, backbone=bb, roi=cfg.roi())
        app.model.use_graph = graph
        ms = app.process_frames(frames)
        outs.append([(m.get("error"), m["stitch_count"], m["edge_distance_mm"], m["stitch_width_mm"]) for m in ms])
        if graph:
            pipe = next(iter(app.model._pipes.values()))
            assert pipe.in_place                                          # K2 reads the head's output buffers directly
            d1 = pipe.outputs[0].clone()
            pipe.replay(frames)
            torch.cuda.synchronize()
            assert torch.equal(d1, pipe.outputs[0])                       # replay is bit-reproducible
            assert len(app.model._pipes) == 1
    assert outs[1] == outs[2]
    assert [o[:2] for o in outs[0]] == [o[:2] for o in outs[1]]          # same decisions eager vs graph

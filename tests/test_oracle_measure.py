"""Pins oracle/measure_port.py against the reference's own code: golden vectors written by oracle/gen_golden.py
from the VERBATIM reference modules (and, when a checkout of the reference is at oracle/_ref/ or
VTI_REFERENCE_DIR, against those modules live)."""
import json
import os

import numpy as np
import pytest

import helpers
from oracle import measure_port as MP
from oracle import ref_verbatim
from vision_textile_inspection_b200 import synth

G = os.path.join(os.path.dirname(__file__), "golden")


def test_known_answer_points(calib):
    ka = json.load(open(os.path.join(G, "known_answers.json")))
    for blk in ka["points"]:
        ex = calib[blk["extrinsics"]]
        c = MP.MeasureConfig(K=calib["camera_matrix"], dist=calib["dist_coeffs"], R=MP.rodrigues(ex["rvec"]),
                             t=ex["tvec"])
        assert np.allclose(c.n_c, blk["n_c"], rtol=0, atol=1e-15) and abs(c.d_c - blk["d_c"]) < 1e-15
        for (u, v), wref in zip(blk["pts"], blk["world"]):
            assert np.array_equal(MP.pixel_to_world(u, v, c), np.array(wref))
            x, y = MP.undistort_point_spec(u, v, c.K, c.dist)          # 5-iteration restatement, <= few ulp
            ray = np.array([x, y, 1.0])
            Xw = c.R.T.dot((-c.d_c / c.n_c.dot(ray)) * ray - c.t)
            assert np.abs(Xw - np.array(wref)).max() < 1e-15
    # survey 8c known answers
    assert abs(ka["points"][0]["width_mm"] - 4.1265102173035775) < 1e-12
    assert abs(ka["points"][0]["edge_mm"] - 8.850401225635439) < 1e-12
    assert abs(ka["points"][1]["width_mm"] - 3.194003887559879) < 1e-12


def test_known_answer_kmeans():
    ka = json.load(open(os.path.join(G, "known_answers.json")))
    for case in ka["kmeans"]:
        v = np.array(case["values"], dtype=np.float64)
        assert MP.kmeans2(v, update_on_break=False).tolist() == case["labels_v0"]
        assert MP.kmeans2(v, update_on_break=True).tolist() == case["labels_v1"]
    assert MP.kmeans2(np.array([10.0, 50.0]), False).tolist() == [0, 0]      # the first-iteration-break quirk


def test_port_matches_verbatim_goldens(calib):
    g = json.load(open(os.path.join(G, "scenes.json")))
    for s in g["scenes"]:
        cfg = synth.CONFIGS[s["config"]]
        _, res, m = helpers.oracle_scene(cfg, s["seed"], calib)
        assert res.boxes.cls.shape[0] == s["n_det"]
        assert ([m["avg_dist"]] if m["avg_dist"] is not None else []) == s["buf_dist"]
        assert ([m["avg_width"]] if m["avg_width"] is not None else []) == s["buf_width"]
        if "stitch_count" in s:
            assert m["n_dist"] == s["stitch_count"]


def test_temporal_sequence_matches_verbatim(calib):
    g = json.load(open(os.path.join(G, "scenes.json")))["sequence"]
    cfg = synth.CONFIGS[g["config"]]
    tm = MP.TemporalMedian()
    for fr in g["frames"]:
        _, _, m = helpers.oracle_scene(cfg, fr["seed"], calib)
        d = MP.result_dict(m, tm)
        assert d["edge_distance_mm"] == fr["edge_distance_mm"]
        assert d["stitch_width_mm"] == fr["stitch_width_mm"]
        assert d["stitch_count"] == fr["stitch_count"]


@pytest.mark.skipif(not ref_verbatim.available(),
                    reason="needs a checkout of the reference at oracle/_ref/ or VTI_REFERENCE_DIR")
def test_port_matches_reference_live_with_error_paths(calib):
    """Live run of the verbatim reference, including the 'Fabric not detected' / 'No stitches detected' returns."""
    from oracle import gen_golden
    cfg = synth.CONFIGS["native"]
    hd, res, _ = helpers.oracle_scene(cfg, 5, calib)
    frame = synth.fabric_frame(cfg, 5)
    K, dist, R, t = gen_golden.camera_for(cfg, calib)
    mod, app = ref_verbatim.make_app(0, K, dist, R, t, roi=cfg.roi())
    mc = helpers.measure_config(cfg, calib)
    cls = res.boxes.cls.numpy()
    for name, keep in (("all", np.ones_like(cls, bool)), ("no_fabric", cls == 0), ("no_stitch", cls == 1)):
        class R_:  # sliced Results
            pass
        r = R_()
        r.boxes = type("B", (), dict(cls=res.boxes.cls[keep], xyxy=res.boxes.xyxy[keep]))()
        r.masks = type("M", (), dict(data=res.masks.data[keep]))()
        app.frame_buf_dist.clear(); app.frame_buf_width.clear()
        _, ret = ref_verbatim.run_frame(app, frame, r)
        m = MP.measure_frame(cls[keep], res.boxes.xyxy.numpy()[keep], res.masks.data.numpy()[keep], cfg.frame_h,
                             cfg.frame_w, mc)
        d = MP.result_dict(m, MP.TemporalMedian())
        assert d.get("error") == ret.get("error")
        assert d["edge_distance_mm"] == ret["edge_distance_mm"] and d["stitch_width_mm"] == ret["stitch_width_mm"]
        assert d["stitch_count"] == ret["stitch_count"]

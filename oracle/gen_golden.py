"""TEST INFRASTRUCTURE ONLY -- writes tests/golden/*.json by running the VERBATIM reference modules.

Needs a checkout of the reference application at oracle/_ref/ (or VTI_REFERENCE_DIR=<checkout>):
    python -m oracle.gen_golden

Outputs
  vision_textile_inspection_b200/data/reference_calibration.json   K / dist / rvec / tvec values of the three
        reference calibration JSONs (camera_calibration.json, extrinsics.json, camera_extrinsics.json), regenerated
        as one fixture (values are data the product needs; the files themselves are not copied)
  tests/golden/known_answers.json    pixel->world, width/edge mm, k-means label vectors from the reference's own
        functions (measurement.py:50-65, 88-113; check_stitch_distance.py:143-171)
  tests/golden/scenes.json           per (config, seed): the dict process_frame returned + the deque contents, with
        model.predict replaced by oracle/ultra_ref.py on seeded synthetic head tensors (inputs regenerate from seeds)
"""
from __future__ import annotations

import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import cv_fixed, measure_port, ref_verbatim, ultra_ref  # noqa: E402
from vision_textile_inspection_b200 import synth  # noqa: E402

SCENES = [("native", 0), ("native", 1), ("native", 2), ("cfg1", 1000), ("cfg1", 1001), ("cfg1", 1002), ("cfg2", 2000),
          ("cfg2", 2001), ("cfg3", 3000), ("cfg3", 3001), ("cfg4", 4000), ("cfg5", 5000), ("cfg5", 5001)]
SEQUENCE = ("native", list(range(10, 22)))


def load_calibration():
    ref = ref_verbatim.REF
    c = json.load(open(os.path.join(ref, "camera_calibration.json")))
    e = json.load(open(os.path.join(ref, "extrinsics.json")))
    ce = json.load(open(os.path.join(ref, "camera_extrinsics.json")))
    return dict(camera_matrix=c["camera_matrix"], dist_coeffs=np.asarray(c["dist_coeffs"]).ravel().tolist(),
                image_size=c["image_size"], extrinsics=dict(rvec=e["rvec"], tvec=e["tvec"]),
                camera_extrinsics=dict(rvec=ce["rvec"], tvec=ce["tvec"]))


def camera_for(cfg, calib):
    K = cv_fixed.scale_K(np.array(calib["camera_matrix"]), cfg.frame_w, cfg.frame_h)
    dist = np.zeros(5) if cfg.undistort else np.array(calib["dist_coeffs"])
    ex = calib[cfg.extrinsics]
    R = measure_port.rodrigues(ex["rvec"])
    return K, dist, R, np.array(ex["tvec"], np.float64)


def run_scene(name, seed, calib, app_cache):
    cfg = synth.CONFIGS[name]
    sc = synth.make_scene(cfg, seed)
    hd = synth.planted_head(cfg, seed, sc)
    frame = synth.fabric_frame(cfg, seed, sc)
    res = ultra_ref.postprocess([l[None] for l in hd["levels"]], hd["coef"][None], hd["proto"][None],
                                (cfg.frame_h, cfg.frame_w), cfg.conf, cfg.iou, cfg.max_det, cfg.nc)[0]
    K, dist, R, t = camera_for(cfg, calib)
    key = (name,)
    if key not in app_cache:
        app_cache[key] = ref_verbatim.make_app(cfg.variant, K, dist, R, t, roi=cfg.roi() if cfg.variant == 0 else None)
    mod, app = app_cache[key]
    if cfg.variant == 0:
        mod.ROI_ENABLED, mod.ROI_X_MIN, mod.ROI_X_MAX, mod.ROI_Y_MIN, mod.ROI_Y_MAX = cfg.roi()
    _, ret = ref_verbatim.run_frame(app, frame, res)
    exp = dict(config=name, seed=seed, n_det=int(res.boxes.cls.shape[0]),
               buf_dist=list(app.frame_buf_dist), buf_width=list(app.frame_buf_width))
    if cfg.variant == 0:
        exp.update(edge_distance_mm=ret["edge_distance_mm"], stitch_width_mm=ret["stitch_width_mm"],
                   stitch_count=ret["stitch_count"], error=ret.get("error"))
    else:
        exp.update(info_text=ret)
    return exp


def main():
    assert ref_verbatim.available(), "needs a checkout of the reference at oracle/_ref/ or VTI_REFERENCE_DIR"
    calib = load_calibration()
    os.makedirs(os.path.join(ROOT, "vision_textile_inspection_b200", "data"), exist_ok=True)
    with open(os.path.join(ROOT, "vision_textile_inspection_b200", "data", "reference_calibration.json"), "w") as f:
        json.dump(calib, f, indent=1)

    # ---- known answers from the reference's own helper functions
    ka = dict(points=[], kmeans=[])
    m0 = ref_verbatim.load(0)
    m1 = ref_verbatim.load(1)
    K = np.array(calib["camera_matrix"])
    dist = np.array(calib["dist_coeffs"])
    for exname in ("extrinsics", "camera_extrinsics"):
        R = measure_port.rodrigues(calib[exname]["rvec"])
        t = np.array(calib[exname]["tvec"])
        n_c, d_c = m0.compute_camera_plane(R, t)
        pts = [(0, 0), (640, 480), (100.5, 400.25), (1279, 959), (500, 600), (531, 600), (500, 655)]
        world = [m0.pixel_to_world_using_camera_plane(u, v, K, dist, R, t, n_c, d_c).tolist() for u, v in pts]
        wl = np.array(world[4]); wr = np.array(world[5]); we = np.array(world[6])
        ka["points"].append(dict(extrinsics=exname, n_c=n_c.tolist(), d_c=d_c, pts=pts, world=world,
                                 width_mm=float(np.linalg.norm(wr - wl)) * 1000.0,
                                 edge_mm=float(np.linalg.norm(wl - we)) * 1000.0))
    rng = np.random.default_rng(5)
    cases = [[10, 50], [10, 11, 50], [1, 2, 3, 10, 11, 12, 30], [5], [7, 7, 7], [10, 30, 50]]
    cases += [rng.normal(400, 3, 12).tolist() + rng.normal(460, 3, 9).tolist() for _ in range(3)]
    cases += [rng.uniform(0, 900, int(n)).tolist() for n in (2, 3, 8, 9, 40, 130, 200)]
    for v in cases:
        a = np.array(v, dtype=np.float64)
        ka["kmeans"].append(dict(values=v, labels_v0=np.asarray(m0.kmeans_1d_two_clusters(a)[0]).tolist(),
                                 labels_v1=np.asarray(m1.kmeans_1d_two_clusters(a)[0]).tolist()))
    os.makedirs(os.path.join(ROOT, "tests", "golden"), exist_ok=True)
    with open(os.path.join(ROOT, "tests", "golden", "known_answers.json"), "w") as f:
        json.dump(ka, f, indent=1)

    # ---- scenes through the verbatim process_frame
    out = dict(scenes=[], sequence=None)
    for name, seed in SCENES:
        cache = {}
        out["scenes"].append(run_scene(name, seed, calib, cache))
        print(out["scenes"][-1])
    cache = {}
    seq = [run_scene(SEQUENCE[0], s, calib, cache) for s in SEQUENCE[1]]
    out["sequence"] = dict(config=SEQUENCE[0], seeds=SEQUENCE[1], frames=seq)
    with open(os.path.join(ROOT, "tests", "golden", "scenes.json"), "w") as f:
        json.dump(out, f, indent=1)
    print("sequence:", [(s["edge_distance_mm"], s["stitch_width_mm"], s["stitch_count"]) for s in seq])


if __name__ == "__main__":
    main()

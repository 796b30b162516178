"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle on the same seeded inputs.

Bars (BASELINE.json north_star): K1 output bit-exact; NMS keep indices + defect counts bit-exact; boxes <= 1e-3 px
(here: bit-exact against the float32 spec); per-instance mask IoU >= 0.999; mm measurements within 0.1 %.
"""
import json
import os

import cv2
import numpy as np
import pytest
import torch

import helpers
from oracle import cv_fixed, measure_port, post_spec, ultra_ref
from vision_textile_inspection_b200 import _lib, synth
from vision_textile_inspection_b200.engine import EngineConfig, InspectionEngine

pytestmark = pytest.mark.gpu
MM_RTOL = 1e-3          # 0.1 %  (north star); observed differences are ~1e-12
IOU_BAR = 0.999
TIE_EPS = 1e-5          # a mask pixel may differ from torch only if torch's value is this close to the threshold
FLIPS = __import__("collections").defaultdict(lambda: dict(instances=0, pixels=0, flipped_instances=0, flipped_pixels=0,
                                                           max_margin=0.0))


@pytest.fixture(scope="module", autouse=True)
def _report_mask_flips():
    """Prints, per config, how many instances / pixels differed from torch and the largest distance of such a pixel
    from the threshold (run with -s or read gpurun_out/mask_flips.json)."""
    yield
    if FLIPS:
        rep = {k: dict(v) for k, v in FLIPS.items()}
        print("\nmask flips vs torch (per config):", json.dumps(rep))
        try:
            os.makedirs(os.path.join(helpers.ROOT, "gpurun_out"), exist_ok=True)
            with open(os.path.join(helpers.ROOT, "gpurun_out", "mask_flips.json"), "w") as f:
                json.dump(rep, f, indent=1)
        except OSError:
            pass


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def make_engine(cfg, max_batch, **over):
    ec = EngineConfig.for_workload(cfg, helpers.load_calib(), max_batch=max_batch)
    for k, v in over.items():
        setattr(ec, k, v)
    return InspectionEngine(ec)


# ------------------------------------------------------------------------------------------------------------ K1
K1_CASES = [("native", 0, 0), ("cfg1", 0, 0), ("cfg2", 1, 0), ("cfg2", 0, 1), ("cfg3", 0, 0), ("cfg3", 1, 0),
            ("cfg4", 0, 0), ("cfg5", 0, 0), ("cfg5", 1, 0)]


@pytest.mark.parametrize("name,undistort,flip", K1_CASES)
def test_k1_bit_exact(name, undistort, flip):
    cfg = synth.CONFIGS[name]
    B = 2
    frames = np.stack([synth.fabric_frame(cfg, 1000 * cfg.cfg_id + i) for i in range(B)])
    eng = make_engine(cfg, B, undistort=undistort, channel_flip=flip)
    got = eng.preprocess(dev(frames)).cpu().numpy()
    und = (eng.cfg.K, eng.cfg.dist) if undistort else None
    ref = ultra_ref.preprocess(list(frames), cfg.imgsz, undistort=und, flip_channels=bool(flip)).numpy()
    assert got.shape == ref.shape
    assert np.array_equal(got, ref), f"max diff {np.abs(got - ref).max()} at {(got != ref).sum()} px"


@pytest.mark.parametrize("h,w,imgsz", [(1080, 1920, 960), (480, 640, 960), (123, 457, 960), (960, 960, 960),
                                        (300, 1000, 640)])
def test_k1_odd_shapes(h, w, imgsz):
    """exact-2x (INTER_AREA switch), upscale, ragged sizes, identity (no resize), random noise frames."""
    calib = helpers.load_calib()
    rng = np.random.default_rng(h + w)
    frames = rng.integers(0, 256, (2, h, w, 3), dtype=np.uint8)
    K = cv_fixed.scale_K(np.array(calib["camera_matrix"]), w, h)
    for undistort in (0, 1):
        ec = EngineConfig(frame_h=h, frame_w=w, K=K, dist=np.array(calib["dist_coeffs"]), R=np.eye(3),
                          t=np.array([0, 0, 0.1]), imgsz=imgsz, max_batch=2, undistort=undistort)
        eng = InspectionEngine(ec)
        got = eng.preprocess(dev(frames)).cpu().numpy()
        ref = ultra_ref.preprocess(list(frames), imgsz, undistort=(K, ec.dist) if undistort else None).numpy()
        assert np.array_equal(got, ref)


# ---------------------------------------------------------------------------------------------------- post + measure
POST_CASES = [("native", [0, 1, 2]), ("cfg1", [1000, 1001, 1002]), ("cfg2", [2000, 2001, 2002]), ("cfg3", [3000, 3001]),
              ("cfg4", [4000, 4001]), ("cfg5", [5000, 5001])]      # cfg5 = 4K frames: largest multiplicity LUTs / sums


def run_gpu(cfg, seeds, export_masks=True):
    heads = [synth.planted_head(cfg, s) for s in seeds]
    eng = make_engine(cfg, len(seeds))
    lv = [dev(np.stack([h["levels"][l] for h in heads])) for l in range(3)]
    coef = dev(np.stack([h["coef"] for h in heads]))
    proto = dev(np.stack([h["proto"] for h in heads]))
    dets, counts, results, masks = eng.post_measure(lv[0], lv[1], lv[2], coef, proto, export_masks=export_masks)
    torch.cuda.synchronize()
    return eng, heads, eng.dets_to_numpy(dets), counts.cpu().numpy(), eng.results_to_numpy(results), masks


@pytest.mark.parametrize("name,seeds", POST_CASES)
def test_decode_nms_bit_exact(name, seeds):
    cfg = synth.CONFIGS[name]
    eng, heads, dets, counts, results, _ = run_gpu(cfg, seeds, export_masks=False)
    for b, hd in enumerate(heads):
        sp = post_spec.postprocess_spec(hd["levels"], hd["coef"], cfg.conf, cfg.iou, cfg.max_det, cfg.nc, cfg.LH,
                                        cfg.LW, cfg.frame_h, cfg.frame_w)
        n = int(counts[b])
        assert n == len(sp["keep_anchor"])                                  # defect count
        assert results["n_cand"][b] == sp["n_cand"]
        d = dets[b, :n]
        assert np.array_equal(d["anchor"], sp["keep_anchor"])               # NMS keep indices, score order
        assert np.array_equal(d["cls"], sp["cls"])
        assert np.array_equal(d["conf"].view(np.uint32), sp["conf"].view(np.uint32))
        assert np.array_equal(d["box_lb"].view(np.uint32), sp["box_lb"].view(np.uint32))
        assert np.array_equal(d["box_frame"].view(np.uint32), sp["box_frame"].view(np.uint32))
        assert np.array_equal(d["box_int"], sp["box_frame"].astype(np.int32))
        # and against the real torch / torchvision operators
        res = ultra_ref.postprocess([l[None] for l in hd["levels"]], hd["coef"][None], hd["proto"][None],
                                    (cfg.frame_h, cfg.frame_w), cfg.conf, cfg.iou, cfg.max_det, cfg.nc,
                                    with_masks=False)[0]
        assert np.array_equal(d["anchor"], res.keep_anchor.numpy())
        assert np.abs(d["box_frame"] - res.boxes.xyxy.numpy()).max() <= 1e-3
        assert np.abs(d["box_lb"] - res.box_lb.numpy()).max() <= 1e-3


def _iou(a, b):
    u = np.logical_or(a, b).sum()
    return 1.0 if u == 0 else np.logical_and(a, b).sum() / u


@pytest.mark.parametrize("name,seeds", POST_CASES)
def test_masks_and_measurements(name, seeds, calib):
    cfg = synth.CONFIGS[name]
    eng, heads, dets, counts, results, masks = run_gpu(cfg, seeds, export_masks=True)
    h, w = cfg.frame_h, cfg.frame_w
    my, mx = cv_fixed.nearest_map(h, cfg.LH), cv_fixed.nearest_map(w, cfg.LW)
    mc = helpers.measure_config(cfg, calib)
    for b, seed in enumerate(seeds):
        n = int(counts[b])
        _, res, m = helpers.oracle_scene(cfg, seed, calib, return_soft=True)
        ref_masks = res.masks.data.numpy() > 0
        soft = res.soft.numpy()
        got_masks = eng.unpack_masks(masks, b, n).cpu().numpy() > 0
        assert got_masks.shape == ref_masks.shape
        d = dets[b, :n]
        for k in range(n):
            iou_lb = _iou(got_masks[k], ref_masks[k])
            iou_fr = _iou(got_masks[k][my][:, mx], ref_masks[k][my][:, mx])
            diff = np.logical_xor(got_masks[k], ref_masks[k])
            FLIPS[name]["instances"] += 1
            FLIPS[name]["pixels"] += int(ref_masks[k].sum())
            if diff.any():
                # a pixel may differ from torch ONLY where torch's own value sits on the threshold to within float
                # rounding (the kernel sums the 32 products and interpolates in another order): |value - 0.5| <= 1e-5
                margin = np.abs(soft[k][diff] - 0.5)
                FLIPS[name]["flipped_instances"] += 1
                FLIPS[name]["flipped_pixels"] += int(diff.sum())
                FLIPS[name]["max_margin"] = max(FLIPS[name]["max_margin"], float(margin.max()))
                assert margin.max() <= TIE_EPS, (k, int(diff.sum()), float(margin.max()))
            if ref_masks[k].sum() >= 1000:          # the north-star bar, literally, wherever 0.999 is resolvable
                assert iou_lb >= IOU_BAR and iou_fr >= IOU_BAR, (k, iou_lb, iou_fr)
            else:                                   # < 1000 px: one pixel is already > 0.1 % -- only threshold ties
                assert diff.sum() <= 1, (k, iou_lb)
            # statistics are EXACT given the mask the GPU produced (cv2.resize NEAREST + cv2.moments on it)
            bm = measure_port.instance_bitmap(got_masks[k].astype(np.float32), h, w)
            if bm is None:
                assert d["m00"][k] == 0 and not (d["flags"][k] & _lib.F_HAS_MASK) and np.isnan(d["area_mm2"][k])
            else:
                M = cv2.moments(bm)
                cols = np.where(bm.any(axis=0))[0]
                assert (d["m00"][k], d["m10"][k], d["m01"][k]) == (int(M["m00"]), int(M["m10"]), int(M["m01"]))
                assert (d["col_min"][k], d["col_max"][k]) == (cols.min(), cols.max())
                # defect area on the fabric plane (north-star "area"): numpy spec in oracle/measure_port.py
                area = measure_port.defect_area_mm2(bm, mc)
                assert area is not None and abs(d["area_mm2"][k] - area) <= 1e-9 * area, (k, d["area_mm2"][k], area)
        # the measure stage run by the oracle on the GPU's own masks must agree on every decision and to ~1 ulp
        mg = measure_port.measure_frame(d["cls"], d["box_frame"], got_masks.astype(np.float32), h, w, mc)
        r = results[b]
        st = {"ok": _lib.ST_OK, "no_fabric": _lib.ST_NO_FABRIC, "no_stitch": _lib.ST_NO_STITCH}[mg["status"]]
        assert r["status"] == st
        if st == _lib.ST_OK:
            assert (r["n_dist"], r["n_width"]) == (mg["n_dist"], mg["n_width"])
            st_idx = [k for k in range(n) if (d["flags"][k] & _lib.F_STITCH) and (d["flags"][k] & _lib.F_IN_ROI)]
            assert len(st_idx) == len(mg["stitches"]) == r["n_stitch"]
            sel = [i for i, k in enumerate(st_idx) if d["flags"][k] & _lib.F_SELECTED]
            fin = [i for i, k in enumerate(st_idx) if d["flags"][k] & _lib.F_FINAL]
            assert sel == mg["selected"] and sorted(fin) == sorted(mg["final"])
            for i, k in enumerate(st_idx):
                s = mg["stitches"][i]
                assert d["cx"][k] == s["cx"] and d["cy"][k] == s["cy"]
                assert (d["left_px"][k], d["right_px"][k]) == (s["left"], s["right"])
                if s.get("width_mm") is not None:
                    assert abs(d["width_mm"][k] - s["width_mm"]) <= 1e-9 * s["width_mm"]
                if s.get("dist_mm") is not None:
                    assert abs(d["dist_mm"][k] - s["dist_mm"]) <= 1e-9 * max(s["dist_mm"], 1e-3)
                    assert d["edge_y"][k] == s["edge_y"]
            for key, ref in (("avg_dist", mg["avg_dist"]), ("avg_width", mg["avg_width"])):
                if ref is None:
                    assert np.isnan(r[key])
                else:
                    assert abs(r[key] - ref) <= 1e-9 * ref
        # end to end against the oracle's own masks: the north-star bar, 0.1 %
        assert r["status"] == {"ok": 0, "no_fabric": 2, "no_stitch": 3}[m["status"]]
        if m["status"] == "ok":
            assert r["n_dist"] == m["n_dist"] and r["n_width"] == m["n_width"]
            for key, ref in (("avg_dist", m["avg_dist"]), ("avg_width", m["avg_width"])):
                if ref is None:
                    assert np.isnan(r[key])
                else:
                    assert abs(r[key] - ref) <= MM_RTOL * ref, (key, r[key], ref)


@pytest.mark.parametrize("name,seeds", [("native", [0, 1]), ("cfg2", [2000]), ("cfg4", [4000])])
def test_mask_variant_b(name, seeds, calib):
    """Newer-Ultralytics masks (SURVEY 8a U6 variant B): logits, no sigmoid, > 0.0, empty-mask detections dropped.
    Oracle: ultra_ref.process_mask(variant="B") on the real torch operators."""
    cfg = synth.CONFIGS[name]
    heads = [synth.planted_head(cfg, s) for s in seeds]
    eng = make_engine(cfg, len(seeds), mask_variant=1)
    lv = [dev(np.stack([h["levels"][l] for h in heads])) for l in range(3)]
    dets, counts, results, masks = eng.post_measure(lv[0], lv[1], lv[2], dev(np.stack([h["coef"] for h in heads])),
                                                    dev(np.stack([h["proto"] for h in heads])), export_masks=True)
    torch.cuda.synchronize()
    dets, counts, results = eng.dets_to_numpy(dets), counts.cpu().numpy(), eng.results_to_numpy(results)
    mc = helpers.measure_config(cfg, calib)
    for b, seed in enumerate(seeds):
        n = int(counts[b])
        d = dets[b, :n]
        _, res, m = helpers.oracle_scene(cfg, seed, calib, return_soft=True, mask_variant="B")
        kept = np.array([not (f & _lib.F_DROPPED) for f in d["flags"]], bool)
        assert np.array_equal(d["anchor"][kept], res.keep_anchor.numpy())        # the same detections survive the drop
        assert results["n_det"][b] == kept.sum() == res.boxes.cls.shape[0]
        got = (eng.unpack_masks(masks, b, n).cpu().numpy() > 0)[kept]
        ref, soft = res.masks.data.numpy() > 0, res.soft.numpy()
        for k in range(ref.shape[0]):
            diff = np.logical_xor(got[k], ref[k])
            if diff.any():                # only on threshold ties of torch's own logit map (|logit| within rounding of 0)
                assert np.abs(soft[k][diff]).max() <= 1e-4, (k, int(diff.sum()), float(np.abs(soft[k][diff]).max()))
            if ref[k].sum() >= 1000:
                assert _iou(got[k], ref[k]) >= IOU_BAR
            else:
                assert diff.sum() <= 1
        r = results[b]
        assert r["status"] == {"ok": 0, "no_fabric": 2, "no_stitch": 3}[m["status"]]
        if m["status"] == "ok":
            assert (r["n_dist"], r["n_width"]) == (m["n_dist"], m["n_width"])
            for key, refv in (("avg_dist", m["avg_dist"]), ("avg_width", m["avg_width"])):
                if refv is None:
                    assert np.isnan(r[key])
                else:
                    assert abs(r[key] - refv) <= MM_RTOL * refv


def test_against_verbatim_reference_goldens(calib):
    """tests/golden/scenes.json was written by the VERBATIM reference process_frame (oracle/gen_golden.py)."""
    g = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "scenes.json")))
    for s in g["scenes"]:
        cfg = synth.CONFIGS[s["config"]]
        _, _, dets, counts, results, _ = run_gpu(cfg, [s["seed"]], export_masks=False)
        r = results[0]
        assert counts[0] == s["n_det"]
        for key, buf in (("avg_dist", s["buf_dist"]), ("avg_width", s["buf_width"])):
            if buf:
                assert abs(r[key] - buf[0]) <= MM_RTOL * buf[0], (s["config"], s["seed"], key, r[key], buf[0])
            else:
                assert np.isnan(r[key])
        if "stitch_count" in s:
            assert r["n_dist"] == s["stitch_count"]


def test_fused_path_equals_export_path():
    cfg = synth.CONFIGS["cfg2"]
    seeds = [2000, 2001, 2002, 2003]
    _, _, d1, c1, r1, _ = run_gpu(cfg, seeds, export_masks=True)
    _, _, d2, c2, r2, _ = run_gpu(cfg, seeds, export_masks=False)
    assert np.array_equal(c1, c2)
    for key in ("status", "n_dist", "n_width", "n_stitch"):
        assert np.array_equal(r1[key], r2[key])
    assert np.array_equal(r1["avg_dist"], r2["avg_dist"], equal_nan=True)
    assert np.array_equal(r1["avg_width"], r2["avg_width"], equal_nan=True)


# ----------------------------------------------------------------------------------------------------- edge cases
def _empty_head(cfg, B):
    shapes = [(cfg.LH // s, cfg.LW // s) for s in (8, 16, 32)]
    lv = [np.full((B, 64 + cfg.nc, hh, ww), -20.0, np.float32) for hh, ww in shapes]
    coef = np.zeros((B, 32, cfg.anchors), np.float32)
    proto = np.zeros((B, 32, cfg.LH // 4, cfg.LW // 4), np.float32)
    return lv, coef, proto


def test_empty_and_ragged_batches(calib):
    cfg = synth.CONFIGS["cfg2"]
    B = 4
    lv, coef, proto = _empty_head(cfg, B)
    hd = synth.planted_head(cfg, 2000)
    for l in range(3):
        lv[l][2] = hd["levels"][l]           # frame 2 has detections, the others are empty
    coef[2], proto[2] = hd["coef"], hd["proto"]
    hd_s = synth.planted_head(cfg, 2001)      # frame 3: stitches only (fabric class logits removed)
    for l in range(3):
        x = hd_s["levels"][l].copy()
        x[64 + 1] = -20.0
        lv[l][3] = x
    coef[3], proto[3] = hd_s["coef"], hd_s["proto"]
    eng = make_engine(cfg, B)
    dets, counts, results, _ = eng.post_measure(dev(lv[0]), dev(lv[1]), dev(lv[2]), dev(coef), dev(proto))
    counts = counts.cpu().numpy()
    res = eng.results_to_numpy(results)
    assert counts[0] == 0 and counts[1] == 0 and counts[2] > 0 and counts[3] > 0
    assert res["status"][0] == _lib.ST_NO_FABRIC and res["status"][1] == _lib.ST_NO_FABRIC
    assert res["status"][2] == _lib.ST_OK
    assert res["status"][3] == _lib.ST_NO_FABRIC
    # fabric only -> 'No stitches detected'
    for l in range(3):
        x = hd["levels"][l].copy()
        x[64 + 0] = -20.0
        lv[l][0] = x
    coef[0], proto[0] = hd["coef"], hd["proto"]
    dets, counts, results, _ = eng.post_measure(dev(lv[0]), dev(lv[1]), dev(lv[2]), dev(coef), dev(proto))
    assert eng.results_to_numpy(results)["status"][0] == _lib.ST_NO_STITCH


def test_max_det_truncation_and_candidate_overflow():
    cfg = synth.CONFIGS["cfg4"]
    hd = synth.planted_head(cfg, 4000)
    lv = [dev(hd["levels"][l][None]) for l in range(3)]
    eng = make_engine(cfg, 1)
    dets, counts, results, _ = eng.post_measure(lv[0], lv[1], lv[2], dev(hd["coef"][None]), dev(hd["proto"][None]))
    assert int(counts[0]) == cfg.max_det == 300
    eng2 = make_engine(cfg, 1, max_candidates=256)          # too small on purpose: must be reported, not silent
    _, _, results2, _ = eng2.post_measure(lv[0], lv[1], lv[2], dev(hd["coef"][None]), dev(hd["proto"][None]))
    assert eng2.results_to_numpy(results2)["status"][0] & _lib.ST_OVERFLOW


def test_process_host_matches_device_path(calib):
    cfg = synth.CONFIGS["cfg2"]
    B = 3
    batch = synth.make_batch(cfg, B, seed0=2000)
    eng = make_engine(cfg, B)
    dets, counts, results, net_in = eng.process_host(batch["frames"], *batch["levels"], batch["coef"], batch["proto"],
                                                     want_net_in=True)
    d2, c2, r2, _ = eng.post_measure(*[dev(x) for x in batch["levels"]], dev(batch["coef"]), dev(batch["proto"]))
    n2 = eng.preprocess(dev(batch["frames"])).cpu().numpy()
    assert np.array_equal(net_in, n2)
    assert np.array_equal(counts, c2.cpu().numpy())
    r2 = eng.results_to_numpy(r2)
    assert np.array_equal(results["avg_dist"], r2["avg_dist"], equal_nan=True)
    assert np.array_equal(results["n_dist"], r2["n_dist"])
    d2 = eng.dets_to_numpy(d2)
    for b in range(B):
        assert np.array_equal(dets[b, :counts[b]]["anchor"], d2[b, :counts[b]]["anchor"])


def test_process_host_zero_copy_pinned_buffers(calib):
    """Pinned (device-mapped) head tensors are read in place by K2/K3 instead of being copied: same records."""
    cfg = synth.CONFIGS["cfg2"]
    B = 5
    batch = synth.make_batch(cfg, B, seed0=2000)
    eng = make_engine(cfg, B)
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    keep = [pin(batch["frames"])] + [pin(l) for l in batch["levels"]] + [pin(batch["coef"]), pin(batch["proto"])]
    d1, c1, r1 = eng.process_host(*[t.numpy() for t in keep])                      # pinned: zero copy for p3/p4/p5/coef
    d2, c2, r2 = eng.process_host(batch["frames"], *batch["levels"], batch["coef"], batch["proto"])   # pageable: copies
    assert np.array_equal(c1, c2) and r1.tobytes() == r2.tobytes()
    for b in range(B):
        assert d1[b, :c1[b]].tobytes() == d2[b, :c2[b]].tobytes()


def test_errors_are_reported_not_raised_into_cuda():
    cfg = synth.CONFIGS["cfg2"]
    eng = make_engine(cfg, 1)
    with pytest.raises(ValueError):
        eng.preprocess(torch.zeros((1, 10, 10, 3), dtype=torch.uint8, device="cuda"))
    with pytest.raises(_lib.VtiError):
        eng.preprocess(torch.zeros((2, cfg.frame_h, cfg.frame_w, 3), dtype=torch.uint8, device="cuda"))  # B > max_batch
    # a frame so large for its imgsz that a K4 work unit's 32-bit moment sums could overflow is refused at creation
    calib = helpers.load_calib()
    huge = EngineConfig(frame_h=16000, frame_w=16000, K=np.array(calib["camera_matrix"]), dist=np.array(calib["dist_coeffs"]),
                        R=np.eye(3), t=np.array([0, 0, 0.1]), imgsz=640, max_batch=1)
    with pytest.raises(_lib.VtiError, match="too large"):
        InspectionEngine(huge)


# ------------------------------------------------------------------------- BASELINE-size, size-independent properties
def test_full_size_batch_properties(calib):
    """BASELINE.json configs[1] at its full size (64 x 1280x720, undistort on) through the C ABI.  The oracle cannot
    run 64 frames in seconds, so this checks properties: (a) batch-position invariance -- the batch holds 8 unique
    frames repeated 8 times and every copy must give bit-identical network input, records and results; (b) the
    first 2 frames equal the oracle exactly (K1) / to the parity bars (post + measure); (c) idempotence of a second
    call; (d) a checksum of checksums over the whole K1 output equals 8 x the checksum of the unique part."""
    cfg = synth.CONFIGS["cfg2"]
    B, U = 64, 8
    batch = synth.make_batch(cfg, B, seed0=2000, n_unique=U)
    eng = make_engine(cfg, B)
    d_frames = dev(batch["frames"])
    net = eng.preprocess(d_frames)
    args = [dev(x) for x in batch["levels"]] + [dev(batch["coef"]), dev(batch["proto"])]
    dets, counts, results, _ = eng.post_measure(*args)
    torch.cuda.synchronize()
    d, c, r = eng.dets_to_numpy(dets), counts.cpu().numpy(), eng.results_to_numpy(results)
    # (a) every repetition of a unique frame is bit-identical, wherever it sits in the batch
    net_u = net[:U]
    for k in range(1, B // U):
        assert torch.equal(net[k * U:(k + 1) * U], net_u)
        assert np.array_equal(c[k * U:(k + 1) * U], c[:U])
        for b in range(U):
            n = c[b]
            assert d[k * U + b, :n].tobytes() == d[b, :n].tobytes()
            assert r[k * U + b].tobytes() == r[b].tobytes()
    # (d) checksum of checksums (uint32 view, wrap-around sum) over all 64 frames = 8 x the unique part
    cs = net.view(torch.int32).to(torch.int64).sum(dim=(1, 2, 3))
    assert int(cs.sum()) == (B // U) * int(cs[:U].sum())
    # (b) the first frames against the oracle
    und = (eng.cfg.K, eng.cfg.dist)
    ref = ultra_ref.preprocess(list(batch["frames"][:2]), cfg.imgsz, undistort=und).numpy()
    assert np.array_equal(net[:2].cpu().numpy(), ref)
    for b in range(2):
        sp = post_spec.postprocess_spec([l[b] for l in batch["levels"]], batch["coef"][b], cfg.conf, cfg.iou,
                                        cfg.max_det, cfg.nc, cfg.LH, cfg.LW, cfg.frame_h, cfg.frame_w)
        assert np.array_equal(d[b, :c[b]]["anchor"], sp["keep_anchor"])
    assert (r["status"] == _lib.ST_OK).all()
    # (c) idempotence: a second call on the same inputs reproduces every byte
    dets2, counts2, results2, _ = eng.post_measure(*args)
    net2 = eng.preprocess(d_frames)
    torch.cuda.synchronize()
    assert torch.equal(net2, net) and torch.equal(counts2, counts)
    d2 = eng.dets_to_numpy(dets2)
    for b in range(B):
        assert d2[b, :c[b]].tobytes() == d[b, :c[b]].tobytes()
    assert eng.results_to_numpy(results2).tobytes() == r.tobytes()


@pytest.mark.parametrize("name,B", [("cfg3", 128), ("cfg4", 32), ("cfg5", 32)])
def test_other_configs_batch_invariance(name, B, calib):
    """BASELINE configs 3 and 4 at their full batch (128 x 1080p, 32 x stress) and one 8-GPU shard of config 5
    (32 of 256 x 4K): records of a frame do not depend on its position in the batch, the stress config saturates
    max_det, and K1 on the 4K / 1080p frames stays bit-exact against cv2."""
    cfg = synth.CONFIGS[name]
    batch = synth.make_batch(cfg, B, seed0=1000 * cfg.cfg_id, n_unique=2)
    eng = make_engine(cfg, B)
    net = eng.preprocess(dev(batch["frames"]))
    dets, counts, results, _ = eng.post_measure(*[dev(x) for x in batch["levels"]], dev(batch["coef"]),
                                                dev(batch["proto"]))
    torch.cuda.synchronize()
    d, c, r = eng.dets_to_numpy(dets), counts.cpu().numpy(), eng.results_to_numpy(results)
    for b in range(2, B):
        assert torch.equal(net[b], net[b % 2]) and c[b] == c[b % 2]
        assert d[b, :c[b]].tobytes() == d[b % 2, :c[b]].tobytes() and r[b].tobytes() == r[b % 2].tobytes()
    und = (eng.cfg.K, eng.cfg.dist) if cfg.undistort else None
    assert np.array_equal(net[:1].cpu().numpy(), ultra_ref.preprocess(list(batch["frames"][:1]), cfg.imgsz, undistort=und).numpy())
    if name == "cfg4":
        assert (c == cfg.max_det).all()


@pytest.mark.parametrize("n_equal", [1500, 3000])
def test_nms_thousands_of_equal_scores(n_equal):
    """Lazy score buckets of K3: thousands of candidates with the SAME score fall into one histogram bin -- 1500 of
    them sort in the shared-memory buffer, 3000 overflow it and take the whole-set global sort.  Equal scores must
    come out in ascending anchor order exactly like torchvision's stable sort, whatever the path."""
    cfg = synth.CONFIGS["cfg4"]
    rng = np.random.default_rng(n_equal)
    shapes = [(cfg.LH // s, cfg.LW // s) for s in (8, 16, 32)]
    lv = [np.full((64 + cfg.nc, hh, ww), -20.0, np.float32) for hh, ww in shapes]
    for l in range(3):
        lv[l][:64] = rng.normal(0, 1.5, lv[l][:64].shape).astype(np.float32)      # random DFL logits: overlapping boxes
    flat = lv[0][64].reshape(-1)
    flat[rng.choice(flat.size, n_equal, replace=False)] = 1.25                     # identical class-0 logits
    lv[1][65].reshape(-1)[rng.choice(lv[1][65].size, 300, replace=False)] = rng.normal(2, 1, 300)   # plus a spread
    coef = rng.normal(0, 1, (32, cfg.anchors)).astype(np.float32)
    proto = rng.normal(0, 1, (32, cfg.LH // 4, cfg.LW // 4)).astype(np.float32)
    eng = make_engine(cfg, 1)
    dets, counts, results, _ = eng.post_measure(*[dev(x[None]) for x in lv], dev(coef[None]), dev(proto[None]))
    torch.cuda.synchronize()
    sp = post_spec.postprocess_spec(lv, coef, cfg.conf, cfg.iou, cfg.max_det, cfg.nc, cfg.LH, cfg.LW, cfg.frame_h,
                                    cfg.frame_w)
    assert sp["n_cand"] >= n_equal
    n = int(counts[0])
    d = eng.dets_to_numpy(dets)[0, :n]
    assert n == len(sp["keep_anchor"]) and np.array_equal(d["anchor"], sp["keep_anchor"])
    assert np.array_equal(d["conf"].view(np.uint32), sp["conf"].view(np.uint32))
    assert eng.results_to_numpy(results)["n_cand"][0] == sp["n_cand"]


@pytest.mark.parametrize("nc", [3, 5, 200])      # 200: class ids >= 128 (the key's class byte must not sign-extend)
def test_decode_nms_other_class_counts(nc):
    """nc != 2 (the reference model has two classes): K2's generic class loop (nc > 4) and the unrolled one (nc <= 4),
    first-maximum tie rule and class-offset NMS stay bit-exact against the spec."""
    import dataclasses
    cfg = dataclasses.replace(synth.CONFIGS["cfg3"], nc=nc)
    rng = np.random.default_rng(nc)
    hd = synth.planted_head(cfg, 3000)
    for l in range(3):                                   # spread the planted class-0/1 evidence over all classes
        x = hd["levels"][l]
        perm = rng.integers(0, nc, x.shape[1:])
        cls_part = x[64:].copy()
        top = cls_part.max(axis=0)
        cls_part[:] = rng.normal(-7, 1, cls_part.shape)
        np.put_along_axis(cls_part, perm[None], top[None], axis=0)
        x[64:] = cls_part
    ec = EngineConfig.for_workload(cfg, helpers.load_calib(), max_batch=1)
    eng = InspectionEngine(ec)
    dets, counts, results, _ = eng.post_measure(*[dev(x[None]) for x in hd["levels"]], dev(hd["coef"][None]),
                                                dev(hd["proto"][None]))
    torch.cuda.synchronize()
    sp = post_spec.postprocess_spec(hd["levels"], hd["coef"], cfg.conf, cfg.iou, cfg.max_det, nc, cfg.LH, cfg.LW,
                                    cfg.frame_h, cfg.frame_w)
    n = int(counts[0])
    d = eng.dets_to_numpy(dets)[0, :n]
    assert n == len(sp["keep_anchor"]) and n > 10
    assert np.array_equal(d["anchor"], sp["keep_anchor"]) and np.array_equal(d["cls"], sp["cls"])
    assert np.array_equal(d["box_lb"].view(np.uint32), sp["box_lb"].view(np.uint32))


def test_misaligned_frames_are_refused_not_faulted():
    cfg = synth.CONFIGS["cfg2"]
    eng = make_engine(cfg, 1)
    raw = torch.zeros((cfg.frame_h * cfg.frame_w * 3 + 16,), dtype=torch.uint8, device="cuda")
    out = torch.empty((1, 3, eng.LH, eng.LW), dtype=torch.float32, device="cuda")
    rc = eng.lib.vti_preprocess(eng._h, raw.data_ptr() + 3, 1, out.data_ptr(), None)       # odd address
    assert rc == -1 and b"aligned" in eng.lib.vti_last_error()
    torch.cuda.synchronize()                                                                # no sticky CUDA error
    assert eng.preprocess(raw[:cfg.frame_h * cfg.frame_w * 3].view(1, cfg.frame_h, cfg.frame_w, 3)).shape[0] == 1


@pytest.mark.parametrize("name,first,count", [("cfg2", 2100, 24), ("cfg3", 3100, 16), ("native", 100, 8)])
def test_seed_sweep_keep_indices_and_mm(name, first, count, calib):
    """A wider sweep of planted scenes than POST_CASES: keep indices / counts / boxes bit-exact against the float32
    spec for every seed, and the fused (no mask export) measurements within 0.1 % of the oracle path for a few."""
    cfg = synth.CONFIGS[name]
    seeds = list(range(first, first + count))
    eng, heads, dets, counts, results, _ = run_gpu(cfg, seeds, export_masks=False)
    for b, hd in enumerate(heads):
        sp = post_spec.postprocess_spec(hd["levels"], hd["coef"], cfg.conf, cfg.iou, cfg.max_det, cfg.nc, cfg.LH,
                                        cfg.LW, cfg.frame_h, cfg.frame_w)
        n = int(counts[b])
        assert n == len(sp["keep_anchor"]), (seeds[b], n)
        d = dets[b, :n]
        assert np.array_equal(d["anchor"], sp["keep_anchor"]), seeds[b]
        assert np.array_equal(d["conf"].view(np.uint32), sp["conf"].view(np.uint32))
        assert np.array_equal(d["box_lb"].view(np.uint32), sp["box_lb"].view(np.uint32))
    for b in range(0, count, max(count // 4, 1)):
        _, _, m = helpers.oracle_scene(cfg, seeds[b], calib)
        r = results[b]
        assert r["status"] == {"ok": 0, "no_fabric": 2, "no_stitch": 3}[m["status"]], seeds[b]
        if m["status"] == "ok":
            assert r["n_dist"] == m["n_dist"] and r["n_width"] == m["n_width"]
            for key, ref in (("avg_dist", m["avg_dist"]), ("avg_width", m["avg_width"])):
                if ref is None:
                    assert np.isnan(r[key])
                else:
                    assert abs(r[key] - ref) <= MM_RTOL * ref, (seeds[b], key, r[key], ref)


def test_peer_gather_single_rank_roundtrip():
    """shard.PeerGather (the NVLink peer-memory gather-to-root of bench.py --gpus N) wired through a 1-rank NCCL group:
    what is pushed into a slot is what root reads back, slot by slot, and unpack_packed() returns the typed views."""
    import torch.distributed as dist
    from vision_textile_inspection_b200 import shard
    created = not dist.is_initialized()
    if created:
        dist.init_process_group("nccl", init_method="tcp://127.0.0.1:29533", rank=0, world_size=1)
    try:
        B, max_det = 4, 16
        packed, (dets, counts, results, _) = shard.alloc_packed(B, max_det, torch.device("cuda", 0))
        pg = shard.PeerGather(packed.numel(), torch.device("cuda", 0))
        for step in range(4):
            packed.copy_(torch.randint(0, 256, (packed.numel(),), dtype=torch.uint8, device="cuda"))
            pg.push(packed, step & 1)
            torch.cuda.synchronize()
            got = pg.gathered(step & 1)
            assert got.shape == (1, packed.numel()) and torch.equal(got[0], packed)
            d, c, r = shard.unpack_packed(got, B, max_det)
            assert torch.equal(d.reshape(-1), dets.reshape(-1)) and torch.equal(c, counts) and torch.equal(r, results)
    finally:
        if created:
            dist.destroy_process_group()


def test_cuda_graph_step_replays_bit_identically():
    """K1 || K2..K5 captured as one CUDA graph (engine.capture_step): a replay reproduces the eager records byte for
    byte, and a replay after the input buffers were overwritten in place reflects the new inputs."""
    cfg = synth.CONFIGS["cfg2"]
    seeds_a, seeds_b = [2000, 2001], [2002, 2003]

    def inputs(seeds):
        heads = [synth.planted_head(cfg, s) for s in seeds]
        frames = np.stack([synth.fabric_frame(cfg, s) for s in seeds])
        return (dev(frames), *[dev(np.stack([h["levels"][l] for h in heads])) for l in range(3)],
                dev(np.stack([h["coef"] for h in heads])), dev(np.stack([h["proto"] for h in heads])))

    eng = make_engine(cfg, 2)
    bufs = inputs(seeds_a)
    graph, net_in, (dets, counts, results, _) = eng.capture_step(*bufs)
    for seeds in (seeds_a, seeds_b):
        fresh = inputs(seeds)
        for dst, src in zip(bufs, fresh):
            dst.copy_(src)
        graph.replay()
        torch.cuda.synchronize()
        got = (net_in.clone(), dets.clone(), counts.clone(), results.clone())
        ref_in = eng.preprocess(fresh[0])
        rd, rc, rr, _ = eng.post_measure(*fresh[1:])
        torch.cuda.synchronize()
        assert torch.equal(got[0], ref_in) and torch.equal(got[2], rc) and torch.equal(got[3], rr)
        for b in range(2):
            n = int(rc[b])
            assert n > 0 and torch.equal(got[1][b, :n], rd[b, :n])


def test_mask_variant_b_fused_path_drops_like_the_oracle(calib):
    """Found by the soak run (tests/test_soak.py, VTI_SOAK_VARIANT_B=1): without mask export only ROUTED detections had
    their masks evaluated, so in variant B every other detection looked empty and was flagged DROPPED.  Variant B now
    evaluates all kept detections: the survivors are the oracle's, with and without export."""
    cfg = synth.CONFIGS["cfg4"]
    seed = 60000
    hd = synth.planted_head(cfg, seed)
    eng = make_engine(cfg, 1, mask_variant=1)
    args = [dev(l[None]) for l in hd["levels"]] + [dev(hd["coef"][None]), dev(hd["proto"][None])]
    _, res, m = helpers.oracle_scene(cfg, seed, calib, mask_variant="B")
    for export in (False, True):
        dets, counts, results, _ = eng.post_measure(*args, export_masks=export)
        torch.cuda.synchronize()
        n = int(counts[0])
        d = eng.dets_to_numpy(dets)[0, :n]
        kept = (d["flags"] & _lib.F_DROPPED) == 0
        assert np.array_equal(d["anchor"][kept], res.keep_anchor.numpy()), export
        assert eng.results_to_numpy(results)["n_det"][0] == kept.sum() == res.boxes.cls.shape[0]


def test_two_geometries_alive_at_once():
    """Advisor r1: cudaFuncAttributeMaxDynamicSharedMemorySize belongs to the kernel function, not to a handle -- a later
    handle with a smaller shared-memory need must not lower the limit under an earlier one (B200Predictor keeps one
    engine per frame shape).  Two engines with different K1 / K3 footprints, used alternately."""
    big, small = synth.CONFIGS["cfg2"], synth.CONFIGS["cfg1"]
    e_big = make_engine(big, 1)                                   # undistort: raw box + footprint, the largest K1 request
    e_small = make_engine(small, 1, max_candidates=512)           # created later, asks for less
    f_big, f_small = dev(synth.fabric_frame(big, 1)[None]), dev(synth.fabric_frame(small, 2)[None])
    ref_big = ultra_ref.preprocess([f_big[0].cpu().numpy()], big.imgsz, undistort=(e_big.cfg.K, e_big.cfg.dist)).numpy()
    ref_small = ultra_ref.preprocess([f_small[0].cpu().numpy()], small.imgsz).numpy()
    hd = synth.planted_head(big, 2000)
    for _ in range(3):
        assert np.array_equal(e_big.preprocess(f_big).cpu().numpy(), ref_big)
        assert np.array_equal(e_small.preprocess(f_small).cpu().numpy(), ref_small)
        _, counts, _, _ = e_big.post_measure(*[dev(l[None]) for l in hd["levels"]], dev(hd["coef"][None]), dev(hd["proto"][None]))
        assert int(counts[0]) > 10
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------------------------ K0
def test_k0_yuyv_ingest_bit_exact_and_host_path(calib):
    """Camera-native ingest (SURVEY 8f rank 2): K0 = cv2.cvtColor(.., COLOR_YUV2BGR_YUY2) bit for bit -- every (Y, U, V)
    triple, random frames, an even-but-not-multiple-of-4 width (the 2-pixel kernel) -- and vti_process_host_yuyv gives the
    records vti_process_host gives on the frames cv2 decodes from the same bytes."""
    u, v = np.meshgrid(np.arange(256, dtype=np.uint8), np.arange(256, dtype=np.uint8), indexing="ij")
    cases = []
    img = np.empty((65536, 256, 2), np.uint8)                   # all 2^24 triples: run = (U, V), position in the run = Y
    img[..., 0] = np.arange(256, dtype=np.uint8)
    img[:, 0::2, 1] = u.reshape(-1, 1)
    img[:, 1::2, 1] = v.reshape(-1, 1)
    cases.append(img.reshape(16, 1024, 1024, 2))                # as 16 frames of 1024 x 1024 (4 runs per row)
    rng = np.random.default_rng(11)
    cases.append(rng.integers(0, 256, (3, 720, 1280, 2), dtype=np.uint8))
    cases.append(rng.integers(0, 256, (3, 33, 70, 2), dtype=np.uint8))      # 3 * 33 * 70 pixels: not a multiple of 4
    for yuyv in cases:
        B, h, w, _ = yuyv.shape
        K = cv_fixed.scale_K(np.array(calib["camera_matrix"]), w, h)
        eng = InspectionEngine(EngineConfig(frame_h=h, frame_w=w, K=K, dist=np.array(calib["dist_coeffs"]), R=np.eye(3),
                                            t=np.array([0, 0, 0.1]), imgsz=960, max_batch=B, roi=(0, 0, 0, 0, 0)))
        got = eng.ingest_yuyv(dev(yuyv)).cpu().numpy()
        for b in range(B):
            assert np.array_equal(got[b], cv2.cvtColor(yuyv[b], cv2.COLOR_YUV2BGR_YUY2)), (h, w, b)
    assert np.array_equal(cv_fixed.yuyv_to_bgr(cases[1][0]), cv2.cvtColor(cases[1][0], cv2.COLOR_YUV2BGR_YUY2))

    cfg = synth.CONFIGS["cfg2"]
    B = 5
    batch = synth.make_batch(cfg, B, seed0=2000)
    yuyv = np.stack([synth.bgr_to_yuyv(f) for f in batch["frames"]])
    bgr = np.stack([cv2.cvtColor(y, cv2.COLOR_YUV2BGR_YUY2) for y in yuyv])
    eng = make_engine(cfg, B)
    heads = (*batch["levels"], batch["coef"], batch["proto"])
    d1, c1, r1, n1 = eng.process_host(yuyv, *heads, want_net_in=True)
    d2, c2, r2, n2 = eng.process_host(bgr, *heads, want_net_in=True)
    assert np.array_equal(n1, n2) and np.array_equal(c1, c2) and r1.tobytes() == r2.tobytes()
    for b in range(B):
        assert d1[b, :c1[b]].tobytes() == d2[b, :c2[b]].tobytes()
    with pytest.raises(ValueError):
        eng.process_host(yuyv[:, :, :, :1], *heads)


"""Several cameras behind one handle (vti_create_multi): every frame of a mixed batch is undistorted by K1 and measured
by K5 with its own camera's calibration, and gives exactly what a one-camera handle of that camera gives."""
import json

import cv2
import numpy as np
import pytest
import torch

import helpers
from oracle import ultra_ref
from vision_textile_inspection_b200 import _lib, synth
from vision_textile_inspection_b200 import app as A
from vision_textile_inspection_b200.engine import EngineConfig, InspectionEngine

pytestmark = pytest.mark.gpu
IDS = [2, 0, 1, 2, 3, 0]


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def rot_z(deg):
    c, s = np.cos(np.radians(deg)), np.sin(np.radians(deg))
    return np.array([[c, -s, 0.0], [s, c, 0.0], [0.0, 0.0, 1.0]])


def camera_set(h, w, n=4):
    """Genuinely different cameras of one frame size: the reference calibration scaled to the frame, a shifted principal
    point, the distortion scaled by 0.6 and 1.3, both reference extrinsics and rotated variants of them."""
    calib = helpers.load_calib()
    K0 = np.diag([w / 1280.0, h / 960.0, 1.0]) @ np.array(calib["camera_matrix"], np.float64)
    K1 = K0.copy()
    K1[0, 2] += 0.02 * w
    K1[1, 2] -= 0.015 * h
    dist = np.array(calib["dist_coeffs"], np.float64)
    ex = [(cv2.Rodrigues(np.asarray(calib[k]["rvec"], np.float64).reshape(3, 1))[0], np.array(calib[k]["tvec"], np.float64))
          for k in ("extrinsics", "camera_extrinsics")]
    cams = [dict(K=K0, dist=dist, R=ex[0][0], t=ex[0][1]),
            dict(K=K1, dist=dist, R=ex[1][0], t=ex[1][1]),
            dict(K=K0, dist=dist * 0.6, R=rot_z(4.0) @ ex[0][0], t=ex[0][1]),
            dict(K=K1, dist=dist * 1.3, R=rot_z(-3.0) @ ex[1][0], t=ex[1][1] * 1.1)]
    for i in range(4, n):                                   # more cameras: principal point and distortion sweeps
        K = K0.copy()
        K[0, 2] += (i - n / 2) * 0.002 * w
        cams.append(dict(K=K, dist=dist * (0.5 + i / n), R=rot_z(i * 0.5) @ ex[i % 2][0], t=ex[i % 2][1]))
    return cams[:n]


def base_config(cfg=None, shape=None, max_batch=len(IDS), **over):
    if cfg is not None:
        ec = EngineConfig.for_workload(cfg, helpers.load_calib(), max_batch=max_batch)
    else:
        h, w, imgsz = shape
        ec = EngineConfig(frame_h=h, frame_w=w, K=np.eye(3), dist=np.zeros(5), R=np.eye(3), t=np.array([0, 0, 0.1]),
                          imgsz=imgsz, max_batch=max_batch)
    for k, v in over.items():
        setattr(ec, k, v)
    return ec


def multi_engine(ec, cams):
    ec.cameras = cams
    eng = InspectionEngine(ec)
    assert eng.n_cameras == len(cams)
    return eng


def single_engines(ec, cams):
    out = []
    for c in cams:
        e = EngineConfig(**{**ec.__dict__, "cameras": None, "K": c["K"], "dist": c["dist"], "R": c["R"], "t": c["t"]})
        out.append(InspectionEngine(e))
        assert out[-1].n_cameras == 1
    return out


def k1_kernels(fn):
    """Names of the K1 kernels `fn` launches (torch.profiler's CUDA activity)."""
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.key for e in prof.key_averages() if "k1_" in e.key]


def is_multi(name):
    """The last template argument (MULTI) of a demangled or mangled fast-kernel name."""
    if name.startswith("_Z"):
        return "Lb1EEEv" in name
    args = name.split("<", 1)[1].split(">", 1)[0]
    return args.split(",")[-1].strip() in ("true", "(bool)1", "1")


# ------------------------------------------------------------------------------------------------------------ K1
# (workload or (h, w, imgsz), the K1 form it takes).  Fast remap path at LW 960 and 640; cfg3 (a 3x shrink: footprints
# not contiguous) and a 457-pixel-wide frame take the generic kernel's per-pixel gather (MODE_GATHER = 2); a width that is
# a multiple of 4 but not of 8 takes its staged raw box (MODE_RAW = 1).
K1_CASES = [("cfg2", None, "k1_fast_kernel<true, false, 960,"), ("native", None, "k1_fast_kernel<true, false, 960,"),
            (None, (768, 1024, 640), "k1_fast_kernel<true, false, 640,"), ("cfg3", None, "k1_letterbox_kernel<2>"),
            (None, (123, 457, 960), "k1_letterbox_kernel<2>"), (None, (300, 1004, 640), "k1_letterbox_kernel<1>")]


@pytest.mark.parametrize("name,shape,kernel", K1_CASES)
def test_k1_each_frame_is_undistorted_with_its_own_camera(name, shape, kernel):
    cfg = synth.CONFIGS[name] if name else None
    h, w = (cfg.frame_h, cfg.frame_w) if cfg else shape[:2]
    imgsz = cfg.imgsz if cfg else shape[2]
    B = len(IDS)
    if cfg:
        frames = np.stack([synth.fabric_frame(cfg, 1000 * cfg.cfg_id + 7 + i) for i in range(B)])
    else:
        frames = np.random.default_rng(h + w).integers(0, 256, (B, h, w, 3), dtype=np.uint8)
    cams = camera_set(h, w)
    eng = multi_engine(base_config(cfg, shape, undistort=1), cams)
    ids = dev(np.array(IDS, np.int32))
    got = eng.preprocess(dev(frames), camera=ids).cpu().numpy()
    for b, c in enumerate(IDS):
        ref = ultra_ref.preprocess([frames[b]], imgsz, undistort=(cams[c]["K"], cams[c]["dist"])).numpy()
        assert np.array_equal(got[b], ref[0]), (b, c)
    singles = single_engines(base_config(cfg, shape, undistort=1), cams)
    per_cam = [e.preprocess(dev(frames)).cpu().numpy() for e in singles]
    for b, c in enumerate(IDS):
        assert np.array_equal(got[b], per_cam[c][b]), (b, c)
    # the path taken: the fast kernel's per-frame camera form beside the form the one-camera handle runs; the generic
    # kernel is one form for both
    names = k1_kernels(lambda: eng.preprocess(dev(frames), camera=ids))
    one = k1_kernels(lambda: singles[0].preprocess(dev(frames)))
    print(f"\n{name or shape}: multi {names}  single {one}")
    assert len(names) == 1 and kernel in names[0], names
    assert len(one) == 1 and kernel in one[0], one
    if kernel.startswith("k1_fast_kernel"):
        assert is_multi(names[0]) and not is_multi(one[0]), (names, one)
    else:
        assert one == names, (one, names)
    # without undistort K1 does not depend on the camera
    plain = multi_engine(base_config(cfg, shape, undistort=0), cams)
    assert torch.equal(plain.preprocess(dev(frames), camera=ids), plain.preprocess(dev(frames)))


# ---------------------------------------------------------------------------------------------------- K2..K5 records
def heads_of(cfg, seeds):
    hs = [synth.planted_head(cfg, s) for s in seeds]
    return [dev(np.stack([x["levels"][l] for x in hs])) for l in range(3)] + \
        [dev(np.stack([x["coef"] for x in hs])), dev(np.stack([x["proto"] for x in hs]))]


def records(eng, heads, camera=None):
    dets, counts, results, _ = eng.post_measure(*heads, camera=camera)
    return eng.dets_to_numpy(dets), counts.cpu().numpy(), eng.results_to_numpy(results)


def assert_frame_equal(a, b, fa, fb):
    """Frame fa of records a == frame fb of records b, byte for byte (the used det slots and every result field)."""
    (da, ca, ra), (db, cb, rb) = a, b
    assert ca[fa] == cb[fb]
    for f in ra.dtype.names:
        assert ra[fa][f].tobytes() == rb[fb][f].tobytes(), f
    for f in da.dtype.names:
        assert da[fa, :ca[fa]][f].tobytes() == db[fb, :cb[fb]][f].tobytes(), f


@pytest.mark.parametrize("name", ["native", "cfg1", "cfg2", "cfg3"])
@pytest.mark.parametrize("undistort", [0, 1])
def test_records_match_one_handle_per_camera(name, undistort):
    cfg = synth.CONFIGS[name]
    seeds = [1000 * cfg.cfg_id + i for i in range(len(IDS))]
    heads = heads_of(cfg, seeds)
    cams = camera_set(cfg.frame_h, cfg.frame_w)
    ec = base_config(cfg, undistort=undistort)
    eng = multi_engine(ec, cams)
    got = records(eng, heads, dev(np.array(IDS, np.int32)))
    per_cam = [records(e, heads) for e in single_engines(base_config(cfg, undistort=undistort), cams)]
    for b, c in enumerate(IDS):
        assert_frame_equal(got, per_cam[c], b, b)
    # the calibration is really applied: some frame's millimetres differ from what camera 0 would measure
    def mm(rec, b):
        d, c, r = rec
        return r[b]["avg_dist"].tobytes() + r[b]["avg_width"].tobytes() + d[b, :c[b]]["area_mm2"].tobytes()
    assert any(mm(got, b) != mm(per_cam[0], b) for b, c in enumerate(IDS) if c != 0), "no frame depends on its camera"


def test_camera_zero_is_the_handles_own_calibration():
    """The entry points without ids on a multi-camera handle, and camera=None, equal a one-camera handle of camera 0
    byte for byte: K1, the records, the host path and the overlay."""
    cfg = synth.CONFIGS["cfg2"]
    B = 3
    batch = synth.make_batch(cfg, B, seed0=2000)
    heads = heads_of(cfg, range(2000, 2000 + B))
    cams = camera_set(cfg.frame_h, cfg.frame_w)
    eng = multi_engine(base_config(cfg, max_batch=B), cams)
    one = single_engines(base_config(cfg, max_batch=B), cams[:1])[0]
    frames = dev(batch["frames"])
    assert torch.equal(eng.preprocess(frames), one.preprocess(frames))
    a, b = records(eng, heads), records(one, heads)
    for f in range(B):
        assert_frame_equal(a, b, f, f)
    dets_m, counts_m, _, _ = eng.post_measure(*heads)
    ann_m = eng.annotate(frames, dets_m, counts_m)
    dets_o, counts_o, _, _ = one.post_measure(*heads)
    assert torch.equal(ann_m, one.annotate(frames, dets_o, counts_o))
    host = [batch["frames"], *batch["levels"], batch["coef"], batch["proto"]]
    hm, ho = eng.process_host(*host, want_net_in=True), one.process_host(*host, want_net_in=True)
    assert np.array_equal(hm[3], ho[3])
    for f in range(B):
        assert_frame_equal(hm[:3], ho[:3], f, f)


# ------------------------------------------------------------------------------------------------------- host path
@pytest.mark.parametrize("pinned", [False, True])
@pytest.mark.parametrize("yuyv", [False, True])
def test_host_path_matches_device_path(pinned, yuyv):
    cfg = synth.CONFIGS["cfg2"]
    B = 7                                                   # 4 chunks of 1, 2, 2, 2 frames
    ids = np.array([3, 1, 0, 2, 2, 1, 3], np.int32)
    batch = synth.make_batch(cfg, B, seed0=2000)
    frames = np.stack([synth.bgr_to_yuyv(f) for f in batch["frames"]]) if yuyv else batch["frames"]
    heads_np = [*batch["levels"], batch["coef"], batch["proto"]]
    eng = multi_engine(base_config(cfg, max_batch=B), camera_set(cfg.frame_h, cfg.frame_w))
    host = [frames] + heads_np
    if pinned:
        keep = [torch.from_numpy(np.ascontiguousarray(a)).pin_memory() for a in host]
        host = [t.numpy() for t in keep]
    dets, counts, results, net_in = eng.process_host(*host, want_net_in=True, camera=ids)
    cam = dev(ids)
    d_frames = eng.ingest_yuyv(dev(frames)) if yuyv else dev(frames)
    ref_net = eng.preprocess(d_frames, camera=cam).cpu().numpy()
    ref = records(eng, [dev(x) for x in heads_np], cam)
    assert np.array_equal(net_in, ref_net)
    for f in range(B):
        assert_frame_equal((dets, counts, results), ref, f, f)
    for bad in ([0, 1, 2, 3, 4, 0, 0], [0, -1, 0, 0, 0, 0, 0]):
        with pytest.raises(_lib.VtiError, match="camera id"):
            eng.process_host(*host, camera=np.array(bad, np.int32))


# ----------------------------------------------------------------------------------------------------- bad device id
def test_device_id_out_of_range_flags_only_that_frame():
    cfg = synth.CONFIGS["cfg2"]
    cams = camera_set(cfg.frame_h, cfg.frame_w)
    B = 3
    batch = synth.make_batch(cfg, B, seed0=2000)
    heads = heads_of(cfg, range(2000, 2000 + B))
    eng = multi_engine(base_config(cfg, max_batch=B), cams)
    good = records(eng, heads, dev(np.array([0, 2, 1], np.int32)))
    bad_ids = dev(np.array([0, len(cams), 1], np.int32))
    bad = records(eng, heads, bad_ids)
    r = bad[2][1]
    assert r["status"] & _lib.ST_BAD_CAMERA
    assert (r["n_stitch"], r["n_fabric"], r["n_dist"], r["n_width"], r["env_valid"]) == (0, 0, 0, 0, 0)
    assert np.isnan(r["avg_dist"]) and np.isnan(r["avg_width"])
    for f in (0, 2):
        assert not bad[2][f]["status"] & _lib.ST_BAD_CAMERA
        assert_frame_equal(bad, good, f, f)
    frames = dev(batch["frames"])
    n_bad = eng.preprocess(frames, camera=bad_ids)
    n_good = eng.preprocess(frames, camera=dev(np.array([0, 2, 1], np.int32)))
    assert torch.equal(n_bad[0], n_good[0]) and torch.equal(n_bad[2], n_good[2])


# ---------------------------------------------------------------------------------------------------- graph replay
def test_captured_step_follows_the_camera_buffer():
    cfg = synth.CONFIGS["cfg2"]
    B = len(IDS)
    batch = synth.make_batch(cfg, B, seed0=2000)
    heads = heads_of(cfg, range(2000, 2000 + B))
    frames = dev(batch["frames"])
    eng = multi_engine(base_config(cfg, max_batch=B), camera_set(cfg.frame_h, cfg.frame_w))
    cam = dev(np.array(IDS, np.int32))
    graph, net_in, (dets, counts, results, _) = eng.capture_step(frames, *heads, camera=cam)
    for ids in (IDS, [3, 3, 1, 0, 2, 1]):
        cam.copy_(torch.tensor(ids, dtype=torch.int32))
        graph.replay()
        torch.cuda.synchronize()
        got = (eng.dets_to_numpy(dets), counts.cpu().numpy(), eng.results_to_numpy(results))
        eager_cam = dev(np.array(ids, np.int32))
        assert torch.equal(net_in, eng.preprocess(frames, camera=eager_cam))
        ref = records(eng, heads, eager_cam)
        for f in range(B):
            assert_frame_equal(got, ref, f, f)


# ------------------------------------------------------------------------------------------------------------- app
class PlantedBackbone:
    """Stands in for the YOLOv8-seg backbone: the planted raw head tensors of the queued seeds."""

    def __init__(self, cfg):
        self.cfg, self.queue = cfg, []

    def __call__(self, net_in):
        hs = [synth.planted_head(self.cfg, self.queue.pop(0)) for _ in range(net_in.shape[0])]
        d = net_in.device
        return (*[torch.from_numpy(np.stack([x["levels"][l] for x in hs])).to(d) for l in range(3)],
                torch.from_numpy(np.stack([x["coef"] for x in hs])).to(d),
                torch.from_numpy(np.stack([x["proto"] for x in hs])).to(d))


def test_multi_camera_app_equals_one_app_per_camera(tmp_path):
    cfg = synth.CONFIGS["cfg2"]
    calib = helpers.load_calib()
    K = np.array(calib["camera_matrix"], np.float64)
    K2 = K.copy()
    K2[0, 2] += 20.0
    files = []
    for i, (Km, dist, ex) in enumerate([(K, calib["dist_coeffs"], "extrinsics"),
                                       (K2, (np.array(calib["dist_coeffs"]) * 0.6).tolist(), "camera_extrinsics")]):
        cp, ep = tmp_path / f"calib{i}.json", tmp_path / f"extr{i}.json"
        cp.write_text(json.dumps({"camera_matrix": Km.tolist(), "dist_coeffs": dist}))
        ep.write_text(json.dumps(calib[ex]))
        files.append((str(cp), str(ep)))
    ids = [0, 1, 1, 0, 0, 1, 0, 1, 1, 0, 1, 0]
    seeds = [2000 + i for i in range(len(ids))]
    frames = np.stack([synth.fabric_frame(cfg, s) for s in seeds])
    kw = dict(roi=cfg.roi(), imgsz=cfg.imgsz, undistort=1)
    bb = PlantedBackbone(cfg)
    multi = A.MultiCameraApp(files, "best_Model.pt", backbone=bb, **kw)
    got = []
    for b0 in range(0, len(ids), 4):
        bb.queue += seeds[b0:b0 + 4]
        got += multi.process_frames(frames[b0:b0 + 4], ids[b0:b0 + 4])
        assert len(multi.last_records) == 4
    with pytest.raises(ValueError):
        multi.process_frames(frames[:2], [0, 2])
    for c, (cp, ep) in enumerate(files):
        sb = PlantedBackbone(cfg)
        one = A.StitchMeasurementApp(cp, ep, "best_Model.pt", camera_index=None, backbone=sb, annotate=False, **kw)
        for b in [i for i, x in enumerate(ids) if x == c]:
            sb.queue.append(seeds[b])
            m = one.process_frames(frames[b:b + 1])[0]
            g = got[b]
            assert {k: v for k, v in g.items() if k != "timestamp"} == {k: v for k, v in m.items() if k != "timestamp"}, b
        assert list(multi.buffers[c][0]) == list(one.frame_buf_dist)
        assert list(multi.buffers[c][1]) == list(one.frame_buf_width)
    assert any(g.get("edge_distance_mm") is not None for g in got)


# ---------------------------------------------------------------------------------------------------------- memory
def test_memory_returns_after_close():
    """Five rounds of create, process_host, close of a 16-camera cfg2 handle give the device memory back."""
    cfg = synth.CONFIGS["cfg2"]
    B = 2
    batch = synth.make_batch(cfg, B, seed0=2000)
    args = [batch["frames"], *batch["levels"], batch["coef"], batch["proto"]]
    cams = camera_set(cfg.frame_h, cfg.frame_w, 16)

    def one_round():
        eng = multi_engine(base_config(cfg, max_batch=B), cams)
        eng.process_host(*args, camera=np.array([15, 3], np.int32))
        eng.close()

    one_round()
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info()[0]
    for _ in range(5):
        one_round()
    torch.cuda.synchronize()
    drop = free0 - torch.cuda.mem_get_info()[0]
    print(f"\nfree device memory after 5 rounds: {drop / 2**20:+.1f} MB lower")
    assert drop <= 8 << 20

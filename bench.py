#!/usr/bin/env python
"""bench.py -- inspected frames/s over pre + post + measure (the metric BASELINE.json names).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--config cfg2] [--impl b200|reference] [--dump-outputs DIR]

A step = one pass of the hot path (K1 undistort+letterbox, K2 decode/filter, K3 NMS, K4 masks+statistics, K5 measure)
over one batch of synthetic frames + planted head tensors already resident in HBM.  N=1 workload = BASELINE.json
configs[1] (64 x 1280x720, undistort on).  For N>1 the driver launches one rank per GPU with torchrun; every rank runs
its own batch (weak scaling, no data-path collective) and pushes its compact per-defect records to rank 0 each step
through NVLink peer memory (shard.PeerGather; --gather nccl = an all-gather of the same buffers).  At N>1 the line also
carries `cfg5_sharded`: BASELINE.json configs[4], 256 synthetic 4K frames SPLIT over the ranks (shard.shard_range,
strong scaling), resident and end to end, records gathered -- beside the weak-scaled cfg2 headline.
The CPU arm (cpu_baseline / --impl reference) runs the reference's OWN measurement.py (from a checkout at
oracle/_ref/ or VTI_REFERENCE_DIR) behind the Ultralytics restatement on real cv2/torch/torchvision operators;
without one the arm runs the measure-stage port and says kind "port".
Prints ONE JSON line on rank 0.  --dump-outputs DIR also writes what the last timed step computed (dump_arrays()),
so that two builds can be compared output for output on the same seeded inputs.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# A benchmark run leaves the tree as it found it (it may be read-only): no bytecode caches, here or in the spawned
# CPU-arm workers.
sys.dont_write_bytecode = True
os.environ["PYTHONDONTWRITEBYTECODE"] = "1"

import numpy as np  # noqa: E402

# stdout carries exactly ONE JSON line: libraries that chat on file descriptor 1 (NCCL prints its version banner there)
# are sent to stderr, the line itself goes to the saved descriptor.
REAL_STDOUT = sys.stdout


def _protect_stdout():
    global REAL_STDOUT
    sys.stdout.flush()
    REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


METRIC = "inspected frames/sec (pre+post+measure)"
UNIT = "frames/s"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def stage_bytes(cfg, n_det_mean: float, n_cand_mean: float | None = None):
    """Algorithmic bytes per FRAME and stage (SURVEY.md 8d, fused path, no mask export).  With n_cand_mean, K2 is what the
    kernel MUST read -- the class planes of every anchor plus the 64 box logits of each confidence-passing anchor, and
    its key + box outputs -- instead of SURVEY's whole-head figure 4 A (64 + nc), which the kernel never touches (ncu:
    19 MB per 64 frames against 181 MB), so that a K2 "fraction of roofline" can never be flattered by bytes not moved."""
    h, w, LH, LW = cfg.frame_h, cfg.frame_w, cfg.LH, cfg.LW
    ph, pw, A = LH // 4, LW // 4, cfg.anchors
    return {
        "K1": 3 * h * w + 12 * LH * LW,
        "K2": 4 * A * (64 + cfg.nc) if n_cand_mean is None else 4 * A * cfg.nc + n_cand_mean * (64 * 4 + 8 + 16),
        "K3": n_det_mean * (32 + 4 + 2) * 4,
        "K4": 128 * ph * pw,
        "K5": 64 * n_det_mean,
    }


DUMP_BYTES = 64 << 20            # --dump-outputs writes at most this much
DUMP_NET_IN_SAMPLE = 1 << 22     # elements of K1's output it keeps (16 MB of float32; cfg2's whole tensor is 400 MB)


def dump_sample_index(numel: int) -> np.ndarray:
    """Flat indices of K1's output that --dump-outputs keeps: all of them up to DUMP_NET_IN_SAMPLE elements, else the
    sorted, de-duplicated indices default_rng(0) draws -- the same on every run and every build."""
    if numel <= DUMP_NET_IN_SAMPLE:
        return np.arange(numel)
    return np.unique(np.random.default_rng(0).integers(0, numel, DUMP_NET_IN_SAMPLE))


def dump_arrays(net_in_sample, dets, counts, results) -> dict:
    """--dump-outputs: what the last timed step handed its caller, as name -> array (host numpy in: the K1 sample at
    dump_sample_index, the vti_det records (B, max_det), the counts, the vti_frame_result rows).  net_in_sample =
    the K1 sample; counts = records per frame; dets_<field> = every field of the records (rows past a frame's count
    zeroed: a caller never reads them); results_<field> = every field of the per-frame results.  float32 fields stay
    float32, the others become float64 (which holds every integer field exactly).  Every value is finite: K5 marks
    "no value" with NaN (a record without a distance, a frame without an average), so each floating-point array has
    its non-finite entries set to 0 and <name>_nonfinite beside it says where they were (0 finite, 1 NaN, 2 +inf,
    3 -inf).  The set of names does not depend on the data.  Raises SystemExit beyond DUMP_BYTES."""
    arrays = {"net_in_sample": net_in_sample, "counts": counts}
    valid = np.arange(dets.shape[1])[None, :] < counts[:, None]
    for f in dets.dtype.names:
        arrays["dets_" + f] = np.where(valid.reshape(valid.shape + (1,) * (dets[f].ndim - 2)), dets[f], 0)
    for f in results.dtype.names:
        arrays["results_" + f] = results[f]
    for k in [k for k, a in arrays.items() if np.issubdtype(a.dtype, np.floating)]:
        a = arrays[k]
        arrays[k + "_nonfinite"] = np.select([np.isnan(a), a == np.inf, a == -np.inf], [1, 2, 3], 0).astype(np.float32)
        arrays[k] = np.where(np.isfinite(a), a, a.dtype.type(0))
    arrays = {k: a.astype(np.float32 if a.dtype == np.float32 else np.float64) for k, a in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_BYTES:
        raise SystemExit(f"--dump-outputs: {total / 2**20:.0f} MB of outputs at this batch, more than "
                         f"{DUMP_BYTES >> 20} MB; use a smaller --batch")
    return arrays


def write_dump(out_dir, arrays: dict) -> None:
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.idx)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
            t_end = time.time() + 5.0                      # the first sample can take a second to appear
            while not self.lines and time.time() < t_end:
                time.sleep(0.05)
        except Exception:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append((time.time(), ln.strip()))

    def stop(self, t0: float, t1: float):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons, power = [], None, set(), []
        rows = [ln for (t, ln) in self.lines if t0 <= t <= t1 + 0.1] or [ln for (_, ln) in self.lines]
        for ln in rows:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); smax = float(f[2]); power.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(power) if power else None}


# ---------------------------------------------------------------------------------------------------------------
def cpu_reference(cfg, batch, calib, n_frames: int, warm: int = 3, single_thread_frames: int = 0, set_threads: bool = True):
    """The reference CPU path on this host: cv2 undistort+letterbox, torch decode + torchvision NMS + process_mask,
    and the measure-stage port (oracle/), frame by frame like the reference (batch 1, measurement.py:208-211)."""
    import cv2
    import torch
    from oracle import cv_fixed, measure_port, ref_verbatim, ultra_ref
    ncpu = os.cpu_count() or 1
    if set_threads:
        if torch.get_num_threads() < ncpu:      # torchrun exports OMP_NUM_THREADS=1: the CPU arm gets every host thread
            torch.set_num_threads(ncpu)
        cv2.setNumThreads(ncpu)
    K = cv_fixed.scale_K(np.array(calib["camera_matrix"]), cfg.frame_w, cfg.frame_h)
    dist = np.array(calib["dist_coeffs"])
    ex = calib[cfg.extrinsics]
    mc = measure_port.MeasureConfig(K=K, dist=np.zeros(5) if cfg.undistort else dist,
                                    R=measure_port.rodrigues(ex["rvec"]), t=np.array(ex["tvec"]), variant=cfg.variant,
                                    roi=cfg.roi(), max_px_distance=250 if cfg.variant == 0 else 150)

    app = None
    if ref_verbatim.available():           # the reference's own process_frame (measurement.py / check_stitch_distance.py)
        _, app = ref_verbatim.make_app(cfg.variant, mc.K, mc.dist, mc.R, mc.t, roi=cfg.roi() if cfg.variant == 0 else None)

    def one(i):
        f = batch["frames"][i]
        ultra_ref.preprocess([f], cfg.imgsz, undistort=(K, dist) if cfg.undistort else None)
        r = ultra_ref.postprocess([l[i:i + 1] for l in batch["levels"]], batch["coef"][i:i + 1],
                                  batch["proto"][i:i + 1], (cfg.frame_h, cfg.frame_w), cfg.conf, cfg.iou, cfg.max_det,
                                  cfg.nc)[0]
        if app is not None:
            return ref_verbatim.run_frame(app, f, r)
        return measure_port.measure_frame(r.boxes.cls.numpy(), r.boxes.xyxy.numpy(), r.masks.data.numpy(),
                                          cfg.frame_h, cfg.frame_w, mc)
    nb = batch["frames"].shape[0]
    for i in range(warm):
        one(i % nb)
    per = []
    t0 = time.perf_counter()
    for i in range(n_frames):
        t1 = time.perf_counter()
        one(i % nb)
        per.append(time.perf_counter() - t1)
    dt = time.perf_counter() - t0
    cores = {"measure_stage": "verbatim reference (oracle/ref_verbatim.py)" if app is not None else "port (oracle/measure_port.py)",
             "os_cpu_count": os.cpu_count(), "torch_threads": torch.get_num_threads(), "cv2_threads": cv2.getNumThreads(),
             "ms_per_frame_median": 1e3 * float(np.median(per)), "ms_per_frame_p10": 1e3 * float(np.percentile(per, 10)),
             "ms_per_frame_p90": 1e3 * float(np.percentile(per, 90))}
    if single_thread_frames:
        nt, nc = torch.get_num_threads(), cv2.getNumThreads()
        torch.set_num_threads(1)
        cv2.setNumThreads(1)
        one(0)
        t1 = time.perf_counter()
        for i in range(single_thread_frames):
            one(i % nb)
        cores["single_thread_frames_per_s"] = single_thread_frames / (time.perf_counter() - t1)
        cores["single_thread_sample_frames"] = single_thread_frames
        torch.set_num_threads(nt)
        cv2.setNumThreads(nc)
    return n_frames / dt, dt, cores


def _cpu_worker(args):
    """One process of the frame-parallel CPU arm: single-threaded operators, its own frames, `n_frames` timed frames."""
    cfg_name, batch, calib, n_frames, bar = args
    import cv2
    import torch
    torch.set_num_threads(1)
    cv2.setNumThreads(1)
    from vision_textile_inspection_b200 import synth
    cfg = synth.CONFIGS[cfg_name]
    cpu_reference(cfg, batch, calib, 1, warm=0, set_threads=False)         # warm-up (imports, allocator)
    bar.wait(timeout=600)
    t0 = time.perf_counter()
    cpu_reference(cfg, batch, calib, n_frames, warm=0, set_threads=False)
    return time.perf_counter() - t0


def cpu_reference_parallel(cfg_key, batch, calib, frames_per_worker: int, workers: int):
    """The CPU path with FRAME-level parallelism: `workers` processes x 1 thread, every process runs the same batch-1
    loop on its own frames.  The reference itself never does this (one frame per call, main.py:211); it is the strongest
    way to put every host core on the same arithmetic, so it is the baseline the speed-up is quoted against.
    Returns (frames/s, seconds of the slowest worker)."""
    import multiprocessing as mp
    ctx = mp.get_context("spawn")
    small = dict(frames=batch["frames"][:2], coef=batch["coef"][:2], proto=batch["proto"][:2],
                 levels=[l[:2] for l in batch["levels"]])
    with ctx.Manager() as mgr:
        bar = mgr.Barrier(workers)
        with ctx.Pool(workers) as pool:
            ts = pool.map(_cpu_worker, [(cfg_key, small, calib, frames_per_worker, bar)] * workers)
    return workers * frames_per_worker / max(ts), max(ts)


def cpu_kind() -> tuple[str, str]:
    """("reference", ...) when the reference's own measure-stage code is staged and runs, else ("port", ...)."""
    from oracle import ref_verbatim
    if ref_verbatim.available():
        return "reference", ("pre/post = the Ultralytics calls restated on the real cv2 / torch / torchvision operators "
                             "(ultralytics itself is not installable offline), measure = the reference's own "
                             "process_frame run verbatim from " + os.path.relpath(ref_verbatim.REF, ROOT))
    return "port", ("cv2+torch+torchvision operators + measure-stage port "
                    "(no reference checkout at oracle/_ref/ or VTI_REFERENCE_DIR)")


def run_reference(args, cfg, rank, world):
    """--impl reference: the CPU path alone on every host core (frame-parallel, one single-threaded process per core);
    a step is a bounded sample of the workload: `workers` x 2 frames."""
    if rank != 0:
        return
    from vision_textile_inspection_b200 import synth
    from vision_textile_inspection_b200.engine import load_reference_calibration
    calib = load_reference_calibration()
    batch = synth.make_batch(cfg, 2)
    workers = os.cpu_count() or 1
    fpw = 2
    total_steps = args.warmup + args.steps          # the workers' own warm-up frame precedes their timed loop
    fps, secs = cpu_reference_parallel(args.config, batch, calib, fpw * max(args.steps, 1), workers)
    seq_fps, _, cores = cpu_reference(cfg, batch, calib, 6, warm=1)       # the reference as it runs: one process
    n_sample = workers * fpw
    kind, kind_txt = cpu_kind()
    line = {
        "impl": "reference", "metric": METRIC, "value": fps, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * secs / max(args.steps, 1), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": cfg.name, "frames_per_step": n_sample, "frame": [cfg.frame_w, cfg.frame_h],
                   "net_in": [cfg.LW, cfg.LH]},
        "cpu_baseline": {"value": fps, "unit": UNIT, "cores": workers, "kind": kind,
                         "sample": f"{n_sample} frames/step of {cfg.name}: {workers} single-threaded processes x {fpw} "
                                   f"frames, {kind_txt} (frame-parallel; the "
                                   f"reference's own one-process loop with library threading does {seq_fps:.2f} frames/s, "
                                   f"threads={cores})"},
        "e2e": {"value": fps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), file=REAL_STDOUT, flush=True)


def _allgather_floats(vals, world, dev):
    """Every rank's list of floats -> (world, len) numpy array on every rank (NCCL all-gather; identity at world 1)."""
    import torch
    import torch.distributed as dist
    t = torch.tensor([float(v) for v in vals], dtype=torch.float64, device=dev)
    if world == 1:
        return t.cpu().numpy()[None]
    out = torch.empty((world, t.numel()), dtype=torch.float64, device=dev)
    dist.all_gather_into_tensor(out.view(-1), t)
    return out.cpu().numpy()


def h2d_probe(dev, world, barrier, mb: int = 256, reps: int = 4):
    """Plain pinned host -> device copy bandwidth of this rank while EVERY rank copies at the same time: what the host
    (its DRAM, its PCIe root complexes / switches) can feed all N GPUs at once.  GB/s of this rank."""
    import torch
    h = torch.empty(mb << 20, dtype=torch.uint8).pin_memory()
    d = torch.empty(mb << 20, dtype=torch.uint8, device=dev)
    d.copy_(h, non_blocking=True)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        d.copy_(h, non_blocking=True)
    e1.record()
    torch.cuda.synchronize()
    return reps * (mb << 20) / (e0.elapsed_time(e1) * 1e-3) / 1e9


def e2e_host(eng, cfg, h_np, B, steps, world, dev, barrier, yuyv=False):
    """vti_process_host with pinned HOST buffers, H2D + K1..K5 + D2H inside the timed region, in two feeding modes:
    "zero_copy" (frames by DMA, head tensors read in place over PCIe) and "dma" (everything copied).  Per-rank seconds
    are gathered so that the line can say what each rank's PCIe path delivered."""
    import torch
    from vision_textile_inspection_b200 import synth as synth_mod
    from vision_textile_inspection_b200._lib import DET_DTYPE, RESULT_DTYPE
    o_dets = torch.empty((B, cfg.max_det, DET_DTYPE.itemsize), dtype=torch.uint8).pin_memory()
    o_counts = torch.empty((B,), dtype=torch.int32).pin_memory()
    o_res = torch.empty((B, RESULT_DTYPE.itemsize), dtype=torch.uint8).pin_memory()
    out = (o_dets.numpy().view(DET_DTYPE).reshape(B, cfg.max_det), o_counts.numpy(),
           o_res.numpy().view(RESULT_DTYPE).reshape(B))
    modes = {}
    # camera-native frames (SURVEY 8f rank 2): the same scenes as packed YUV 4:2:2, converted on the device by K0
    yuyv_t = torch.from_numpy(np.stack([synth_mod.bgr_to_yuyv(f) for f in h_np[0][:min(B, 8)]])).pin_memory() if yuyv else None
    if yuyv_t is not None and B > yuyv_t.shape[0]:
        yuyv_t = yuyv_t.repeat((B + yuyv_t.shape[0] - 1) // yuyv_t.shape[0], 1, 1, 1)[:B].contiguous().pin_memory()
    for mode in ("zero_copy", "dma") + (("yuyv_zero_copy",) if yuyv_t is not None else ()):
        if mode == "dma":
            os.environ["VTI_NO_ZERO_COPY"] = "1"
        else:
            os.environ.pop("VTI_NO_ZERO_COPY", None)
        args_np = h_np if mode != "yuyv_zero_copy" else [yuyv_t.numpy()] + list(h_np[1:])
        for _ in range(2):
            eng.process_host(*args_np, out=out)
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            eng.process_host(*args_np, out=out)
        mine = time.perf_counter() - t0
        barrier()
        modes[mode] = _allgather_floats([mine], world, dev)[:, 0]          # seconds per rank
    os.environ.pop("VTI_NO_ZERO_COPY", None)
    yuyv_modes = {m: modes.pop(m) for m in list(modes) if m.startswith("yuyv")}
    ed, ec, er = out
    # bytes that cross PCIe per step and rank.  DMA mode: everything presented.  Zero-copy mode: the frames by DMA + what
    # the kernels read in place (class planes, 64 box logits per candidate, kept coefficient rows, the union rectangle
    # of the crop windows of the prototypes; 32-byte sectors), estimated from the records of the last call.
    presented = sum(a.nbytes for a in h_np)
    zc = 0
    for b in range(B):
        n = int(ec[b])
        zc += 4 * cfg.nc * cfg.anchors + 32 * 64 * int(er["n_cand"][b]) + 32 * 32 * n
        if n:
            bx = ed[b, :n]["box_lb"] * 0.25
            x0, y0 = np.maximum(np.ceil(bx[:, 0]), 0).min(), np.maximum(np.ceil(bx[:, 1]), 0).min()
            x1 = np.minimum(np.ceil(bx[:, 2]) - 1, cfg.LW // 4 - 1).max()
            y1 = np.minimum(np.ceil(bx[:, 3]) - 1, cfg.LH // 4 - 1).max()
            zc += int(max(y1 - y0 + 1, 0) * (max(x1 - x0 + 1, 0) + 6)) * 32 * 4
    d2h = o_dets.numel() + 4 * o_counts.numel() + o_res.numel()
    h2d = {"zero_copy": int(h_np[0].nbytes + zc), "dma": int(presented)}
    best = min(modes, key=lambda m: modes[m].max())
    rep = {m: {"frames_per_s": world * B * steps / float(modes[m].max()),
               "h2d_gbs_per_rank": [round(h2d[m] * steps / float(t) / 1e9, 2) for t in modes[m]],
               "h2d_gbs_all_ranks": round(sum(h2d[m] * steps / float(t) / 1e9 for t in modes[m]), 2),
               "h2d_bytes_per_step": h2d[m]} for m in modes}
    ingest = None
    if yuyv_modes:
        t = yuyv_modes["yuyv_zero_copy"]
        nb = int(yuyv_t.numel() + zc)
        ingest = {"frames_per_s": world * B * steps / float(t.max()), "h2d_bytes_per_step": nb,
                  "h2d_gbs_per_rank": [round(nb * steps / float(x) / 1e9, 2) for x in t],
                  "frame_bytes": int(yuyv_t.numel() // B), "bgr_frame_bytes": int(h_np[0].nbytes // B),
                  "api": "vti_process_host_yuyv: camera-native packed YUV 4:2:2 host frames (what a V4L2 camera delivers "
                         "before cv2.VideoCapture.read() converts them), K0 converts on the device in front of K1; head "
                         "tensors zero-copy as in the headline mode.  Informational: the headline e2e stays on BGR frames, "
                         "the reference's process_frame input"}
    return {"value": rep[best]["frames_per_s"], "mode": best, **({"ingest_yuyv": ingest} if ingest else {}), "h2d_bytes_per_step": h2d[best], "d2h_bytes_per_step": int(d2h),
            "h2d_dma_bytes_per_step": int(h_np[0].nbytes if best == "zero_copy" else presented),
            "h2d_zero_copy_bytes_per_step_est": int(zc if best == "zero_copy" else 0),
            "host_bytes_presented_per_step": int(presented), "steps": steps, "modes": rep}, out


def run_cfg5_sharded(args, rank, world, dev, barrier, calib, use_peer):
    """BASELINE.json configs[4]: a 256-frame synthetic 4K stream SPLIT across the ranks (shard.shard_range), every GPU
    runs the whole path on its shard, the per-defect records are gathered on rank 0; resident and end to end."""
    import torch
    import torch.distributed as dist
    from vision_textile_inspection_b200 import shard, synth
    from vision_textile_inspection_b200.engine import EngineConfig, InspectionEngine
    cfg = synth.CONFIGS["cfg5"]
    total = args.cfg5_frames
    lo, hi = shard.shard_range(total, rank, world)
    B = hi - lo
    n_unique = min(B, 8)
    batch = synth.make_batch(cfg, B, seed0=1000 * cfg.cfg_id + lo, n_unique=n_unique)
    eng = InspectionEngine(EngineConfig.for_workload(cfg, calib, max_batch=B), device=dev)
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    host = [pin(batch["frames"])] + [pin(l) for l in batch["levels"]] + [pin(batch["coef"]), pin(batch["proto"])]
    d = [t.to(dev) for t in host]
    net_in = torch.empty((B, 3, eng.LH, eng.LW), dtype=torch.float32, device=dev)
    packed, outs = shard.alloc_packed(B, cfg.max_det, dev)
    peer = None
    if world > 1 and use_peer:
        try:
            peer = shard.PeerGather(packed.numel(), dev)
        except Exception:                                        # noqa: BLE001
            peer = None
        flag = torch.tensor([1 if peer is not None else 0], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if int(flag.item()) == 0:
            peer = None
    gathered = torch.empty((world * packed.numel(),), dtype=torch.uint8, device=dev) if world > 1 and peer is None else None
    graph = eng.capture_step(d[0], d[1], d[2], d[3], d[4], d[5], net_in=net_in, outputs=outs)[0]
    slot = [0]

    def step():
        graph.replay()
        if world > 1:
            if peer is not None:
                slot[0] = peer.push(packed)
                if rank == 0:
                    peer.consume(slot[0], out=consumed)          # root reads every step, on the stream of the waits
            else:
                dist.all_gather_into_tensor(gathered, packed)
    consumed = torch.empty((world, packed.numel()), dtype=torch.uint8, device=dev) if peer is not None and rank == 0 else None
    steps = max(2, min(args.steps, 10))
    for _ in range(3):
        step()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    barrier()
    ms = float(_allgather_floats([e0.elapsed_time(e1)], world, dev).max())
    # what reached rank 0 must be every rank's own counts
    checked = None
    if world > 1:
        mine = outs[1].clone()
        allc = torch.empty((world, B), dtype=torch.int32, device=dev)
        dist.all_gather_into_tensor(allc.view(-1), mine)
        if rank == 0:
            got = consumed if peer is not None else gathered.view(world, -1)
            _, g_counts, _ = shard.unpack_packed(got, B, cfg.max_det)
            checked = bool(torch.equal(g_counts.view(world, B), allc))
            if not checked:
                raise RuntimeError("cfg5_sharded: rank 0 did not receive every rank's records")
    eng.set_profiling(True)
    eng.preprocess(d[0], out=net_in)
    eng.post_measure(d[1], d[2], d[3], d[4], d[5], outputs=outs)
    stage_ms = eng.stage_ms()
    eng.set_profiling(False)
    e2e, _ = e2e_host(eng, cfg, [t.numpy() for t in host], B, max(2, min(args.steps, 4)), world, dev, barrier)
    sb = stage_bytes(cfg, float(outs[1].float().mean().item()))
    peak, _ = peaks()
    return {"workload": cfg.name, "scaling": "strong", "frames_total": total, "frames_per_gpu": B, "unique_frames_per_gpu": n_unique,
            "value": total * steps / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms / steps, "steps": steps,
            "gather": "peer memory push, root consumes every step" if peer is not None else ("NCCL all-gather" if world > 1 else "none (1 GPU)"),
            "gather_checked": checked, "stage_ms": dict(zip(["K1", "K2", "K3", "K4", "K5"], stage_ms)),
            "frac_of_hbm_roofline_per_gpu": (B * sum(sb.values()) / (ms / steps * 1e-3) / 1e9) / peak,
            "e2e": e2e}


def run_b200(args, cfg, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from vision_textile_inspection_b200 import shard, synth
    from vision_textile_inspection_b200.engine import EngineConfig, InspectionEngine, load_reference_calibration

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    calib = load_reference_calibration()
    # One rank = one slice of the host cores: torchrun starts N processes that would otherwise all land on the same
    # cores for their pinned-buffer copies and launch threads (every GPU of this pool reports the same CPU affinity).
    affinity = None
    if world > 1 and hasattr(os, "sched_setaffinity"):
        try:
            cores = sorted(os.sched_getaffinity(0))
            per = max(1, len(cores) // world)
            mine = cores[local_rank * per:(local_rank + 1) * per] or cores
            os.sched_setaffinity(0, mine)
            affinity = f"{mine[0]}-{mine[-1]} of {len(cores)} cores"
        except OSError:
            affinity = None
    B = cfg.batch if args.batch is None else args.batch
    if args.post_streams == 0:
        # auto: when K1 has nothing heavy to do (no undistort, no resize: BASELINE configs[3], the NMS-bound stress case)
        # the K2 -> K3 -> K4 -> K5 chain -- one CTA per frame in K3 / K5 -- is the critical path and leaves most SMs idle;
        # consecutive batches are independent, so two post chains run side by side (two handles, two streams)
        g_ = cfg.geo
        k1_light = (not cfg.undistort) and cfg.frame_w == g_["new_w"] and cfg.frame_h == g_["new_h"]
        args.post_streams = 2 if k1_light else 1
    n_unique = min(B, args.unique)
    batch = synth.make_batch(cfg, B, seed0=1000 * cfg.cfg_id + 100 * rank, n_unique=n_unique)
    eng = InspectionEngine(EngineConfig.for_workload(cfg, calib, max_batch=B), device=dev)
    # --post-streams 2: consecutive batches are independent, so their post stages may overlap -- a second handle (its
    # own candidate lists and unit list) takes the odd steps on a second post stream.  That pays when the
    # K2 -> K3 -> K4 -> K5 chain, not K1, bounds the step (cfg4: 138 -> 208 k frames/s); cfg2 is K1-bound and keeps one.
    engs = [eng, InspectionEngine(EngineConfig.for_workload(cfg, calib, max_batch=B), device=dev)] \
        if args.post_streams == 2 else [eng, eng]

    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    host = {k: pin(batch[k]) for k in ("frames", "coef", "proto")}
    host_lv = [pin(l) for l in batch["levels"]]
    d_frames = host["frames"].to(dev)
    d_lv = [l.to(dev) for l in host_lv]
    d_coef, d_proto = host["coef"].to(dev), host["proto"].to(dev)
    net_in = torch.empty((B, 3, eng.LH, eng.LW), dtype=torch.float32, device=dev)
    # records + results + counts of a step live in ONE buffer (one all-gather); two such buffers alternate so that the
    # gather of step i (its own stream) runs under the kernels of step i+1
    bufs = [shard.alloc_packed(B, cfg.max_det, dev) for _ in range(2)]
    packed, outs = bufs[0]
    gathered = [torch.empty((world * bufs[0][0].numel(),), dtype=torch.uint8, device=dev) for _ in range(2)] if world > 1 else None
    # Records travel to rank 0 through NVLink peer memory (shard.PeerGather: one copy-engine copy + a signal per rank
    # and step, no collective kernel); an NCCL all-gather of the same buffers is the fallback when symmetric memory
    # cannot be set up on this box, and what --gather nccl selects.
    peer = None
    if world > 1 and args.gather == "peer":
        try:
            peer = shard.PeerGather(bufs[0][0].numel(), dev)
        except Exception as e:                                   # noqa: BLE001  (said out loud, then NCCL)
            print(f"[bench] rank {rank}: peer-memory gather unavailable ({type(e).__name__}: {e}); using NCCL all-gather",
                  file=sys.stderr)
        flag = torch.tensor([1 if peer is not None else 0], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)              # all ranks or none
        if int(flag.item()) == 0:
            peer = None
    consumed = (torch.empty((world, bufs[0][0].numel()), dtype=torch.uint8, device=dev)
                if peer is not None and rank == 0 else None)
    peer_slot = {"last": 0}

    def peer_push(pk):
        """This rank's records into root's slot; root copies the slot out on the same stream (flow control of the three
        slots: shard.PeerGather docstring)."""
        peer_slot["last"] = peer.push(pk)
        if consumed is not None:
            peer.consume(peer_slot["last"], out=consumed)
    in_bytes = (d_frames.numel() + 4 * (sum(l.numel() for l in d_lv) + d_coef.numel() + d_proto.numel()))
    out_bytes = 4 * net_in.numel()

    # Pre (K1) and post+measure (K2..K5) of one batch are independent -- the backbone sits between them -- so they are
    # issued on two streams: the latency-bound per-frame CTAs of K3/K5 run under the streaming K1.
    s_pre, s_post = torch.cuda.Stream(dev), torch.cuda.Stream(dev, priority=-1)   # post CTAs win free SM slots
    s_posts = [s_post, torch.cuda.Stream(dev, priority=-1) if args.post_streams == 2 else s_post]
    s_gather = torch.cuda.Stream(dev, priority=-1)
    ev_gather = [None, None]
    state = {"i": 0}

    # --step-form graph (default): one step = ONE CUDA graph (engine.capture_step: K1 beside K2..K5 on a forked
    # high-priority branch, joined at the end), one graph per record buffer, replayed on the current stream.  Measured
    # 2 % faster than issuing the same six kernels on two streams every step (--step-form streams, below).
    graphs, nodes_per_graph = None, 0
    if args.step_form == "graph" and args.post_streams == 1:
        try:
            l_b = eng.launch_count
            graphs = [eng.capture_step(d_frames, d_lv[0], d_lv[1], d_lv[2], d_coef, d_proto, net_in=net_in,
                                       outputs=bufs[k][1])[0] for k in range(2)]
            nodes_per_graph = (eng.launch_count - l_b) // 4        # per graph: one eager warm-up pass + the capture
        except Exception as e:                                     # noqa: BLE001  (said out loud, then the stream form)
            print(f"[bench] rank {rank}: CUDA graph capture failed ({type(e).__name__}: {e}); using the stream form",
                  file=sys.stderr)
            graphs = None
    replays = {"n": 0}

    def step(overlap=True, use_graph=None):
        """One pass of the hot path over one batch.  overlap=True: K1 goes to s_pre, K2..K5 (+ the record gather) to
        s_post and the two streams are NOT joined per step -- consecutive batches are independent, exactly as in a
        pipeline with the backbone between pre and post -- fork()/join() bracket the timed region instead."""
        if not overlap:
            eng.preprocess(d_frames, out=net_in)
            dets, counts, results, _ = eng.post_measure(d_lv[0], d_lv[1], d_lv[2], d_coef, d_proto, outputs=outs)
            if world > 1:
                shard.gather_packed(packed)
            return
        k = state["i"] & 1
        state["i"] += 1
        pk, ot = bufs[k]
        if graphs is not None and use_graph is not False:
            cur = torch.cuda.current_stream(dev)
            if world > 1 and ev_gather[k] is not None:
                cur.wait_event(ev_gather[k])                   # buffer k was gathered two steps ago
            graphs[k].replay()
            replays["n"] += 1
            if world > 1:
                s_gather.wait_stream(cur)
                with torch.cuda.stream(s_gather):
                    if peer is not None:
                        peer_push(pk)
                    else:
                        dist.all_gather_into_tensor(gathered[k], pk)
                    ev_gather[k] = torch.cuda.Event()
                    ev_gather[k].record(s_gather)
            return
        with torch.cuda.stream(s_posts[k]):
            if world > 1 and ev_gather[k] is not None:
                s_posts[k].wait_event(ev_gather[k])            # buffer k was gathered two steps ago
            engs[k].post_measure(d_lv[0], d_lv[1], d_lv[2], d_coef, d_proto, outputs=ot)
        if world > 1:
            s_gather.wait_stream(s_posts[k])
            with torch.cuda.stream(s_gather):
                if peer is not None:
                    peer_push(pk)                              # rank 0 copies the slot out right behind the waits
                else:
                    dist.all_gather_into_tensor(gathered[k], pk)   # ranks in frame order; shard.unpack_packed gives the views
                ev_gather[k] = torch.cuda.Event()
                ev_gather[k].record(s_gather)
        with torch.cuda.stream(s_pre):
            eng.preprocess(d_frames, out=net_in)

    def fork():
        cur = torch.cuda.current_stream(dev)
        s_pre.wait_stream(cur)
        for sp in s_posts:
            sp.wait_stream(cur)
        s_gather.wait_stream(cur)

    def join():
        cur = torch.cuda.current_stream(dev)
        cur.wait_stream(s_pre)
        for sp in s_posts:
            cur.wait_stream(sp)
        cur.wait_stream(s_gather)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # --dump-outputs: the K1 sample and the size of the dump are settled before anything is timed (a dry run on
    # zeros of the real shapes refuses more than DUMP_BYTES here rather than after the run)
    dump_idx = None
    if args.dump_outputs and rank == 0:
        from vision_textile_inspection_b200._lib import DET_DTYPE, RESULT_DTYPE
        idx = dump_sample_index(net_in.numel())
        dump_arrays(np.zeros(idx.size, np.float32), np.zeros((B, cfg.max_det), DET_DTYPE), np.zeros(B, np.int32),
                    np.zeros(B, RESULT_DTYPE))
        dump_idx = torch.from_numpy(idx).to(dev)
    fork()
    for _ in range(args.warmup):
        step()
    join()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    l0 = sum(e.launch_count for e in set(engs)) + nodes_per_graph * replays["n"]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_wall0 = time.time()
    e0.record()
    fork()
    for _ in range(args.steps):
        step()
    join()
    e1.record()
    # what the last timed step produced, for --dump-outputs (the steps below overwrite these buffers)
    last_out = ([net_in.view(-1)[dump_idx]] + [t.clone() for t in bufs[(state["i"] - 1) & 1][1][:3]]
                if dump_idx is not None else None)
    launches = sum(e.launch_count for e in set(engs)) + nodes_per_graph * replays["n"] - l0   # graph kernel nodes count
    # two more regions of K steps, timed the same way: the spread of the number (the reported value is the FIRST region)
    extra_ev = []
    for _ in range(2):
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        a0.record()
        fork()
        for _ in range(args.steps):
            step()
        join()
        a1.record()
        extra_ev.append((a0, a1))
    # The timed region is K steps (a few ms); nvidia-smi samples every 100 ms.  The identical loop keeps running,
    # untimed, until >= 0.5 s of load has been sampled, so "clocks" describes this workload under load.
    fork()
    for _ in range(args.load_steps):                    # same count on every rank: step() may hold a collective
        step()
    join()
    barrier()
    t_wall1 = time.time()
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    region_ms = [ms] + [float(_allgather_floats([a0.elapsed_time(a1)], world, dev).max()) for a0, a1 in extra_ev]
    clocks = sampler.stop(t_wall0, t_wall1) if rank == 0 else None
    value = world * B * args.steps / (ms * 1e-3)
    gather_checked = None
    if world > 1:
        # what reached rank 0 must be every rank's own records (checked on the per-frame counts and result bytes)
        k_last = (state["i"] - 1) & 1
        mine = torch.cat([bufs[k_last][1][1].view(torch.uint8).view(-1), bufs[k_last][1][2].reshape(-1)])
        ref_all = torch.empty((world, mine.numel()), dtype=torch.uint8, device=dev)
        dist.all_gather_into_tensor(ref_all.view(-1), mine)
        if rank == 0:
            got = consumed if peer is not None else gathered[k_last].view(world, -1)
            _, g_counts, g_results = shard.unpack_packed(got, B, cfg.max_det)
            got_cat = torch.cat([g_counts.view(world, -1).view(torch.uint8).view(world, -1),
                                 g_results.reshape(world, -1)], dim=1)
            gather_checked = bool(torch.equal(got_cat, ref_all))
            if not gather_checked:
                raise RuntimeError("record gather: rank 0 did not receive every rank's records")

    # ---- per-kernel durations (CUDA events recorded by the library on the launching stream), same inputs
    eng.set_profiling(True)
    acc = np.zeros(5)
    for _ in range(args.steps):
        step(overlap=False)                  # serialised on one stream so that each event pair brackets one kernel
        acc += np.array(eng.stage_ms())
    eng.set_profiling(False)
    stage_ms = (acc / args.steps).tolist()
    res = eng.results_to_numpy(outs[2])
    n_det_mean = float(outs[1].float().mean().item())

    # ---- end to end through the C ABI with HOST (pinned) buffers: H2D + K1..K5 + D2H every step, both feeding modes
    h_np = [host["frames"].numpy()] + [l.numpy() for l in host_lv] + [host["coef"].numpy(), host["proto"].numpy()]
    e2e_steps = max(2, min(args.steps, 10))
    e2e, e2e_out = e2e_host(eng, cfg, h_np, B, e2e_steps, world, dev, barrier, yuyv=cfg.frame_w % 2 == 0)
    e2e_value, h2d, d2h = e2e["value"], e2e["h2d_bytes_per_step"], e2e["d2h_bytes_per_step"]
    probe = _allgather_floats([h2d_probe(dev, world, barrier)], world, dev)[:, 0]
    # ---- the same, through the Python drop-in (app.B200Predictor.run) with the backbone's output staying on the device:
    #      only the frames cross PCIe (informational; the headline e2e above also ships the head tensors from the host)
    from vision_textile_inspection_b200.app import B200Predictor
    ecfg = eng.cfg
    pred = B200Predictor(lambda net: (d_lv[0], d_lv[1], d_lv[2], d_coef, d_proto), ecfg.K, ecfg.dist, ecfg.R, ecfg.t,
                         device=dev, undistort=cfg.undistort, nc=cfg.nc, roi=cfg.roi(), variant=cfg.variant, channel_flip=0)
    pred.extra = dict(max_px_distance=ecfg.max_px_distance)
    f_host = host["frames"].numpy()
    for _ in range(2):
        pred.run(f_host, cfg.conf, cfg.iou, cfg.max_det, cfg.imgsz, export_masks=False)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        pred.run(f_host, cfg.conf, cfg.iou, cfg.max_det, cfg.imgsz, export_masks=False)
    barrier()
    fo_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([fo_s], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        fo_s = float(t.item())
    e2e_frames_only = {"value": world * B * e2e_steps / fo_s, "unit": UNIT, "h2d_bytes_per_step": int(f_host.nbytes),
                       "d2h_bytes_per_step": int(d2h), "steps": e2e_steps,
                       "api": "app.B200Predictor.run: frames from pinned host memory, head tensors produced on the device"}

    # ---- single-frame latency of the drop-in call path (the reference processes one frame per call, main.py:211)
    pred1 = B200Predictor(lambda net: (d_lv[0][:1], d_lv[1][:1], d_lv[2][:1], d_coef[:1], d_proto[:1]), ecfg.K, ecfg.dist,
                          ecfg.R, ecfg.t, device=dev, undistort=cfg.undistort, nc=cfg.nc, roi=cfg.roi(),
                          variant=cfg.variant, channel_flip=0)
    pred1.extra = dict(max_px_distance=ecfg.max_px_distance)
    f1 = f_host[:1]
    lat = []
    for i in range(33):
        t1 = time.perf_counter()
        pred1.run(f1, cfg.conf, cfg.iou, cfg.max_det, cfg.imgsz, export_masks=False)
        if i >= 3:
            lat.append(1e3 * (time.perf_counter() - t1))
    latency = {"ms_median": float(np.median(lat)), "ms_p90": float(np.percentile(lat, 90)), "frames": 1,
               "api": "app.B200Predictor.run, one frame from host memory to host records (H2D + K1..K5 + D2H)"}

    # ---- the OTHER step form, timed the same way (informational): with --step-form graph this is the two-stream form
    #      (six launches per step, streams joined only at the ends), with --step-form streams the graph form
    other = None
    if world == 1 and args.post_streams == 1:
        if graphs is not None:
            def other_step():
                step(use_graph=False)
            name = "streams"
        else:
            g_alt = eng.capture_step(d_frames, d_lv[0], d_lv[1], d_lv[2], d_coef, d_proto, net_in=net_in, outputs=outs)[0]
            other_step, name = g_alt.replay, "graph"
        fork()
        for _ in range(3):
            other_step()
        join()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        g0.record()
        fork()
        for _ in range(args.steps):
            other_step()
        join()
        g1.record()
        torch.cuda.synchronize()
        o_ms = g0.elapsed_time(g1) / args.steps
        other = {"step_form": name, "ms_per_step": o_ms, "frames_per_s": B / (o_ms * 1e-3)}

    # ---- the whole frame with a stand-in network between pre and post (SURVEY 8f rank 1; informational, --backbone n|s|m)
    full_frame = None
    if args.backbone and world == 1:
        from vision_textile_inspection_b200.backbone import make_standin_backbone
        bb = make_standin_backbone(cfg.nc, args.backbone, dev, dtype=torch.bfloat16)
        pipe = eng.capture_pipeline(bb, B)
        pipe.frames.copy_(d_frames)

        def timed(fn, n):
            for _ in range(3):
                fn()
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            a0.record()
            for _ in range(n):
                fn()
            a1.record()
            torch.cuda.synchronize()
            return a0.elapsed_time(a1) / n
        t_full = timed(pipe.replay, max(3, args.steps // 2))
        g_net = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g_net):
            bb(pipe.net_in, out=pipe.head)
        t_net = timed(g_net.replay, max(3, args.steps // 2))
        t_ours = float(sum(stage_ms))
        full_frame = {"backbone": f"stand-in YOLOv8{args.backbone}-seg topology, random weights, bf16 autocast, channels_last, "
                                  f"{sum(p.numel() for p in bb.net.parameters()) / 1e6:.2f} M parameters (PyTorch / cuDNN)",
                      "one_cuda_graph": "K1 -> backbone -> K2 -> K3 -> K4 -> K5, head tensors written in place into the buffers K2-K4 read",
                      "ms_per_batch_whole_frame": t_full, "ms_per_batch_backbone_alone": t_net,
                      "ms_per_batch_pre_post_measure_serial": t_ours, "frames_per_s_whole_frame": B / (t_full * 1e-3),
                      "share_of_pre_post_measure": t_ours / t_full, "head_in_place": bool(pipe.in_place),
                      "note": "with random weights the head produces few / arbitrary detections: K2-K5 see less work "
                              "than on the planted tensors of the headline; the share uses the headline's stage times"}
    # ---- compressed ingest (SURVEY 8f rank 2; informational, --jpeg): camera MJPEG frames decoded by nvJPEG on the device
    ingest_jpeg = None
    if args.jpeg and world == 1:
        import cv2
        jp = [cv2.imencode(".jpg", f, [cv2.IMWRITE_JPEG_QUALITY, 90])[1].tobytes() for f in batch["frames"]]
        fr = torch.empty_like(d_frames)

        def _time(fn, reps=5):
            for _ in range(2):
                fn()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(reps):
                fn()
            torch.cuda.synchronize()
            return (time.perf_counter() - t0) / reps

        def _whole(**kw):
            eng.decode_jpeg_batch(jp, out=fr, **kw)
            eng.preprocess(fr, out=net_in)
            eng.post_measure(d_lv[0], d_lv[1], d_lv[2], d_coef, d_proto, outputs=outs)
            outs[1].cpu()

        one_s = _time(lambda: eng.decode_jpeg_batch(jp, out=fr, one_by_one=True), reps=3)
        by_lanes = {}
        for lanes in (1, 2, 4, 8):                      # host threads the batch is split over (vti_decode_jpeg_batch lanes)
            os.environ["VTI_JPEG_LANES"] = str(lanes)
            by_lanes[lanes] = B / _time(lambda: eng.decode_jpeg_batch(jp, out=fr))
        best = max(by_lanes, key=by_lanes.get)
        os.environ["VTI_JPEG_LANES"] = str(best)
        dec_s = B / by_lanes[best]
        tot_s = _time(_whole)
        os.environ.pop("VTI_JPEG_LANES")
        ingest_jpeg = {"jpeg_bytes_per_frame": int(np.mean([len(j) for j in jp])), "raw_bytes_per_frame": int(batch["frames"][0].nbytes),
                       "backend": eng.jpeg_backend(),
                       "decode_frames_per_s": B / dec_s, "decode_pre_post_measure_frames_per_s": B / tot_s,
                       "decode_one_by_one_frames_per_s": B / one_s, "lanes": best,
                       "decode_frames_per_s_by_lanes": {str(k): v for k, v in by_lanes.items()},
                       "api": "engine.decode_jpeg_batch (vti_decode_jpeg_batch: nvjpegDecodeBatched, JPEG bytes on the host) -> K1..K5, "
                              "head tensors on the device; one_by_one = vti_decode_jpeg (single-image hybrid decoder)"}
    # ---- BASELINE configs[4]: the 4K stream split over the ranks (every N > 1; --cfg5 forces it at N = 1)
    cfg5 = None
    if (world > 1 or args.cfg5) and not args.no_cfg5:
        cfg5 = run_cfg5_sharded(args, rank, world, dev, barrier, calib, use_peer=(args.gather == "peer"))
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    # ---- roofline of the dominant kernel
    peak, peak_src = peaks()
    sb = stage_bytes(cfg, n_det_mean)                                      # SURVEY 8d figures (whole_path, roofline)
    sb_read = stage_bytes(cfg, n_det_mean, float(res["n_cand"].mean()))   # K2 = what it must read
    names = ["K1", "K2", "K3", "K4", "K5"]
    dom = int(np.argmax(stage_ms))
    achieved = B * sb_read[names[dom]] / (stage_ms[dom] * 1e-3) / 1e9
    traffic = None
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):
        try:
            traffic = json.load(open(tp)).get(cfg.name, {}).get(names[dom])
        except Exception:
            traffic = None
    total_bytes = B * sum(sb.values())
    # ---- CPU baseline on a bounded sample (rank 0, N=1 only)
    cpu = None
    if world == 1 and not args.no_cpu:
        n_cpu = args.cpu_frames
        fps, dt, cores = cpu_reference(cfg, batch, calib, n_cpu, single_thread_frames=6)
        workers = os.cpu_count() or 1
        par_fps, par_s = cpu_reference_parallel(args.config, batch, calib, 4, workers)
        kind, kind_txt = cpu_kind()
        cpu = {"value": par_fps, "unit": UNIT, "cores": workers, "kind": kind,
               "sample": f"frame-parallel: {workers} single-threaded processes x 4 frames of {cfg.name} in {par_s:.1f}s "
                         f"(batch-1 loop per process: {kind_txt}); the reference's own one-process loop with library threading: "
                         f"{fps:.2f} frames/s over {n_cpu} frames in {dt:.1f}s; threads={cores}"}
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8/f32 (integer resize+remap, f32 decode/NMS/masks, f64 measure)", "data": "synthetic",
        "config": {"workload": cfg.name, "frames_per_gpu_per_step": B, "frame": [cfg.frame_w, cfg.frame_h],
                   "net_in": [cfg.LW, cfg.LH], "anchors": cfg.anchors, "undistort": cfg.undistort,
                   "conf": cfg.conf, "iou": cfg.iou, "max_det": cfg.max_det, "mean_dets_per_frame": n_det_mean,
                   "l2": f"inputs+outputs per step {(in_bytes + out_bytes) / 1e6:.0f} MB > 126 MB L2, no flush needed",
                   "unique_frames": n_unique, "rank_cpu_affinity": affinity, "streams": ("one CUDA graph per step: K1 beside K2-K5 on a forked high-priority branch, joined at the end of the graph; the record gather on its own stream (double-buffered records)"
                               if graphs is not None else
                               "K1 || K2-K5 on two streams (post at high priority) + the record gather on a third (double-buffered records), joined at the ends of the timed region"),
                   "step_form": "graph" if graphs is not None else "streams",
                   "post_streams": args.post_streams,
                   "gather": ("none (1 GPU)" if world == 1 else
                              "peer memory: per rank and step one copy-engine copy of the packed records into rank 0's symmetric buffer + signal, no collective kernel"
                              if peer is not None else "NCCL all-gather of the packed records"),
                   "gather_checked": gather_checked,
                   "clock_sampling": "nvidia-smi every 100 ms over the timed steps + an untimed continuation of the same loop",
                   "status_ok_frames": int((res["status"] == 0).sum())},
        "clocks": clocks,
        "spread": {"ms_per_step_regions": [m / args.steps for m in region_ms],
                   "rel_spread": (max(region_ms) - min(region_ms)) / min(region_ms),
                   "note": "three back-to-back timed regions of K steps; `value` is the first"},
        "gpu_launches": int(launches),
        "e2e": dict(e2e, unit=UNIT,
                    h2d_probe_gbs_per_rank=[round(float(v), 2) for v in probe],
                    h2d_probe_gbs_all_ranks=round(float(probe.sum()), 2),
                    api="vti_process_host: pinned host buffers, 4-chunk copy/compute pipeline.  mode zero_copy: the frames "
                        "are DMA-copied, the head tensors are read in place over PCIe: class planes + candidate box logits "
                        "(K2), kept coefficient rows (K3), the union rectangle of the crop windows of the prototypes (fetch "
                        "kernel before K4).  mode dma: every presented byte is copied.  value = the faster mode at this N; "
                        "h2d_probe = plain pinned copies issued by all ranks at once (what the host can feed N GPUs)"),
        "e2e_frames_only": e2e_frames_only,
        "latency_single_frame": latency,
        "other_step_form": other,
        "roofline": {"bound": "hbm", "kernel": names[dom], "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": B * sb_read[names[dom]]},
        "stage_ms": dict(zip(names, stage_ms)),
        "stage_gbs": {n: (B * sb_read[n] / (t * 1e-3) / 1e9 if t > 0 else None) for n, t in zip(names, stage_ms)},
        "whole_path": {"algorithmic_bytes_per_frame": sum(sb.values()),
                       "hbm_roofline_frames_per_s": peak * 1e9 / sum(sb.values()),
                       "frac_of_hbm_roofline": (total_bytes / (ms / args.steps * 1e-3) / 1e9) / peak},
    }
    if cfg5 is not None:
        line["cfg5_sharded"] = cfg5
    if full_frame is not None:
        line["full_frame"] = full_frame
    if ingest_jpeg is not None:
        line["ingest_jpeg"] = ingest_jpeg
    if cpu is not None:
        line["cpu_baseline"] = cpu
    print(json.dumps(line), file=REAL_STDOUT, flush=True)
    if last_out is not None:
        write_dump(args.dump_outputs, dump_arrays(last_out[0].cpu().numpy(), eng.dets_to_numpy(last_out[1]),
                                                  last_out[2].cpu().numpy(), eng.results_to_numpy(last_out[3])))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="cfg2")
    ap.add_argument("--batch", type=int, default=None)
    ap.add_argument("--cpu-frames", type=int, default=24)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--unique", type=int, default=64, help="distinct synthetic frames / head tensors per rank (<= batch)")
    ap.add_argument("--backbone", default=None, choices=["n", "s", "m"],
                    help="also time the whole frame (K1 -> stand-in YOLOv8-seg network -> K2..K5) as one CUDA graph")
    ap.add_argument("--jpeg", action="store_true", help="also time compressed ingest (nvJPEG decode of JPEG frames on the device)")
    ap.add_argument("--cfg5", action="store_true", help="also run the cfg5_sharded block at N = 1")
    ap.add_argument("--no-cfg5", action="store_true", help="skip the cfg5_sharded block at N > 1")
    ap.add_argument("--cfg5-frames", type=int, default=256)
    ap.add_argument("--load-steps", type=int, default=1500, help="untimed continuation for the clock sampler")
    ap.add_argument("--step-form", default="graph", choices=["graph", "streams"],
                    help="graph: one CUDA graph replay per step; streams: the six kernels issued on two streams per step")
    ap.add_argument("--post-streams", type=int, default=0, choices=[0, 1, 2],
                    help="2: the post stages of consecutive batches overlap (two handles, two post streams); measured: no "
                         "gain on cfg2 (K1-bound, 221 vs 226 k frames/s), +50 %% on the post-bound stress config cfg4")
    ap.add_argument("--gather", default="peer", choices=["peer", "nccl"],
                    help="N > 1: records to rank 0 through NVLink peer memory (default) or an NCCL all-gather")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (rank 0's batch) as DIR/<name>.npy, at most 64 MB")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    _protect_stdout()
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    from vision_textile_inspection_b200 import synth
    cfg = synth.CONFIGS[args.config]
    if args.impl == "reference":
        run_reference(args, cfg, rank, world)
    else:
        run_b200(args, cfg, rank, world, local_rank)


if __name__ == "__main__":
    main()

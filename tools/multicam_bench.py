"""What several cameras behind one handle cost: cfg2 (1280x720, undistort, imgsz 960), B = 64, with C cameras assigned
round-robin to the frames of the batch, against the one-camera handle in the same process.

Each camera has its own K1 remap table (about 4.2 MB at cfg2, DESIGN.md 3).  One table stays in L2 across the batch;
at C cameras a batch touches C tables, and past about 30 of them they no longer fit the 126 MB L2.  Per variant this
reports the graph-replay step time (engine.capture_step: K1 beside K2..K5, as bench.py times it) and the K1 time
alone (CUDA events around back-to-back vti_preprocess[_multi] calls), both as the median over rounds in which the
variants alternate, with the spread.  The 64 input frames (177 MB) exceed L2, as in bench.py.

    python tools/multicam_bench.py [--cameras 1,2,8,32,64] [--rounds 5] [--steps 50] [--out result.json]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def gpu_identity(index: int) -> dict:
    """Name, power limit and maximum SM clock of the card, read when the numbers are taken."""
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), f"--query-gpu={q}", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [s.strip() for s in out.split(",")]
        return {"gpu": name, "power_limit": power, "sm_clock_max": clock}
    except Exception as e:  # noqa: BLE001
        return {"gpu": None, "power_limit": None, "sm_clock_max": None, "nvidia_smi": f"unavailable ({e})"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cameras", default="1,2,8,32,64")
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=50, help="graph replays per timed window")
    ap.add_argument("--k1-calls", type=int, default=50, help="K1 calls per timed window")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    from test_multi_camera import camera_set
    from vision_textile_inspection_b200 import synth
    from vision_textile_inspection_b200.engine import EngineConfig, InspectionEngine, load_reference_calibration

    if not torch.cuda.is_available():
        raise SystemExit("multicam_bench needs a CUDA device")
    dev = torch.device("cuda", 0)
    cfg = synth.CONFIGS["cfg2"]
    B = args.batch
    batch = synth.make_batch(cfg, B, seed0=2000, n_unique=8)
    cu = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    frames, lv, coef, proto = cu(batch["frames"]), [cu(x) for x in batch["levels"]], cu(batch["coef"]), cu(batch["proto"])
    calib = load_reference_calibration()

    variants = {"one-camera handle": (InspectionEngine(EngineConfig.for_workload(cfg, calib, max_batch=B), dev), None)}
    for C in [int(c) for c in args.cameras.split(",")]:
        ec = EngineConfig.for_workload(cfg, calib, max_batch=B)
        ec.cameras = camera_set(cfg.frame_h, cfg.frame_w, C)
        ids = torch.arange(B, dtype=torch.int32, device=dev) % C
        variants[f"{C} cameras"] = (InspectionEngine(ec, dev), ids)

    graphs = {}
    for name, (eng, ids) in variants.items():
        net_in = torch.empty((B, 3, eng.LH, eng.LW), dtype=torch.float32, device=dev)
        graphs[name] = (eng.capture_step(frames, *lv, coef, proto, net_in=net_in, camera=ids)[0], net_in)

    def time_graph(name):
        g = graphs[name][0]
        g.replay()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            g.replay()
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1) / args.steps

    def time_k1(name):
        eng, ids = variants[name]
        out = graphs[name][1]
        eng.preprocess(frames, out=out, camera=ids)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.k1_calls):
            eng.preprocess(frames, out=out, camera=ids)
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1) / args.k1_calls

    ident = gpu_identity(0)
    step = {n: [] for n in variants}
    k1 = {n: [] for n in variants}
    for r in range(args.rounds):                               # variants alternate within every round
        order = list(variants) if r % 2 == 0 else list(reversed(variants))
        for n in order:
            step[n].append(time_graph(n))
            k1[n].append(time_k1(n))
    rows = []
    for n, (eng, _) in variants.items():
        s, k = np.array(step[n]), np.array(k1[n])
        rows.append({"variant": n, "cameras": eng.n_cameras,
                     "step_ms_median": round(float(np.median(s)), 4), "step_ms_min": round(float(s.min()), 4),
                     "step_ms_max": round(float(s.max()), 4), "frames_per_s": round(B / float(np.median(s)) * 1e3),
                     "k1_ms_median": round(float(np.median(k)), 4), "k1_ms_min": round(float(k.min()), 4),
                     "k1_ms_max": round(float(k.max()), 4)})
    res = {"workload": "cfg2 1280x720 undistort imgsz 960", "batch": B, "rounds": args.rounds, "steps": args.steps,
           "k1_calls": args.k1_calls, **ident, "torch_device_name": torch.cuda.get_device_name(dev), "rows": rows}
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()

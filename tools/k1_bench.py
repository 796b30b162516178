"""K1-only microbench for kernel tuning (not the headline bench): times vti_preprocess alone on one config with CUDA
events and checks the output bit-exactly against real cv2 (cv2.undistort + resize + copyMakeBorder, as Ultralytics' LetterBox).  Several library variants are
loaded into ONE process and timed in interleaved rounds, so clock ramp-up and order effects hit all of them alike.  Build
each variant side by side, then pass them all:
    VTI_LIB=tools/_variants/libvti_A.so VTI_NVCC_FLAGS="-D..." python vision_textile_inspection_b200/build.py --force
    python tools/k1_bench.py [--libs tools/_variants/libvti_*.so]"""
import argparse
import glob
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="cfg2")
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--libs", nargs="*", default=None)
    ap.add_argument("--check", type=int, default=2, help="frames compared with cv2")
    a = ap.parse_args()
    os.environ["VTI_NO_BUILD"] = "1" if a.libs else os.environ.get("VTI_NO_BUILD", "")
    import torch
    from vision_textile_inspection_b200 import _lib, synth
    from vision_textile_inspection_b200.engine import EngineConfig, InspectionEngine
    cfg = synth.CONFIGS[a.config]
    B = a.batch
    base = np.stack([synth.fabric_frame(cfg, 4242 + i) for i in range(min(B, 4))])
    frames = np.ascontiguousarray(np.concatenate([base] * ((B + len(base) - 1) // len(base)))[:B])
    libs = a.libs or [None]
    engs = []
    for path in libs:
        if path is not None:
            _lib._lib, _lib.LIB_PATH = None, os.path.abspath(path)
        engs.append(InspectionEngine(EngineConfig.for_workload(cfg, max_batch=B), device="cuda:0"))
    d = torch.from_numpy(frames).cuda()
    out = torch.empty((B, 3, engs[0].LH, engs[0].LW), dtype=torch.float32, device="cuda")
    ref = None
    if a.check:
        import cv2
        # Ultralytics LetterBox on real cv2 (tests/ hold the oracle proper; this tool only needs a checker for variants)
        ec, LH, LW = engs[0].cfg, engs[0].LH, engs[0].LW
        r = min(cfg.imgsz / cfg.frame_h, cfg.imgsz / cfg.frame_w)
        nw, nh = int(round(cfg.frame_w * r)), int(round(cfg.frame_h * r))
        top, left = int(round((LH - nh) / 2 - 0.1)), int(round((LW - nw) / 2 - 0.1))
        outs = []
        for f in frames[:a.check]:
            if cfg.undistort:
                f = cv2.undistort(f, np.asarray(ec.K, np.float64), np.asarray(ec.dist, np.float64))
            if (nw, nh) != (cfg.frame_w, cfg.frame_h):
                f = cv2.resize(f, (nw, nh), interpolation=cv2.INTER_LINEAR)
            f = cv2.copyMakeBorder(f, top, LH - nh - top, left, LW - nw - left, cv2.BORDER_CONSTANT, value=(114, 114, 114))
            outs.append(np.ascontiguousarray(f.transpose(2, 0, 1)).astype(np.float32) / np.float32(255.0))
        ref = np.stack(outs)
    ok, ts = [], [[] for _ in engs]
    for eng in engs:
        out.zero_()
        for _ in range(3):
            eng.preprocess(d, out=out)
        torch.cuda.synchronize()
        ok.append(None if ref is None else bool(np.array_equal(out[:a.check].cpu().numpy(), ref)))
    for _ in range(a.rounds):
        for k, eng in enumerate(engs):
            eng.preprocess(d, out=out)
            for _ in range(a.iters):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                eng.preprocess(d, out=out)
                e1.record()
                torch.cuda.synchronize()
                ts[k].append(e0.elapsed_time(e1) * 1e3)
    bytes_alg = B * (3 * cfg.frame_h * cfg.frame_w + 12 * engs[0].LH * engs[0].LW)
    for k, path in enumerate(libs):
        med = float(np.median(ts[k]))
        tag = "default" if path is None else os.path.basename(path).replace("libvti_", "").replace(".so", "")
        print(json.dumps({"tag": tag, "config": a.config, "B": B, "us_median": round(med, 2),
                          "us_min": round(float(np.min(ts[k])), 2), "us_p90": round(float(np.percentile(ts[k], 90)), 2),
                          "bit_exact": ok[k], "frac_of_6543": round(bytes_alg / med / 1e3 / 6543.1, 4)}), flush=True)


if __name__ == "__main__":
    main()

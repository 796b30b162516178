"""Host-layer guarantees of a libvti handle: the host-buffer path issues the same post chain as the stream entry points,
closing a handle leaves the caller's current device alone, and a handle gives back every allocation it made."""
import numpy as np
import pytest
import torch

import helpers
from vision_textile_inspection_b200 import _lib, synth
from vision_textile_inspection_b200.engine import EngineConfig, InspectionEngine

pytestmark = pytest.mark.gpu


def make_engine(cfg, max_batch, device=None, **over):
    ec = EngineConfig.for_workload(cfg, helpers.load_calib(), max_batch=max_batch)
    for k, v in over.items():
        setattr(ec, k, v)
    return InspectionEngine(ec, device=device)


@pytest.mark.parametrize("pinned", [False, True])
def test_host_path_matches_device_path_when_every_mask_is_evaluated(pinned):
    """Mask variant B evaluates every kept detection's mask, routed or not; the host path exports no masks, so this is
    the setting in which it does.  vti_process_host then evaluates the masks of the detections outside the ROI exactly
    as vti_post_measure does, with the head tensors copied or read in place (pinned: zero copy plus the prototype
    fetch, whose rectangle must cover those detections too)."""
    cfg = synth.CONFIGS["cfg2"]
    B = 3
    batch = synth.make_batch(cfg, B, seed0=2000)
    # the synthetic stitch rows span the frame's width: an ROI ending at 3/4 of it leaves the right quarter's outside
    on, x_min, _, y_min, y_max = cfg.roi()
    eng = make_engine(cfg, B, mask_variant=1, roi=(on, x_min, cfg.frame_w * 3 // 4, y_min, y_max))
    heads = [*batch["levels"], batch["coef"], batch["proto"]]
    host = [batch["frames"]] + heads
    if pinned:
        keep = [torch.from_numpy(np.ascontiguousarray(a)).pin_memory() for a in host]
        host = [t.numpy() for t in keep]
    dets, counts, results, net_in = eng.process_host(*host, want_net_in=True)
    cu = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    d2, c2, r2, _ = eng.post_measure(*[cu(x) for x in heads])
    n2 = eng.preprocess(cu(batch["frames"])).cpu().numpy()
    d2, c2, r2 = eng.dets_to_numpy(d2), c2.cpu().numpy(), eng.results_to_numpy(r2)
    outside = [int(((d2[b, :c2[b]]["flags"] & _lib.F_IN_ROI) == 0).sum()) for b in range(B)]
    assert sum(outside) > 0, "the scenes must contain kept detections outside the ROI"
    assert np.array_equal(net_in, n2)
    assert np.array_equal(counts, c2)
    for f in results.dtype.names:                 # field by field, bit for bit: padding belongs to neither buffer
        assert results[f].tobytes() == r2[f].tobytes(), f
    for f in dets.dtype.names:
        for b in range(B):
            assert dets[b, :counts[b]][f].tobytes() == d2[b, :c2[b]][f].tobytes(), (b, f)


def test_close_keeps_the_callers_current_device():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    eng = make_engine(synth.CONFIGS["cfg1"], 1, device="cuda:1")
    torch.cuda.set_device(0)
    eng.close()
    assert torch.cuda.current_device() == 0


def test_memory_returns_after_close():
    """Five rounds of create, process_host (staging buffers), set_profiling(True) (events), close: the device's free
    memory comes back.  One handle per round needs about 60 MB at this size, so a leak of any of its buffers shows."""
    cfg = synth.CONFIGS["cfg2"]
    B = 2
    batch = synth.make_batch(cfg, B, seed0=2000)
    args = [batch["frames"], *batch["levels"], batch["coef"], batch["proto"]]

    def one_round():
        eng = make_engine(cfg, B)
        eng.process_host(*args)
        eng.set_profiling(True)
        eng.close()

    one_round()                                   # warm-up: module loads and context growth stay
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info()[0]
    for _ in range(5):
        one_round()
    torch.cuda.synchronize()
    drop = free0 - torch.cuda.mem_get_info()[0]
    print(f"\nfree device memory after 5 rounds: {drop / 2**20:+.1f} MB lower")
    assert drop <= 8 << 20

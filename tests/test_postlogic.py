"""SURVEY 8f rank 4: the per-frame record logic of main.py:213-293 (offsets, validity window, 5-deep
fallback buffers, travelled distance, DB row) -- product state machine vs the line-by-line restatement, same jitter."""
import random

import numpy as np

from oracle import main_logic_ref
from vision_textile_inspection_b200.postlogic import SeamRecordLogic


def _sequence(seed, n=400):
    rng = np.random.default_rng(seed)
    ms, counts, c = [], [], 0
    for _ in range(n):
        kind = rng.integers(0, 6)
        seam = None if kind == 0 else float(rng.uniform(3.0, 11.0))
        width = None if kind == 1 else float(rng.uniform(3.0, 6.0))
        ms.append({"edge_distance_mm": seam, "stitch_width_mm": width, "stitch_count": int(rng.integers(0, 40))})
        c += int(rng.integers(0, 4)) if rng.random() > 0.1 else 0        # encoder sometimes stands still
        counts.append(c)
    return ms, counts


def test_record_logic_matches_main_py_restatement():
    for seed in range(5):
        ms, counts = _sequence(seed)
        ref = main_logic_ref.run(ms, counts, random.Random(seed).uniform, total_distance_mm=12.5)
        logic = SeamRecordLogic(total_distance_mm=12.5, jitter=random.Random(seed).uniform)
        got = [logic.update(m, c).row for m, c in zip(ms, counts)]
        assert got == ref
        assert any(r is None for r in got) and any(r is not None for r in got)


def test_known_answers():
    logic = SeamRecordLogic(jitter=lambda a, b: 0.0)
    # 6.8 - 1.3 = 5.5 in (3.5, 8.0); 4.4 - 1.0 = 3.4 in (2.8, 4.15): valid, 3 stitches travelled
    r = logic.update({"edge_distance_mm": 6.8, "stitch_width_mm": 4.4}, 3)
    assert r.measured and r.row == dict(total_distance=round(3 * 3.4, 1), stitch_length=3.4, seam_allowance=5.5)
    # invalid seam (9.9 - 1.3 = 8.6 > 8.0): falls back to the buffer means (4 primed values + the one above)
    r = logic.update({"edge_distance_mm": 9.9, "stitch_width_mm": 4.4}, 5)
    assert not r.measured and r.valid
    assert abs(r.seam_allowance_mm - (4 * 6.5 + 5.5) / 5) < 1e-12 and abs(r.stitch_length_mm - (4 * 3.9 + 3.4) / 5) < 1e-12
    # no encoder movement: nothing is inserted even with a valid measurement
    assert logic.update({"edge_distance_mm": 6.8, "stitch_width_mm": 4.4}, 5).row is None
    # process_frame error dict ('Fabric not detected'): both None -> buffered values
    r = logic.update({"edge_distance_mm": None, "stitch_width_mm": None, "error": "Fabric not detected"}, 6)
    assert r.valid and not r.measured and r.row is not None


def test_record_logic_matches_the_verbatim_main_py_block():
    """Pinned against the reference itself: oracle/main_verbatim.py executes main.py:214-293 as it stands in the
    reference's file (constants from the reference's config module), with the same seeded jitter stream."""
    import pytest
    from oracle import main_verbatim
    from vision_textile_inspection_b200 import postlogic
    if not main_verbatim.available():
        pytest.skip("needs a checkout of the reference at oracle/_ref/ or VTI_REFERENCE_DIR")
    for seed in range(5):
        ms, counts = _sequence(seed)
        ref, ns = main_verbatim.run(ms, counts, seed, total_distance_mm=12.5)
        # the product's defaults are the reference's config values
        assert (ns["SEAM_LENGTH_OFFSET"], ns["STITCH_WIDTH_OFFSET"]) == (postlogic.SEAM_LENGTH_OFFSET, postlogic.STITCH_WIDTH_OFFSET)
        assert (ns["Seam_lower_limit"], ns["Seam_upper_limit"]) == postlogic.SEAM_LIMITS
        assert (ns["stitch_lower_limit"], ns["stitch_upper_limit"]) == postlogic.STITCH_LIMITS
        logic = SeamRecordLogic(total_distance_mm=12.5, jitter=random.Random(seed).uniform)
        got = [logic.update(m, c).row for m, c in zip(ms, counts)]
        assert got == ref
        assert abs(logic.total_distance_mm - ns["total_distance_mm"]) < 1e-9
        assert main_logic_ref.run(ms, counts, random.Random(seed).uniform, total_distance_mm=12.5) == ref

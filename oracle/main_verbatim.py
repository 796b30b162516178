"""TEST INFRASTRUCTURE ONLY -- runs the record logic of the reference's main.py VERBATIM.

main.py:main() is one long camera loop and cannot be imported and called piecewise, but the lines that
turn process_frame's dict into a database row (from `current_stitch_count = serial_reader.get_stitch_count()` down to
the `db.insert_measurement(...)` call, main.py:214-293) are plain Python on local names.  This module cuts exactly
those lines out of the reference's own file (where it lies: oracle/_ref/ or VTI_REFERENCE_DIR, see
oracle/ref_verbatim.py), de-indents them and executes them, once per frame, in a namespace that supplies the names
the block reads: the constants from the reference's config module, stub `serial_reader` / `db` objects, the deques and
counters the loop keeps, and `random` (seeded by the caller).  No line of the block is restated here.
"""
from __future__ import annotations

import contextlib
import io
import os
import random
import textwrap
from collections import deque

from . import ref_verbatim

START = "current_stitch_count = serial_reader.get_stitch_count()"
END = "# Update total distance"


def available() -> bool:
    return ref_verbatim.available() and os.path.isfile(os.path.join(ref_verbatim.REF, "main.py"))


def _block() -> str:
    src = open(os.path.join(ref_verbatim.REF, "main.py"), encoding="utf-8").read().splitlines()
    i0 = next(i for i, l in enumerate(src) if START in l)
    i1 = next(i for i, l in enumerate(src) if END in l and i > i0)
    return textwrap.dedent("\n".join(src[i0:i1]))


class _Serial:
    def __init__(self):
        self.count = 0

    def get_stitch_count(self):
        return self.count


class _Db:
    def __init__(self):
        self.rows = []

    def insert_measurement(self, **kw):
        self.rows.append(kw)
        return True


def run(measurements_seq, stitch_counts, seed: int, total_distance_mm: float = 0.0):
    """Returns, per frame, the keyword dict main.py handed to db.insert_measurement (None where it inserted nothing)."""
    ref_verbatim._stubs()
    import sys
    if ref_verbatim.REF not in sys.path:
        sys.path.insert(0, ref_verbatim.REF)
    with contextlib.redirect_stdout(io.StringIO()), contextlib.redirect_stderr(io.StringIO()):
        import config as ref_config                      # the reference's own constants (offsets, validity window)
    code = compile(_block(), "main.py[214:293]", "exec")
    rnd = random.Random(seed)
    ns = {k: getattr(ref_config, k) for k in dir(ref_config) if not k.startswith("_")}
    ns.update(random=rnd, serial_reader=_Serial(), db=_Db(), last_stitch_count=0, total_distance_mm=float(total_distance_mm),
              valid_seam_buffer=deque([6.5] * 5, maxlen=5), valid_width_buffer=deque([3.9] * 5, maxlen=5), LOG_DEBUG=False)
    out = []
    for m, c in zip(measurements_seq, stitch_counts):
        ns["serial_reader"].count = c
        ns["measurements"] = dict(m)
        n0 = len(ns["db"].rows)
        with contextlib.redirect_stdout(io.StringIO()):
            exec(code, ns)
        out.append(ns["db"].rows[-1] if len(ns["db"].rows) > n0 else None)
    return out, ns

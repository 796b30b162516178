"""Post-boundary record logic (SURVEY.md 8f rank 4) -- what main.py does with the dict that
process_frame returns, frame after frame, before the database row is written (main.py:213-293):

  offsets (config.py:156-157) -> validity window (config.py:147-150) -> 5-deep buffers of the last valid values,
  primed with 6.5 / 3.9 (main.py:183-184) -> fallback to the buffer mean + a small random jitter when the frame has
  no valid measurement (main.py:270-275) -> travelled distance = stitch-count delta x stitch width (main.py:280-283)
  -> the row (total_distance, stitch_length, seam_allowance), each rounded to 0.1 (main.py:287-291,
  database.py:98-111).

Pure host state machine, frame-ordered like the temporal median: in a multi-GPU run it is applied to the gathered
per-frame results in frame order.  The jitter source is injectable so that the logic is testable bit-for-bit.
"""
from __future__ import annotations

import random
from collections import deque
from dataclasses import dataclass, field

SEAM_LENGTH_OFFSET, STITCH_WIDTH_OFFSET = -1.3, -1.0            # config.py:156-157 (env-overridable there)
SEAM_LIMITS, STITCH_LIMITS = (3.5, 8.0), (2.8, 4.15)            # config.py:147-150 (exclusive bounds)


@dataclass
class FrameRecord:
    seam_allowance_mm: float | None
    stitch_length_mm: float | None
    valid: bool                    # a measured or buffered value is available
    measured: bool                 # this frame's own measurement passed the validity window
    stitch_delta: int
    moved_distance_mm: float
    total_distance_mm: float
    row: dict | None = None        # what DatabaseHandler.insert_measurement receives, or None when nothing is inserted


@dataclass
class SeamRecordLogic:
    seam_offset: float = SEAM_LENGTH_OFFSET
    width_offset: float = STITCH_WIDTH_OFFSET
    seam_limits: tuple = SEAM_LIMITS
    stitch_limits: tuple = STITCH_LIMITS
    total_distance_mm: float = 0.0            # main.py:168 starts from the last DB row
    last_stitch_count: int = 0
    jitter: object = random.uniform           # main.py:273-274
    seam_buf: deque = field(default_factory=lambda: deque([6.5] * 5, maxlen=5))
    width_buf: deque = field(default_factory=lambda: deque([3.9] * 5, maxlen=5))

    def update(self, measurements: dict, stitch_count: int | None = None) -> FrameRecord:
        """One inspected frame: `measurements` is process_frame's dict, `stitch_count` the encoder reading
        (None = no serial reader: the count does not move, main.py:214)."""
        cur = self.last_stitch_count if stitch_count is None else stitch_count
        delta = cur - self.last_stitch_count
        self.last_stitch_count = cur
        seam = measurements.get("edge_distance_mm", None)
        width = measurements.get("stitch_width_mm", None)
        if seam is not None:
            seam += self.seam_offset
        if width is not None:
            width += self.width_offset
        valid_seam = seam is not None and self.seam_limits[0] < seam < self.seam_limits[1]
        valid_width = width is not None and self.stitch_limits[0] < width < self.stitch_limits[1]
        measured = valid = valid_seam and valid_width
        if measured:
            self.seam_buf.append(seam)
            self.width_buf.append(width)
        elif len(self.seam_buf) > 0 and len(self.width_buf) > 0:
            seam = sum(self.seam_buf) / len(self.seam_buf) + self.jitter(-0.1, 0.1)
            width = sum(self.width_buf) / len(self.width_buf) + self.jitter(-0.08, 0.08)
            valid = True
        moved, row = 0.0, None
        if delta > 0 and valid:
            moved = delta * width
            self.total_distance_mm += moved
            row = dict(total_distance=round(self.total_distance_mm, 1), stitch_length=round(width, 1),
                       seam_allowance=round(seam, 1))
        return FrameRecord(seam, width, valid, measured, delta, moved, self.total_distance_mm, row)

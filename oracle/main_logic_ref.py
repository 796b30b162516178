"""TEST INFRASTRUCTURE ONLY -- line-by-line restatement of the per-frame record logic that lives inline in
main.py:main() (:167-168, :183-184, :213-293).  It cannot be imported from the reference (it is the
body of a `while True` loop around a camera, a serial port and MySQL), so it is restated here with the same variable
names and the same statement order; tests/test_postlogic.py drives it and the product's SeamRecordLogic with the same
measurement sequence and the same jitter stream.  Parity unpinned by the reference (no tests, no recorded rows)."""
from collections import deque

Seam_upper_limit, stitch_upper_limit, Seam_lower_limit, stitch_lower_limit = 8.0, 4.15, 3.5, 2.8   # config.py:147-150
SEAM_LENGTH_OFFSET, STITCH_WIDTH_OFFSET = -1.3, -1.0                                                # config.py:156-157


def run(measurement_dicts, stitch_counts, uniform, total_distance_mm=0.0):
    """Returns the list of insert_measurement keyword dicts (None where main.py inserts nothing)."""
    last_stitch_count = 0                                   # main.py:167
    valid_seam_buffer = deque([6.5] * 5, maxlen=5)          # main.py:183
    valid_width_buffer = deque([3.9] * 5, maxlen=5)         # main.py:184
    rows = []
    for measurements, current_stitch_count in zip(measurement_dicts, stitch_counts):
        stitch_delta = current_stitch_count - last_stitch_count           # :221
        last_stitch_count = current_stitch_count                          # :222
        seam_length_mm = measurements.get('edge_distance_mm', None)       # :225
        stitch_width_mm = measurements.get('stitch_width_mm', None)       # :226
        if seam_length_mm is not None:                                    # :229-232
            seam_length_mm += SEAM_LENGTH_OFFSET
        if stitch_width_mm is not None:
            stitch_width_mm += STITCH_WIDTH_OFFSET
        valid_seam = seam_length_mm is not None and Seam_lower_limit < seam_length_mm < Seam_upper_limit      # :250-253
        valid_stitch = stitch_width_mm is not None and stitch_lower_limit < stitch_width_mm < stitch_upper_limit
        has_valid_measurement = valid_seam and valid_stitch               # :260
        if has_valid_measurement:                                         # :262-265
            valid_seam_buffer.append(seam_length_mm)
            valid_width_buffer.append(stitch_width_mm)
        else:                                                             # :270-275
            if len(valid_seam_buffer) > 0 and len(valid_width_buffer) > 0:
                seam_length_mm = sum(valid_seam_buffer) / len(valid_seam_buffer) + uniform(-0.1, 0.1)
                stitch_width_mm = sum(valid_width_buffer) / len(valid_width_buffer) + uniform(-0.08, 0.08)
                has_valid_measurement = True
        row = None
        if stitch_delta > 0 and has_valid_measurement:                    # :280-291
            moved_distance_mm = stitch_delta * stitch_width_mm
            total_distance_mm += moved_distance_mm
            row = dict(total_distance=round(total_distance_mm, 1), stitch_length=round(stitch_width_mm, 1),
                       seam_allowance=round(seam_length_mm, 1))
        rows.append(row)
    return rows

"""TEST INFRASTRUCTURE ONLY -- CPU port of the reference's measure stage (the part of the hot path that lives in
the reference's own files).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import this.

Follows, step by step (SURVEY.md 8a rows M1-M8):
  variant 0: measurement.py:44-65 (plane, pixel->world), :70-86 (instance bitmap), :88-113 (k-means),
             :160-185 (union, lower envelope), :188-511 (process_frame, numbers only -- no drawing)
  variant 1: Utils/check_stitch_distance.py:57-80, :85-111, :143-171, :226-251, :281-553

It makes the same library calls in the same order as the reference (cv2.resize INTER_NEAREST on the full
letterboxed mask, cv2.moments, np.any/np.where, cv2.undistortPoints, np.median/np.mean), so timing it is timing the
reference's algorithm, and it is pinned against the reference itself: oracle/gen_golden.py imports the verbatim
reference modules (oracle/ref_verbatim.py) and tests/test_oracle_measure.py checks this port against the
vectors it wrote to tests/golden/ (plus the known-answer vectors of SURVEY.md 8c).

Unlike the reference it returns every intermediate (per-stitch centroids, widths, selections) so the CUDA
records can be compared field by field.
"""
from __future__ import annotations

from collections import deque
from dataclasses import dataclass, field

import cv2
import numpy as np


@dataclass
class MeasureConfig:
    K: np.ndarray
    dist: np.ndarray
    R: np.ndarray
    t: np.ndarray
    variant: int = 0                      # 0 measurement.py, 1 check_stitch_distance.py
    roi: tuple = (1, 10, 1270, 300, 760)  # enabled, x_min, x_max, y_min, y_max   (config.py:91-95)
    stitch_id: int = 0
    fabric_id: int = 1
    min_stitches: int = 3                 # config.py:79
    max_px_distance: int = 250            # config.py:81 (150 in check_stitch_distance.py:38)
    neighborhood: int = 3                 # config.py:82
    n_c: np.ndarray = field(default=None)
    d_c: float = 0.0

    def __post_init__(self):
        self.K = np.asarray(self.K, np.float64).reshape(3, 3)
        self.dist = np.asarray(self.dist, np.float64).ravel()
        self.R = np.asarray(self.R, np.float64).reshape(3, 3)
        self.t = np.asarray(self.t, np.float64).reshape(3)
        self.n_c, self.d_c = camera_plane(self.R, self.t)


def rodrigues(rvec) -> np.ndarray:
    R, _ = cv2.Rodrigues(np.asarray(rvec, np.float64).reshape(3, 1))
    return R


def camera_plane(R, t):
    """measurement.py:44-48."""
    n_c = np.asarray(R)[:, 2].astype(np.float64)
    return n_c, -float(n_c.dot(t))


def undistort_point_spec(u, v, K, dist):
    """cv2.undistortPoints(P=None) restated: exactly 5 fixed-point iterations (SURVEY 8a M5)."""
    k1, k2, p1, p2, k3 = [float(x) for x in np.asarray(dist).ravel()[:5]]
    x0 = (float(u) - K[0, 2]) * (1.0 / K[0, 0])          # OpenCV multiplies by ifx = 1./fx: bit-exact this way
    y0 = (float(v) - K[1, 2]) * (1.0 / K[1, 1])
    x, y = x0, y0
    for _ in range(5):
        r2 = x * x + y * y
        icd = 1.0 / (1.0 + ((k3 * r2 + k2) * r2 + k1) * r2)
        dx = 2.0 * p1 * x * y + p2 * (r2 + 2.0 * x * x)
        dy = p1 * (r2 + 2.0 * y * y) + 2.0 * p2 * x * y
        x = (x0 - dx) * icd
        y = (y0 - dy) * icd
    return x, y


def pixel_to_world(u, v, c: MeasureConfig):
    """measurement.py:50-65 -- ray through the undistorted pixel intersected with the fabric plane."""
    pts = np.array([[[float(u), float(v)]]], dtype=np.float64)
    und = cv2.undistortPoints(pts, c.K, c.dist, P=None)
    ray = np.array([float(und[0, 0, 0]), float(und[0, 0, 1]), 1.0], dtype=np.float64)
    den = float(c.n_c.dot(ray))
    if abs(den) < 1e-9:
        return None
    return c.R.T.dot((-c.d_c / den) * ray - c.t)


def defect_area_mm2(bitmap: np.ndarray, c: MeasureConfig):
    """Spec of vti_det.area_mm2 (the north-star's "area"; the reference itself never outputs one -- it only uses m00 as
    a centroid denominator, measurement.py:304-307 -- so this numpy function IS the definition, not a restatement).

    Area of the frame-resolution bitmap on the fabric plane: (number of set pixels) x (plane area of one pixel at the
    bitmap's centroid), the latter as |dP/du x dP/dv| by central differences (+-0.5 px) of the reference's own
    pixel -> world projection (pixel_to_world above = measurement.py:50-65).  mm^2; None if the bitmap is empty."""
    M = cv2.moments(bitmap)
    if M["m00"] <= 0:
        return None
    cx, cy = M["m10"] / M["m00"], M["m01"] / M["m00"]
    pts = [pixel_to_world(cx - 0.5, cy, c), pixel_to_world(cx + 0.5, cy, c),
           pixel_to_world(cx, cy - 0.5, c), pixel_to_world(cx, cy + 0.5, c)]
    if any(p is None for p in pts):
        return None
    du, dv = pts[1] - pts[0], pts[3] - pts[2]
    return float(M["m00"]) * float(np.linalg.norm(np.cross(du, dv))) * 1e6


def instance_bitmap(mask_lb: np.ndarray, h: int, w: int):
    """measurement.py:70-86 -- nearest-resize the WHOLE letterboxed mask (pad rows included) to the frame."""
    arr = np.asarray(mask_lb)
    if arr.shape != (h, w):
        arr = cv2.resize(arr, (w, h), interpolation=cv2.INTER_NEAREST)
    m = (arr > 0).astype(np.uint8)
    return m if np.count_nonzero(m) > 0 else None


def kmeans2(values: np.ndarray, update_on_break: bool, max_iters: int = 10) -> np.ndarray:
    """measurement.py:88-113 (labels NOT updated on break) / check_stitch_distance.py:143-171 (updated)."""
    if values.size < 2:
        return np.zeros(values.shape[0], dtype=int)
    c0, c1 = float(values.min()), float(values.max())
    labels = np.zeros(values.shape[0], dtype=int)
    for _ in range(max_iters):
        nl = (np.abs(values - c1) < np.abs(values - c0)).astype(int)
        if nl.sum() == 0 or nl.sum() == len(values):
            if update_on_break:
                labels = nl
            break
        n0 = float(values[nl == 0].mean()) if (nl == 0).any() else c0
        n1 = float(values[nl == 1].mean()) if (nl == 1).any() else c1
        if n0 == c0 and n1 == c1:
            if update_on_break:
                labels = nl
            break
        c0, c1, labels = n0, n1, nl
    return labels


def fabric_envelope(fabric: np.ndarray, upper: bool) -> np.ndarray:
    """measurement.py:170-185 (bottom-most row per column) / check_stitch_distance.py:238-251 (top-most); -1 = none."""
    h, w = fabric.shape
    if upper:
        has = fabric.any(axis=0)
        idx = np.argmax(fabric > 0, axis=0)
        return np.where(has, idx, -1).astype(int)
    rev = fabric[::-1, :]
    has = rev.any(axis=0)
    idx = np.argmax(rev > 0, axis=0)
    return np.where(has, h - 1 - idx, -1).astype(int)


def _neigh_env(envelope, cx_int, w, nb):
    xs = [int(np.clip(cx_int + dx, 0, w - 1)) for dx in range(-nb, nb + 1)]
    return [envelope[x] for x in xs if envelope[x] >= 0]


def measure_frame(cls_arr, boxes, masks, h: int, w: int, c: MeasureConfig) -> dict:
    """Everything process_frame computes after model.predict, minus drawing and the temporal median.

    cls_arr (N,), boxes (N,4) frame px float32, masks (N,LH,LW) nonzero=set (or None)."""
    out = dict(status="ok", stitches=[], widths=[], dists=[], selected=[], final=[], avg_dist=None, avg_width=None,
               n_dist=0, n_width=0, envelope=None, det_route=[])
    cls_arr = np.asarray(cls_arr)
    boxes = np.asarray(boxes)
    roi = None
    if c.variant == 0 and c.roi[0]:
        x_min = max(0, min(int(c.roi[1]), w - 1))
        x_max = max(0, min(int(c.roi[2]), w - 1))
        y_min = max(0, min(int(c.roi[3]), h - 1))
        y_max = max(0, min(int(c.roi[4]), h - 1))
        if x_min < x_max and y_min < y_max:
            roi = (x_min, y_min, x_max, y_max)
    st_masks, st_boxes, fab_masks = [], [], []
    for i, cid in enumerate(cls_arr):
        cid = int(cid)
        x1, y1, x2, y2 = map(int, boxes[i])
        if roi is not None:
            bx, by = 0.5 * (x1 + x2), 0.5 * (y1 + y2)
            if not (roi[0] <= bx <= roi[2] and roi[1] <= by <= roi[3]):
                out["det_route"].append(-1)
                continue
        m = instance_bitmap(masks[i], h, w) if masks is not None else None
        if cid == c.stitch_id:
            st_masks.append(m)
            st_boxes.append((x1, y1, x2, y2))
            out["det_route"].append(0)
        elif cid == c.fabric_id:
            if m is not None:
                fab_masks.append(m)
            elif c.variant == 1:
                tmp = np.zeros((h, w), dtype=np.uint8)
                cv2.rectangle(tmp, (x1, y1), (x2, y2), 1, -1)
                fab_masks.append(tmp)
            out["det_route"].append(1)
        else:
            out["det_route"].append(-2)
    fabric = None
    if fab_masks:
        fabric = np.zeros((h, w), dtype=np.uint8)
        for m in fab_masks:
            fabric = cv2.bitwise_or(fabric, m)
    if fabric is None or np.count_nonzero(fabric) == 0:
        out["status"] = "no_fabric"
        return out
    env = fabric_envelope(fabric, upper=(c.variant == 1))
    out["envelope"] = env
    cys = []
    for k, m in enumerate(st_masks):
        x1, y1, x2, y2 = st_boxes[k]
        if m is not None and m.sum() > 0:
            M = cv2.moments((m > 0).astype(np.uint8))
            ok = (M["m00"] > 1e-6) if c.variant == 0 else (M["m00"] != 0)
            if ok:
                cx, cy = float(M["m10"] / M["m00"]), float(M["m01"] / M["m00"])
            else:
                cx, cy = float((x1 + x2) / 2), float((y1 + y2) / 2)
            cols = np.where(np.any(m > 0, axis=0))[0]
            if cols.size > 0:
                left, right = float(cols.min()), float(cols.max())
            else:
                left, right = float(x1), float(x2)
            m00 = int(M["m00"])
        else:
            cx, cy = float((x1 + x2) / 2), float((y1 + y2) / 2)
            left, right = float(x1), float(x2)
            m00 = 0
        out["stitches"].append(dict(cx=cx, cy=cy, left=left, right=right, m00=m00, box=(x1, y1, x2, y2)))
        cys.append(cy)
    if not cys:
        out["status"] = "no_stitch"
        return out
    n = len(cys)

    def width_of(i):
        s = out["stitches"][i]
        pl = pixel_to_world(s["left"], s["cy"], c)
        pr = pixel_to_world(s["right"], s["cy"], c)
        if pl is not None and pr is not None:
            return float(np.linalg.norm(pr - pl)) * 1000.0
        if c.variant == 1:
            pa = pixel_to_world(s["cx"], s["cy"], c)
            pb = pixel_to_world(s["cx"] + 10, s["cy"], c)
            if pa is not None and pb is not None:
                return ((s["right"] - s["left"]) / 10.0) * float(np.linalg.norm(pb - pa)) * 1000.0
        return None

    if c.variant == 0:
        for i in range(n):
            wmm = width_of(i)
            out["stitches"][i]["width_mm"] = wmm
            if wmm is not None:
                out["widths"].append(wmm)
    # row selection
    labels = np.zeros(n, dtype=int)
    chosen = 0
    if n >= 2:
        vals = np.array(cys)
        labels = kmeans2(vals, update_on_break=(c.variant == 1))
        valid = env[env >= 0]
        if valid.size > 0:
            fm = float(np.mean(valid))
            m0 = float(vals[labels == 0].mean()) if (labels == 0).any() else 1e9
            m1 = float(vals[labels == 1].mean()) if (labels == 1).any() else 1e9
            chosen = 0 if abs(m0 - fm) < abs(m1 - fm) else 1
        selected = [i for i, lab in enumerate(labels) if lab == chosen]
    else:
        selected = list(range(n))
    final = []
    for i in selected:
        s = out["stitches"][i]
        ev = _neigh_env(env, int(round(s["cx"])), w, c.neighborhood)
        if not ev:
            continue
        env_y = int(round(float(np.median(ev))))
        if c.variant == 0:
            ok = abs(float(s["cy"]) - float(env_y)) < c.max_px_distance
        else:
            ok = 0 < (float(s["cy"]) - float(env_y)) < c.max_px_distance
        if ok:
            final.append(i)
    if not final:
        final = selected
    out["selected"], out["final"] = selected, final
    for i in final:
        s = out["stitches"][i]
        cx_int = int(np.clip(int(round(s["cx"])), 0, w - 1))
        ev = _neigh_env(env, cx_int, w, c.neighborhood)
        if ev:
            edge_y = float(np.median(ev))
            ps = pixel_to_world(s["cx"], s["cy"], c)
            pe = pixel_to_world(s["cx"], edge_y, c)
            if ps is not None and pe is not None:
                d = float(np.linalg.norm(ps - pe)) * 1000.0
                s["dist_mm"], s["edge_y"] = d, edge_y
                out["dists"].append(d)
        if c.variant == 1:
            wmm = width_of(i)
            s["width_mm"] = wmm
            if wmm is not None:
                out["widths"].append(wmm)
    out["n_dist"], out["n_width"] = len(out["dists"]), len(out["widths"])
    if out["n_dist"] >= c.min_stitches:
        out["avg_dist"] = float(np.mean(out["dists"]))
    if out["n_width"] >= c.min_stitches:
        out["avg_width"] = float(np.mean(out["widths"]))
    return out


class TemporalMedian:
    """measurement.py:149-150, 474-484 -- two 8-deep deques, median over the valid averages, frame order."""

    def __init__(self, depth: int = 8):
        self.d = deque(maxlen=depth)
        self.w = deque(maxlen=depth)

    def push(self, avg_dist, avg_width):
        sd = sw = None
        if avg_dist is not None:
            self.d.append(avg_dist)
            sd = float(np.median(self.d))
        if avg_width is not None:
            self.w.append(avg_width)
            sw = float(np.median(self.w))
        return sd, sw


_ERR = {"no_fabric": "Fabric not detected", "no_stitch": "No stitches detected"}


def result_dict(m: dict, smooth: TemporalMedian) -> dict:
    """The dict process_frame returns (measurement.py:285-287, 335-337, 506-511), minus the timestamp."""
    if m["status"] != "ok":
        return dict(edge_distance_mm=None, stitch_width_mm=None, stitch_count=0, error=_ERR[m["status"]])
    sd, sw = smooth.push(m["avg_dist"], m["avg_width"])
    return dict(edge_distance_mm=sd, stitch_width_mm=sw, stitch_count=m["n_dist"])

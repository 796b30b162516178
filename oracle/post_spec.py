"""TEST INFRASTRUCTURE ONLY -- deterministic float32 specification of the YOLOv8-seg head post-processing.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import this.

The arithmetic restated here lives in `ultralytics` (unpinned, requirements.txt:13), reached from
measurement.py:208-210 (`self.model.predict(rgb, conf=..., iou=..., max_det=..., imgsz=960)`) and
Utils/check_stitch_distance.py:286.  `ultralytics` is not vendored in the reference and is not
installed, so this restates its published algorithm (SURVEY.md 8a rows U3-U7):

  U3  Detect/Segment head tail: DFL softmax-expectation over 16 bins, dist2bbox(xywh), x stride, class sigmoid
  U4  ops.non_max_suppression: best class, `> conf` (strict), xywh->xyxy, class offset 7680, torchvision nms, [:max_det]
  U5  torchvision.ops.nms CPU kernel: stable descending sort, greedy, suppress iff IoU > thr (float vs double compare)
  U7  ops.scale_boxes + clip_boxes

Every float32 operation is a single IEEE-754 rounded mul/add/sub/div in a fixed order (no FMA), and exp() is a fully
specified Cody-Waite + degree-7 polynomial (`exp_spec`), so a CUDA kernel using __fmul_rn/__fadd_rn/__fdiv_rn is
*bit-identical* to this file.  oracle/ultra_ref.py runs the same stages with the real torch / torchvision operators;
tests/test_oracle_post.py pins this spec against it (exact where the operators are exactly rounded, <= 2 ulp where
torch's vectorised expf is involved).
"""
from __future__ import annotations

import numpy as np

F32 = np.float32
REG_MAX = 16
MAX_WH = F32(7680.0)

_LOG2E = F32(1.4426950408889634)
_LN2_HI = F32(0.693359375)             # 9 significant bits: n * LN2_HI is exact for |n| < 2^15
_LN2_LO = F32(-2.12194440e-4)
_EXP_C = [F32(1.0 / 5040.0), F32(1.0 / 720.0), F32(1.0 / 120.0), F32(1.0 / 24.0), F32(1.0 / 6.0), F32(0.5),
          F32(1.0), F32(1.0)]


def exp_spec(x: np.ndarray) -> np.ndarray:
    """exp(x) in float32, bit-reproducible: clamp to [-86, 88], n = rint(x*log2e), r = x - n*ln2 (two-step),
    Horner degree 7 with separately rounded mul and add, scale by 2^n."""
    x = np.clip(np.asarray(x, F32), F32(-86.0), F32(88.0)).astype(F32)
    n = np.rint(x * _LOG2E).astype(F32)
    r = (x - n * _LN2_HI).astype(F32)
    r = (r - n * _LN2_LO).astype(F32)
    p = np.full_like(r, _EXP_C[0])
    for c in _EXP_C[1:]:
        p = (p * r).astype(F32)
        p = (p + c).astype(F32)
    return np.ldexp(p, n.astype(np.int32)).astype(F32)


def sigmoid_spec(x: np.ndarray) -> np.ndarray:
    """1 / (1 + exp_spec(-x)), IEEE division."""
    e = exp_spec(-np.asarray(x, F32))
    return (F32(1.0) / (F32(1.0) + e)).astype(F32)


def level_shapes(LH: int, LW: int, strides=(8, 16, 32)):
    return [(LH // s, LW // s) for s in strides]


def decode_spec(levels, nc: int, strides=(8, 16, 32)):
    """U3.  levels: list of (64+nc, Hl, Wl) float32 for ONE frame.

    Returns xywh (A,4) float32 in letterbox px, cls_prob (A,nc) float32.  Anchor order: level 8 first, row-major."""
    xywh_all, cls_all = [], []
    karr = np.arange(REG_MAX, dtype=F32)
    for p, s in zip(levels, strides):
        p = np.asarray(p, F32)
        C, Hl, Wl = p.shape
        assert C == 4 * REG_MAX + nc
        box = p[:4 * REG_MAX].reshape(4, REG_MAX, Hl * Wl)
        m = box.max(axis=1, keepdims=True)
        e = exp_spec((box - m).astype(F32))
        S = np.zeros((4, Hl * Wl), F32)
        for k in range(REG_MAX):
            S = (S + e[:, k]).astype(F32)
        d = np.zeros((4, Hl * Wl), F32)
        for k in range(REG_MAX):
            pk = (e[:, k] / S).astype(F32)
            d = (d + (karr[k] * pk).astype(F32)).astype(F32)
        ys, xs = np.divmod(np.arange(Hl * Wl), Wl)
        ax = (xs.astype(F32) + F32(0.5)).astype(F32)
        ay = (ys.astype(F32) + F32(0.5)).astype(F32)
        x1 = (ax - d[0]).astype(F32)
        y1 = (ay - d[1]).astype(F32)
        x2 = (ax + d[2]).astype(F32)
        y2 = (ay + d[3]).astype(F32)
        cx = ((x1 + x2).astype(F32) / F32(2.0)).astype(F32)
        cy = ((y1 + y2).astype(F32) / F32(2.0)).astype(F32)
        w = (x2 - x1).astype(F32)
        h = (y2 - y1).astype(F32)
        st = F32(s)
        xywh_all.append(np.stack([cx * st, cy * st, w * st, h * st], 1).astype(F32))
        cls_all.append(sigmoid_spec(p[4 * REG_MAX:].reshape(nc, Hl * Wl)).T.astype(F32))
    return np.concatenate(xywh_all, 0), np.concatenate(cls_all, 0)


def candidates_spec(xywh: np.ndarray, cls_prob: np.ndarray, conf_thres: float):
    """U4 prelude: best class, strict `> conf`, xywh->xyxy.  Order preserved (ascending anchor index)."""
    conf = cls_prob.max(axis=1)
    j = cls_prob.argmax(axis=1)                       # first maximum, as torch.max on CPU
    sel = np.nonzero(conf > F32(conf_thres))[0]
    hw = (xywh[sel, 2] / F32(2.0)).astype(F32)
    hh = (xywh[sel, 3] / F32(2.0)).astype(F32)
    xyxy = np.stack([xywh[sel, 0] - hw, xywh[sel, 1] - hh, xywh[sel, 0] + hw, xywh[sel, 1] + hh], 1).astype(F32)
    return sel.astype(np.int32), xyxy, conf[sel].astype(F32), j[sel].astype(np.int32)


def nms_spec(xyxy: np.ndarray, scores: np.ndarray, cls: np.ndarray, iou_thres: float, max_det: int):
    """U4/U5: class-offset greedy NMS.  Returns indices into the candidate list, in descending-score order."""
    n = xyxy.shape[0]
    if n == 0:
        return np.zeros((0,), np.int64)
    off = (cls.astype(F32) * MAX_WH).astype(F32)[:, None]
    b = (xyxy + off).astype(F32)
    x1, y1, x2, y2 = b[:, 0], b[:, 1], b[:, 2], b[:, 3]
    areas = ((x2 - x1).astype(F32) * (y2 - y1).astype(F32)).astype(F32)
    order = np.argsort(-scores.astype(np.float64), kind="stable")     # ties -> lower candidate index first
    suppressed = np.zeros(n, bool)
    keep = []
    thr = float(iou_thres)                                             # compared in double, like the C++ kernel
    for _i in range(n):
        i = order[_i]
        if suppressed[i]:
            continue
        keep.append(i)
        if len(keep) >= max_det:
            break
        rest = order[_i + 1:]
        xx1 = np.maximum(x1[i], x1[rest])
        yy1 = np.maximum(y1[i], y1[rest])
        xx2 = np.minimum(x2[i], x2[rest])
        yy2 = np.minimum(y2[i], y2[rest])
        w = np.maximum(F32(0.0), (xx2 - xx1).astype(F32))
        h = np.maximum(F32(0.0), (yy2 - yy1).astype(F32))
        inter = (w * h).astype(F32)
        den = ((areas[i] + areas[rest]).astype(F32) - inter).astype(F32)
        with np.errstate(divide="ignore", invalid="ignore"):
            ovr = (inter / den).astype(F32)
        suppressed[rest[ovr.astype(np.float64) > thr]] = True
    return np.asarray(keep, np.int64)


def scale_boxes_spec(xyxy_lb: np.ndarray, LH: int, LW: int, h: int, w: int) -> np.ndarray:
    """U7: letterbox px -> frame px, clipped.  gain/pad are Python doubles; the tensor math is float32."""
    gain = min(LH / h, LW / w)
    padx = int(round((LW - w * gain) / 2 - 0.1))
    pady = int(round((LH - h * gain) / 2 - 0.1))
    b = np.array(xyxy_lb, F32, copy=True)
    b[:, [0, 2]] = (b[:, [0, 2]] - F32(padx)).astype(F32)
    b[:, [1, 3]] = (b[:, [1, 3]] - F32(pady)).astype(F32)
    b = (b / F32(gain)).astype(F32)
    b[:, [0, 2]] = np.clip(b[:, [0, 2]], F32(0), F32(w))
    b[:, [1, 3]] = np.clip(b[:, [1, 3]], F32(0), F32(h))
    return b


def postprocess_spec(levels, coef, conf_thres, iou_thres, max_det, nc, LH, LW, h, w):
    """U3+U4+U5+U7 for one frame.  coef: (32, A).  Returns a dict of numpy arrays (kept detections, score order)."""
    xywh, cls_prob = decode_spec(levels, nc)
    sel, xyxy, conf, cls = candidates_spec(xywh, cls_prob, conf_thres)
    keep = nms_spec(xyxy, conf, cls, iou_thres, max_det)
    anchors = sel[keep]
    return dict(
        n_cand=int(sel.size), cand_anchor=sel, cand_xyxy=xyxy, cand_conf=conf, cand_cls=cls,
        keep_anchor=anchors.astype(np.int32), box_lb=xyxy[keep], conf=conf[keep], cls=cls[keep],
        box_frame=scale_boxes_spec(xyxy[keep], LH, LW, h, w) if keep.size else np.zeros((0, 4), F32),
        coef=np.ascontiguousarray(np.asarray(coef, F32)[:, anchors].T),
    )

"""TEST INFRASTRUCTURE ONLY -- the reference CPU pre/post path, assembled from the REAL third-party operators.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import this.

measurement.py:208-210 calls `ultralytics` `YOLO.predict`; ultralytics is a pip dependency
(requirements.txt:13, unpinned), absent from the reference and not installed here.  This module
restates what that call does around the backbone (SURVEY.md 8a U0-U7), using the same operators ultralytics itself
calls -- cv2.resize / cv2.copyMakeBorder / cv2.undistort, torch softmax / sigmoid / matmul / F.interpolate,
torchvision.ops.nms -- so the third-party CPU kernels stay in the loop.  It is both the parity oracle for the CUDA
path and the timed CPU baseline.  parity unpinned by the reference (it has no tests); pinned instead against
cv2/torch/torchvision themselves and against oracle/post_spec.py + oracle/cv_fixed.py.

Mask variant: "A" of SURVEY 8a U6 (sigmoid -> crop -> bilinear upsample -> > 0.5), no empty-mask drop.
"""
from __future__ import annotations

import cv2
import numpy as np
import torch
import torch.nn.functional as Fnn
import torchvision

from .cv_fixed import letterbox_geometry

REG_MAX = 16
MAX_WH = 7680


def letterbox(img: np.ndarray, imgsz: int = 960, stride: int = 32) -> np.ndarray:
    """ultralytics.data.augment.LetterBox(auto=True, scaleup=True, center=True) [U1]."""
    h, w = img.shape[:2]
    g = letterbox_geometry(h, w, imgsz, stride)
    if (w, h) != (g["new_w"], g["new_h"]):
        img = cv2.resize(img, (g["new_w"], g["new_h"]), interpolation=cv2.INTER_LINEAR)
    return cv2.copyMakeBorder(img, g["top"], g["bottom"], g["left"], g["right"], cv2.BORDER_CONSTANT,
                              value=(114, 114, 114))


def preprocess(frames, imgsz: int = 960, stride: int = 32, undistort=None, flip_channels: bool = False) -> torch.Tensor:
    """U0+U1+U2 for a list/array of HxWx3 uint8 frames -> (B,3,LH,LW) float32 in [0,1].

    `frames` are what the network should see in plane order 0,1,2 unless flip_channels (see SURVEY N1: the reference
    converts BGR->RGB at measurement.py:205 and ultralytics flips it back, so the planes are the camera's B,G,R).
    `undistort` = (K, dist) enables the north-star image-level cv2.undistort before the letterbox."""
    out = []
    for f in frames:
        if undistort is not None:
            f = cv2.undistort(f, np.asarray(undistort[0], np.float64), np.asarray(undistort[1], np.float64))
        out.append(letterbox(f, imgsz, stride))
    im = np.stack(out)
    if flip_channels:
        im = im[..., ::-1]
    im = np.ascontiguousarray(im.transpose(0, 3, 1, 2))
    t = torch.from_numpy(im).float()
    t /= 255
    return t


def decode(levels, nc: int, strides=(8, 16, 32)) -> torch.Tensor:
    """Detect._inference + DFL + dist2bbox [U3].  levels: list of (B, 64+nc, Hl, Wl).  -> (B, 4+nc, A)."""
    B = levels[0].shape[0]
    no = 4 * REG_MAX + nc
    x_cat = torch.cat([xi.reshape(B, no, -1) for xi in levels], 2)
    anchors, strides_t = [], []
    for xi, s in zip(levels, strides):
        Hl, Wl = xi.shape[2:]
        sx = torch.arange(Wl, dtype=torch.float32) + 0.5
        sy = torch.arange(Hl, dtype=torch.float32) + 0.5
        sy, sx = torch.meshgrid(sy, sx, indexing="ij")
        anchors.append(torch.stack((sx, sy), -1).view(-1, 2))
        strides_t.append(torch.full((Hl * Wl, 1), float(s), dtype=torch.float32))
    anchors = torch.cat(anchors).transpose(0, 1)
    strides_t = torch.cat(strides_t).transpose(0, 1)
    box, cls = x_cat.split((4 * REG_MAX, nc), 1)
    b, _, a = box.shape
    p = box.view(b, 4, REG_MAX, a).transpose(2, 1).softmax(1)          # (b,16,4,a)
    wgt = torch.arange(REG_MAX, dtype=torch.float32).view(1, REG_MAX, 1, 1)
    dist = Fnn.conv2d(p, wgt).view(b, 4, a)                              # DFL's frozen 1x1 conv
    lt, rb = dist.chunk(2, 1)
    x1y1 = anchors.unsqueeze(0) - lt
    x2y2 = anchors.unsqueeze(0) + rb
    c_xy = (x1y1 + x2y2) / 2
    wh = x2y2 - x1y1
    dbox = torch.cat((c_xy, wh), 1) * strides_t
    return torch.cat((dbox, cls.sigmoid()), 1)


def non_max_suppression(pred: torch.Tensor, conf_thres: float, iou_thres: float, max_det: int, nc: int):
    """ops.non_max_suppression (agnostic=False, multi_label=False, no time limit) [U4/U5].

    pred: (B, 4+nc+nm, A).  Returns per image (rows (x1,y1,x2,y2,conf,cls,coef...), anchor index per row)."""
    mi = 4 + nc
    xc = pred[:, 4:mi].amax(1) > conf_thres
    pred = pred.transpose(-1, -2).clone()
    xy, wh = pred[..., :2].clone(), pred[..., 2:4] / 2
    pred[..., :2] = xy - wh
    pred[..., 2:4] = xy + wh
    out = []
    for xi, x in enumerate(pred):
        idx = torch.nonzero(xc[xi]).view(-1)
        x = x[xc[xi]]
        if not x.shape[0]:
            out.append((x.new_zeros((0, 6 + x.shape[1] - mi)), idx))
            continue
        box, cls, mask = x.split((4, nc, x.shape[1] - mi), 1)
        conf, j = cls.max(1, keepdim=True)
        keep0 = conf.view(-1) > conf_thres
        x = torch.cat((box, conf, j.float(), mask), 1)[keep0]
        idx = idx[keep0]
        c = x[:, 5:6] * MAX_WH
        i = torchvision.ops.nms(x[:, :4] + c, x[:, 4], iou_thres)[:max_det]
        out.append((x[i], idx[i]))
    return out


def crop_mask(masks: torch.Tensor, boxes: torch.Tensor) -> torch.Tensor:
    n, h, w = masks.shape
    x1, y1, x2, y2 = torch.chunk(boxes[:, :, None], 4, 1)
    r = torch.arange(w, dtype=x1.dtype)[None, None, :]
    c = torch.arange(h, dtype=x1.dtype)[None, :, None]
    return masks * ((r >= x1) * (r < x2) * (c >= y1) * (c < y2))


def process_mask(proto: torch.Tensor, coef: torch.Tensor, boxes_lb: torch.Tensor, shape, variant: str = "A",
                 return_soft: bool = False):
    """ops.process_mask(upsample=True) [U6].  proto (32,ph,pw), coef (N,32), boxes (N,4) letterbox px.

    variant "A" (Ultralytics <= 8.0.x, the north-star wording): sigmoid -> crop -> bilinear x4 -> > 0.5.
    variant "B" (newer releases, SURVEY 8a U6): NO sigmoid, crop, bilinear x4, > 0.0 (the caller additionally drops
    detections whose mask is empty: see postprocess(mask_variant="B")).  The crop is the float-compare crop_mask in
    both (the rounded-slice crop newer releases use for n < 50 on CPU is not reproduced: SURVEY 8a marks it optional).
    return_soft: also return the float map before the threshold (tests check that a pixel that differs from the CUDA
    path sits on the threshold to within float rounding)."""
    c, mh, mw = proto.shape
    ih, iw = shape
    masks = (coef @ proto.float().view(c, -1))
    if variant == "A":
        masks = masks.sigmoid()
    masks = masks.view(-1, mh, mw)
    db = boxes_lb.clone()
    db[:, 0] *= mw / iw
    db[:, 2] *= mw / iw
    db[:, 3] *= mh / ih
    db[:, 1] *= mh / ih
    masks = crop_mask(masks, db)
    if masks.shape[0]:
        masks = Fnn.interpolate(masks[None], shape, mode="bilinear", align_corners=False)[0]
    else:
        masks = masks.new_zeros((0, ih, iw))
    soft = masks.clone() if return_soft else None
    hard = masks.gt_(0.5 if variant == "A" else 0.0)
    return (hard, soft) if return_soft else hard


def scale_boxes(img1_shape, boxes: torch.Tensor, img0_shape) -> torch.Tensor:
    """ops.scale_boxes + clip_boxes [U7] (in place on a clone)."""
    boxes = boxes.clone()
    gain = min(img1_shape[0] / img0_shape[0], img1_shape[1] / img0_shape[1])
    pad = (round((img1_shape[1] - img0_shape[1] * gain) / 2 - 0.1),
           round((img1_shape[0] - img0_shape[0] * gain) / 2 - 0.1))
    boxes[..., [0, 2]] -= pad[0]
    boxes[..., [1, 3]] -= pad[1]
    boxes[..., :4] /= gain
    boxes[..., 0].clamp_(0, img0_shape[1])
    boxes[..., 1].clamp_(0, img0_shape[0])
    boxes[..., 2].clamp_(0, img0_shape[1])
    boxes[..., 3].clamp_(0, img0_shape[0])
    return boxes


class _Boxes:
    def __init__(self, xyxy, conf, cls):
        self.xyxy, self.conf, self.cls = xyxy, conf, cls


class _Masks:
    def __init__(self, data):
        self.data = data


class RefResults:
    """Shaped like ultralytics Results where measurement.py reads it (measurement.py:74-75, 242-245)."""

    def __init__(self, xyxy, conf, cls, masks, box_lb, anchors):
        self.boxes = _Boxes(xyxy, conf, cls)
        self.masks = _Masks(masks) if masks is not None else None
        self.box_lb = box_lb
        self.keep_anchor = anchors


def postprocess(levels, coef, proto, frame_hw, conf_thres, iou_thres, max_det, nc, with_masks=True, mask_variant="A",
                return_soft=False):
    """U3..U7 for a batch.  levels: list of (B,64+nc,Hl,Wl); coef (B,32,A); proto (B,32,ph,pw).  -> [RefResults]
    mask_variant "B": newer-Ultralytics masks, and detections whose mask is empty are dropped (construct_result's
    `keep = masks.amax((-2, -1)) > 0`)."""
    levels = [torch.as_tensor(l, dtype=torch.float32) for l in levels]
    coef = torch.as_tensor(coef, dtype=torch.float32)
    proto = torch.as_tensor(proto, dtype=torch.float32)
    LH, LW = proto.shape[2] * 4, proto.shape[3] * 4
    pred = torch.cat((decode(levels, nc), coef), 1)
    res = []
    for b, (x, anchors) in enumerate(non_max_suppression(pred, conf_thres, iou_thres, max_det, nc)):
        masks = soft = None
        if with_masks:
            masks = process_mask(proto[b], x[:, 6:], x[:, :4], (LH, LW), mask_variant, return_soft)
            if return_soft:
                masks, soft = masks
            if mask_variant == "B":
                keep = masks.amax((-2, -1)) > 0
                x, anchors, masks = x[keep], anchors[keep], masks[keep]
                soft = soft[keep] if soft is not None else None
        xyxy = scale_boxes((LH, LW), x[:, :4], frame_hw)
        r = RefResults(xyxy, x[:, 4], x[:, 5], masks, x[:, :4].clone(), anchors)
        r.soft = soft
        res.append(r)
    return res

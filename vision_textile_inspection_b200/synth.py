"""Seeded synthetic inputs for the inspection hot path (SURVEY.md 8d).

The reference's weights (best_Model.pt / single_needle_model.pt) are absent, so the YOLOv8-seg head tensors are
*planted*: a scene of fabric regions and stitch dashes is drawn in letterbox space, and raw head logits are
constructed so that decoding them yields 5-30 overlapping candidates per instance, plus background clutter.
Frames are woven-fabric textures with the same scene geometry.  Everything is numpy + default_rng => identical
bytes on every machine for a given (config, seed).

Shapes follow BASELINE.md section 3 (configs 1-5) plus the reference deployment ("native", 1280x960,
config.py:59-60).
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field

import numpy as np

REG_MAX = 16
NM = 32
STRIDES = (8, 16, 32)


def _py_round(x: float) -> int:
    return int(round(x))


def letterbox_geometry(h: int, w: int, imgsz: int, stride: int = 32):
    """Ultralytics LetterBox(auto=True) geometry (host-side mirror of csrc/plan.cpp; SURVEY 8a U1)."""
    r = min(imgsz / h, imgsz / w)
    new_w, new_h = _py_round(w * r), _py_round(h * r)
    dw, dh = (imgsz - new_w) % stride, (imgsz - new_h) % stride
    dw /= 2
    dh /= 2
    top, bottom = _py_round(dh - 0.1), _py_round(dh + 0.1)
    left, right = _py_round(dw - 0.1), _py_round(dw + 0.1)
    return dict(new_w=new_w, new_h=new_h, top=top, bottom=bottom, left=left, right=right,
                LH=new_h + top + bottom, LW=new_w + left + right)


@dataclass
class WorkloadConfig:
    """One BASELINE.json config as concrete numbers."""
    name: str
    frame_w: int
    frame_h: int
    batch: int
    imgsz: int
    conf: float
    iou: float
    max_det: int
    variant: int = 0            # 0 = measurement.py, 1 = Utils/check_stitch_distance.py
    undistort: int = 0          # image-level cv2.undistort before the letterbox (north-star addition)
    extrinsics: str = "extrinsics"
    n_stitch: tuple = (20, 60)
    n_fabric: tuple = (1, 2)
    clutter: bool = False       # config 4: thousands of background candidates
    nc: int = 2
    cfg_id: int = 0
    geo: dict = field(default_factory=dict)

    def __post_init__(self):
        self.geo = letterbox_geometry(self.frame_h, self.frame_w, self.imgsz)

    @property
    def LH(self):
        return self.geo["LH"]

    @property
    def LW(self):
        return self.geo["LW"]

    @property
    def anchors(self):
        return sum((self.LH // s) * (self.LW // s) for s in STRIDES)

    def roi(self):
        """ROI of config.py:91-95 scaled from the 1280x960 calibration size to this frame."""
        if self.variant == 1:
            return (0, 0, 0, 0, 0)
        sx, sy = self.frame_w / 1280.0, self.frame_h / 960.0
        return (1, int(10 * sx), int(1270 * sx), int(300 * sy), int(760 * sy))


CONFIGS = {
    "native": WorkloadConfig("native-1280x960", 1280, 960, 1, 960, 0.20, 0.25, 200, cfg_id=0),
    "cfg1": WorkloadConfig("cfg1-640x640-main", 640, 640, 1, 960, 0.20, 0.25, 200, cfg_id=1),
    "cfg2": WorkloadConfig("cfg2-1280x720-b64-undistort", 1280, 720, 64, 960, 0.20, 0.25, 200, undistort=1, cfg_id=2),
    "cfg3": WorkloadConfig("cfg3-1920x1080-b128-stitchdist", 1920, 1080, 128, 640, 0.20, 0.45, 200, variant=1,
                           extrinsics="camera_extrinsics", cfg_id=3),
    "cfg4": WorkloadConfig("cfg4-640x640-b32-stress", 640, 640, 32, 640, 0.05, 0.25, 300, n_stitch=(400, 440),
                           clutter=True, cfg_id=4),
    "cfg5": WorkloadConfig("cfg5-3840x2160-b256-sharded", 3840, 2160, 256, 960, 0.20, 0.25, 200, cfg_id=5),
}


# ----------------------------------------------------------------------------------------------------------------
# scene
# ----------------------------------------------------------------------------------------------------------------
@dataclass
class Scene:
    LH: int
    LW: int
    instances: list            # (cls, x1, y1, x2, y2) letterbox px
    fabric_ind: np.ndarray     # (LH, LW) bool, union of fabric regions
    stitch_ind: np.ndarray     # (LH, LW) bool


def make_scene(cfg: WorkloadConfig, seed: int) -> Scene:
    rng = np.random.default_rng(seed)
    LH, LW = cfg.LH, cfg.LW
    top, new_h = cfg.geo["top"], cfg.geo["new_h"]
    X = np.arange(LW)[None, :]
    Y = np.arange(LH)[:, None]
    n_fab = int(rng.integers(cfg.n_fabric[0], cfg.n_fabric[1] + 1))
    n_st = int(rng.integers(cfg.n_stitch[0], cfg.n_stitch[1] + 1))
    inst = []
    fabric = np.zeros((LH, LW), bool)
    phase = rng.uniform(0, 2 * math.pi)
    wav = 3.0 * np.sin(X * (2 * math.pi / 180.0) + phase)
    if cfg.variant == 0:
        # fabric occupies 10 % .. ~66 % of the image height; its LOWER edge is the seam-allowance reference
        y_top = top + 0.10 * new_h
        y_edge = top + (0.64 + 0.04 * rng.random()) * new_h
        band = (Y >= y_top) & (Y <= y_edge + wav)
        stitch_y0 = y_edge - (0.055 + 0.02 * rng.random()) * new_h
        row_gap = -0.05 * new_h
    else:
        # check_stitch_distance: UPPER edge, stitches 0..150 frame px below it
        y_edge = top + (0.38 + 0.04 * rng.random()) * new_h
        y_bot = top + 0.97 * new_h
        band = (Y >= y_edge + wav) & (Y <= y_bot)
        stitch_y0 = y_edge + (0.05 + 0.02 * rng.random()) * new_h
        row_gap = 0.05 * new_h
    xs0 = 0.02 * LW
    xs1 = 0.98 * LW
    for f in range(n_fab):
        lo = xs0 if f == 0 else 0.5 * LW - 8
        hi = xs1 if n_fab == 1 else (0.5 * LW + 8 if f == 0 else xs1)
        reg = band & (X >= lo) & (X <= hi)
        ys, xs = np.nonzero(reg)
        inst.append((1, float(xs.min()), float(ys.min()), float(xs.max() + 1), float(ys.max() + 1)))
        fabric |= reg
    stitch = np.zeros((LH, LW), bool)
    rows = 2 if (cfg.clutter or rng.random() < 0.5) else 1
    if cfg.clutter:
        rows = 8
    per_row = int(math.ceil(n_st / rows))
    k = 0
    for r in range(rows):
        yc = stitch_y0 + r * row_gap + rng.uniform(-1.0, 1.0)
        pitch = (0.92 * LW) / per_row
        for j in range(per_row):
            if k >= n_st:
                break
            sw = float(np.clip(0.6 * pitch, 6.0, 24.0)) + rng.uniform(-1.0, 1.0)
            sh = 8.0 + rng.uniform(-1.0, 1.0)
            xc = 0.04 * LW + (j + 0.5) * pitch + rng.uniform(-1.5, 1.5)
            ycj = yc + rng.uniform(-1.0, 1.0)
            x1, y1, x2, y2 = xc - sw / 2, ycj - sh / 2, xc + sw / 2, ycj + sh / 2
            if y1 < 1 or y2 > LH - 1:
                continue
            stitch[int(round(y1)):int(round(y2)), int(round(x1)):int(round(x2))] = True
            inst.append((0, float(round(x1)), float(round(y1)), float(round(x2)), float(round(y2))))
            k += 1
    return Scene(LH, LW, inst, fabric, stitch)


# ----------------------------------------------------------------------------------------------------------------
# frames
# ----------------------------------------------------------------------------------------------------------------
def fabric_frame(cfg: WorkloadConfig, seed: int, scene: Scene | None = None) -> np.ndarray:
    """uint8 BGR h x w x 3 woven-fabric texture with a straight fabric edge and dark stitch dashes."""
    rng = np.random.default_rng(seed + 7919)
    h, w = cfg.frame_h, cfg.frame_w
    if scene is None:
        scene = make_scene(cfg, seed)
    py, px = rng.uniform(6, 10, 2)
    yy = np.arange(h, dtype=np.float32)[:, None]
    xx = np.arange(w, dtype=np.float32)[None, :]
    weave = (0.5 + 0.5 * np.sin(xx * (2 * np.pi / px))) * (0.5 + 0.5 * np.sin(yy * (2 * np.pi / py)))
    illum = 0.75 + 0.25 * np.sin(xx * (np.pi / w) + 0.3) * np.cos(yy * (0.7 * np.pi / h))
    # scene indicators are in letterbox space: gather them to frame space with the nearest map
    g = cfg.geo
    ymap = np.clip(((np.arange(h) + 0.5) * g["new_h"] / h).astype(int) + g["top"], 0, cfg.LH - 1)
    xmap = np.clip(((np.arange(w) + 0.5) * g["new_w"] / w).astype(int) + g["left"], 0, cfg.LW - 1)
    fab = scene.fabric_ind[ymap][:, xmap]
    sti = scene.stitch_ind[ymap][:, xmap]
    base = np.where(fab, 150.0 + 70.0 * weave, 40.0 + 10.0 * weave) * illum
    base = np.where(sti, 25.0, base)
    img = np.empty((h, w, 3), np.float32)
    tint = (0.92, 1.0, 0.96)
    noise = rng.normal(0.0, 4.0, (h, w)).astype(np.float32)
    for c in range(3):
        img[..., c] = base * tint[c] + noise
    return np.clip(np.rint(img), 0, 255).astype(np.uint8)


# ----------------------------------------------------------------------------------------------------------------
# head tensors
# ----------------------------------------------------------------------------------------------------------------
def _lowpass_noise(rng, shape, k=9):
    a = rng.normal(0.0, 1.0, (shape[0] + k - 1, shape[1] + k - 1))
    c = np.cumsum(np.cumsum(a, 0), 1)
    c = np.pad(c, ((1, 0), (1, 0)))
    out = c[k:, k:] - c[:-k, k:] - c[k:, :-k] + c[:-k, :-k]
    out = out / (out.std() + 1e-9)
    return out.astype(np.float32)


def planted_head(cfg: WorkloadConfig, seed: int, scene: Scene | None = None):
    """Raw YOLOv8-seg head tensors for one frame.

    Returns dict(levels=[(64+nc,Hl,Wl) f32]*3, coef=(32,A) f32, proto=(32,ph,pw) f32, scene=Scene).
    Layout is what ultralytics' Segment head hands to Detect._inference: per level cat(cv2(x), cv3(x)) with box
    channel = side*16+bin (sides l,t,r,b), mask coefficients cat over levels, prototypes at 1/4 resolution."""
    rng = np.random.default_rng(seed + 104729)
    if scene is None:
        scene = make_scene(cfg, seed)
    LH, LW, nc = cfg.LH, cfg.LW, cfg.nc
    ph, pw = LH // 4, LW // 4
    shapes = [(LH // s, LW // s) for s in STRIDES]
    levels, coefs = [], []
    bg_mu, bg_sd = (-4.0, 1.5) if cfg.clutter else (-7.0, 1.0)
    for (Hl, Wl) in shapes:
        lv = np.empty((4 * REG_MAX + nc, Hl, Wl), np.float32)
        lv[:4 * REG_MAX] = rng.normal(0.0, 1.0, (4 * REG_MAX, Hl, Wl))
        lv[4 * REG_MAX:] = rng.normal(bg_mu, bg_sd, (nc, Hl, Wl))
        levels.append(lv)
        coefs.append(rng.normal(0.0, 0.5, (NM, Hl, Wl)).astype(np.float32))
    kbins = np.arange(REG_MAX, dtype=np.float32)

    def plant(li, gy, gx, cls, box):
        s = STRIDES[li]
        Hl, Wl = shapes[li]
        if not (0 <= gy < Hl and 0 <= gx < Wl):
            return
        ax, ay = (gx + 0.5) * s, (gy + 0.5) * s
        x1, y1, x2, y2 = box
        tgt = np.array([ax - x1, ay - y1, x2 - ax, y2 - ay], np.float32) / s
        tgt = np.clip(tgt + rng.uniform(-0.5, 0.5, 4), 0.0, REG_MAX - 1.0)
        lv = levels[li]
        for side in range(4):
            lv[side * REG_MAX:(side + 1) * REG_MAX, gy, gx] = -6.0 * (kbins - tgt[side]) ** 2 / 4.0 \
                + rng.normal(0.0, 0.05, REG_MAX)
        lv[4 * REG_MAX:, gy, gx] = rng.normal(-6.0, 1.0, nc)
        lv[4 * REG_MAX + cls, gy, gx] = rng.normal(2.0, 1.0)
        c = rng.normal(0.0, 0.15, NM)
        c[0] = (4.0 if cls == 1 else 0.0) + rng.normal(0.0, 0.05)
        c[1] = (4.0 if cls == 0 else 0.0) + rng.normal(0.0, 0.05)
        coefs[li][:, gy, gx] = c

    for (cls, x1, y1, x2, y2) in scene.instances:
        cx, cy = 0.5 * (x1 + x2), 0.5 * (y1 + y2)
        if cls == 1:
            li = 2
            gx, gy = int(cx // 32), int(cy // 32)
            for dy in (-1, 0, 1):
                for dx in (-1, 0, 1):
                    plant(li, gy + dy, gx + dx, cls, (x1, y1, x2, y2))
        else:
            gx, gy = int(cx // 8), int(cy // 8)
            for dy in (-1, 0, 1):
                for dx in (-1, 0, 1):
                    if rng.random() < 0.75:
                        plant(0, gy + dy, gx + dx, cls, (x1, y1, x2, y2))
            plant(1, int(cy // 16), int(cx // 16), cls, (x1, y1, x2, y2))
    # prototypes: ch0 = fabric coverage, ch1 = stitch coverage (area-averaged to 1/4 res, mapped to [-1,1]),
    # ch2.. = low-pass noise so all 32 channels of the contraction carry signal
    proto = np.empty((NM, ph, pw), np.float32)
    proto[0] = scene.fabric_ind.reshape(ph, 4, pw, 4).mean((1, 3)) * 2.0 - 1.0
    proto[1] = scene.stitch_ind.reshape(ph, 4, pw, 4).mean((1, 3)) * 2.0 - 1.0
    for c in range(2, NM):
        proto[c] = _lowpass_noise(rng, (ph, pw))
    coef = np.concatenate([c.reshape(NM, -1) for c in coefs], 1)
    return dict(levels=levels, coef=np.ascontiguousarray(coef), proto=proto, scene=scene)


def make_batch(cfg: WorkloadConfig, batch: int, seed0: int | None = None, n_unique: int | None = None,
               with_frames: bool = True):
    """Batch of frames + head tensors.  n_unique < batch repeats content (bench: content does not affect timing).

    Seeds follow SURVEY 8d: seed = 1000*config + frame_idx."""
    if seed0 is None:
        seed0 = 1000 * cfg.cfg_id
    n_unique = batch if n_unique is None else min(n_unique, batch)
    frames, heads = [], []
    for i in range(n_unique):
        sc = make_scene(cfg, seed0 + i)
        if with_frames:
            frames.append(fabric_frame(cfg, seed0 + i, sc))
        heads.append(planted_head(cfg, seed0 + i, sc))
    idx = [i % n_unique for i in range(batch)]
    out = dict(
        levels=[np.stack([heads[i]["levels"][l] for i in idx]) for l in range(3)],
        coef=np.stack([heads[i]["coef"] for i in idx]),
        proto=np.stack([heads[i]["proto"] for i in idx]),
        scenes=[heads[i]["scene"] for i in idx],
    )
    if with_frames:
        out["frames"] = np.stack([frames[i] for i in idx])
    return out


def bgr_to_yuyv(bgr: np.ndarray) -> np.ndarray:
    """A YUYV camera stand-in for tests and the bench (SURVEY 8f rank 2, K0): (h, w, 3) BGR -> (h, w, 2) packed YUYV (BT.601 studio range, chroma of a
    pixel pair averaged).  Not an OpenCV restatement -- only the decode direction has a parity bar."""
    f = bgr.astype(np.float64)
    b, g, r = f[..., 0], f[..., 1], f[..., 2]
    y = 16 + (65.481 * r + 128.553 * g + 24.966 * b) / 255
    u = 128 + (-37.797 * r - 74.203 * g + 112.0 * b) / 255
    v = 128 + (112.0 * r - 93.786 * g - 18.214 * b) / 255
    out = np.empty(bgr.shape[:2] + (2,), np.uint8)
    out[..., 0] = np.clip(np.rint(y), 0, 255)
    out[:, 0::2, 1] = np.clip(np.rint((u[:, 0::2] + u[:, 1::2]) / 2), 0, 255)
    out[:, 1::2, 1] = np.clip(np.rint((v[:, 0::2] + v[:, 1::2]) / 2), 0, 255)
    return out


"""Stand-in YOLOv8-seg network in plain PyTorch (SURVEY.md 8f rank 1): the step BETWEEN pre and post.

The reference loads `best_Model.pt` through Ultralytics (measurement.py:145, :208); neither the weights
nor the package exist offline (the reference's .MISSING_LARGE_BLOBS), so this module rebuilds the published YOLOv8-seg
TOPOLOGY (Conv-BN-SiLU stem, C2f stages, SPPF, PAN-FPN neck, Segment head with DFL box branch, class branch, mask
coefficient branch and the Proto module) with random weights and the head-bias initialisation Ultralytics uses, and
returns the RAW head tensors in the layouts include/vti.h names:

    p3, p4, p5 : B x (64 + nc) x Hl x Wl   (cat(box branch, class branch), strides 8 / 16 / 32)
    coef       : B x 32 x A                (mask coefficient branch, levels concatenated)
    proto      : B x 32 x LH/4 x LW/4

It exists so that the whole frame -- K1 -> backbone -> K2..K5 -- can be captured as ONE CUDA graph and the share of the
accelerated stages in a full frame can be measured; it makes no accuracy claim.  The head writes its concatenations
straight into preallocated output buffers (`torch.cat(..., out=)`), so K2 / K3 / K4 read the head's output IN PLACE: no
copy sits between the network and the post kernels.  PyTorch is the plumbing here, as the north star says ("the YOLOv8
backbone stays in PyTorch only to produce raw head tensors").
"""
from __future__ import annotations

import math

import torch
import torch.nn as nn
import torch.nn.functional as F


class Conv(nn.Module):
    def __init__(self, c1, c2, k=1, s=1):
        super().__init__()
        self.conv = nn.Conv2d(c1, c2, k, s, k // 2, bias=False)
        self.bn = nn.BatchNorm2d(c2)

    def forward(self, x):
        return F.silu(self.bn(self.conv(x)))


class Bottleneck(nn.Module):
    def __init__(self, c, shortcut=True):
        super().__init__()
        self.cv1, self.cv2, self.add = Conv(c, c, 3), Conv(c, c, 3), shortcut

    def forward(self, x):
        y = self.cv2(self.cv1(x))
        return x + y if self.add else y


class C2f(nn.Module):
    def __init__(self, c1, c2, n=1, shortcut=False):
        super().__init__()
        self.c = c2 // 2
        self.cv1 = Conv(c1, 2 * self.c, 1)
        self.cv2 = Conv((2 + n) * self.c, c2, 1)
        self.m = nn.ModuleList(Bottleneck(self.c, shortcut) for _ in range(n))

    def forward(self, x):
        y = list(self.cv1(x).chunk(2, 1))
        y.extend(m(y[-1]) for m in self.m)
        return self.cv2(torch.cat(y, 1))


class SPPF(nn.Module):
    def __init__(self, c1, c2, k=5):
        super().__init__()
        self.cv1, self.cv2 = Conv(c1, c1 // 2, 1), Conv(c1 // 2 * 4, c2, 1)
        self.m = nn.MaxPool2d(k, 1, k // 2)

    def forward(self, x):
        y = [self.cv1(x)]
        y.extend(self.m(y[-1]) for _ in range(3))
        return self.cv2(torch.cat(y, 1))


class Proto(nn.Module):
    def __init__(self, c1, c_=64, c2=32):
        super().__init__()
        self.cv1 = Conv(c1, c_, 3)
        self.upsample = nn.ConvTranspose2d(c_, c_, 2, 2, 0, bias=True)
        self.cv2, self.cv3 = Conv(c_, c_, 3), Conv(c_, c2, 1)

    def forward(self, x):
        return self.cv3(self.cv2(self.upsample(self.cv1(x))))


class SegmentHead(nn.Module):
    """Ultralytics `Segment(Detect)` in training-mode form: raw per-level maps, coefficients, prototypes."""

    def __init__(self, nc, ch, nm=32, npr=64, reg_max=16):
        super().__init__()
        self.nc, self.nm, self.reg_max = nc, nm, reg_max
        c2, c3, c4 = max(16, ch[0] // 4, reg_max * 4), max(ch[0], min(nc, 100)), max(ch[0] // 4, nm)
        self.cv2 = nn.ModuleList(nn.Sequential(Conv(x, c2, 3), Conv(c2, c2, 3), nn.Conv2d(c2, 4 * reg_max, 1)) for x in ch)
        self.cv3 = nn.ModuleList(nn.Sequential(Conv(x, c3, 3), Conv(c3, c3, 3), nn.Conv2d(c3, nc, 1)) for x in ch)
        self.cv4 = nn.ModuleList(nn.Sequential(Conv(x, c4, 3), Conv(c4, c4, 3), nn.Conv2d(c4, nm, 1)) for x in ch)
        self.proto = Proto(ch[0], npr, nm)
        for a, b, s in zip(self.cv2, self.cv3, (8, 16, 32)):       # Detect.bias_init
            a[-1].bias.data[:] = 1.0
            b[-1].bias.data[:nc] = math.log(5 / nc / (640 / s) ** 2)


class YoloV8SegStandIn(nn.Module):
    """width / depth multiples of the published scales: n (0.25, 0.33), s (0.50, 0.33), m (0.75, 0.67)."""
    SCALES = {"n": (0.25, 0.33, 1024), "s": (0.50, 0.33, 1024), "m": (0.75, 0.67, 768)}

    def __init__(self, nc=2, scale="n"):
        super().__init__()
        w, d, mc = self.SCALES[scale]
        ch = lambda c: max(8, int(math.ceil(min(c, mc) * w / 8) * 8))
        dp = lambda n: max(1, round(n * d))
        c1, c2, c3, c4, c5 = ch(64), ch(128), ch(256), ch(512), ch(1024)
        self.stem = nn.Sequential(Conv(3, c1, 3, 2), Conv(c1, c2, 3, 2), C2f(c2, c2, dp(3), True))
        self.s3 = nn.Sequential(Conv(c2, c3, 3, 2), C2f(c3, c3, dp(6), True))
        self.s4 = nn.Sequential(Conv(c3, c4, 3, 2), C2f(c4, c4, dp(6), True))
        self.s5 = nn.Sequential(Conv(c4, c5, 3, 2), C2f(c5, c5, dp(3), True), SPPF(c5, c5))
        self.n4 = C2f(c5 + c4, c4, dp(3))
        self.n3 = C2f(c4 + c3, c3, dp(3))
        self.d3 = Conv(c3, c3, 3, 2)
        self.p4 = C2f(c3 + c4, c4, dp(3))
        self.d4 = Conv(c4, c4, 3, 2)
        self.p5 = C2f(c4 + c5, c5, dp(3))
        self.head = SegmentHead(nc, (c3, c4, c5))
        self.nc = nc

    def features(self, x):
        f2 = self.stem(x)
        f3 = self.s3(f2)
        f4 = self.s4(f3)
        f5 = self.s5(f4)
        u4 = self.n4(torch.cat((F.interpolate(f5, scale_factor=2.0, mode="nearest"), f4), 1))
        o3 = self.n3(torch.cat((F.interpolate(u4, scale_factor=2.0, mode="nearest"), f3), 1))
        o4 = self.p4(torch.cat((self.d3(o3), u4), 1))
        o5 = self.p5(torch.cat((self.d4(o4), f5), 1))
        return o3, o4, o5

    def forward(self, x, out=None):
        """x: B x 3 x LH x LW float32 in [0, 1].  out = (p3, p4, p5, coef, proto) preallocated float32 buffers or None."""
        feats = self.features(x)
        h = self.head
        B = x.shape[0]
        lv, co = [], []
        for i, f in enumerate(feats):
            box, cls, cf = h.cv2[i](f).float(), h.cv3[i](f).float(), h.cv4[i](f).float()
            # (channels_last inputs make torch.cat return a channels_last result: the ABI wants contiguous NCHW)
            lv.append(torch.cat((box, cls), 1, out=out[i]) if out is not None else torch.cat((box, cls), 1).contiguous())
            co.append(cf.reshape(B, h.nm, -1))
        coef = torch.cat(co, 2, out=out[3]) if out is not None else torch.cat(co, 2)
        proto = h.proto(feats[0]).float()
        if out is not None:
            out[4].copy_(proto)
            proto = out[4]
        else:
            proto = proto.contiguous()
        return lv[0], lv[1], lv[2], coef, proto


def make_standin_backbone(nc=2, scale="n", device="cuda", dtype=torch.float32, seed=0, channels_last=True):
    """Random-weight stand-in as a `backbone` callable for app.B200Predictor / app.StitchMeasurementApp.

    dtype torch.bfloat16 / float16 runs the convolutions under autocast (the head tensors are float32 either way).
    The returned callable accepts `out=` (the static head buffers of a captured pipeline)."""
    g = torch.Generator().manual_seed(seed)
    with torch.random.fork_rng():
        torch.manual_seed(int(g.initial_seed()))
        net = YoloV8SegStandIn(nc, scale)
    net = net.to(device).eval()
    if channels_last:
        net = net.to(memory_format=torch.channels_last)

    @torch.no_grad()
    def run(net_in, out=None):
        x = net_in.contiguous(memory_format=torch.channels_last) if channels_last else net_in
        if dtype != torch.float32:
            with torch.autocast("cuda", dtype=dtype):
                return net(x, out)
        return net(x, out)
    run.net = net
    return run

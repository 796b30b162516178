"""InspectionEngine -- host-side owner of one libvti handle on one GPU.

PyTorch is plumbing here (device memory, streams); every stage runs in the hand-written kernels behind the C ABI
(include/vti.h).  There is no CPU or eager-PyTorch fallback: without libvti.so or without a CUDA device the engine
raises.
"""
from __future__ import annotations

import ctypes as C
import json
import os
from dataclasses import dataclass

import numpy as np
import torch

from . import _lib
from ._lib import DET_DTYPE, RESULT_DTYPE, VtiCamera, VtiGeometry, VtiParams, check

DATA = os.path.join(os.path.dirname(os.path.abspath(__file__)), "data")


def load_reference_calibration() -> dict:
    """K / dist / rvec / tvec values of the reference's calibration JSONs (regenerated fixture, see oracle/gen_golden.py)."""
    with open(os.path.join(DATA, "reference_calibration.json")) as f:
        return json.load(f)


def rodrigues(rvec) -> np.ndarray:
    """Rotation vector -> matrix (same formula as cv2.Rodrigues; measurement.py:139)."""
    r = np.asarray(rvec, np.float64).reshape(3)
    th = float(np.linalg.norm(r))
    if th < 1e-300:
        return np.eye(3)
    k = r / th
    Kx = np.array([[0, -k[2], k[1]], [k[2], 0, -k[0]], [-k[1], k[0], 0]])
    return np.cos(th) * np.eye(3) + (1 - np.cos(th)) * np.outer(k, k) + np.sin(th) * Kx


def _dist5(dist, what: str) -> list:
    """Distortion coefficients as the 5 of the implemented model (k1, k2, p1, p2, k3), zero-padded."""
    d = np.asarray(dist, np.float64).reshape(-1)
    if d.size > 5 and np.any(d[5:] != 0.0):
        raise ValueError(f"{what}: only the 5-coefficient model (k1, k2, p1, p2, k3) is implemented; "
                         f"got {d.size} coefficients with non-zero higher terms")
    return np.concatenate([d[:5], np.zeros(max(0, 5 - d.size))]).tolist()


@dataclass
class EngineConfig:
    frame_h: int
    frame_w: int
    K: np.ndarray
    dist: np.ndarray
    R: np.ndarray
    t: np.ndarray
    imgsz: int = 960
    stride: int = 32
    nc: int = 2
    conf: float = 0.20            # config.py:71
    iou: float = 0.25             # config.py:72
    max_det: int = 200            # config.py:73
    max_batch: int = 1
    variant: int = 0              # 0 measurement.py, 1 Utils/check_stitch_distance.py
    undistort: int = 0
    channel_flip: int = 0
    stitch_id: int = 0
    fabric_id: int = 1
    roi: tuple = (1, 10, 1270, 300, 760)
    min_stitches: int = 3
    max_px_distance: int = 250
    neighborhood: int = 3
    max_candidates: int = 0
    mask_variant: int = 0         # 0 = "A" (sigmoid, > 0.5), 1 = "B" (newer Ultralytics: logits, > 0.0, empty masks dropped)
    cameras: list | None = None   # several cameras of this frame size: [{K, dist, R, t}, ...]; K / dist / R / t are then unused

    @staticmethod
    def for_workload(cfg, calib: dict | None = None, max_batch: int | None = None) -> "EngineConfig":
        """EngineConfig for a synth.WorkloadConfig: K scaled from the 1280x960 calibration size (SURVEY 7)."""
        calib = calib or load_reference_calibration()
        K = np.diag([cfg.frame_w / 1280.0, cfg.frame_h / 960.0, 1.0]) @ np.array(calib["camera_matrix"], np.float64)
        ex = calib[cfg.extrinsics]
        try:
            import cv2
            R = cv2.Rodrigues(np.asarray(ex["rvec"], np.float64).reshape(3, 1))[0]
        except Exception:  # pragma: no cover
            R = rodrigues(ex["rvec"])
        return EngineConfig(
            frame_h=cfg.frame_h, frame_w=cfg.frame_w, K=K, dist=np.array(calib["dist_coeffs"], np.float64), R=R,
            t=np.array(ex["tvec"], np.float64), imgsz=cfg.imgsz, nc=cfg.nc, conf=cfg.conf, iou=cfg.iou,
            max_det=cfg.max_det, max_batch=max_batch or cfg.batch, variant=cfg.variant, undistort=cfg.undistort,
            roi=cfg.roi(), max_px_distance=250 if cfg.variant == 0 else 150)

    def to_params(self) -> VtiParams:
        p = VtiParams()
        p.struct_size = C.sizeof(VtiParams)
        p.frame_h, p.frame_w, p.imgsz, p.stride = self.frame_h, self.frame_w, self.imgsz, self.stride
        p.nc, p.max_det, p.max_batch = self.nc, self.max_det, self.max_batch
        p.variant, p.undistort, p.channel_flip = self.variant, self.undistort, self.channel_flip
        p.stitch_id, p.fabric_id = self.stitch_id, self.fabric_id
        p.roi_enabled, p.roi_x_min, p.roi_x_max, p.roi_y_min, p.roi_y_max = [int(v) for v in self.roi]
        p.min_stitches, p.max_px_distance, p.neighborhood = self.min_stitches, self.max_px_distance, self.neighborhood
        p.max_candidates = self.max_candidates
        p.mask_variant = int(self.mask_variant)
        p.conf, p.iou = self.conf, self.iou
        p.iou_threshold = float(self.iou)          # the Python float torchvision.ops.nms receives (a C++ double)
        p.K[:] = np.asarray(self.K, np.float64).reshape(9).tolist()
        p.dist[:] = _dist5(self.dist, "EngineConfig.dist")
        p.R[:] = np.asarray(self.R, np.float64).reshape(9).tolist()
        p.t[:] = np.asarray(self.t, np.float64).reshape(3).tolist()
        return p

    def to_cameras(self):
        """`cameras` as a ctypes array of VtiCamera (vti_create_multi)."""
        arr = (VtiCamera * len(self.cameras))()
        for i, cam in enumerate(self.cameras):
            c = arr[i]
            c.struct_size = C.sizeof(VtiCamera)
            c.K[:] = np.asarray(cam["K"], np.float64).reshape(9).tolist()
            c.dist[:] = _dist5(cam["dist"], f"EngineConfig.cameras[{i}].dist")
            c.R[:] = np.asarray(cam["R"], np.float64).reshape(9).tolist()
            c.t[:] = np.asarray(cam["t"], np.float64).reshape(3).tolist()
        return arr


class InspectionEngine:
    """One libvti handle bound to one CUDA device.  All tensor arguments are CUDA tensors on that device."""

    def __init__(self, cfg: EngineConfig, device: int | str | torch.device | None = None):
        if not torch.cuda.is_available():
            raise _lib.VtiError("InspectionEngine needs a CUDA device: the hot path has no CPU fallback")
        self.lib = _lib.load()
        self.cfg = cfg
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        if self.device.type != "cuda":
            raise _lib.VtiError("InspectionEngine device must be CUDA")
        self._h = C.c_void_p()
        with torch.cuda.device(self.device):
            if cfg.cameras:
                check(self.lib.vti_create_multi(C.byref(cfg.to_params()), len(cfg.cameras), cfg.to_cameras(),
                                                C.byref(self._h)), "vti_create_multi")
            else:
                check(self.lib.vti_create(C.byref(cfg.to_params()), C.byref(self._h)), "vti_create")
        self.n_cameras = int(self.lib.vti_camera_count(self._h))
        g = VtiGeometry()
        check(self.lib.vti_get_geometry(self._h, C.byref(g)), "vti_get_geometry")
        self.g = g
        self.LH, self.LW, self.ph, self.pw, self.A = g.LH, g.LW, g.ph, g.pw, g.A
        self.level_shapes = [(g.lvl_h[i], g.lvl_w[i]) for i in range(3)]

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self.lib.vti_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------------------------------------ helpers
    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _chk(self, t: torch.Tensor, dtype, shape, name):
        if t.device != self.device or t.dtype != dtype or tuple(t.shape) != tuple(shape) or not t.is_contiguous():
            raise ValueError(f"{name}: expected contiguous {dtype} {tuple(shape)} on {self.device}, got "
                             f"{t.dtype} {tuple(t.shape)} on {t.device}")

    def _chk_camera(self, camera, B):
        """Device pointer of a per-frame camera id tensor (int32 (B,) on the engine's device), or None."""
        if camera is None:
            return None
        self._chk(camera, torch.int32, (B,), "camera")
        return camera.data_ptr()

    def alloc_outputs(self, B: int, masks: bool = False):
        dets = torch.empty((B, self.cfg.max_det, DET_DTYPE.itemsize), dtype=torch.uint8, device=self.device)
        counts = torch.empty((B,), dtype=torch.int32, device=self.device)
        results = torch.empty((B, RESULT_DTYPE.itemsize), dtype=torch.uint8, device=self.device)
        m = None
        if masks:
            m = torch.empty((B, self.cfg.max_det, self.LH, self.LW // 32), dtype=torch.int32, device=self.device)
        return dets, counts, results, m

    # ------------------------------------------------------------------------------------------------- stages
    def preprocess(self, frames: torch.Tensor, out: torch.Tensor | None = None, camera=None) -> torch.Tensor:
        """K1.  frames (B,h,w,3) uint8 -> (B,3,LH,LW) float32.  camera: int32 (B,) device tensor of camera ids (None:
        camera 0 for every frame)."""
        B = frames.shape[0]
        self._chk(frames, torch.uint8, (B, self.cfg.frame_h, self.cfg.frame_w, 3), "frames")
        cam = self._chk_camera(camera, B)
        if out is None:
            out = torch.empty((B, 3, self.LH, self.LW), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            check(self.lib.vti_preprocess_multi(self._h, frames.data_ptr(), cam, B, out.data_ptr(), self._stream()),
                  "vti_preprocess_multi")
        return out

    def _check_head(self, p3, p4, p5, coef, proto):
        B = p3.shape[0]
        for t, (hh, ww), nm in zip((p3, p4, p5), self.level_shapes, ("p3", "p4", "p5")):
            self._chk(t, torch.float32, (B, 64 + self.cfg.nc, hh, ww), nm)
        self._chk(coef, torch.float32, (B, 32, self.A), "coef")
        self._chk(proto, torch.float32, (B, 32, self.ph, self.pw), "proto")
        return B

    def postprocess(self, p3, p4, p5, coef, proto, outputs=None, export_masks: bool = False):
        """K2+K3+K4.  Returns (dets, counts, masks) device tensors (see alloc_outputs)."""
        B = self._check_head(p3, p4, p5, coef, proto)
        dets, counts, results, masks = outputs if outputs is not None else self.alloc_outputs(B, export_masks)
        with torch.cuda.device(self.device):
            check(self.lib.vti_postprocess(self._h, p3.data_ptr(), p4.data_ptr(), p5.data_ptr(), coef.data_ptr(),
                                           proto.data_ptr(), B, dets.data_ptr(), counts.data_ptr(),
                                           masks.data_ptr() if masks is not None else None, self._stream()),
                  "vti_postprocess")
        return dets, counts, masks

    def measure(self, dets, counts, results=None, camera=None):
        """K5.  Completes the records in place; returns the per-frame result tensor.  camera: as in preprocess."""
        B = dets.shape[0]
        cam = self._chk_camera(camera, B)
        if results is None:
            results = torch.empty((B, RESULT_DTYPE.itemsize), dtype=torch.uint8, device=self.device)
        with torch.cuda.device(self.device):
            check(self.lib.vti_measure_multi(self._h, B, cam, dets.data_ptr(), counts.data_ptr(), results.data_ptr(),
                                             self._stream()), "vti_measure_multi")
        return results

    def post_measure(self, p3, p4, p5, coef, proto, outputs=None, export_masks: bool = False, camera=None):
        B = self._check_head(p3, p4, p5, coef, proto)
        cam = self._chk_camera(camera, B)
        dets, counts, results, masks = outputs if outputs is not None else self.alloc_outputs(B, export_masks)
        head = [p3.data_ptr(), p4.data_ptr(), p5.data_ptr(), coef.data_ptr(), proto.data_ptr()]
        mptr = masks.data_ptr() if masks is not None else None
        with torch.cuda.device(self.device):
            check(self.lib.vti_post_measure_multi(self._h, *head, B, cam, dets.data_ptr(), counts.data_ptr(), mptr,
                                                  results.data_ptr(), self._stream()), "vti_post_measure_multi")
        return dets, counts, results, masks

    def capture_step(self, frames, p3, p4, p5, coef, proto, net_in=None, outputs=None, export_masks: bool = False,
                     camera=None):
        """One pass of the hot path as ONE CUDA graph: K1 on a forked branch beside K2 -> K3 -> K4 -> K5, joined at the
        end.  The stage entry points only launch kernels on the stream they are handed (no allocation, no
        synchronisation), so they are capturable as they are.  Returns (graph, net_in, (dets, counts, results, masks));
        `graph.replay()` re-runs the step on the CURRENT contents of the captured buffers, the camera ids included."""
        B = self._check_head(p3, p4, p5, coef, proto)
        self._chk(frames, torch.uint8, (B, self.cfg.frame_h, self.cfg.frame_w, 3), "frames")
        if net_in is None:
            net_in = torch.empty((B, 3, self.LH, self.LW), dtype=torch.float32, device=self.device)
        if outputs is None:
            outputs = self.alloc_outputs(B, export_masks)
        with torch.cuda.device(self.device):
            self.preprocess(frames, out=net_in, camera=camera)     # warm-up outside the capture (lazy module loading)
            self.post_measure(p3, p4, p5, coef, proto, outputs=outputs, camera=camera)
            torch.cuda.synchronize(self.device)
            graph = torch.cuda.CUDAGraph()
            side = torch.cuda.Stream(self.device, priority=-1)   # kernel nodes keep the priority of their stream:
            with torch.cuda.graph(graph):                        # the post CTAs win free SM slots over K1's 16 k CTAs
                cur = torch.cuda.current_stream(self.device)
                side.wait_stream(cur)                        # fork: K1 does not depend on the post stage
                with torch.cuda.stream(side):
                    self.post_measure(p3, p4, p5, coef, proto, outputs=outputs, camera=camera)
                self.preprocess(frames, out=net_in, camera=camera)
                cur.wait_stream(side)                        # join
        return graph, net_in, outputs

    # ------------------------------------------------------------------------------- overlay + JPEG (off the hot path)
    def annotate(self, frames: torch.Tensor, dets: torch.Tensor, counts: torch.Tensor, texts=None, out=None) -> torch.Tensor:
        """K6: the reference's overlay drawn on the GPU into a copy of `frames` (B,h,w,3 uint8 BGR, device).  Call right
        after post_measure() of the same batch.  texts: optional list (per frame) of (x, y, string, scale, (b, g, r))."""
        B = frames.shape[0]
        self._chk(frames, torch.uint8, (B, self.cfg.frame_h, self.cfg.frame_w, 3), "frames")
        if out is None:
            out = torch.empty_like(frames)
        with torch.cuda.device(self.device):
            check(self.lib.vti_annotate(self._h, frames.data_ptr(), B, dets.data_ptr(), counts.data_ptr(), out.data_ptr(),
                                        self._stream()), "vti_annotate")
            for b, items in enumerate(texts or []):
                for (x, y, text, scale, col) in items or []:
                    check(self.lib.vti_draw_text(self._h, out.data_ptr(), b, int(x), int(y), text.encode("ascii", "replace"),
                                                 int(scale), int(col[0]), int(col[1]), int(col[2]), self._stream()),
                          "vti_draw_text")
        return out

    def encode_jpeg(self, image: torch.Tensor, quality: int = 95) -> bytes:
        """nvJPEG encode of one (h,w,3) uint8 BGR device frame (main.py:314 saves the annotated frame as a JPEG)."""
        self._chk(image, torch.uint8, (self.cfg.frame_h, self.cfg.frame_w, 3), "image")
        cap = self.cfg.frame_h * self.cfg.frame_w * 3 + 65536
        buf = (C.c_uint8 * cap)()
        with torch.cuda.device(self.device):
            n = self.lib.vti_encode_jpeg(self._h, image.data_ptr(), int(quality), buf, cap, self._stream())
        if n < 0:
            check(int(n), "vti_encode_jpeg")
        return bytes(buf[:n])

    def decode_jpeg_batch(self, jpegs, out: torch.Tensor | None = None, one_by_one: bool = False) -> torch.Tensor:
        """Compressed ingest: a list of JPEG byte strings (camera MJPEG frames) -> (B,h,w,3) uint8 BGR frames ON THE DEVICE
        (nvJPEG, the whole batch in one nvjpegDecodeBatched call on the best backend the box offers; `one_by_one` = the
        single-image hybrid decoder), ready for preprocess().  Only the compressed bytes cross PCIe."""
        B = len(jpegs)
        if out is None:
            out = torch.empty((B, self.cfg.frame_h, self.cfg.frame_w, 3), dtype=torch.uint8, device=self.device)
        self._chk(out, torch.uint8, (B, self.cfg.frame_h, self.cfg.frame_w, 3), "out")
        with torch.cuda.device(self.device):
            if one_by_one:
                for b, j in enumerate(jpegs):
                    check(self.lib.vti_decode_jpeg(self._h, j, len(j), out[b].data_ptr(), self._stream()), "vti_decode_jpeg")
            else:
                ptrs = (C.c_char_p * B)(*jpegs)
                lens = (C.c_int64 * B)(*[len(j) for j in jpegs])
                check(self.lib.vti_decode_jpeg_batch(self._h, ptrs, lens, B, out.data_ptr(), self._stream()),
                      "vti_decode_jpeg_batch")
        return out

    def jpeg_backend(self) -> str:
        """Which nvJPEG backend decoded the last batch ("nvjpeg-hardware" | "nvjpeg-gpu-hybrid" | "nvjpeg-hybrid" | "none")."""
        return self.lib.vti_jpeg_backend().decode()

    def capture_pipeline(self, backbone, B: int, export_masks: bool = False) -> "GraphedPipeline":
        """The WHOLE frame -- K1 -> backbone -> K2 -> K3 -> K4 -> K5 -- for a fixed batch as ONE CUDA graph."""
        return GraphedPipeline(self, backbone, B, export_masks)

    def ingest_yuyv(self, yuyv: torch.Tensor, out: torch.Tensor | None = None) -> torch.Tensor:
        """K0: camera-native packed YUV 4:2:2 frames (B,h,w,2) uint8 on the device -> (B,h,w,3) BGR, bit-exact against
        cv2.cvtColor(.., COLOR_YUV2BGR_YUY2) (what cv2.VideoCapture.read() does on the CPU, main.py:188)."""
        B = yuyv.shape[0]
        self._chk(yuyv, torch.uint8, (B, self.cfg.frame_h, self.cfg.frame_w, 2), "yuyv")
        if out is None:
            out = torch.empty((B, self.cfg.frame_h, self.cfg.frame_w, 3), dtype=torch.uint8, device=self.device)
        self._chk(out, torch.uint8, (B, self.cfg.frame_h, self.cfg.frame_w, 3), "out")
        with torch.cuda.device(self.device):
            check(self.lib.vti_ingest_yuyv(self._h, yuyv.data_ptr(), B, out.data_ptr(), self._stream()), "vti_ingest_yuyv")
        return out

    def process_host(self, frames: np.ndarray, p3, p4, p5, coef, proto, want_net_in: bool = False, out=None, camera=None):
        """End-to-end with HOST numpy buffers (ideally pinned): H2D, K1..K5, D2H.  Returns (dets, counts, results[, net_in]).
        `frames` is (B,h,w,3) BGR, or (B,h,w,2) camera-native YUYV (converted on the device by K0).  camera: host array of
        B camera ids (None: camera 0 for every frame); an id out of range raises VtiError before any work."""
        B = frames.shape[0]
        if frames.dtype != np.uint8 or frames.ndim != 4 or frames.shape[1:3] != (self.cfg.frame_h, self.cfg.frame_w) or frames.shape[3] not in (2, 3):
            raise ValueError(f"process_host: frames must be uint8 (B,{self.cfg.frame_h},{self.cfg.frame_w},3) BGR or (..,2) YUYV, got {frames.dtype} {frames.shape}")
        cam = None
        if camera is not None:
            cam = np.ascontiguousarray(camera, dtype=np.int32)
            if cam.shape != (B,):
                raise ValueError(f"process_host: camera must hold {B} ids, got shape {cam.shape}")
        entry = self.lib.vti_process_host_multi if frames.shape[3] == 3 else self.lib.vti_process_host_yuyv_multi
        if out is None:
            out = (np.empty((B, self.cfg.max_det), DET_DTYPE), np.empty((B,), np.int32), np.empty((B,), RESULT_DTYPE))
        dets, counts, results = out
        net_in = np.empty((B, 3, self.LH, self.LW), np.float32) if want_net_in else None
        arrs = [frames, p3, p4, p5, coef, proto]
        for a_ in arrs:
            if not a_.flags["C_CONTIGUOUS"]:
                raise ValueError("process_host needs C-contiguous host arrays")
        with torch.cuda.device(self.device):
            check(entry(self._h, *[a_.ctypes.data for a_ in arrs], B, cam.ctypes.data if cam is not None else None,
                        net_in.ctypes.data if net_in is not None else None, dets.ctypes.data,
                        counts.ctypes.data, results.ctypes.data), "vti_process_host")
        return (dets, counts, results, net_in) if want_net_in else (dets, counts, results)

    @property
    def launch_count(self) -> int:
        return int(self.lib.vti_launch_count(self._h))

    def set_profiling(self, on: bool):
        check(self.lib.vti_set_profiling(self._h, int(on)), "vti_set_profiling")

    def stage_ms(self) -> list:
        """[K1, K2, K3, K4, K5] durations (ms) of the most recent calls, CUDA events on the launching stream."""
        ms = (C.c_float * 5)()
        check(self.lib.vti_get_stage_ms(self._h, ms), "vti_get_stage_ms")
        return [float(v) for v in ms]

    # ------------------------------------------------------------------------------------------------ readback
    @staticmethod
    def dets_to_numpy(dets: torch.Tensor) -> np.ndarray:
        return dets.cpu().numpy().view(DET_DTYPE).reshape(dets.shape[0], dets.shape[1])

    @staticmethod
    def results_to_numpy(results: torch.Tensor) -> np.ndarray:
        return results.cpu().numpy().view(RESULT_DTYPE).reshape(results.shape[0])

    def unpack_masks(self, masks: torch.Tensor, b: int, n: int) -> torch.Tensor:
        """Bit-packed (max_det, LH, LW/32) int32 -> (n, LH, LW) float32 0/1, like Results.masks.data."""
        w = masks[b, :n].to(torch.int64) & 0xFFFFFFFF
        bits = (w.unsqueeze(-1) >> torch.arange(32, device=masks.device)) & 1
        return bits.reshape(n, self.LH, self.LW).to(torch.float32)


class GraphedPipeline:
    """K1 -> backbone (PyTorch) -> K2..K5 of a fixed batch captured as ONE CUDA graph (SURVEY.md 8f rank 1).

    Static buffers: `frames` (B,h,w,3) uint8 in, `net_in`, the five head tensors, the record outputs.  The backbone is
    any callable `net_in -> (p3, p4, p5, coef, proto)`; if it accepts `out=` (backbone.make_standin_backbone does) it
    writes the head tensors straight into the static buffers K2 / K3 / K4 read -- no copy between the network and the
    post kernels -- otherwise its results are copied there inside the graph.  `replay(frames)` copies new frames in
    (host or device tensor) and re-runs the graph; the outputs are overwritten in place."""

    def __init__(self, eng: InspectionEngine, backbone, B: int, export_masks: bool = False):
        self.eng, self.B = eng, B
        dev, c = eng.device, eng.cfg
        self.frames = torch.zeros((B, c.frame_h, c.frame_w, 3), dtype=torch.uint8, device=dev)
        self.net_in = torch.empty((B, 3, eng.LH, eng.LW), dtype=torch.float32, device=dev)
        self.head = tuple(torch.empty((B, 64 + c.nc, hh, ww), dtype=torch.float32, device=dev) for hh, ww in eng.level_shapes) + (
            torch.empty((B, 32, eng.A), dtype=torch.float32, device=dev),
            torch.empty((B, 32, eng.ph, eng.pw), dtype=torch.float32, device=dev))
        self.outputs = eng.alloc_outputs(B, export_masks)
        self.in_place = True

        def body():
            eng.preprocess(self.frames, out=self.net_in)
            if self.in_place:
                got = backbone(self.net_in, out=self.head)
            else:
                got = backbone(self.net_in)
            for dst, src in zip(self.head, got):
                if src.data_ptr() != dst.data_ptr():
                    dst.copy_(src)
            eng.post_measure(*self.head, outputs=self.outputs)
        with torch.cuda.device(dev):
            side = torch.cuda.Stream(dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):                          # warm-up off the capture (cuDNN autotuning, lazy loads)
                try:
                    body()
                except TypeError:
                    self.in_place = False
                    body()
                body()
            torch.cuda.current_stream(dev).wait_stream(side)
            torch.cuda.synchronize(dev)
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph):
                body()

    def replay(self, frames=None):
        if frames is not None:
            if isinstance(frames, np.ndarray):
                frames = torch.from_numpy(np.ascontiguousarray(frames))
            self.frames.copy_(frames, non_blocking=True)
        self.graph.replay()
        return self.outputs

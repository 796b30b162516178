"""Drop-in host side of the reference's detect-and-measure call (SURVEY.md 8b), above the C ABI.

Two boundaries are mirrored, same names / argument meaning / error behaviour as the reference:

  outer   StitchMeasurementApp(calib_path, extr_path, model_path, camera_index=0, calib_w=640, calib_h=640,
                               frame_buffer=8, min_stitches=3, stitch_id=0, fabric_id=1)
          .process_frame(frame) -> (annotated, measurements)          measurement.py:123-126, 188-511
          (constructed at main.py:80-91, called at main.py:211); force_camera_resolution(cap, w, h)
          is importable from here as well (main.py:16, 198).
  inner   B200Predictor.predict(rgb, verbose=False, conf=, iou=, max_det=, imgsz=) -> [Results]
          with r.boxes.cls / r.boxes.xyxy / r.masks.data                measurement.py:208-210, 244-245, 74-75
          Assigning a B200Predictor to the reference app's `.model` accelerates pre + post with zero edits there.

The YOLOv8-seg backbone stays in PyTorch and only produces the raw head tensors: a `backbone` is any callable
`net_in (B,3,LH,LW) float32 cuda -> (p3, p4, p5, coef, proto)` (see include/vti.h for the layouts).  Everything around
it -- letterbox, decode, NMS, masks, measurement -- runs in libvti.so on the GPU; there is no CPU fallback.
The only host arithmetic kept here is what the reference keeps as frame-ordered state: the two 8-deep median deques
(measurement.py:149-150, 474-484).
"""
from __future__ import annotations

import json
import os
import time
from collections import deque
from datetime import datetime

import numpy as np
import torch

from . import _lib
from .engine import EngineConfig, InspectionEngine

# config.py:59-95 defaults (the reference star-imports them; here they are constructor keywords)
CALIB_W, CALIB_H = 1280, 960
CONF_THRESH, IOU_THRESH, MAX_DETECTIONS = 0.20, 0.25, 200
FRAME_BUFFER, MIN_STITCHES = 8, 3
MAX_PX_DISTANCE, ENVELOPE_NEIGHBORHOOD = 250, 3
STITCH_CLASS_ID, FABRIC_CLASS_ID = 0, 1
ROI_DEFAULT = (1, 10, CALIB_W - 10, 300, CALIB_H - 200)      # enabled, x_min, x_max, y_min, y_max
ROI_BORDER_COLOR, ROI_BORDER_THICKNESS = (144, 238, 144), 2
CAMERA_AUTO_EXPOSURE, CAMERA_EXPOSURE = 1, 150

_ERRORS = {_lib.ST_NO_FABRIC: "Fabric not detected", _lib.ST_NO_STITCH: "No stitches detected"}


def load_json(path):
    with open(path, "r") as f:
        return json.load(f)


def load_camera(calib_path, extr_path):
    """(K, dist, R, t) of one camera from the reference's two JSON files, with its errors (measurement.py:127-146)."""
    if not os.path.exists(calib_path):
        raise FileNotFoundError(f"Calibration file missing: {calib_path}")
    calib = load_json(calib_path)
    K = np.array(calib["camera_matrix"], dtype=np.float64)
    dist = np.array(calib["dist_coeffs"], dtype=np.float64).ravel()
    if not os.path.exists(extr_path):
        raise FileNotFoundError(f"Extrinsics file missing: {extr_path}")
    extr = load_json(extr_path)
    rvec = np.array(extr["rvec"], dtype=np.float64).reshape(3, 1)
    t = np.array(extr["tvec"], dtype=np.float64).reshape(3,)
    from .engine import rodrigues
    try:
        import cv2
        R = cv2.Rodrigues(rvec)[0]
    except Exception:  # pragma: no cover
        R = rodrigues(rvec)
    return K, dist, R, t


def smooth(buf_dist: deque, buf_width: deque, avg_dist, avg_width):
    """measurement.py:474-484 -- frame-ordered state, hence on the host."""
    sd = sw = None
    if avg_dist is not None:
        buf_dist.append(avg_dist)
        sd = float(np.median(buf_dist))
    if avg_width is not None:
        buf_width.append(avg_width)
        sw = float(np.median(buf_width))
    return sd, sw


def measurement_dict(r, buf_dist: deque, buf_width: deque) -> dict:
    """process_frame's dict (measurement.py:281-287, 332-337, 474-511) for one vti_frame_result, smoothing with the
    camera's two deques."""
    if int(r["status"]) & _lib.ST_OVERFLOW:
        # more confidence-passing anchors than the handle's candidate capacity: the kept subset is not the
        # top-scoring one (Ultralytics keeps the best max_nms) -- never silent
        import warnings
        warnings.warn(f"vti: candidate list overflow ({int(r['n_cand'])} candidates): raise max_candidates or conf",
                      RuntimeWarning, stacklevel=3)
    status = int(r["status"]) & 0xFF
    if status in _ERRORS:
        return {"edge_distance_mm": None, "stitch_width_mm": None, "stitch_count": 0,
                "timestamp": datetime.now(), "error": _ERRORS[status]}
    ad = None if np.isnan(r["avg_dist"]) else float(r["avg_dist"])
    aw = None if np.isnan(r["avg_width"]) else float(r["avg_width"])
    sd, sw = smooth(buf_dist, buf_width, ad, aw)
    return {"edge_distance_mm": sd, "stitch_width_mm": sw, "stitch_count": int(r["n_dist"]),
            "timestamp": datetime.now()}


def force_camera_resolution(cap, w, h):
    """Same contract as measurement.py:23-42: set the capture size, report what the camera gave."""
    import cv2
    cap.set(cv2.CAP_PROP_FRAME_WIDTH, w)
    cap.set(cv2.CAP_PROP_FRAME_HEIGHT, h)
    time.sleep(2)
    aw, ah = int(cap.get(cv2.CAP_PROP_FRAME_WIDTH)), int(cap.get(cv2.CAP_PROP_FRAME_HEIGHT))
    cap.set(cv2.CAP_PROP_AUTO_EXPOSURE, CAMERA_AUTO_EXPOSURE)
    cap.set(cv2.CAP_PROP_EXPOSURE, CAMERA_EXPOSURE)
    if aw != w or ah != h:
        print(f"Warning: camera resolution {aw}x{ah}, expected {w}x{h}")
    return aw, ah


def backbone_from_ultralytics(model_path: str, device="cuda"):
    """Wrap an Ultralytics YOLOv8-seg checkpoint so that it returns RAW head tensors (no decode, no NMS).

    Needs the `ultralytics` package and the weight file, neither of which exists in the build container
    (the reference's .MISSING_LARGE_BLOBS): this adapter is provided for integration and is NOT covered by tests.
    """
    try:
        from ultralytics import YOLO
    except Exception as e:  # pragma: no cover
        raise RuntimeError("ultralytics is not installed: pass backbone=<callable> instead") from e
    net = YOLO(model_path).model.to(device).eval()  # pragma: no cover
    head = net.model[-1]                            # pragma: no cover

    @torch.no_grad()
    def run(net_in):                                # pragma: no cover
        head.training, head.export = True, False     # training-mode forward = raw per-level maps, coefficients, protos
        try:
            out = net(net_in)
        finally:
            head.training = False
        feats, coef, proto = out[0], out[1], out[2]
        return feats[0].contiguous(), feats[1].contiguous(), feats[2].contiguous(), coef.contiguous(), proto.contiguous()
    return run


class _Boxes:
    def __init__(self, cls, xyxy, conf):
        self.cls, self.xyxy, self.conf = cls, xyxy, conf


class _Masks:
    def __init__(self, data):
        self.data = data


class Results:
    """The slice of ultralytics' Results that measurement.py reads (:242-245, :74-75)."""

    def __init__(self, boxes, masks, records=None, frame_result=None):
        self.boxes, self.masks = boxes, masks
        self.records, self.frame_result = records, frame_result


class B200Predictor:
    """Inner boundary: `.predict()` with the keyword arguments measurement.py:208-210 passes.

    One InspectionEngine per (frame shape, imgsz, conf, iou, max_det) is created on first use and kept.
    `channel_flip=1` reproduces BasePredictor.preprocess's `im[..., ::-1]` on the array it is handed (the reference
    hands it RGB, so the network sees B,G,R planes -- SURVEY 8a U2).
    """

    def __init__(self, backbone, K, dist, R=None, t=None, device=None, undistort=0, nc=2, roi=(0, 0, 0, 0, 0),
                 variant=0, channel_flip=1, mask_variant=0):
        if not torch.cuda.is_available():
            raise _lib.VtiError("B200Predictor needs a CUDA device: the hot path has no CPU fallback")
        self.backbone = backbone
        self.K, self.dist = np.asarray(K, np.float64), np.asarray(dist, np.float64).ravel()
        self.R = np.eye(3) if R is None else np.asarray(R, np.float64)
        self.t = np.array([0.0, 0.0, 1.0]) if t is None else np.asarray(t, np.float64)
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        self.undistort, self.nc, self.roi, self.variant, self.channel_flip = undistort, nc, roi, variant, channel_flip
        self.mask_variant = mask_variant      # 0: Ultralytics <= 8.0.x masks (sigmoid, > 0.5); 1: newer (logits, > 0, drop)
        self.extra = {}
        self._engines = {}
        self.use_graph = False                # True: K1 -> backbone -> K2..K5 of a batch shape run as ONE CUDA graph
        self._pipes = {}
        self.last_device = None

    def engine_for(self, h, w, imgsz, conf, iou, max_det, batch=1) -> InspectionEngine:
        key = (h, w, imgsz, float(conf), float(iou), int(max_det), batch)
        eng = self._engines.get(key)
        if eng is None:
            ec = EngineConfig(frame_h=h, frame_w=w, K=self.K, dist=self.dist, R=self.R, t=self.t, imgsz=imgsz,
                              nc=self.nc, conf=conf, iou=iou, max_det=max_det, max_batch=batch, variant=self.variant,
                              undistort=self.undistort, channel_flip=self.channel_flip, roi=self.roi,
                              mask_variant=self.mask_variant, **self.extra)
            eng = self._engines[key] = InspectionEngine(ec, self.device)
        return eng

    @torch.no_grad()
    def run(self, frames: np.ndarray, conf, iou, max_det, imgsz, export_masks=True):
        """frames (B,h,w,3) uint8 BGR host array -- or (B,h,w,2) packed YUYV as a V4L2 camera delivers it -> (engine, dets,
        counts, results, masks) with records on the host."""
        B, h, w = frames.shape[:3]
        eng = self.engine_for(h, w, imgsz, conf, iou, max_det, B)
        if frames.shape[3] == 2 and self.use_graph:
            raise ValueError("use_graph takes BGR frames; YUYV frames go through the stream path")
        if self.use_graph:
            key = (id(eng), B, bool(export_masks))
            pipe = self._pipes.get(key)
            if pipe is None:
                pipe = self._pipes[key] = eng.capture_pipeline(self.backbone, B, export_masks)
            dets, counts, results, masks = pipe.replay(frames)
            self.last_device = (eng, pipe.frames, dets, counts)
            return eng, eng.dets_to_numpy(dets), counts.cpu().numpy(), eng.results_to_numpy(results), masks
        d_frames = torch.from_numpy(np.ascontiguousarray(frames)).to(self.device, non_blocking=True)
        if frames.shape[3] == 2:                                            # camera-native YUYV (main.py:188's cap.read()
            d_frames = eng.ingest_yuyv(d_frames)                            # conversion, on the device): K0
        net_in = eng.preprocess(d_frames)                                   # K1
        p3, p4, p5, coef, proto = self.backbone(net_in)                     # PyTorch backbone -> raw head tensors
        dets, counts, results, masks = eng.post_measure(p3, p4, p5, coef, proto, export_masks=export_masks)  # K2..K5
        self.last_device = (eng, d_frames, dets, counts)       # for the GPU overlay (engine.annotate) of this batch
        return eng, eng.dets_to_numpy(dets), counts.cpu().numpy(), eng.results_to_numpy(results), masks

    def predict(self, source, verbose=False, conf=0.25, iou=0.7, max_det=300, imgsz=640, **_ignored):
        frames = source[None] if isinstance(source, np.ndarray) and source.ndim == 3 else np.stack(list(source))
        eng, dets, counts, results, masks = self.run(frames, conf, iou, max_det, imgsz, export_masks=True)
        out = []
        for b in range(frames.shape[0]):
            n = int(counts[b])
            d = dets[b, :n]
            md = eng.unpack_masks(masks, b, n).cpu() if n else None
            if n and self.mask_variant == 1:              # newer Ultralytics removes detections with an empty mask
                keep = (d["flags"] & _lib.F_DROPPED) == 0
                d, md = d[keep], md[torch.from_numpy(keep)]
            boxes = _Boxes(torch.from_numpy(d["cls"].astype(np.float32)), torch.from_numpy(d["box_frame"].copy()),
                           torch.from_numpy(d["conf"].copy()))
            m = _Masks(md) if len(d) else None
            out.append(Results(boxes, m, d, results[b]))
        return out


class StitchMeasurementApp:
    """Outer boundary: what main.py:80-91 constructs and main.py:211 calls.

    Extra keywords (all optional) carry what the reference reads from config.py / the camera: `backbone` (callable, see
    module docstring; default = backbone_from_ultralytics(model_path)), `roi`, `conf`, `iou`, `max_det`, `imgsz`,
    `undistort`, `annotate`, `device`.  `camera_index=None` skips opening a camera (`.cap` is then None).
    """
    VARIANT = 0          # measure-stage semantics: 0 = measurement.py, 1 = Utils/check_stitch_distance.py (subclass below)

    def __init__(self, calib_path, extr_path, model_path, camera_index=0, calib_w=640, calib_h=640, frame_buffer=8,
                 min_stitches=MIN_STITCHES, stitch_id=STITCH_CLASS_ID, fabric_id=FABRIC_CLASS_ID, *, backbone=None,
                 roi=ROI_DEFAULT, conf=CONF_THRESH, iou=IOU_THRESH, max_det=MAX_DETECTIONS, imgsz=960, undistort=0,
                 max_px_distance=MAX_PX_DISTANCE, neighborhood=ENVELOPE_NEIGHBORHOOD, annotate=True, device=None,
                 mask_variant=0, jpeg_quality=0):
        self.K, self.dist, self.R, self.t = load_camera(calib_path, extr_path)
        self.n_c = self.R[:, 2].astype(np.float64)                  # measurement.py:44-48
        self.d_c = -float(self.n_c.dot(self.t))

        if backbone is None:
            backbone = backbone_from_ultralytics(model_path)
        self.model = B200Predictor(backbone, self.K, self.dist, self.R, self.t, device=device, undistort=undistort,
                                   roi=tuple(int(v) for v in roi), channel_flip=0,   # frames arrive BGR: no flip
                                   variant=self.VARIANT, mask_variant=mask_variant)
        self.model.extra = dict(min_stitches=min_stitches, stitch_id=stitch_id, fabric_id=fabric_id,
                                max_px_distance=max_px_distance, neighborhood=neighborhood)
        self.conf, self.iou, self.max_det, self.imgsz = conf, iou, max_det, imgsz
        self.annotate = annotate               # True: minimal cv2 overlay on the host; "gpu": K6 overlay (+ nvJPEG); False: none
        self.jpeg_quality, self.last_jpeg = jpeg_quality, None

        self.cap, self.aw, self.ah = None, calib_w, calib_h
        if camera_index is not None:
            try:
                import cv2
                self.cap = cv2.VideoCapture(camera_index, cv2.CAP_V4L2)
                self.aw, self.ah = force_camera_resolution(self.cap, calib_w, calib_h)
            except Exception as e:  # pragma: no cover
                print("Camera unavailable:", e)
        self.frame_buf_dist = deque(maxlen=frame_buffer)
        self.frame_buf_width = deque(maxlen=frame_buffer)
        self.min_stitches, self.stitch_id, self.fabric_id = min_stitches, stitch_id, fabric_id
        self.running = True
        self.last_records = None

    # ------------------------------------------------------------------------------------------------------------
    def _smooth(self, avg_dist, avg_width):
        return smooth(self.frame_buf_dist, self.frame_buf_width, avg_dist, avg_width)

    def _finish(self, r) -> dict:
        return measurement_dict(r, self.frame_buf_dist, self.frame_buf_width)

    def process_frames(self, frames: np.ndarray):
        """Batched form of process_frame: (B,h,w,3) uint8 -> list of measurement dicts, smoothing in frame order."""
        eng, dets, counts, results, _ = self.model.run(frames, self.conf, self.iou, self.max_det, self.imgsz,
                                                       export_masks=False)
        self.last_records = [dets[b, :int(counts[b])] for b in range(frames.shape[0])]
        return [self._finish(results[b]) for b in range(frames.shape[0])]

    def process_frame(self, frame):
        """frame: h x w x 3 uint8 BGR (not mutated), or h x w x 2 packed YUYV straight from the camera (converted on the
        device, bit-exact cv2.cvtColor).  Returns (annotated BGR, measurements); never raises."""
        try:
            m = self.process_frames(np.ascontiguousarray(frame)[None])[0]
        except Exception as e:
            print("Model inference error:", e)
            return frame.copy(), {"edge_distance_mm": None, "stitch_width_mm": None, "stitch_count": 0,
                                  "timestamp": datetime.now(), "error": "Model inference failed"}
        if self.annotate == "gpu":
            return self._annotate_gpu(frame, m), m
        # a YUYV frame comes back as the BGR frame K0 made of it on the device (what cap.read() would have returned)
        annotated = frame.copy() if frame.shape[2] == 3 else self.model.last_device[1][0].cpu().numpy()
        if self.annotate:
            self._draw(annotated, m)
        return annotated, m

    def _annotate_gpu(self, frame, m):
        """annotate="gpu": the overlay rasterised by libvti (K6) on the frame that is already on the device, optionally
        JPEG-encoded there as well (`jpeg_quality`; main.py:314 writes the annotated frame with cv2.imwrite) -- the last
        per-frame CPU cost of the reference's loop.  `self.last_jpeg` holds the encoded bytes."""
        eng, d_frames, dets, counts = self.model.last_device
        h = frame.shape[0]
        sd, sw = m.get("edge_distance_mm"), m.get("stitch_width_mm")
        if "error" in m:
            text = m["error"]
        elif sd is not None and sw is not None:
            text = f"Edge Dist: {sd:.2f}mm | Avg Width: {sw:.2f}mm (n_d={m['stitch_count']})"
        elif sd is not None:
            text = f"Edge Distance: {sd:.2f}mm (n={m['stitch_count']})"
        elif sw is not None:
            text = f"Avg Width: {sw:.2f}mm"
        else:
            text = f"Insufficient stitches (need {self.min_stitches})"
        rec = self.last_records[0] if self.last_records else []
        info = f"Stitches: {int(sum(1 for d in rec if d['flags'] & _lib.F_STITCH and d['flags'] & _lib.F_IN_ROI))} | " \
               f"Fabric: {int(sum(1 for d in rec if d['flags'] & _lib.F_FABRIC and d['flags'] & _lib.F_IN_ROI and d['flags'] & _lib.F_HAS_MASK))}"
        ann = eng.annotate(d_frames[:1], dets[:1], counts[:1],
                           texts=[[(10, 14, text, 2, (0, 0, 255)), (10, h - 18, info, 1, (0, 0, 0))]])
        self.last_jpeg = eng.encode_jpeg(ann[0], self.jpeg_quality) if self.jpeg_quality else None
        return ann[0].cpu().numpy()

    def _draw(self, img, m):
        """Overlay (OUT of the hot path, SURVEY 8f rank 3): ROI box, per-stitch edge lines, the info line."""
        try:
            import cv2
        except Exception:  # pragma: no cover
            return
        h, w = img.shape[:2]
        en, x0, x1, y0, y1 = self.model.roi
        if en:
            x0, x1 = max(0, min(x0, w - 1)), max(0, min(x1, w - 1))
            y0, y1 = max(0, min(y0, h - 1)), max(0, min(y1, h - 1))
            if x0 < x1 and y0 < y1:
                cv2.rectangle(img, (x0, y0), (x1, y1), ROI_BORDER_COLOR, ROI_BORDER_THICKNESS)
        rec = self.last_records[0] if self.last_records else []
        for d in rec:
            if d["flags"] & _lib.F_HAS_DIST:
                cx, cy, ey = int(round(d["cx"])), int(round(d["cy"])), int(round(d["edge_y"]))
                cv2.line(img, (cx, ey), (cx, cy), (0, 255, 0), 1)
                cv2.circle(img, (cx, ey), 2, (255, 0, 255), -1)
        sd, sw = m.get("edge_distance_mm"), m.get("stitch_width_mm")
        if "error" in m:
            text = m["error"]
        elif sd is not None and sw is not None:
            text = f"Edge Dist: {sd:.2f}mm | Avg Width: {sw:.2f}mm (n_d={m['stitch_count']})"
        elif sd is not None:
            text = f"Edge Distance: {sd:.2f}mm (n={m['stitch_count']})"
        elif sw is not None:
            text = f"Avg Width: {sw:.2f}mm"
        else:
            text = f"Insufficient stitches (need {self.min_stitches})"
        cv2.putText(img, text, (10, 30), cv2.FONT_HERSHEY_SIMPLEX, 0.7, (0, 0, 255), 2)

    def _info_text(self, r) -> str:
        """Utils/check_stitch_distance.py:513-540 (smoothing + the text line it returns and draws)."""
        ad = None if np.isnan(r["avg_dist"]) else float(r["avg_dist"])
        aw = None if np.isnan(r["avg_width"]) else float(r["avg_width"])
        sd, sw = self._smooth(ad, aw)
        n_found = int(r["n_width"])
        if sd is not None and sw is not None:
            return f"Edge Dist: {sd:.2f}mm | Avg Width: {sw:.2f}mm (n={n_found})"
        if sd is not None:
            return f"Edge Distance: {sd:.2f}mm (n={n_found})"
        if sw is not None:
            return f"Avg Width: {sw:.2f}mm (n={n_found})"
        return f"Insufficient stitches (found {n_found}, need {self.min_stitches})"

    def run(self):  # pragma: no cover - camera loop of measurement.py:513-560, needs hardware
        last = 0.0
        while self.running and self.cap is not None:
            ret, frame = self.cap.read()
            if not ret:
                continue
            if time.time() - last >= 2.0:
                _, m = self.process_frame(frame)
                print(f"Edge: {m.get('edge_distance_mm', 'N/A')}mm | Width: {m.get('stitch_width_mm', 'N/A')}mm")
                last = time.time()
        if self.cap is not None:
            self.cap.release()


class CheckStitchDistanceApp(StitchMeasurementApp):
    """Outer drop-in for BASELINE config 3: the class Utils/check_stitch_distance.py:176 also calls
    StitchMeasurementApp, whose process_frame (:281-553) returns `(annotated, info_text)` -- a string, not a dict.

    Same constructor signature (:177-187); semantics of that file: no ROI, predict() without imgsz (Ultralytics'
    default 640, :286), upper fabric envelope, mask-less fabric detections as filled boxes, `0 < d < 150` proximity
    rule, widths of the final stitches only, k-means labels updated on break -- all inside libvti (variant = 1).
    Error returns: "Model error" (:291), "Fabric not detected" (:347), "No stitches detected" (:406)."""
    VARIANT = 1

    def __init__(self, calib_path, extr_path, model_path, camera_index=0, calib_w=640, calib_h=640, frame_buffer=8,
                 min_stitches=MIN_STITCHES, stitch_id=STITCH_CLASS_ID, fabric_id=FABRIC_CLASS_ID, **kw):
        kw.setdefault("roi", (0, 0, 0, 0, 0))
        kw.setdefault("imgsz", 640)
        kw.setdefault("max_px_distance", 150)              # check_stitch_distance.py:38
        super().__init__(calib_path, extr_path, model_path, camera_index, calib_w, calib_h, frame_buffer, min_stitches,
                         stitch_id, fabric_id, **kw)

    def process_frames(self, frames: np.ndarray):
        """(B,h,w,3) uint8 -> list of info_text strings, smoothing in frame order."""
        eng, dets, counts, results, _ = self.model.run(frames, self.conf, self.iou, self.max_det, self.imgsz,
                                                       export_masks=False)
        self.last_records = [dets[b, :int(counts[b])] for b in range(frames.shape[0])]
        out = []
        for b in range(frames.shape[0]):
            status = int(results[b]["status"]) & 0xFF
            out.append(_ERRORS[status] if status in _ERRORS else self._info_text(results[b]))
        return out

    def process_frame(self, frame):
        """frame: h x w x 3 uint8 BGR (not mutated).  Returns (annotated, info_text); never raises."""
        try:
            text = self.process_frames(np.ascontiguousarray(frame)[None])[0]
        except Exception as e:
            print("Model inference error:", e)
            return frame.copy(), "Model error"
        annotated = frame.copy()
        if self.annotate and text not in _ERRORS.values():
            try:
                import cv2
                cv2.putText(annotated, text, (10, 30), cv2.FONT_HERSHEY_SIMPLEX, 0.7, (0, 0, 255), 2)
            except Exception:  # pragma: no cover
                pass
        return annotated, text


class MultiCameraApp:
    """Several cameras of one frame size behind ONE libvti handle: the reference's per-frame measurement
    (StitchMeasurementApp.process_frame's dict, measurement.py semantics) for batches that mix cameras.

    `cameras` = [(calib_path, extr_path), ...], one pair per camera as the reference reads them (FileNotFoundError
    like StitchMeasurementApp).  Keywords as StitchMeasurementApp's (`backbone`, `roi`, `conf`, `iou`, `max_det`,
    `imgsz`, `undistort`, `frame_buffer`, `min_stitches`, ...).  Each frame is undistorted (undistort=1) and measured
    with its own camera's calibration; each camera keeps its own two median deques, fed in batch order.  The ROI,
    thresholds and classes are shared by all cameras.  Opens no capture device and draws no overlay.
    """

    def __init__(self, cameras, model_path, frame_buffer=8, min_stitches=MIN_STITCHES, stitch_id=STITCH_CLASS_ID,
                 fabric_id=FABRIC_CLASS_ID, *, backbone=None, roi=ROI_DEFAULT, conf=CONF_THRESH, iou=IOU_THRESH,
                 max_det=MAX_DETECTIONS, imgsz=960, undistort=0, max_px_distance=MAX_PX_DISTANCE,
                 neighborhood=ENVELOPE_NEIGHBORHOOD, device=None, mask_variant=0):
        if not cameras or len(cameras) > _lib.MAX_CAMERAS:
            raise ValueError(f"MultiCameraApp: 1..{_lib.MAX_CAMERAS} cameras, got {len(cameras or [])}")
        self.cameras = [dict(zip(("K", "dist", "R", "t"), load_camera(cp, ep))) for cp, ep in cameras]
        if not torch.cuda.is_available():
            raise _lib.VtiError("MultiCameraApp needs a CUDA device: the hot path has no CPU fallback")
        self.backbone = backbone if backbone is not None else backbone_from_ultralytics(model_path)
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        self.config = dict(imgsz=imgsz, conf=conf, iou=iou, max_det=max_det, undistort=undistort,
                           roi=tuple(int(v) for v in roi), min_stitches=min_stitches, stitch_id=stitch_id,
                           fabric_id=fabric_id, max_px_distance=max_px_distance, neighborhood=neighborhood,
                           mask_variant=mask_variant)
        self.min_stitches = min_stitches
        self.buffers = [(deque(maxlen=frame_buffer), deque(maxlen=frame_buffer)) for _ in self.cameras]
        self._engines = {}
        self.last_records = None

    def engine_for(self, h, w, batch) -> InspectionEngine:
        """The handle for (frame size, batch): every camera's tables, built once and kept."""
        key = (h, w, batch)
        eng = self._engines.get(key)
        if eng is None:
            c0 = self.cameras[0]
            ec = EngineConfig(frame_h=h, frame_w=w, K=c0["K"], dist=c0["dist"], R=c0["R"], t=c0["t"], nc=2,
                              max_batch=batch, channel_flip=0, cameras=self.cameras, **self.config)
            eng = self._engines[key] = InspectionEngine(ec, self.device)
        return eng

    @torch.no_grad()
    def process_frames(self, frames: np.ndarray, camera_ids) -> list:
        """frames (B,h,w,3) uint8 BGR (or (B,h,w,2) packed YUYV) and camera_ids (B ints) -> B measurement dicts."""
        frames = np.ascontiguousarray(frames)
        B, h, w = frames.shape[:3]
        ids = np.asarray(camera_ids).reshape(-1)
        if ids.shape != (B,) or not np.issubdtype(ids.dtype, np.integer):
            raise ValueError(f"process_frames: {B} integer camera ids expected, got {ids.dtype} {ids.shape}")
        if B and (ids.min() < 0 or ids.max() >= len(self.cameras)):
            raise ValueError(f"process_frames: camera ids must be in [0, {len(self.cameras)}), got {ids.tolist()}")
        eng = self.engine_for(h, w, B)
        cam = torch.from_numpy(ids.astype(np.int32)).to(self.device)
        d_frames = torch.from_numpy(frames).to(self.device, non_blocking=True)
        if frames.shape[3] == 2:
            d_frames = eng.ingest_yuyv(d_frames)                            # K0
        net_in = eng.preprocess(d_frames, camera=cam)                       # K1, each frame with its camera's remap
        p3, p4, p5, coef, proto = self.backbone(net_in)
        dets, counts, results, _ = eng.post_measure(p3, p4, p5, coef, proto, camera=cam)    # K2..K5
        dets, counts, results = eng.dets_to_numpy(dets), counts.cpu().numpy(), eng.results_to_numpy(results)
        self.last_records = [dets[b, :int(counts[b])] for b in range(B)]
        return [measurement_dict(results[b], *self.buffers[int(ids[b])]) for b in range(B)]

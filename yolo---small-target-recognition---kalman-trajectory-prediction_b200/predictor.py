"""Host-side mirror of the reference's detect API: ``YOLO(cfg).predict(source, ...) -> list[Results]``.

Follows, for the detect path only,
  Model.predict / __call__             ultralytics/engine/model.py:158-187, :498-557
  BasePredictor.preprocess/inference   ultralytics/engine/predictor.py:152-204 (LetterBox, data/augment.py:1667-1743)
  DetectionPredictor.postprocess       ultralytics/models/yolo/detect/predict.py:34-125
  Results / Boxes                      ultralytics/engine/results.py:192-290, :855-1072
with the three stages executed by the CUDA library: stem-fused preprocess + forward (engine), DFL decode
+ candidate filter, NMS + scale_boxes.  The reference package is not imported; INTEGRATION.md shows the
``DetectionPredictor`` subclass a maintainer would register through ``model.predict(predictor=...)``.
"""
from __future__ import annotations

import ctypes as C
import math
import os
import time

import numpy as np

from . import _lib, cfg, ops, weights
from .engine import Engine


# ---------------------------------------------------------------------------------------------------
# Results containers (engine/results.py)
# ---------------------------------------------------------------------------------------------------

# Annotator colours (utils/plotting.py:95-120 hex palette, as BGR tuples) and the plate colours that get dark / white ink (:255-278)
_PALETTE_BGR = tuple((int(h[4:6], 16), int(h[2:4], 16), int(h[0:2], 16)) for h in (
    "042AFF 0BDBEB F3F3F3 00DFB7 111F68 FF6FDD FF444F CCED00 00F344 BD00FF 00B4FF DD00BA 00FFFF 26C000 01FFB3 7D24FF 7B0068 FF1B6C "
    "FC6D2F A2FF0B").split())
_DARK_INK_ON = frozenset({(235, 219, 11), (243, 243, 243), (183, 223, 0), (221, 111, 255), (0, 237, 204), (68, 243, 0), (255, 255, 0),
                          (179, 255, 1), (11, 255, 162)})
_WHITE_INK_ON = frozenset({(255, 42, 4), (79, 68, 255), (255, 0, 189), (255, 180, 0), (186, 0, 221), (0, 192, 38), (255, 36, 125),
                           (104, 0, 123), (108, 27, 255), (47, 109, 252), (104, 31, 17)})


class Boxes:
    """Detection boxes: ``data`` is (n, 6) [x1, y1, x2, y2, conf, cls] or (n, 7) with a track id in column 4."""

    def __init__(self, boxes, orig_shape):
        if boxes.ndim == 1:
            boxes = boxes[None, :]
        n = boxes.shape[-1]
        assert n in {6, 7}, f"expected 6 or 7 values but got {n}"
        self.data = boxes
        self.orig_shape = orig_shape
        self.is_track = n == 7

    # -- BaseTensor protocol (results.py:23-190)
    @property
    def shape(self):
        return self.data.shape

    def _wrap(self, d):
        return self.__class__(d, self.orig_shape)

    def cpu(self):
        return self if isinstance(self.data, np.ndarray) else self._wrap(self.data.cpu())

    def numpy(self):
        return self if isinstance(self.data, np.ndarray) else self._wrap(self.data.cpu().numpy())

    def cuda(self):
        import torch

        return self._wrap(torch.as_tensor(self.data).cuda())

    def to(self, *a, **k):
        import torch

        return self._wrap(torch.as_tensor(self.data).to(*a, **k))

    def __len__(self):
        return len(self.data)

    def __getitem__(self, idx):
        return self._wrap(self.data[idx])

    # -- views
    @property
    def xyxy(self):
        return self.data[:, :4]

    @property
    def conf(self):
        return self.data[:, -2]

    @property
    def cls(self):
        return self.data[:, -1]

    @property
    def id(self):
        return self.data[:, -3] if self.is_track else None

    @property
    def xywh(self):
        d = self.xyxy
        out = d.copy() if isinstance(d, np.ndarray) else d.clone()
        out[:, 0] = (d[:, 0] + d[:, 2]) / 2
        out[:, 1] = (d[:, 1] + d[:, 3]) / 2
        out[:, 2] = d[:, 2] - d[:, 0]
        out[:, 3] = d[:, 3] - d[:, 1]
        return out

    @property
    def xyxyn(self):
        d = self.xyxy
        out = d.copy() if isinstance(d, np.ndarray) else d.clone()
        out[:, [0, 2]] /= self.orig_shape[1]
        out[:, [1, 3]] /= self.orig_shape[0]
        return out

    @property
    def xywhn(self):
        out = self.xywh
        out[:, [0, 2]] /= self.orig_shape[1]
        out[:, [1, 3]] /= self.orig_shape[0]
        return out


class Results:
    """engine/results.py:192-290 restricted to the detect task."""

    def __init__(self, orig_img, path, names, boxes=None, speed=None):
        self.orig_img = orig_img
        self.orig_shape = orig_img.shape[:2]
        self.boxes = Boxes(boxes, self.orig_shape) if boxes is not None else None
        self.masks = self.probs = self.keypoints = self.obb = None
        self.speed = speed or {"preprocess": None, "inference": None, "postprocess": None}
        self.names = names
        self.path = path
        self.save_dir = None

    def __len__(self):
        return 0 if self.boxes is None else len(self.boxes)

    def update(self, boxes=None, **_):
        """results.py:340-368: replace the boxes (used by trackers to attach ids)."""
        if boxes is not None:
            self.boxes = Boxes(boxes, self.orig_shape)

    def cpu(self):
        r = Results(self.orig_img, self.path, self.names, speed=self.speed)
        r.boxes = self.boxes.cpu() if self.boxes is not None else None
        return r

    def numpy(self):
        r = Results(self.orig_img, self.path, self.names, speed=self.speed)
        r.boxes = self.boxes.numpy() if self.boxes is not None else None
        return r

    def summary(self, normalize=False, decimals=5):
        """results.py:788-860 for detections: one dict per box {name, class, confidence, box{x1,y1,x2,y2}[, track_id]}."""
        out = []
        if self.boxes is None:
            return out
        h, w = self.orig_shape if normalize else (1, 1)
        d = self.boxes.numpy()
        for row in d.data:
            cls, conf = int(row[-1]), round(float(row[-2]), decimals)
            r = {"name": self.names[cls], "class": cls, "confidence": conf,
                 "box": {"x1": round(float(row[0]) / w, decimals), "y1": round(float(row[1]) / h, decimals),
                         "x2": round(float(row[2]) / w, decimals), "y2": round(float(row[3]) / h, decimals)}}
            if d.is_track:
                r["track_id"] = int(row[4])
            out.append(r)
        return out

    def to_json(self, normalize=False, decimals=5):
        """results.py: to_json."""
        import json

        return json.dumps(self.summary(normalize=normalize, decimals=decimals), indent=2)

    tojson = to_json

    def save_txt(self, txt_file, save_conf=False):
        """results.py:695-750 for detections: one line per box, ``class x_center y_center width height [conf] [track_id]`` with
        normalised coordinates in '%g' format, APPENDED to the file."""
        import os

        texts = []
        if self.boxes is not None and len(self.boxes):
            d = self.boxes.numpy()
            for row, nb in zip(d.data, d.xywhn):
                line = (int(row[-1]), *[float(v) for v in nb]) + ((float(row[-2]),) if save_conf else ()) + ((int(row[4]),) if d.is_track else ())
                texts.append(("%g " * len(line)).rstrip() % line)
        if texts:
            os.makedirs(os.path.dirname(os.path.abspath(str(txt_file))), exist_ok=True)
            with open(txt_file, "a", encoding="utf-8") as f:
                f.writelines(t + "\n" for t in texts)
        return str(txt_file)

    def plot(self, conf=True, labels=True, line_width=None, img=None, boxes=True, color_mode="class", txt_color=(255, 255, 255), **_):
        """results.py:475-613 restricted to boxes, drawn the way the reference's Annotator draws them with OpenCV
        (utils/plotting.py:170-364, the path taken for ASCII class names): same pixels as `Results.plot()` of the reference for
        the same boxes -- palette colour by class (or by track id / row with color_mode="instance"), anti-aliased rectangle of
        the image-scaled line width, label plate above the box (inside it at the top edge, pulled left at the right edge), ink
        chosen against the plate colour, rows painted last-to-first.  Host-side drawing, not part of the hot path.  Non-ASCII
        names make the reference switch to PIL and a TrueType font; here they are drawn with the same OpenCV calls."""
        import cv2

        assert color_mode in {"instance", "class"}, f"Expected color_mode='instance' or 'class', not {color_mode}."
        im = np.ascontiguousarray((self.orig_img if img is None else img).copy())
        if self.boxes is None or not boxes:
            return im
        lw = line_width or max(round(sum(im.shape) / 2 * 0.003), 2)
        thick, scale = max(lw - 1, 1), lw / 3
        d = self.boxes.numpy()
        rows = d.data
        for i in range(len(rows)):
            row = rows[len(rows) - 1 - i]                              # reversed(pred_boxes), i counts from the end (:568)
            c = int(row[-1])
            tid = int(row[4]) if d.is_track else None
            key = c if color_mode == "class" else (tid if tid is not None else i)
            plate = _PALETTE_BGR[int(key) % len(_PALETTE_BGR)]
            ink = (104, 31, 17) if plate in _DARK_INK_ON else ((255, 255, 255) if plate in _WHITE_INK_ON else tuple(txt_color))
            p1 = (int(row[0]), int(row[1]))
            cv2.rectangle(im, p1, (int(row[2]), int(row[3])), plate, thickness=lw, lineType=cv2.LINE_AA)
            if labels:
                name = ("" if tid is None else f"id:{tid} ") + str(self.names[c])
                text = f"{name} {float(row[-2]):.2f}" if conf else name
                w, h = cv2.getTextSize(text, 0, fontScale=scale, thickness=thick)[0]
                h += 3
                above = p1[1] >= h                                      # room for the plate above the box?
                if p1[0] > im.shape[1] - w:
                    p1 = (im.shape[1] - w, p1[1])
                cv2.rectangle(im, p1, (p1[0] + w, p1[1] - h if above else p1[1] + h), plate, -1, cv2.LINE_AA)
                cv2.putText(im, text, (p1[0], p1[1] - 2 if above else p1[1] + h - 1), 0, scale, ink, thickness=thick, lineType=cv2.LINE_AA)
        return im

    def verbose(self):
        """results.py:663-693."""
        if not len(self):
            return "(no detections), "
        cls = self.boxes.numpy().cls.astype(int)
        counts = np.bincount(cls)
        return "".join(f"{n} {self.names[c]}{'s' * int(n > 1)}, " for c, n in enumerate(counts) if n)


# ---------------------------------------------------------------------------------------------------
# letterbox geometry (data/augment.py:1692-1733)
# ---------------------------------------------------------------------------------------------------
def check_imgsz(imgsz, stride=32):
    """utils/checks.py check_imgsz(min_dim=2): int -> [s, s]; every side rounded up to a stride multiple."""
    if isinstance(imgsz, int):
        imgsz = [imgsz, imgsz]
    imgsz = [max(math.ceil(int(x) / stride) * stride, stride) for x in imgsz]
    return imgsz if len(imgsz) == 2 else [imgsz[0], imgsz[0]]


def letterbox_geometry(h0, w0, new_shape, auto, stride=32):
    """Returns (resized (h, w), canvas (H, W), top, left) exactly as LetterBox computes them (scaleup, center)."""
    r = min(new_shape[0] / h0, new_shape[1] / w0)
    new_unpad = int(round(w0 * r)), int(round(h0 * r))
    dw, dh = new_shape[1] - new_unpad[0], new_shape[0] - new_unpad[1]
    if auto:
        dw, dh = dw % stride, dh % stride
    dw, dh = dw / 2, dh / 2
    top, bottom = int(round(dh - 0.1)), int(round(dh + 0.1))
    left, right = int(round(dw - 0.1)), int(round(dw + 0.1))
    return (new_unpad[1], new_unpad[0]), (new_unpad[1] + top + bottom, new_unpad[0] + left + right), top, left


def scale_params(canvas_hw, orig_hw):
    """gain / pad of scale_boxes (utils/ops.py:105-138, ratio_pad=None) + clip bounds."""
    gain = min(canvas_hw[0] / orig_hw[0], canvas_hw[1] / orig_hw[1])
    pad_x = round((canvas_hw[1] - orig_hw[1] * gain) / 2 - 0.1)
    pad_y = round((canvas_hw[0] - orig_hw[0] * gain) / 2 - 0.1)
    return gain, pad_x, pad_y, orig_hw[1], orig_hw[0]


def letterbox_table(shapes, imgsz):
    """LetterBox of a batch of frames of ``shapes`` [(h, w), ...] as BasePredictor.pre_transform (engine/predictor.py) chooses it:
    ``auto`` (minimal stride padding) only when every shape is the same, else every frame into the full ``imgsz`` canvas.
    Returns (canvas (H, W), geom int32 [B][6] {h, w, rh, rw, top, left} for ``ops.letterbox_u8``, scale float32 [B][5] of
    ``scale_params`` per frame for the NMS epilogue)."""
    shapes = [(int(h), int(w)) for h, w in shapes]
    auto = len(set(shapes)) == 1
    geom, scale, canvas = [], [], set()
    for h0, w0 in shapes:
        (rh, rw), hw, top, left = letterbox_geometry(h0, w0, imgsz, auto)
        canvas.add(hw)
        geom.append((h0, w0, rh, rw, top, left))
        scale.append(scale_params(hw, (h0, w0)))
    (H, W), = canvas
    return (H, W), np.asarray(geom, np.int32).reshape(-1, 6), np.asarray(scale, np.float32).reshape(-1, 5)


# ---------------------------------------------------------------------------------------------------
# model facade
# ---------------------------------------------------------------------------------------------------
class DetectPipeline:
    """Engine + decode + NMS for a fixed (batch, canvas H x W): every launch of one detect step."""

    def __init__(self, spec, state_dict, batch, H, W, max_det=300, fuse_head=True):
        self.engine = Engine(spec, state_dict, batch, H, W, fuse_head=fuse_head)
        e = self.engine
        self.post = ops.DetectPost(batch, e.level_h, e.level_w, e.level_stride, e.nc, e.lstride, max_det=max_det)
        self.B, self.H, self.W = batch, H, W
        self.feats = None
        self.canvas = None          # [B][H][W][3] uint8, allocated by the first ``letterbox``

    def __call__(self, frames_u8, conf, iou, pad_top=0, pad_left=0, orig_hw=None, classes_mask=None, agnostic=False,
                 mode="exact", stream=None):
        """frames_u8: CUDA uint8 [B][h][w][3] BGR.  Returns (dets [B][max_det][6], counts [B]) device tensors."""
        self.engine.forward_u8(frames_u8, pad_top, pad_left, stream=stream)
        return self.finish(conf, iou, orig_hw, classes_mask, agnostic, mode, stream)

    def run_tensor(self, x, conf, iou, orig_hw=None, classes_mask=None, agnostic=False, mode="exact", stream=None):
        self.engine.forward_tensor(x, stream=stream)
        return self.finish(conf, iou, orig_hw, classes_mask, agnostic, mode, stream)

    def letterbox(self, packed, offsets, geom, stream=None):
        """LetterBox frames of individual shapes (``ops.pack_frames`` layout, CUDA tables of ``letterbox_table``) into
        ``self.canvas``."""
        import torch

        if self.canvas is None:
            self.canvas = torch.empty((self.B, self.H, self.W, 3), dtype=torch.uint8, device=packed.device)
        return ops.letterbox_u8(packed, offsets, geom, self.H, self.W, out=self.canvas, stream=stream)

    def run_ragged(self, packed, offsets, geom, scale, conf, iou, classes_mask=None, agnostic=False, mode="exact", stream=None):
        """A batch of frames of individual shapes: letterbox, forward on the canvas, candidates, NMS with each image's
        scale_boxes (``scale``: CUDA float32 [B][5]).  Returns (dets [B][max_det][6], counts [B]) like ``__call__``."""
        self.letterbox(packed, offsets, geom, stream)
        self.engine.forward_u8(self.canvas, 0, 0, stream=stream)
        return self.finish(conf, iou, None, classes_mask, agnostic, mode, stream, scale)

    def finish(self, conf, iou, orig_hw, classes_mask, agnostic, mode, stream, scale=None):
        self.candidates(conf, classes_mask, stream)
        return self.nms(iou, orig_hw, agnostic, mode, stream, scale)

    def candidates(self, conf, classes_mask=None, stream=None):
        """Head outputs -> per-image candidate lists (the only post-processing launch that reads engine buffers)."""
        if self.engine.fused_head:
            self.post.candidates_from_head(self.engine.head_dist, self.engine.head_cls, conf, classes_mask, stream=stream)
        else:
            self.post.decode(self.engine.level_ptrs, conf, classes_mask, stream=stream)

    def nms(self, iou, orig_hw=None, agnostic=False, mode="exact", stream=None, scale=None):
        """scale_boxes to ``orig_hw`` (one shape for the batch), or per image with ``scale`` (CUDA float32 [B][5])."""
        if scale is None and orig_hw is not None:
            scale = scale_params((self.H, self.W), orig_hw)
        return self.post.nms(iou, agnostic=agnostic, mode=mode, scale=scale, stream=stream)

    def embed(self, stream=None):
        """get_obj_feats (models/yolo/detect/predict.py) for the detections ``nms`` kept: [B][max_det][s] fp32 device tensor, row k
        of image b valid for k < count[b].  Reads the Detect inputs in the engine arena, so it must follow ``nms`` on the same
        stream before the next forward."""
        import torch

        lv = self.engine.detect_inputs()
        s = min(c for *_, c in lv)
        if self.feats is None:
            self.feats = torch.empty((self.B, self.post.max_det, s), dtype=torch.float32, device="cuda")
        n = len(lv)
        arr = lambda k: (C.c_int * n)(*[d[k] for d in lv])
        _lib.check(self.engine.lib.b2_reid_gather((C.c_void_p * n)(*[d[0] for d in lv]), arr(1), arr(2), arr(3), arr(4), arr(5), n,
                                                  _lib.ptr(self.post.out_idx), _lib.ptr(self.post.out_count), self.B, self.post.max_det, s,
                                                  _lib.ptr(self.feats), _lib.stream_ptr(stream)))
        return self.feats


class YOLO:
    """``YOLO('yolov8s-p2.yaml')`` facade (models/yolo/model.py:26, engine/model.py:29) for the detect task.

    ``model``: a model name / YAML path understood by :func:`cfg.resolve`.  Weights: ``state_dict`` (a torch or
    numpy state_dict with the reference's key names) or, by default, the seeded synthetic recipe of
    :mod:`weights` (the reference ships no checkpoint).
    """

    def __init__(self, model="yolov8n-p2.yaml", task="detect", verbose=False, state_dict=None, nc=None, seed=0):
        if task not in (None, "detect"):
            raise NotImplementedError(f"task {task!r}: only 'detect' is on the hot path")
        _lib.require_cuda()
        ckpt_names = None
        if isinstance(model, str) and model.endswith(".pt"):           # engine/model.py:_load -> nn/tasks.py load_checkpoint
            model, ckpt_sd, ckpt_names = weights.load_checkpoint(model)
            state_dict = ckpt_sd if state_dict is None else state_dict
        self.spec = cfg.resolve(model, nc=nc)
        self.names = ckpt_names if ckpt_names and len(ckpt_names) == self.spec["nc"] else self.spec["names"]
        self.state_dict = weights.to_numpy_state_dict(state_dict) if state_dict is not None else weights.synthetic_state_dict(self.spec, seed)
        self.overrides = {"conf": 0.25, "iou": 0.7, "imgsz": 640, "max_det": 300, "agnostic_nms": False, "classes": None,
                          "batch": 1, "verbose": verbose, "nms_mode": "exact"}
        self._pipes = {}
        self.task = "detect"

    def load_state_dict(self, sd):
        self.state_dict = weights.to_numpy_state_dict(sd)
        self._pipes.clear()
        return self

    def _pipe(self, batch, H, W, max_det):
        key = (batch, H, W, max_det)
        if key not in self._pipes:
            self._pipes[key] = DetectPipeline(self.spec, self.state_dict, batch, H, W, max_det)
        return self._pipes[key]

    def __call__(self, source=None, stream=False, **kwargs):
        return self.predict(source, stream, **kwargs)

    def predict(self, source=None, stream=False, **kwargs):
        """engine/model.py:498-557.  source: HWC BGR uint8 ndarray, list of them, a BCHW float tensor in [0,1], or a path / glob /
        directory / .txt list of image and video files (data/loaders.py LoadImagesAndVideos; ``batch`` frames per forward,
        ``vid_stride``; with ``stream=True`` a generator, as the reference asks for long videos)."""
        import torch

        if isinstance(source, (str, os.PathLike)) or (isinstance(source, (list, tuple)) and source and isinstance(source[0], (str, os.PathLike))):
            from .loaders import LoadImagesAndVideos, LoadStreams

            batch, stride = int(kwargs.pop("batch", self.overrides["batch"])), int(kwargs.pop("vid_stride", 1))
            src = str(source) if isinstance(source, os.PathLike) else source
            if isinstance(src, str) and (src.endswith(".streams") or src.lower().startswith(("rtsp://", "rtmp://", "http://", "https://", "tcp://")) or src.isnumeric()):
                ds = LoadStreams(src, vid_stride=stride, buffer=bool(kwargs.pop("stream_buffer", False)))       # data/build.py check_source
            else:
                kwargs.pop("stream_buffer", None)
                ds = LoadImagesAndVideos(src, batch=batch, vid_stride=stride)
            self.dataset = ds

            def gen():
                for paths, imgs, _ in ds:
                    for r, pth in zip(self.predict(imgs, False, **kwargs), paths):
                        r.path = pth
                        yield r

            return gen() if stream else list(gen())

        a = {**self.overrides, **kwargs}
        want_feats = bool(a.pop("_feats", False))      # internal (YOLO.track with BoT-SORT ReID): Results.feats per image
        if a.get("predictor") is not None:
            # engine/model.py:549 swaps the predictor class; this facade IS the predictor -- to put the engine behind an installed
            # Ultralytics model use b200dt.ultra_plugin.predictor_class()
            raise TypeError("predictor= is not supported by b200dt.YOLO; pass b200dt.ultra_plugin.predictor_class() to ultralytics' own YOLO.predict")
        dv = a.get("device")
        if dv not in (None, "", "cuda") and not (isinstance(dv, int) and dv == _lib.require_cuda().index) and str(dv) != f"cuda:{_lib.require_cuda().index}" and str(dv) != str(_lib.require_cuda().index):
            raise ValueError(f"device={dv!r}: b200dt runs on the current CUDA device ({_lib.require_cuda()}); there is no CPU path")
        for k in ("half", "device", "save", "show", "rect", "mode", "augment", "visualize", "embed", "predictor"):
            a.pop(k, None)          # half: the engine always computes in bf16 with fp32 accumulation; the rest do not touch the hot path
        conf, iou, max_det = float(a["conf"]), float(a["iou"]), int(a["max_det"])
        assert 0 <= conf <= 1, f"Invalid Confidence threshold {conf}, valid values are between 0.0 and 1.0"
        assert 0 <= iou <= 1, f"Invalid IoU {iou}, valid values are between 0.0 and 1.0"
        imgsz = check_imgsz(a["imgsz"])
        dev = _lib.require_cuda()
        cmask = ops._classes_mask(a["classes"], self.spec["nc"], dev)
        results = []
        if isinstance(source, torch.Tensor):
            # LoadTensor (data/loaders.py:566-638): BCHW float 0-1, sides divisible by the stride
            x = source[None] if source.ndim == 3 else source
            if x.shape[2] % 32 or x.shape[3] % 32:
                raise ValueError(f"input tensor shape {tuple(x.shape)} must be divisible by stride 32")
            t0 = time.perf_counter()
            x = x.to(dev).contiguous()
            if x.dtype not in (torch.float32, torch.bfloat16):
                x = x.float()
            B, _, H, W = x.shape
            pipe = self._pipe(B, H, W, max_det)
            dets, counts = pipe.run_tensor(x, conf, iou, (H, W), cmask, a["agnostic_nms"], a["nms_mode"])
            feats = pipe.embed() if want_feats else None
            cnt = counts.cpu().tolist()
            ms = (time.perf_counter() - t0) * 1e3 / B
            imgs = (x.float().permute(0, 2, 3, 1).flip(-1) * 255).to(torch.uint8).cpu().numpy()    # loaders convert_torch2numpy_batch
            for b in range(B):
                results.append(Results(imgs[b], f"image{b}.jpg", self.names, dets[b, :cnt[b]].clone(),
                                       {"preprocess": 0.0, "inference": ms, "postprocess": 0.0}))
                if want_feats:
                    results[-1].feats = feats[b, :cnt[b]].clone()
        else:
            frames = [source] if isinstance(source, np.ndarray) else list(source)
            if not frames:
                return []
            for f in frames:
                if not (isinstance(f, np.ndarray) and f.ndim == 3 and f.shape[2] == 3 and f.dtype == np.uint8):
                    raise TypeError("source must be HWC BGR uint8 ndarray(s) or a BCHW float tensor")
            t0 = time.perf_counter()
            if len({f.shape for f in frames}) == 1:
                h0, w0 = frames[0].shape[:2]
                (rh, rw), (H, W), top, left = letterbox_geometry(h0, w0, imgsz, auto=True)
                batch = torch.from_numpy(np.ascontiguousarray(np.stack(frames))).to(dev, non_blocking=True)
                if (rh, rw) != (h0, w0):
                    batch = ops.resize_bilinear_u8(batch, rh, rw)
                if H % 32 or W % 32:
                    raise ValueError(f"letterboxed size {H}x{W} is not a multiple of 32")
                pipe = self._pipe(len(frames), H, W, max_det)
                dets, counts = pipe(batch, conf, iou, top, left, (h0, w0), cmask, a["agnostic_nms"], a["nms_mode"])
            else:
                # frames of different shapes: each letterboxed into the imgsz canvas (auto=False), all in one forward
                (H, W), geom, scale = letterbox_table([f.shape[:2] for f in frames], imgsz)
                packed, offs = ops.pack_frames(frames)
                up = lambda arr: torch.from_numpy(arr).to(dev)
                pipe = self._pipe(len(frames), H, W, max_det)
                dets, counts = pipe.run_ragged(up(packed), up(offs), up(geom), up(scale), conf, iou, cmask, a["agnostic_nms"], a["nms_mode"])
            feats = pipe.embed() if want_feats else None
            cnt = counts.cpu().tolist()
            ms = (time.perf_counter() - t0) * 1e3 / len(frames)
            for i, f in enumerate(frames):
                results.append(Results(f, f"image{i}.jpg", self.names, dets[i, :cnt[i]].clone(),
                                       {"preprocess": 0.0, "inference": ms, "postprocess": 0.0}))
                if want_feats:
                    results[-1].feats = feats[i, :cnt[i]].clone()
        if a.get("verbose"):
            for r in results:
                print(f"{r.orig_shape[0]}x{r.orig_shape[1]} {r.verbose()}{r.speed['inference']:.1f}ms")
        return iter(results) if stream else results

    def track(self, source=None, stream=False, persist=False, **kwargs):
        """engine/model.py:559-591 + trackers/track.py: predict with conf 0.1 by default (ByteTrack wants the low-confidence boxes),
        then the tracker's update attaches ids (``Results.boxes.id``).  ``tracker``: 'bytetrack.yaml' / 'botsort.yaml' (the defaults),
        the path of a tracker YAML file (its keys over the defaults of its ``tracker_type``) or a dict of the keys.  BoT-SORT with
        ``with_reid: True`` (``model: auto``) gets each detection's appearance vector from the detector (``Results.feats``).
        A list of frames is one video, walked in order by ONE tracker (the reference's non-stream datasets); ``persist=True`` keeps
        the tracker between calls."""
        from . import byte_tracker

        tracker = kwargs.pop("tracker", "bytetrack.yaml")
        cls = byte_tracker.BYTETracker
        if isinstance(tracker, (str, os.PathLike)) and str(tracker) not in ("bytetrack.yaml", "botsort.yaml") and os.path.isfile(tracker):
            import yaml

            with open(tracker, encoding="utf-8") as fh:
                tracker = yaml.safe_load(fh) or {}
            kind = tracker.get("tracker_type")
            if kind not in ("bytetrack", "botsort"):
                raise AssertionError(f"Only 'bytetrack' and 'botsort' are supported for now, but got '{kind}'")
        if isinstance(tracker, str):
            if "botsort" in tracker:
                cls = byte_tracker.BOTSORT
            elif "bytetrack" not in tracker:
                raise AssertionError(f"Only 'bytetrack' and 'botsort' are supported for now, but got '{tracker}'")
            tracker = None
        elif isinstance(tracker, dict) and tracker.get("tracker_type") == "botsort":
            cls = byte_tracker.BOTSORT
        kwargs["conf"] = kwargs.get("conf") or 0.1
        if not (persist and getattr(self, "trackers", None)):
            self.trackers = [cls(tracker, frame_rate=30)]
        if self.trackers[0].reid:
            kwargs["_feats"] = True
        if isinstance(source, (str, os.PathLike)) or (isinstance(source, (list, tuple)) and source and isinstance(source[0], (str, os.PathLike))):
            # file sources: frames arrive batch by batch; the tracker is reset when the file changes (track.py:87-89, persist=False)
            def gen():
                last, slot = None, 0
                for r in self.predict(source, True, **kwargs):
                    ds = self.dataset
                    if getattr(ds, "mode", "") == "stream":               # one tracker per source (track.py:62-68), results arrive source by source
                        if len(self.trackers) != ds.bs:
                            self.trackers = [cls(tracker, frame_rate=30) for _ in range(ds.bs)]
                        byte_tracker.update_results([self.trackers[slot]], [r], is_stream=False)
                        slot = (slot + 1) % ds.bs
                        yield r
                        continue
                    if not persist and last is not None and r.path != last:
                        self.trackers[0].reset()
                    last = r.path
                    byte_tracker.update_results(self.trackers, [r], is_stream=False)
                    yield r

            return gen() if stream else list(gen())
        results = list(self.predict(source, False, **kwargs))
        byte_tracker.update_results(self.trackers, results, is_stream=False)
        return iter(results) if stream else results

    def fuse(self):
        return self          # BN is always folded at lowering time (engine.lower)

    def to(self, *_a, **_k):
        return self

    def info(self):
        return {"layers": len(self.spec["layers"]), "gflops_640": cfg.conv_flops(self.spec, 640, 640) / 1e9}

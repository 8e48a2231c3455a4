"""Plug the B200 detect path into an installed Ultralytics through its own extension point.

``Model.predict(source, predictor=CustomPredictorClass, ...)`` (ultralytics/engine/model.py:549) instantiates the class once,
caches it on ``model.predictor`` and from then on every ``model(frame)`` call (kalman/aircraft_detection_tracking.py:98) runs
its three stages from ``BasePredictor.stream_inference`` (engine/predictor.py:331-343):

    preprocess(im)                      replaces engine/predictor.py:152-175   (LetterBox, BGR->RGB, /255: fused into the stem kernel)
    inference(im)                       replaces AutoBackend.forward           (nn/autobackend.py:608-637: the engine's launch plan)
    postprocess(preds, img, orig_imgs)  replaces models/yolo/detect/predict.py:34-125 (NMS + scale_boxes) and returns genuine
                                        ``ultralytics.engine.results.Results`` objects

Ultralytics is imported lazily: this repository does not depend on it (the GPU test box has no copy), the class is built by
:func:`predictor_class` where it is installed.  Usage::

    from ultralytics import YOLO
    from b200dt.ultra_plugin import predictor_class
    model = YOLO("yolov8s-p2.yaml")
    model.predict(frame, predictor=predictor_class(), conf=0.15, iou=0.6)     # first call installs the predictor
    results = model(frame, verbose=False)                                      # the project's driver loop, unchanged
"""
from __future__ import annotations

import numpy as np

_CLASS = None


def results_from_dets(dets_per_image, orig_imgs, paths, names):
    """(n_i, 6) [x1, y1, x2, y2, conf, cls] tensors in original-frame pixels -> ``ultralytics.engine.results.Results``
    (construct_result, models/yolo/detect/predict.py:111-125)."""
    from ultralytics.engine.results import Results

    return [Results(o, path=p, names=names, boxes=d) for d, o, p in zip(dets_per_image, orig_imgs, paths)]


def predictor_class():
    """The ``DetectionPredictor`` subclass to pass as ``predictor=`` (built on first use, needs ``ultralytics`` importable)."""
    global _CLASS
    if _CLASS is not None:
        return _CLASS
    from ultralytics.models.yolo.detect import DetectionPredictor        # models/yolo/detect/predict.py:8

    from . import _lib, cfg, ops, weights
    from .predictor import DetectPipeline, check_imgsz, letterbox_geometry, letterbox_table

    class B200DetectionPredictor(DetectionPredictor):
        """DetectionPredictor whose three stages run on the CUDA engine of this package (no Ultralytics module executes)."""

        _b200_pipe = None

        def _pipe_for(self, batch, H, W):
            key = (batch, H, W, int(self.args.max_det))
            if self._b200_pipe is None or self._b200_pipe[0] != key:
                net = self.model.model if hasattr(self.model, "model") else self.model        # AutoBackend -> DetectionModel
                yaml_d = dict(getattr(net, "yaml", {}) or {})
                spec = cfg.resolve(yaml_d if yaml_d.get("backbone") else yaml_d.get("yaml_file", "yolov8n-p2"), nc=len(self.model.names))
                sd = weights.to_numpy_state_dict(net.state_dict())
                self._b200_pipe = (key, DetectPipeline(spec, sd, batch, H, W, int(self.args.max_det)))
            return self._b200_pipe[1]

        def preprocess(self, im):
            """im: list of HWC BGR uint8 frames (LoadPilAndNumpy, data/loaders.py:519-558).  Uploads them; the letterbox border,
            the channel swap and the /255 happen inside the stem kernel.  Frames of different shapes (pre_transform's auto=False
            case) are packed, uploaded once and letterboxed into the imgsz canvas on the GPU; NMS then scales boxes per frame."""
            import torch

            dev = _lib.require_cuda()                                  # raises without a CUDA device: there is no CPU fallback
            if isinstance(im, torch.Tensor):
                raise NotImplementedError("tensor sources: use b200dt.predictor.YOLO.predict")
            frames = list(im)
            if len({f.shape for f in frames}) != 1:
                (H, W), geom, scale = letterbox_table([f.shape[:2] for f in frames], check_imgsz(self.imgsz))
                packed, offs = ops.pack_frames(frames)
                up = lambda arr: torch.from_numpy(arr).to(dev)
                pipe = self._pipe_for(len(frames), H, W)
                canvas = pipe.letterbox(up(packed), up(offs), up(geom))
                self._b200_geom = (len(frames), H, W, 0, 0, None, up(scale))
                return canvas
            h0, w0 = frames[0].shape[:2]
            (rh, rw), (H, W), top, left = letterbox_geometry(h0, w0, check_imgsz(self.imgsz), auto=True)
            u8 = torch.from_numpy(np.ascontiguousarray(np.stack(frames))).to(dev, non_blocking=True)
            if (rh, rw) != (h0, w0):
                u8 = ops.resize_bilinear_u8(u8, rh, rw)
            self._b200_geom = (len(frames), H, W, top, left, (h0, w0), None)
            return u8

        def inference(self, im, *args, **kwargs):
            B, H, W, top, left, _, _ = self._b200_geom
            self._pipe_for(B, H, W).engine.forward_u8(im, top, left)
            return im

        def postprocess(self, preds, img, orig_imgs, **kwargs):
            B, H, W, _, _, orig_hw, scale = self._b200_geom
            pipe = self._pipe_for(B, H, W)
            cmask = ops._classes_mask(self.args.classes, len(self.model.names), img.device)
            dets, counts = pipe.finish(float(self.args.conf), float(self.args.iou), orig_hw, cmask, bool(self.args.agnostic_nms), "exact", None,
                                       scale)
            n = counts.cpu().tolist()
            return results_from_dets([dets[i, :n[i]].clone() for i in range(B)], orig_imgs, self.batch[0], self.model.names)

    _CLASS = B200DetectionPredictor
    return _CLASS

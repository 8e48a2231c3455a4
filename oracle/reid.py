"""Oracle (numpy, CPU) for BoT-SORT ReID on the detector's own features -- TEST INFRASTRUCTURE ONLY (tests/).

Restates, for botsort.yaml ``with_reid: True`` with ``model: auto`` (Ultralytics 8.3.193):
  get_obj_feats          ultralytics/models/yolo/detect/predict.py DetectionPredictor.get_obj_feats (the features of the maps that
                         feed Detect, kept by the forward pre-hook of trackers/track.py on_predict_start)
  BOTrack.update_features ultralytics/trackers/bot_sort.py BOTrack (:20-151): update / re_activate refresh the features
  BOTSORT.get_dists      ultralytics/trackers/bot_sort.py BOTSORT (:154-232) with matching.embedding_distance
                         (scipy.spatial.distance.cdist, third party) between iou_distance and fuse_score
  BYTETracker.update     byte_tracker.py: feats split with the boxes' masks (feats[remain_inds], feats[inds_second])
on top of oracle/byte_tracker.py (BOTSORT without ReID, unchanged).

These functions are restated from the reference's description without a reference checkout: they are NOT pinned by
reference-generated goldens.  If a detail turns out to differ from the reference, the reference wins.  ``BOTSORT.gaps`` records
how far each combined-cost decision is from a floating-point tie, so a test can state its margin.
"""
from __future__ import annotations

from collections import deque

import numpy as np
from scipy.spatial.distance import cdist

from . import byte_tracker as obt


def get_obj_feats(feat_maps, idxs):
    """DetectionPredictor.get_obj_feats: feat_maps = the Detect inputs [(B, C_l, h, w), ...] in Detect order, idxs = per image the
    kept anchor ids of NMS (return_idxs=True).  s = min(C_l); each level's anchor rows are averaged over groups of C_l / s
    CONSECUTIVE channels (x.permute(0, 2, 3, 1).reshape(B, -1, s, C_l // s).mean(-1)), the levels concatenated along the anchor
    axis.  Per image a float32 (n, s) array, or [] without detections, as the reference returns."""
    s = min(int(x.shape[1]) for x in feat_maps)
    B = feat_maps[0].shape[0]
    obj = np.concatenate([np.asarray(x, np.float32).transpose(0, 2, 3, 1).reshape(B, -1, s, x.shape[1] // s).mean(-1)
                          for x in feat_maps], axis=1)
    return [f[np.asarray(i, np.int64)] if len(i) else [] for f, i in zip(obj, idxs)]


def embedding_distance(tracks, detections, metric="cosine"):
    """matching.embedding_distance: max(0, cdist(track smooth_feat, detection curr_feat)) -- float64 (cdist converts)."""
    cost = np.zeros((len(tracks), len(detections)), dtype=np.float32)
    if cost.size == 0:
        return cost
    det_features = np.asarray([t.curr_feat for t in detections], dtype=np.float32)
    track_features = np.asarray([t.smooth_feat for t in tracks], dtype=np.float32)
    return np.maximum(0.0, cdist(track_features, det_features, metric))


class BOTrack(obt.BOTrack):
    """bot_sort.py BOTrack with an appearance feature: curr_feat / smooth_feat / the last 50 features, refreshed by every update
    and re_activate."""

    def __init__(self, xywh, score, cls, counter, feat=None):
        super().__init__(xywh, score, cls, counter)
        self.smooth_feat = self.curr_feat = None
        self.features = deque([], maxlen=50)
        self.alpha = 0.9
        if feat is not None:
            self.update_features(feat)

    def update_features(self, feat):
        """BOTrack.update_features, float32 and in place exactly as the reference: the first smooth_feat IS curr_feat."""
        feat /= np.linalg.norm(feat)
        self.curr_feat = feat
        if self.smooth_feat is None:
            self.smooth_feat = feat
        else:
            self.smooth_feat = self.alpha * self.smooth_feat + (1 - self.alpha) * feat
        self.features.append(feat)
        self.smooth_feat /= np.linalg.norm(self.smooth_feat)

    def re_activate(self, new_track, frame_id):
        if new_track.curr_feat is not None:
            self.update_features(new_track.curr_feat)
        super().re_activate(new_track, frame_id)

    def update(self, new_track, frame_id):
        if new_track.curr_feat is not None:
            self.update_features(new_track.curr_feat)
        super().update(new_track, frame_id)


class BOTSORT(obt.BOTSORT):
    """bot_sort.py BOTSORT with ``with_reid=True``, ``model: auto``.  update(xywh, conf, cls, img=None, feats=None): feats (n, D)
    float32 are the rows' appearance vectors; stages 1 and 3 use get_dists' combined cost."""

    def __init__(self, gmc_method="sparseOptFlow", proximity_thresh=0.5, appearance_thresh=0.8, **kw):
        super().__init__(gmc_method=gmc_method, **kw)
        self.proximity_thresh, self.appearance_thresh = proximity_thresh, appearance_thresh
        self.gaps = dict(match=np.inf, appearance=np.inf, competing=np.inf)
        self._pending = []

    def update(self, xywh, conf, cls, img=None, feats=None):
        """Splits ``feats`` like byte_tracker.py (high-score rows, then the low-score rows of the second association); the base
        update builds those two detection lists, in that order, through ``_init_track``, which takes them from here."""
        if feats is None:
            raise ValueError("BOTSORT(with_reid=True) needs the detections' features")
        conf = np.asarray(conf, np.float32)
        feats = np.asarray(feats, np.float32).reshape(len(conf), -1)
        remain = conf >= self.high
        second = (conf > self.low) & (conf < self.high)
        self._pending = [feats[remain], feats[second]]
        return super().update(xywh, conf, cls, img)

    def _init_track(self, xywh, conf, cls, idx):
        feats = self._pending.pop(0)
        return [BOTrack(list(b) + [i], s, c, self._counter, f.copy()) for b, s, c, i, f in zip(xywh, conf, cls, idx, feats)]

    def _dists(self, tracks, dets):
        """BOTSORT.get_dists."""
        dists = obt.iou_distance(tracks, dets)
        dists_mask = dists > (1 - self.proximity_thresh)
        if self.fuse:
            dists = obt.fuse_score(dists, dets)
        raw = embedding_distance(tracks, dets) / 2.0
        emb = raw.copy()
        emb[emb > (1 - self.appearance_thresh)] = 1.0
        emb[dists_mask] = 1.0
        dists = np.minimum(dists, emb)
        self._record_gaps(dists, raw[~dists_mask] if raw.size else raw)
        return dists

    def _record_gaps(self, cost, raw_emb):
        """Decision gaps of one combined cost matrix: distance of every entry to the stage thresholds (match_thresh, 0.7), of every
        unmasked embedding term to the appearance gate, and between the two smallest entries below match_thresh of every row and
        column (the pairs an assignment chooses between)."""
        if cost.size == 0:
            return
        self.gaps["match"] = min(self.gaps["match"], float(np.abs(cost - self.match_thresh).min()), float(np.abs(cost - 0.7).min()))
        if raw_emb.size:
            self.gaps["appearance"] = min(self.gaps["appearance"], float(np.abs(raw_emb - (1 - self.appearance_thresh)).min()))
        for axis in (0, 1):
            if cost.shape[axis] > 1:
                two = np.sort(np.where(cost < self.match_thresh, cost, np.inf), axis=axis)
                with np.errstate(invalid="ignore"):                 # inf - inf where a row / column has < 2 candidates
                    d = np.diff(two.take([0, 1], axis=axis), axis=axis)
                d = d[np.isfinite(d)]
                if d.size:
                    self.gaps["competing"] = min(self.gaps["competing"], float(d.min()))

"""Upstream tracker plug-in (ByteTrack, BoT-SORT with or without ReID) over the B200 kernels: mirror of ``ultralytics/trackers/byte_tracker.py`` (STrack
:14-237, BYTETracker :240-485), ``trackers/utils/matching.py`` (linear_assignment :20-63, iou_distance :66-113, fuse_score
:135-157) and the ``trackers/track.py`` callback contract (:72-102: ``tracker.update(boxes) -> (k, 8)`` rows
``[x1, y1, x2, y2, track_id, score, cls, idx]``, ``Results.update(boxes=rows[:, :-1])``).

Same names, arguments and control flow as the reference; the numeric work of a frame runs on the GPU through the C ABI:
``b2_kf_predict`` (STrack.multi_predict), ``b2_iou_cost`` (iou_distance + fuse_score), ``b2_linear_assignment`` (the
``lap.lapjv(extend_cost=True, cost_limit=thresh)`` branch -- an exact float64 shortest-augmenting-path solver, no ``lap``
dependency), ``b2_kf_update`` / ``b2_kf_initiate`` batched over the matches of a stage (the reference updates matched tracks one
by one; the stages only ever look at tracks that were NOT matched before, so batching per stage is the same computation).
Track state is float32 on the device (float64 numpy in the reference).  No CPU fallback: every call needs the CUDA library.

BoT-SORT ReID (botsort.yaml ``with_reid: True`` with ``model: auto``, bot_sort.py BOTrack.update_features, BOTSORT.get_dists,
matching.embedding_distance): the appearance vectors are the detector's own Detect-input features (``Results.feats``, gathered
by ``b2_reid_gather``) and stay on the device as float32 rows; ``b2_reid_update`` normalises / smooths them for all of a stage's
pairs in one launch, ``b2_botsort_cost`` forms the combined float64 cost of stages 1 and 3 and ``b2_linear_assignment_f64``
solves it.  A separate ReID network (``model: yolo11n-cls.pt``, ...) is not provided.
"""
from __future__ import annotations

from collections import deque
from types import SimpleNamespace

import numpy as np

from . import _lib
from .kalman_filter import KalmanFilterXYAH


class TrackState:
    """basetrack.py:9-26."""
    New, Tracked, Lost, Removed = 0, 1, 2, 3


# ---------------------------------------------------------------------------------------------------
# matching (trackers/utils/matching.py)
# ---------------------------------------------------------------------------------------------------
def _boxes_of(tracks):
    if len(tracks) and isinstance(tracks[0], np.ndarray):
        return np.ascontiguousarray(tracks, dtype=np.float32).reshape(-1, 4)
    return np.ascontiguousarray([t.xyxy for t in tracks], dtype=np.float32).reshape(-1, 4)


def iou_distance(atracks, btracks, _scores=None):
    """matching.py:66-113: 1 - IoU cost matrix (N, M), float32.  Lists of STrack or of xyxy arrays."""
    import torch

    n, m = len(atracks), len(btracks)
    if n == 0 or m == 0:
        return np.zeros((n, m), dtype=np.float32)
    _lib.require_cuda()
    lib = _lib.load()
    a = torch.as_tensor(_boxes_of(atracks), device="cuda")
    b = torch.as_tensor(_boxes_of(btracks), device="cuda")
    sc = None if _scores is None else torch.as_tensor(np.ascontiguousarray(_scores, np.float32), device="cuda")
    cost = torch.empty((n, m), dtype=torch.float32, device="cuda")
    _lib.check(lib.b2_iou_cost(_lib.ptr(a), _lib.ptr(b), _lib.ptr(sc), None, None, 1, n, m, _lib.ptr(cost), _lib.stream_ptr()))
    return cost.cpu().numpy()


def fuse_score(cost_matrix, detections):
    """matching.py:135-157 (host form, for callers that hold a cost matrix already; BYTETracker fuses inside b2_iou_cost)."""
    if cost_matrix.size == 0:
        return cost_matrix
    det_scores = np.array([d.score for d in detections], dtype=np.float32)[None].repeat(cost_matrix.shape[0], axis=0)
    return 1 - (1 - cost_matrix) * det_scores


def linear_assignment(cost_matrix, thresh, use_lap=True):
    """matching.py:20-63 -> (matches [[row, col], ...], unmatched rows, unmatched cols).  Both of the reference's branches
    return the optimum of the same thresholded problem; one exact GPU solver serves both."""
    import torch

    cost_matrix = np.asarray(cost_matrix)
    if cost_matrix.size == 0:
        return np.empty((0, 2), dtype=int), tuple(range(cost_matrix.shape[0])), tuple(range(cost_matrix.shape[1]))
    dt = np.float64 if cost_matrix.dtype == np.float64 else np.float32          # lapjv solves a float64 cost as it is
    x, y = linear_assignment_device(torch.as_tensor(np.ascontiguousarray(cost_matrix, dt), device="cuda")[None], thresh)
    x, y = x[0].cpu().numpy(), y[0].cpu().numpy()
    matches = [[ix, int(mx)] for ix, mx in enumerate(x) if mx >= 0]
    return matches, np.where(x < 0)[0], np.where(y < 0)[0]


def linear_assignment_device(cost, thresh, na=None, nb=None):
    """Batched form: cost CUDA float32 or float64 [S][n_max][m_max] (problem s uses its na[s] x nb[s] corner) -> (x [S][n_max],
    y [S][m_max]) int32 CUDA tensors, -1 = unmatched."""
    import torch

    _lib.require_cuda()
    lib = _lib.load()
    S, n, m = cost.shape
    x = torch.empty((S, n), dtype=torch.int32, device="cuda")
    y = torch.empty((S, m), dtype=torch.int32, device="cuda")
    solve = lib.b2_linear_assignment_f64 if cost.dtype == torch.float64 else lib.b2_linear_assignment
    if cost.dtype not in (torch.float32, torch.float64):
        raise TypeError(f"linear_assignment: cost dtype {cost.dtype} (float32 or float64)")
    _lib.check(solve(_lib.ptr(cost.contiguous()), _lib.ptr(na), _lib.ptr(nb), S, n, m, float(thresh), _lib.ptr(x), _lib.ptr(y), _lib.stream_ptr()))
    return x, y


def botsort_distance(tracks, detections, scores, proximity_thresh, appearance_thresh):
    """BOTSORT.get_dists with ReID (bot_sort.py:154-232, matching.embedding_distance) in one b2_botsort_cost launch: the IoU
    distance (fused with ``scores`` when given) where it is below the combined appearance / proximity gate of the float64 cosine
    distance between track ``smooth_feat`` and detection ``curr_feat``.  Returns the float64 (N, M) matrix."""
    import torch

    n, m = len(tracks), len(detections)
    if n == 0 or m == 0:
        return np.zeros((n, m), dtype=np.float64)
    _lib.require_cuda()
    lib = _lib.load()
    a = torch.as_tensor(_boxes_of(tracks), device="cuda")
    b = torch.as_tensor(_boxes_of(detections), device="cuda")
    sc = None if scores is None else torch.as_tensor(np.ascontiguousarray(scores, np.float32), device="cuda")
    fa = torch.stack([t.smooth_feat for t in tracks])
    fb = torch.stack([d.curr_feat for d in detections])
    if fa.shape[1] != fb.shape[1]:
        raise ValueError(f"feature widths differ: tracks {fa.shape[1]}, detections {fb.shape[1]}")
    cost = torch.empty((n, m), dtype=torch.float64, device="cuda")
    # dists > (1 - proximity_thresh) compares a float32 matrix with a Python float: NumPy 2 rounds the scalar to float32;
    # emb > (1 - appearance_thresh) compares float64 with float64
    _lib.check(lib.b2_botsort_cost(_lib.ptr(a), _lib.ptr(b), _lib.ptr(sc), None, None, _lib.ptr(fa), _lib.ptr(fb), fa.shape[1], 1, n, m,
                                   float(np.float32(1 - proximity_thresh)), float(1 - appearance_thresh), _lib.ptr(cost), _lib.stream_ptr()))
    return cost.cpu().numpy()


def reid_update(curr, smooth=None, has_smooth=None):
    """BOTrack.update_features for every row of ``curr`` (CUDA float32 [N][D], normalised in place) in one b2_reid_update launch.
    ``smooth``: the rows' previous smooth features (float32 [N][D], updated in place) with ``has_smooth`` (bool per row) telling
    which exist; None: first features only.  Returns (curr, smooth)."""
    import torch

    _lib.require_cuda()
    N, D = curr.shape
    if smooth is None:
        smooth = torch.empty_like(curr)
    mask = None if has_smooth is None else torch.as_tensor(np.asarray(has_smooth, np.uint8), device="cuda")
    _lib.check(_lib.load().b2_reid_update(_lib.ptr(curr), _lib.ptr(smooth), _lib.ptr(mask), N, D, _lib.stream_ptr()))
    return curr, smooth


# ---------------------------------------------------------------------------------------------------
# STrack / BYTETracker
# ---------------------------------------------------------------------------------------------------
class STrack:
    """byte_tracker.py:14-237 for axis-aligned boxes.  mean (8,) / covariance (8, 8) are numpy copies of the device state."""

    shared_kalman = None
    _count = 0

    def __init__(self, xywh, score, cls):
        assert len(xywh) in {5, 6}, f"expected 5 or 6 values but got {len(xywh)}"
        x, y, w, h = (np.float32(v) for v in xywh[:4])
        self._tlwh = np.asarray([x - w / 2, y - h / 2, w, h], dtype=np.float32)
        self.kalman_filter = None
        self.mean, self.covariance = None, None
        self.is_activated = False
        self.score, self.cls, self.idx = score, cls, xywh[-1]
        self.tracklet_len = 0
        self.angle = xywh[4] if len(xywh) == 6 else None
        self.track_id = 0
        self.state = TrackState.New
        self.start_frame = self.frame_id = 0

    @staticmethod
    def next_id():
        STrack._count += 1
        return STrack._count

    @staticmethod
    def reset_id():
        STrack._count = 0

    @property
    def end_frame(self):
        return self.frame_id

    def mark_lost(self):
        self.state = TrackState.Lost

    def mark_removed(self):
        self.state = TrackState.Removed

    @staticmethod
    def multi_predict(stracks):
        """:94-107 -- one b2_kf_predict launch for the pool."""
        if len(stracks) <= 0:
            return
        mm = np.asarray([st.mean.copy() for st in stracks])
        mc = np.asarray([st.covariance for st in stracks])
        for i, st in enumerate(stracks):
            if st.state != TrackState.Tracked:
                mm[i][7] = 0
        mm, mc = STrack.shared_kalman.multi_predict(mm, mc)
        for i, st in enumerate(stracks):
            st.mean, st.covariance = mm[i], mc[i]

    @staticmethod
    def multi_gmc(stracks, H=np.eye(2, 3)):
        """:109-125 -- the camera-motion warp applied to every state and covariance (8 x 8 products on the host, as the reference)."""
        if stracks:
            R8x8 = np.kron(np.eye(4, dtype=float), H[:2, :2])
            t = H[:2, 2]
            for st in stracks:
                mean = R8x8.dot(st.mean)
                mean[:2] += t
                st.mean, st.covariance = mean, R8x8.dot(st.covariance).dot(R8x8.transpose())

    # the three state changes of the reference take the Kalman result computed for the whole stage (see BYTETracker._apply)
    def activate(self, kalman_filter, frame_id, mean, covariance):
        self.kalman_filter = kalman_filter
        self.track_id = self.next_id()
        self.mean, self.covariance = mean, covariance
        self.tracklet_len = 0
        self.state = TrackState.Tracked
        if frame_id == 1:
            self.is_activated = True
        self.frame_id = self.start_frame = frame_id

    def re_activate(self, new_track, frame_id, mean, covariance, new_id=False):
        self.mean, self.covariance = mean, covariance
        self.tracklet_len = 0
        self.state = TrackState.Tracked
        self.is_activated = True
        self.frame_id = frame_id
        if new_id:
            self.track_id = self.next_id()
        self.score, self.cls, self.angle, self.idx = new_track.score, new_track.cls, new_track.angle, new_track.idx

    def update(self, new_track, frame_id, mean, covariance):
        self.frame_id = frame_id
        self.tracklet_len += 1
        self.mean, self.covariance = mean, covariance
        self.state = TrackState.Tracked
        self.is_activated = True
        self.score, self.cls, self.angle, self.idx = new_track.score, new_track.cls, new_track.angle, new_track.idx

    @property
    def tlwh(self):
        if self.mean is None:
            return self._tlwh.copy()
        ret = self.mean[:4].copy()
        ret[2] *= ret[3]
        ret[:2] -= ret[2:] / 2
        return ret

    @property
    def xyxy(self):
        ret = self.tlwh.copy()
        ret[2:] += ret[:2]
        return ret

    @staticmethod
    def tlwh_to_xyah(tlwh):
        ret = np.asarray(tlwh).copy()
        ret[:2] += ret[2:] / 2
        ret[2] /= ret[3]
        return ret

    def convert_coords(self, tlwh):
        return self.tlwh_to_xyah(tlwh)

    @property
    def xywh(self):
        ret = np.asarray(self.tlwh).copy()
        ret[:2] += ret[2:] / 2
        return ret

    @property
    def result(self):
        return self.xyxy.tolist() + [self.track_id, self.score, self.cls, self.idx]

    def __repr__(self):
        return f"OT_{self.track_id}_({self.start_frame}-{self.end_frame})"


DEFAULT_ARGS = dict(tracker_type="bytetrack", track_high_thresh=0.25, track_low_thresh=0.1, new_track_thresh=0.25, track_buffer=30,
                    match_thresh=0.8, fuse_score=True)          # ultralytics/cfg/trackers/bytetrack.yaml


class BYTETracker:
    """byte_tracker.py:240-485.  ``args``: a namespace / dict with the bytetrack.yaml keys (None: the yaml's defaults)."""

    reid = False                # BOTSORT with_reid: detections carry appearance features

    def __init__(self, args=None, frame_rate=30):
        if args is None:
            args = DEFAULT_ARGS
        if isinstance(args, dict):
            args = SimpleNamespace(**{**DEFAULT_ARGS, **args})
        self.tracked_stracks, self.lost_stracks, self.removed_stracks = [], [], []
        self.frame_id = 0
        self.args = args
        self.max_time_lost = int(frame_rate / 30.0 * args.track_buffer)
        self.kalman_filter = self.get_kalmanfilter()
        STrack.shared_kalman = self.kalman_filter
        self.reset_id()

    def get_kalmanfilter(self):
        return KalmanFilterXYAH()

    def init_track(self, results, img=None):
        if len(results) == 0:
            return []
        bboxes = np.asarray(results.xywh, dtype=np.float32)
        bboxes = np.concatenate([bboxes, np.arange(len(bboxes), dtype=np.float32).reshape(-1, 1)], axis=-1)
        return [STrack(xywh, s, c) for (xywh, s, c) in zip(bboxes, np.asarray(results.conf), np.asarray(results.cls))]

    def get_dists(self, tracks, detections):
        """Cost of stages 1 and 3: iou_distance (+ fuse_score) in one launch."""
        return iou_distance(tracks, detections, [d.score for d in detections] if self.args.fuse_score else None)

    def multi_predict(self, tracks):
        STrack.multi_predict(tracks)

    @staticmethod
    def reset_id():
        STrack.reset_id()

    def reset(self):
        self.tracked_stracks, self.lost_stracks, self.removed_stracks = [], [], []
        self.frame_id = 0
        self.kalman_filter = self.get_kalmanfilter()
        STrack.shared_kalman = self.kalman_filter
        self.reset_id()

    def _apply(self, pairs, touched):
        """KalmanFilter.update for every (track, detection) pair of one association stage in ONE launch, then the reference's
        per-pair state change: ``update`` for tracked tracks, ``re_activate`` for lost ones (:346-353, :361-368, :380-382).
        ``touched`` collects the tracks, re-found ones flagged."""
        if not pairs:
            return
        if self.reid:
            self._update_features(pairs)
        means, covs = self.kalman_filter.update(np.asarray([t.mean for t, _ in pairs]), np.asarray([t.covariance for t, _ in pairs]),
                                                np.asarray([t.convert_coords(d.tlwh) for t, d in pairs], dtype=np.float32))
        for (trk, det), m, c in zip(pairs, means, covs):
            was_tracked = trk.state == TrackState.Tracked
            if was_tracked:
                trk.update(det, self.frame_id, m, c)
            else:
                trk.re_activate(det, self.frame_id, m, c, new_id=False)
            touched.append((trk, not was_tracked))

    def _stage(self, tracks, dets, thresh, dists):
        """One association stage: cost launch (``dists(tracks, dets)``) + assignment launch -> (pairs, unmatched track indices,
        unmatched detection indices)."""
        cost = dists(tracks, dets)
        matches, free_t, free_d = linear_assignment(cost, thresh=thresh)
        return [(tracks[a], dets[b]) for a, b in matches], list(free_t), list(free_d)

    def update(self, results, img=None, feats=None):
        """:299-410.  results: a ``Boxes``-like object on the host (``.conf``, ``.cls``, ``.xywh``, boolean-mask indexing);
        feats: the rows' appearance vectors (``Results.feats``; read by BOTSORT with ReID only), split like the boxes.
        Stages as in the reference: high-score boxes against tracked + lost tracks (threshold ``match_thresh``, scores fused when
        ``fuse_score``), low-score boxes against the still-unmatched TRACKED tracks (plain IoU, 0.5), the remaining high-score
        boxes against the one-frame-old unconfirmed tracks (0.7), then births, time-outs and de-duplication."""
        self.frame_id += 1
        cfg_ = self.args
        conf = np.asarray(results.conf)
        high = conf >= cfg_.track_high_thresh
        low = (conf > cfg_.track_low_thresh) & (conf < cfg_.track_high_thresh)
        feats_high = feats_low = None
        if self.reid:
            feats_high, feats_low = self._split_feats(feats, len(conf), high, low)
        dets_high = self.init_track(results[high], feats_high)
        confirmed = [t for t in self.tracked_stracks if t.is_activated]
        tentative = [t for t in self.tracked_stracks if not t.is_activated]
        pool = self.joint_stracks(confirmed, self.lost_stracks)
        self.multi_predict(pool)
        if hasattr(self, "gmc") and img is not None:              # BoT-SORT: global motion compensation (:329-337)
            try:
                warp = self.gmc.apply(img, None)
            except Exception:
                warp = np.eye(2, 3)
            STrack.multi_gmc(pool, warp)
            STrack.multi_gmc(tentative, warp)
        touched, newly_lost, dropped = [], [], []
        # stage 1
        pairs, free_t, free_d = self._stage(pool, dets_high, cfg_.match_thresh, self.get_dists)
        self._apply(pairs, touched)
        # stage 2: only tracks that were being tracked compete for the low-score boxes; the rest of stage 1's leftovers stay lost
        dets_low = self.init_track(results[low], feats_low)
        still_tracked = [pool[k] for k in free_t if pool[k].state == TrackState.Tracked]
        pairs, free_t2, _ = self._stage(still_tracked, dets_low, 0.5, iou_distance)
        self._apply(pairs, touched)
        for k in free_t2:
            trk = still_tracked[k]
            if trk.state != TrackState.Lost:
                trk.mark_lost()
                newly_lost.append(trk)
        # stage 3
        leftovers = [dets_high[k] for k in free_d]
        pairs, free_u, free_d = self._stage(tentative, leftovers, 0.7, self.get_dists)
        self._apply(pairs, touched)
        for k in free_u:
            tentative[k].mark_removed()
            dropped.append(tentative[k])
        # births: one b2_kf_initiate launch
        born = [leftovers[k] for k in free_d if leftovers[k].score >= cfg_.new_track_thresh]
        if born:
            means, covs = self.kalman_filter.initiate(np.asarray([t.convert_coords(t._tlwh) for t in born], dtype=np.float32))
            for trk, m, c in zip(born, means, covs):
                trk.activate(self.kalman_filter, self.frame_id, m, c)
                touched.append((trk, False))
        for trk in self.lost_stracks:                              # time-outs
            if self.frame_id - trk.end_frame > self.max_time_lost:
                trk.mark_removed()
                dropped.append(trk)
        # list bookkeeping (:397-408): survivors, then this frame's updated / born tracks, then the re-found ones
        alive = [t for t in self.tracked_stracks if t.state == TrackState.Tracked]
        alive = self.joint_stracks(alive, [t for t, refound in touched if not refound])
        alive = self.joint_stracks(alive, [t for t, refound in touched if refound])
        lost = self.sub_stracks(self.lost_stracks, alive) + newly_lost
        lost = self.sub_stracks(lost, self.removed_stracks)
        self.tracked_stracks, self.lost_stracks = self.remove_duplicate_stracks(alive, lost)
        self.removed_stracks = (self.removed_stracks + dropped)
        if len(self.removed_stracks) > 1000:
            self.removed_stracks = self.removed_stracks[-999:]
        return np.asarray([t.result for t in self.tracked_stracks if t.is_activated], dtype=np.float32)

    @staticmethod
    def joint_stracks(tlista, tlistb):
        """:450-463: union keeping the first occurrence of every track id."""
        seen, merged = set(), []
        for trk in list(tlista) + list(tlistb):
            if trk.track_id not in seen:
                seen.add(trk.track_id)
                merged.append(trk)
        return merged

    @staticmethod
    def sub_stracks(tlista, tlistb):
        """:465-469."""
        gone = {trk.track_id for trk in tlistb}
        return [trk for trk in tlista if trk.track_id not in gone]

    @staticmethod
    def remove_duplicate_stracks(stracksa, stracksb):
        """:471-485: of a tracked / lost pair that overlaps with IoU > 0.85 the one with the shorter history goes."""
        close = np.argwhere(iou_distance(stracksa, stracksb) < 0.15)
        drop_a, drop_b = set(), set()
        for ia, ib in close:
            span_a = stracksa[ia].frame_id - stracksa[ia].start_frame
            span_b = stracksb[ib].frame_id - stracksb[ib].start_frame
            (drop_b if span_a > span_b else drop_a).add(int(ib if span_a > span_b else ia))
        return ([t for k, t in enumerate(stracksa) if k not in drop_a], [t for k, t in enumerate(stracksb) if k not in drop_b])


# ---------------------------------------------------------------------------------------------------
# BoT-SORT without ReID (trackers/bot_sort.py: BOTrack :20-151, BOTSORT :154-232; utils/gmc.py)
# ---------------------------------------------------------------------------------------------------
class GMC:
    """utils/gmc.py:14-350 for the methods 'sparseOptFlow' (botsort.yaml's default) and none.  Host-side OpenCV exactly as in the
    reference (goodFeaturesToTrack, calcOpticalFlowPyrLK, estimateAffinePartial2D): one 2 x 3 matrix per frame, not a GPU path."""

    def __init__(self, method="sparseOptFlow", downscale=2):
        self.method = None if method in ("none", "None", None) else method
        if self.method not in (None, "sparseOptFlow"):
            raise NotImplementedError(f"GMC method {method!r}: only 'sparseOptFlow' and 'none' are provided")
        self.downscale = max(1, downscale)
        self.feature_params = dict(maxCorners=1000, qualityLevel=0.01, minDistance=1, blockSize=3, useHarrisDetector=False, k=0.04)
        self.reset_params()

    def reset_params(self):
        self.prevFrame = self.prevKeyPoints = None
        self.initializedFirstFrame = False

    def apply(self, raw_frame, detections=None):
        import copy

        import cv2

        if self.method is None:
            return np.eye(2, 3)
        height, width, c = raw_frame.shape
        frame = cv2.cvtColor(raw_frame, cv2.COLOR_BGR2GRAY) if c == 3 else raw_frame
        H = np.eye(2, 3)
        if self.downscale > 1.0:
            frame = cv2.resize(frame, (width // self.downscale, height // self.downscale))
        keypoints = cv2.goodFeaturesToTrack(frame, mask=None, **self.feature_params)
        if not self.initializedFirstFrame or self.prevKeyPoints is None:
            self.prevFrame, self.prevKeyPoints, self.initializedFirstFrame = frame.copy(), copy.copy(keypoints), True
            return H
        matched, status, _ = cv2.calcOpticalFlowPyrLK(self.prevFrame, frame, self.prevKeyPoints, None)
        prev = np.array([self.prevKeyPoints[i] for i in range(len(status)) if status[i]])
        curr = np.array([matched[i] for i in range(len(status)) if status[i]])
        if prev.shape[0] > 4 and prev.shape[0] == curr.shape[0]:
            H, _ = cv2.estimateAffinePartial2D(prev, curr, cv2.RANSAC)
            if self.downscale > 1.0:
                H[0, 2] *= self.downscale
                H[1, 2] *= self.downscale
        self.prevFrame, self.prevKeyPoints = frame.copy(), copy.copy(keypoints)
        return H


class BOTrack(STrack):
    """bot_sort.py:20-151: XYWH filter, both size velocities zeroed while a track is not Tracked.  With ReID: ``curr_feat`` /
    ``smooth_feat`` (CUDA float32 rows) and the last 50 ``features``, set by BOTSORT in batches (``b2_reid_update``)."""

    shared_kalman = None

    def __init__(self, xywh, score, cls):
        super().__init__(xywh, score, cls)
        self.smooth_feat = self.curr_feat = None
        self.features = deque([], maxlen=50)
        self.alpha = 0.9

    @staticmethod
    def multi_predict(stracks):
        if len(stracks) <= 0:
            return
        mm = np.asarray([st.mean.copy() for st in stracks])
        mc = np.asarray([st.covariance for st in stracks])
        for i, st in enumerate(stracks):
            if st.state != TrackState.Tracked:
                mm[i][6] = 0
                mm[i][7] = 0
        mm, mc = BOTrack.shared_kalman.multi_predict(mm, mc)
        for i, st in enumerate(stracks):
            st.mean, st.covariance = mm[i], mc[i]

    @property
    def tlwh(self):
        if self.mean is None:
            return self._tlwh.copy()
        ret = self.mean[:4].copy()
        ret[:2] -= ret[2:] / 2
        return ret

    def convert_coords(self, tlwh):
        return self.tlwh_to_xywh(tlwh)

    @staticmethod
    def tlwh_to_xywh(tlwh):
        ret = np.asarray(tlwh).copy()
        ret[:2] += ret[2:] / 2
        return ret


BOTSORT_DEFAULT_ARGS = dict(DEFAULT_ARGS, tracker_type="botsort", gmc_method="sparseOptFlow", proximity_thresh=0.5, appearance_thresh=0.8,
                            with_reid=False, model="auto")          # ultralytics/cfg/trackers/botsort.yaml


class BOTSORT(BYTETracker):
    """bot_sort.py:154-232: ByteTrack's association on the XYWH filter plus global motion compensation from the frame handed to
    ``update(results, img, feats)``.  ``with_reid=True`` with ``model: auto``: ``feats`` (n, D) are the detections' appearance
    vectors and stages 1 and 3 use the combined IoU / appearance cost (``botsort_distance``)."""

    def __init__(self, args=None, frame_rate=30):
        from .kalman_filter import KalmanFilterXYWH

        self._kf_cls = KalmanFilterXYWH
        if args is None:
            args = BOTSORT_DEFAULT_ARGS
        if isinstance(args, dict):
            args = SimpleNamespace(**{**BOTSORT_DEFAULT_ARGS, **args})
        self.reid = bool(getattr(args, "with_reid", False))
        if self.reid and getattr(args, "model", "auto") != "auto":
            raise NotImplementedError(f"BoT-SORT ReID model {args.model!r}: only the detector's own features (model: auto) are provided")
        super().__init__(args, frame_rate)
        self.gmc = GMC(method=args.gmc_method)
        self.proximity_thresh, self.appearance_thresh = args.proximity_thresh, args.appearance_thresh
        self.encoder = None

    def get_kalmanfilter(self):
        kf = self._kf_cls()
        BOTrack.shared_kalman = kf
        return kf

    def init_track(self, results, img=None):
        """``img``: with ReID, the rows' features (CUDA float32, a private copy): normalised as the BOTrack constructor's
        update_features does, in one launch."""
        if len(results) == 0:
            return []
        bboxes = np.asarray(results.xywh, dtype=np.float32)
        bboxes = np.concatenate([bboxes, np.arange(len(bboxes), dtype=np.float32).reshape(-1, 1)], axis=-1)
        tracks = [BOTrack(xywh, s, c) for (xywh, s, c) in zip(bboxes, np.asarray(results.conf), np.asarray(results.cls))]
        if self.reid and img is not None:
            curr, smooth = reid_update(img)
            for t, c, sm in zip(tracks, curr, smooth):
                t.curr_feat, t.smooth_feat = c, sm
                t.features.append(c)
        return tracks

    def get_dists(self, tracks, detections):
        if not self.reid:
            return super().get_dists(tracks, detections)
        return botsort_distance(tracks, detections, [d.score for d in detections] if self.args.fuse_score else None,
                                self.proximity_thresh, self.appearance_thresh)

    @staticmethod
    def _split_feats(feats, n, high, low):
        """feats[remain_inds], feats[inds_second] (byte_tracker.py update) as CUDA float32 copies."""
        import torch

        if feats is None:
            raise ValueError("BOTSORT(with_reid=True).update needs the detections' features (Results.feats)")
        f = torch.as_tensor(feats, dtype=torch.float32, device="cuda")
        if f.ndim != 2 or f.shape[0] != n:
            raise ValueError(f"feats of shape {tuple(f.shape)} for {n} detections")
        pick = lambda m: f.index_select(0, torch.as_tensor(np.flatnonzero(m), device="cuda"))
        return pick(high), pick(low)

    def _update_features(self, pairs):
        """update_features(det.curr_feat) of every track of one stage's pairs (BOTrack.update / re_activate) in one launch."""
        import torch

        curr = torch.stack([d.curr_feat for _, d in pairs])
        smooth = torch.stack([t.smooth_feat if t.smooth_feat is not None else d.curr_feat for t, d in pairs])
        curr, smooth = reid_update(curr, smooth, [t.smooth_feat is not None for t, _ in pairs])
        for (t, _), c, sm in zip(pairs, curr, smooth):
            t.curr_feat, t.smooth_feat = c, sm
            t.features.append(c)

    def multi_predict(self, tracks):
        BOTrack.multi_predict(tracks)

    def reset(self):
        super().reset()
        self.gmc.reset_params()


# ---------------------------------------------------------------------------------------------------
# trackers/track.py:72-102: attach ids to a list of Results
# ---------------------------------------------------------------------------------------------------
def update_results(trackers, results, is_stream=True):
    """on_predict_postprocess_end: results[i].boxes -> tracker.update -> results[i] = results[i][idx] with boxes replaced by the
    (k, 7) track rows [x1, y1, x2, y2, id, conf, cls].  Results without tracks are left untouched, as in the reference."""
    for i, result in enumerate(results):
        tracker = trackers[i if is_stream else 0]
        det = result.boxes.cpu().numpy()
        tracks = tracker.update(det, getattr(result, "orig_img", None), getattr(result, "feats", None))
        if len(tracks) == 0:
            continue
        result.update(boxes=tracks[:, :-1])
    return results

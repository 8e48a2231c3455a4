"""Host-side mirror of the project's tracker API over the CUDA Kalman track bank (csrc/tracker.cu).

  EnhancedMultiTargetTracker   same constructor, ``update(detections) -> list[dict]``, ``stats``,
                               ``frame_count``, ``next_track_id``, ``trackers``, ``get_statistics()`` as
                               kalman/enhanced_multi_target_tracker.py:4-304 (one video stream).
  TrackerBank                  the batched form the B200 pipeline uses: S independent streams advanced by
                               one launch sequence per frame, detections and results resident on the GPU.

All Kalman / association / lifecycle arithmetic runs in the CUDA library; this module only marshals
arguments and formats the output dicts (get_track_info, enhanced_aircraft_kalman_tracker.py:335-383).
"""
from __future__ import annotations

import ctypes as C
import math

import numpy as np

from . import _lib

TRACK_COLS, TRAJ_LEN = _lib.TRACK_COLS, _lib.TRAJ_LEN
_STAT_KEYS = ("total_tracks_created", "total_tracks_terminated", "current_active_tracks",
              "long_term_predictions", "successful_recoveries")


class TrackerBank:
    """S independent multi-target trackers (one per video stream) resident on one GPU.

    ``capacity`` bounds the simultaneously live tracks per stream (the reference's list is unbounded,
    enhanced_multi_target_tracker.py:92-101): ``grow()`` enlarges the bank in place, ``stats_async()`` /
    ``export()`` expose the ``dropped`` counter, and the callers in this package (EnhancedMultiTargetTracker,
    DetectTrackPipeline) grow ahead of need and raise if a detection was ever dropped.
    ``max_out`` (default: capacity) is the number of rows per stream the output block holds."""

    def __init__(self, n_streams, capacity=256, max_dets=300, max_lost_frames=450, min_hits=3, iou_threshold=0.3, device=None,
                 max_out=None, mode=0):
        """mode 1: the rules of camera_motion_compensation's MotionCompensatedMultiTracker / MotionResetKalmanTracker."""
        self.device = device or _lib.require_cuda()
        self.lib = _lib.load()
        self.mode = int(mode)
        self.S, self.capacity, self.max_dets = int(n_streams), int(capacity), int(max_dets)
        self.max_lost_frames, self.min_hits, self.iou_threshold = int(max_lost_frames), int(min_hits), float(iou_threshold)
        self._follow_capacity = max_out is None
        self.max_out = self.capacity if max_out is None else int(max_out)
        self._h = C.c_void_p()
        _lib.check(self.lib.b2_tracker_create_ex(self.S, self.capacity, self.max_dets, self.max_lost_frames, self.min_hits,
                                                 self.iou_threshold, self.mode, C.byref(self._h)))
        self._alloc_outputs()

    def _alloc_outputs(self):
        import torch

        self.rows = torch.zeros((self.S, self.max_out, TRACK_COLS), dtype=torch.float32, device=self.device)
        self.counts = torch.zeros((self.S,), dtype=torch.int32, device=self.device)
        self.traj = self.traj_len = None
        self.extra = torch.zeros((self.S, self.max_out, 4), dtype=torch.float32, device=self.device) if self.mode else None
        self.stats_dev = torch.zeros((self.S, 8), dtype=torch.int64, device=self.device)

    def close(self):
        if getattr(self, "_h", None):
            self.lib.b2_tracker_destroy(self._h)
            self._h = None

    __del__ = close

    def reset(self):
        _lib.check(self.lib.b2_tracker_reset(self._h, _lib.stream_ptr()))

    def reset_streams(self, flags, stream=None):
        """``reset()`` for the streams whose CUDA int32 ``flags`` [S] entry is non-zero, ordered on the stream (no synchronisation)."""
        assert flags.is_cuda and flags.dtype.itemsize == 4 and flags.numel() == self.S
        _lib.check(self.lib.b2_tracker_reset_streams(self._h, _lib.ptr(flags), _lib.stream_ptr(stream)))

    def grow(self, new_capacity):
        """Enlarge every stream's bank to ``new_capacity`` slots (state, ids and slot indices are kept; synchronises)."""
        _lib.check(self.lib.b2_tracker_grow(self._h, int(new_capacity), _lib.stream_ptr()))
        self.capacity = int(new_capacity)
        if self._follow_capacity:
            self.max_out = self.capacity
            self._alloc_outputs()

    def update(self, dets, det_counts, with_trajectory=True, stream=None):
        """dets: CUDA float32 [S][max_dets][cols>=4] rows x1,y1,x2,y2,...; det_counts: CUDA int32 [S].
        Returns (rows [S][max_out][20], counts [S]) device tensors (views of internal buffers)."""
        import torch

        assert dets.is_cuda and dets.is_contiguous() and dets.shape[0] == self.S and dets.shape[1] == self.max_dets
        if with_trajectory and self.traj is None:
            self.traj = torch.zeros((self.S, self.max_out, TRAJ_LEN, 2), dtype=torch.float32, device=self.device)
            self.traj_len = torch.zeros((self.S, self.max_out), dtype=torch.int32, device=self.device)
        _lib.check(self.lib.b2_tracker_update_ex(self._h, _lib.ptr(dets), dets.shape[2], _lib.ptr(det_counts), _lib.ptr(self.rows),
                                                 _lib.ptr(self.counts), _lib.ptr(self.traj) if with_trajectory else None,
                                                 _lib.ptr(self.traj_len) if with_trajectory else None, _lib.ptr(self.extra), self.max_out,
                                                 _lib.stream_ptr(stream)))
        return self.rows, self.counts

    def stats_async(self, stream=None, out=None):
        """[S][8] int64 device snapshot {created, terminated, active, long_term, recoveries, dropped, 0, 0} (mode 1: [6], [7] =
        individual_resets, tracking_recoveries), stream-ordered, into ``out`` (default: an internal buffer)."""
        out = self.stats_dev if out is None else out
        _lib.check(self.lib.b2_tracker_stats(self._h, _lib.ptr(out), _lib.stream_ptr(stream)))
        return out

    def predict_only(self, stream=None):
        """AircraftKalmanTracker.predict alone on every live track."""
        _lib.check(self.lib.b2_tracker_bank_predict(self._h, _lib.stream_ptr(stream)))

    def export(self, stream_idx=0):
        """Dense state of one stream (synchronises): x (n,8), P (n,8,8), meta (n,8) int32, stats (8,) int64."""
        cap = self.capacity
        x = np.zeros((cap, 8), np.float32)
        P = np.zeros((cap, 64), np.float32)
        meta = np.zeros((cap, 8), np.int32)
        n = C.c_int32()
        stats = (C.c_longlong * 8)()
        _lib.check(self.lib.b2_tracker_export(self._h, stream_idx, x.ctypes.data_as(C.c_void_p), P.ctypes.data_as(C.c_void_p),
                                              meta.ctypes.data_as(C.c_void_p), C.byref(n), stats))
        k = n.value
        order = np.argsort(meta[:k, 0], kind="stable")          # reference list order == ascending track id
        return x[:k][order], P[:k].reshape(k, 8, 8)[order], meta[:k][order], np.array(list(stats), np.int64)

    def export_motion(self, stream_idx=0):
        """prediction_confidence of one stream's live tracks, ascending track id (synchronises)."""
        m = np.zeros((self.capacity, 8), np.float32)
        n = C.c_int32()
        _lib.check(self.lib.b2_tracker_export_motion(self._h, stream_idx, m.ctypes.data_as(C.c_void_p), C.byref(n)))
        m = m[:n.value]
        return m[np.argsort(m[:, 0].copy().view(np.int32), kind="stable"), 6]

    def export_reset(self, stream_idx=0):
        """mode 1: (n, 7) {id, reset_count, last_reset_frame, motion_consistency, len(position_history), len(motion_scores),
        len(bbox_history)} of one stream's live tracks, ascending track id (synchronises)."""
        m = np.zeros((self.capacity, 8), np.float32)
        n = C.c_int32()
        _lib.check(self.lib.b2_tracker_export_reset(self._h, stream_idx, m.ctypes.data_as(C.c_void_p), C.byref(n)))
        m = m[:n.value]
        iv = m.view(np.int32)
        order = np.argsort(iv[:, 0], kind="stable")
        out = np.stack([iv[:, 0], iv[:, 1], iv[:, 2], m[:, 3], iv[:, 4], iv[:, 5], iv[:, 6]], 1).astype(np.float64)
        return out[order]

    @staticmethod
    def bytes_per_track():
        a, b = C.c_int(), C.c_int()
        _lib.load().b2_tracker_bytes_per_track(C.byref(a), C.byref(b))
        return a.value, b.value


def rows_to_dicts(rows, traj=None, traj_len=None):
    """(n, 20) float32 rows (+ trajectories) of one stream -> list of get_track_info dicts, ascending id."""
    rows = np.ascontiguousarray(rows, np.float32)
    irows = rows.view(np.int32)
    order = np.argsort(irows[:, 0], kind="stable")
    out = []
    for k in order:
        r, ir = rows[k], irows[k]
        predicted = bool(ir[6])
        d = {
            "track_id": f"T{int(ir[0]):03d}",
            "bbox": r[1:5].astype(np.float64),
            "confidence": float(r[5]),
            "status": "predicted" if predicted else "detected",
            "age": int(ir[7]), "hits": int(ir[8]), "hit_streak": int(ir[9]),
            "time_since_update": int(ir[10]), "lost_frames": int(ir[11]), "is_lost": bool(ir[12]),
            "trajectory": [] if traj is None else [(float(a), float(b)) for a, b in traj[k][:int(traj_len[k])]],
            "velocity": r[13:15].astype(np.float64),
            "motion_confidence": float(r[15]), "is_stable_motion": bool(ir[16]),
            "speed": float(r[17]), "direction": float(r[18]),
        }
        out.append(d)
    return out


class _TrackView:
    """Read-only view of one track, with the attributes callers of ``tracker.trackers`` read
    (kalman/enhanced_multi_target_tracker.py:288-304, camera_motion_compensation subclasses)."""

    def __init__(self, x, P, meta):
        self.track_id = f"T{int(meta[0]):03d}"
        self.x, self.P = x.astype(np.float64), P.astype(np.float64)
        self.age, self.hits, self.hit_streak = int(meta[1]), int(meta[2]), int(meta[3])
        self.time_since_update, self.lost_frames, self.is_lost = int(meta[4]), int(meta[5]), bool(meta[6])


class EnhancedMultiTargetTracker:
    """Drop-in for kalman/enhanced_multi_target_tracker.py:4 (single stream).

    The reference's track list is unbounded; the bank behind this class starts at ``capacity`` slots and doubles
    (``TrackerBank.grow``) before a frame could overflow it, so no detection is ever dropped.  ``max_dets`` bounds the
    detections of one frame (the NMS cap of the detector, 300); more raise ``ValueError``.
    """

    def __init__(self, max_lost_frames=450, min_hits=3, iou_threshold=0.3, capacity=512, max_dets=300, verbose=False):
        import torch

        self.max_lost_frames, self.min_hits, self.iou_threshold = max_lost_frames, min_hits, iou_threshold
        self.bank = TrackerBank(1, capacity, max_dets, max_lost_frames, min_hits, iou_threshold)
        self.frame_count = 0
        self.next_track_id = 1
        self.stats = {k: 0 for k in _STAT_KEYS}
        self.verbose = verbose
        self._dets = torch.zeros((1, max_dets, 4), dtype=torch.float32, device=self.bank.device)
        self._host = torch.zeros((max_dets, 4), dtype=torch.float32).pin_memory()
        self._cnt = torch.zeros((1,), dtype=torch.int32, device=self.bank.device)

    def update(self, detections):
        """detections: list of [x1, y1, x2, y2, conf] -> list of track-info dicts (ascending track id)."""
        import torch

        n = len(detections)
        if n > self.bank.max_dets:
            raise ValueError(f"{n} detections exceed max_dets={self.bank.max_dets}")
        # every detection may found a track: make room first (the reference appends without bound, :92-101)
        need = self.stats["current_active_tracks"] + n
        if need > self.bank.capacity:
            self.bank.grow(min(65535, max(2 * self.bank.capacity, need)))
        if n:
            self._host[:n] = torch.as_tensor(np.asarray([list(d)[:4] for d in detections], dtype=np.float32))
            self._dets[0, :n].copy_(self._host[:n], non_blocking=True)
        self._cnt.fill_(n)
        rows, counts = self.bank.update(self._dets, self._cnt)
        k = int(counts[0].item())
        r = rows[0, :k].cpu().numpy()
        tr = self.bank.traj[0, :k].cpu().numpy()
        tl = self.bank.traj_len[0, :k].cpu().numpy()
        self._refresh_stats()
        return rows_to_dicts(r, tr, tl)

    def _refresh_stats(self):
        st = (C.c_longlong * 8)()
        _lib.check(self.bank.lib.b2_tracker_export(self.bank._h, 0, None, None, None, None, st))
        for k, v in zip(_STAT_KEYS, list(st)[:5]):
            self.stats[k] = int(v)
        self.frame_count, self.next_track_id = int(st[5]), int(st[6])
        if st[7]:      # cannot happen below 65535 live tracks: update() grows the bank first
            raise RuntimeError(f"track bank overflow: {int(st[7])} detections found no free slot (capacity={self.bank.capacity})")

    @property
    def trackers(self):
        x, P, meta, _ = self.bank.export(0)
        return [_TrackView(x[i], P[i], meta[i]) for i in range(len(x))]

    def get_statistics(self):
        """enhanced_multi_target_tracker.py:288-304."""
        x, P, meta, stats = self.bank.export(0)
        conf = self.bank.export_motion(0)
        d = dict(self.stats)
        d["frame_count"] = self.frame_count
        d["tracker_details"] = [{"track_id": f"T{int(m[0]):03d}", "age": int(m[1]), "hits": int(m[2]), "lost_frames": int(m[5]),
                                 "is_lost": bool(m[6]), "confidence": float(c)} for m, c in zip(meta, conf)]
        return d


class MotionCompensatedMultiTracker(EnhancedMultiTargetTracker):
    """Drop-in for camera_motion_compensation/motion_compensated_multi_tracker.py:18 on the CUDA track bank (mode 1):
    MotionResetKalmanTracker tracks (per-track jump / velocity / size reset detectors, cooldown, covariance rescale, blended
    association box), the subclass's own association (IoU > threshold, ties to the larger indices) and reporting of every
    live track.  ``update(detections, frame)``: the frame feeds :class:`GlobalMotionDetector` (global_motion_detector.py: sparse
    optical flow, OpenCV on the host exactly as the reference -- one decision per frame); when it asks for a reset and
    ``_should_global_reset`` agrees (motion_compensated_multi_tracker.py:119-146) every track of the stream is dropped and the
    frame's detections found new ones (:148-166): ``b2_tracker_reset`` + a normal update on the empty bank."""

    def __init__(self, max_lost_frames=150, min_hits=1, iou_threshold=0.1, capacity=512, max_dets=300):
        import torch

        self.max_lost_frames, self.min_hits, self.iou_threshold = max_lost_frames, min_hits, iou_threshold
        self.bank = TrackerBank(1, capacity, max_dets, max_lost_frames, min_hits, iou_threshold, mode=1)
        self.frame_count = 0
        self.next_track_id = 1
        self.stats = {"total_frames": 0, "global_motion_events": 0, "individual_resets": 0, "tracking_recoveries": 0, "global_resets": 0}
        self._active = 0
        from collections import deque

        self.motion_detector = GlobalMotionDetector()
        self.global_motion_compensation = True
        self.global_motion_history, self.detection_stability_history = deque(maxlen=20), deque(maxlen=10)
        self.frame_motion_info = None
        self._base = [0, 0]            # individual resets / recoveries counted by banks that a global reset has cleared since
        self._dets = torch.zeros((1, max_dets, 4), dtype=torch.float32, device=self.bank.device)
        self._host = torch.zeros((max_dets, 4), dtype=torch.float32).pin_memory()
        self._cnt = torch.zeros((1,), dtype=torch.int32, device=self.bank.device)

    def update(self, detections, frame=None):
        import torch

        self.frame_count += 1
        global_motion = False
        if frame is not None and self.global_motion_compensation:
            is_motion, mag, vec, should_reset = self.motion_detector.detect_motion(frame)
            self.frame_motion_info = {"is_motion": bool(is_motion), "magnitude": float(mag), "vector": np.asarray(vec).tolist(), "should_reset": bool(should_reset)}
            self.global_motion_history.append(float(mag))
            if should_reset:
                global_motion = True
                self.stats["global_motion_events"] += 1
        self.detection_stability_history.append(len(detections))
        if global_motion and self._should_global_reset():
            self.stats["global_resets"] += 1
            self._base = [self.stats["individual_resets"], self.stats["tracking_recoveries"]]
            self.bank.reset()
            self._active = 0
        n = len(detections)
        if n > self.bank.max_dets:
            raise ValueError(f"{n} detections exceed max_dets={self.bank.max_dets}")
        if self._active + n > self.bank.capacity:
            self.bank.grow(min(65535, max(2 * self.bank.capacity, self._active + n)))
        if n:
            self._host[:n] = torch.as_tensor(np.asarray([list(d)[:4] for d in detections], dtype=np.float32))
            self._dets[0, :n].copy_(self._host[:n], non_blocking=True)
        self._cnt.fill_(n)
        rows, counts = self.bank.update(self._dets, self._cnt)
        k = int(counts[0].item())
        r = rows[0, :k].cpu().numpy()
        ex = self.bank.extra[0, :k].cpu().numpy()
        tr, tl = self.bank.traj[0, :k].cpu().numpy(), self.bank.traj_len[0, :k].cpu().numpy()
        st = (C.c_longlong * 8)()
        _lib.check(self.bank.lib.b2_tracker_export(self.bank._h, 0, None, None, None, None, st))
        self._active = int(st[2])
        self.next_track_id = int(st[6])
        self.stats.update(total_frames=self.frame_count, individual_resets=self._base[0] + int(st[3]), tracking_recoveries=self._base[1] + int(st[4]))
        if st[7]:
            raise RuntimeError(f"track bank overflow: {int(st[7])} detections found no free slot")
        out = rows_to_dicts(r, tr, tl)
        order = np.argsort(r.view(np.int32)[:, 0], kind="stable")
        for d, j in zip(out, order):
            d["reset_count"] = int(ex[j].view(np.int32)[0])
            d["frames_since_reset"] = int(ex[j].view(np.int32)[1])
            d["motion_consistency"] = float(ex[j][2])
        return out

    def _should_global_reset(self):
        """motion_compensated_multi_tracker.py:119-146."""
        info = self.frame_motion_info
        if not info or not info["should_reset"]:
            return False
        if len(self.detection_stability_history) >= 5:
            recent = list(self.detection_stability_history)[-5:]
            if np.std(recent) / (np.mean(recent) + 1) > 0.5:
                return True
        if len(self.global_motion_history) >= 3 and np.mean(list(self.global_motion_history)[-3:]) > 30.0:
            return True
        return info["magnitude"] > 60.0

    def get_statistics(self):
        d = dict(self.stats)
        d["frame_count"] = self.frame_count
        d["active_trackers"] = self._active
        d["motion_detector"] = dict(self.motion_detector.stats)
        return d


MOTION_STAT_KEYS = ("total_detections", "motion_events", "reset_triggers", "avg_motion_magnitude", "global_motion_events", "global_resets")


class GlobalMotionBank:
    """:class:`GlobalMotionDetector` and the global-reset decision of :class:`MotionCompensatedMultiTracker` for S streams on the GPU
    (csrc/motion.cu): per frame ``flow(frames)`` (gray pyramid, corners of the previous frame, pyramidal LK into this one; frames
    only) then ``decide(det_counts)`` (the detector's vector and thresholds, ``_should_global_reset``).  ``decide`` returns device
    tensors: flags int32 [S] (1 where the stream's tracks are to be dropped: ``TrackerBank.reset_streams``) and info float32 [S][8]
    {magnitude, vx, vy, is_motion, should_reset, global_reset, corners, tracked corners}.  frame_shapes: one (h, w) or S of them;
    frames are CUDA uint8 [S][h][w][3] or, for mixed shapes, packed by ``ops.pack_frames``."""

    def __init__(self, n_streams, frame_shapes, device=None):
        import torch

        from . import ops

        self.device = device or _lib.require_cuda()
        self.lib = _lib.load()
        self.S = int(n_streams)
        shapes = [tuple(hw) for hw in frame_shapes] if hasattr(frame_shapes[0], "__len__") else [tuple(frame_shapes)] * self.S
        if len(shapes) != self.S:
            raise ValueError(f"frame_shapes lists {len(shapes)} shapes for {self.S} streams")
        self.frame_shapes = [(int(h), int(w)) for h, w in shapes]
        sh = np.ascontiguousarray(np.asarray(self.frame_shapes, np.int32))
        self._h = C.c_void_p()
        _lib.check(self.lib.b2_motion_create(self.S, sh.ctypes.data_as(C.c_void_p), C.byref(self._h)))
        self.uniform = len(set(self.frame_shapes)) == 1
        offs = (np.arange(self.S, dtype=np.int64) * (self.frame_shapes[0][0] * self.frame_shapes[0][1] * 3) if self.uniform
                else ops.pack_layout(self.frame_shapes)[0])
        self.offsets = torch.from_numpy(offs).to(self.device)
        self.flags = torch.zeros((self.S,), dtype=torch.int32, device=self.device)
        self.info = torch.zeros((self.S, 8), dtype=torch.float32, device=self.device)
        self.stats_dev = torch.zeros((self.S, 8), dtype=torch.float64, device=self.device)

    def close(self):
        if getattr(self, "_h", None):
            self.lib.b2_motion_destroy(self._h)
            self._h = None

    __del__ = close

    def reset(self, stream=None):
        """Forget every stream's previous frame and decision history."""
        _lib.check(self.lib.b2_motion_reset(self._h, _lib.stream_ptr(stream)))

    def flow(self, frames, offsets=None, stream=None):
        """frames: CUDA uint8, [S][h][w][3] or the packed layout (``offsets``: CUDA int64 [S] byte offsets, default: ``ops.pack_layout``)."""
        assert frames.is_cuda and frames.is_contiguous() and frames.dtype.itemsize == 1
        offsets = self.offsets if offsets is None else offsets
        _lib.check(self.lib.b2_motion_flow(self._h, _lib.ptr(frames), _lib.ptr(offsets), _lib.stream_ptr(stream)))

    def decide(self, det_counts=None, tracker_stats=None, stream=None):
        """det_counts: CUDA int32 [S] detections of this frame (None: 0); tracker_stats: ``TrackerBank.stats_async()`` before the
        reset (feeds the individual-resets / recoveries base), or None.  Returns (flags, info) device tensors."""
        _lib.check(self.lib.b2_motion_decide(self._h, _lib.ptr(det_counts), _lib.ptr(tracker_stats), _lib.ptr(self.flags), _lib.ptr(self.info),
                                             _lib.stream_ptr(stream)))
        return self.flags, self.info

    def stats_async(self, stream=None):
        """[S][8] float64 device snapshot {total_detections, motion_events, reset_triggers, avg_motion_magnitude, global_motion_events,
        global_resets, individual-resets base, recoveries base}, stream-ordered."""
        _lib.check(self.lib.b2_motion_stats(self._h, _lib.ptr(self.stats_dev), _lib.stream_ptr(stream)))
        return self.stats_dev

    def stats(self):
        """Per stream: the detector's ``stats`` dict plus the tracker's global_motion_events / global_resets (synchronises)."""
        st = self.stats_async().cpu().numpy()
        return [{k: (float(v) if k == "avg_motion_magnitude" else int(v)) for k, v in zip(MOTION_STAT_KEYS, row)} for row in st]


class GlobalMotionDetector:
    """camera_motion_compensation/global_motion_detector.py for its default method 'optical_flow' (:113-184): corners of the previous
    frame (goodFeaturesToTrack) followed into the current one (calcOpticalFlowPyrLK); the global vector is the mean flow of the
    points within the 75th percentile of the distance to the median flow; ``is_motion`` above 30 px, ``should_reset`` above 50 px, or
    above 45 px when the last three vectors point the same way (consistency > 0.7, :262-280).  Host-side OpenCV as in the reference:
    one small decision per frame in front of the GPU tracker, not a GPU path."""

    def __init__(self, method="optical_flow"):
        from collections import deque

        if method != "optical_flow":
            raise NotImplementedError(f"motion detection method {method!r}: only 'optical_flow' (the reference's default) is provided")
        self.method = method
        self.prev_gray = None
        self.motion_history, self.motion_vectors = deque(maxlen=10), deque(maxlen=5)
        self.global_motion_threshold, self.reset_motion_threshold, self.consistency_threshold = 30.0, 50.0, 0.7
        self.stats = {"total_detections": 0, "motion_events": 0, "reset_triggers": 0, "avg_motion_magnitude": 0.0}

    def detect_motion(self, frame):
        """-> (is_motion, magnitude, vector, should_reset)."""
        import cv2

        gray = cv2.cvtColor(frame, cv2.COLOR_BGR2GRAY)
        if self.prev_gray is None:
            self.prev_gray = gray
            return False, 0.0, np.array([0.0, 0.0]), False
        res = self._detect_by_optical_flow(gray)
        self.prev_gray = gray
        st = self.stats
        st["total_detections"] += 1
        st["motion_events"] += int(bool(res[0]))
        st["reset_triggers"] += int(bool(res[3]))
        st["avg_motion_magnitude"] = (st["avg_motion_magnitude"] * (st["total_detections"] - 1) + float(res[1])) / st["total_detections"]
        return res

    def _detect_by_optical_flow(self, gray):
        import cv2

        nothing = (False, 0.0, np.array([0.0, 0.0]), False)
        corners = cv2.goodFeaturesToTrack(self.prev_gray, maxCorners=200, qualityLevel=0.01, minDistance=15, blockSize=7)
        if corners is None or len(corners) < 20:
            return nothing
        nxt, status, _ = cv2.calcOpticalFlowPyrLK(self.prev_gray, gray, corners, None, winSize=(21, 21), maxLevel=3,
                                                  criteria=(cv2.TERM_CRITERIA_EPS | cv2.TERM_CRITERIA_COUNT, 30, 0.01))
        if status is None:
            return nothing
        ok = status.flatten() == 1
        if ok.sum() < 10:
            return nothing
        flow = nxt[ok].reshape(-1, 2) - corners[ok].reshape(-1, 2)
        if len(flow) <= 8:
            return nothing
        dist = np.linalg.norm(flow - np.median(flow, axis=0), axis=1)
        near = dist < np.percentile(dist, 75)
        if near.sum() <= 5:
            return nothing
        vec = np.mean(flow[near], axis=0)
        mag = np.linalg.norm(vec)
        self.motion_history.append(mag)
        self.motion_vectors.append(vec)
        is_motion, should_reset = mag > self.global_motion_threshold, mag > self.reset_motion_threshold
        if len(self.motion_vectors) >= 3 and is_motion and self._consistency(list(self.motion_vectors)[-3:]) > self.consistency_threshold:
            should_reset = should_reset or mag > self.global_motion_threshold * 1.5
        return is_motion, mag, vec, should_reset

    @staticmethod
    def _consistency(vectors):
        ang = [np.arctan2(v[1], v[0]) for v in vectors]
        d = [abs(a - b) for a, b in zip(ang[1:], ang[:-1])]
        d = [2 * np.pi - x if x > np.pi else x for x in d]
        return max(0.0, 1.0 - np.mean(d) / np.pi)


def direction_wrap(c):
    """The wrap rule of _calculate_direction_consistency (enhanced_aircraft_kalman_tracker.py:165-182)."""
    return c if abs(c) < math.pi else c - 2 * math.pi * (1 if c > 0 else -1 if c < 0 else 0)

"""The per-frame detect+track step for many concurrent video streams on one GPU, and its sharding over GPUs.

This is the loop body of the project driver (kalman/aircraft_detection_tracking.py:88-109:
``model(frame)`` -> ``boxes.xyxy/conf`` -> ``tracker.update(dets)``) for S streams at once:

    uint8 frames [S][h][w][3] --stem+forward--> head logits --decode--> candidates --NMS+scale--> dets [S][300][6]
        --Kalman bank (sweep: predict / IoU candidates / coasting tracks; resolve: match / update / create)-->
        track rows [S][max_tracks_out][20] + counts [S] + bank counters [S][8]

Everything between the frame upload and the result download stays on the GPU, on one CUDA stream, with no
host synchronisation.  Streams are independent (one tracker per stream in the reference), so multi-GPU
execution shards streams across ranks with no collective on the data path; NCCL only gathers results.
"""
from __future__ import annotations

from . import _lib, cfg, ops, weights
from .predictor import DetectPipeline, letterbox_table
from .tracker import GlobalMotionBank, TrackerBank


def bind_host_to_gpu(gpu_index):
    """Pin this process to the CPU cores NVML reports as local to the GPU, so that the pinned frame / result buffers it
    allocates afterwards are first-touched on that GPU's NUMA node (eight ranks uploading 21 GB/s each otherwise cross the
    socket interconnect).  Returns the core list, or None when NVML / sched_setaffinity is unavailable."""
    import os

    try:
        import pynvml

        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(int(gpu_index))
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = [i * 64 + b for i, m in enumerate(words) for b in range(64) if (int(m) >> b) & 1]
        allowed = sorted(set(cpus) & set(os.sched_getaffinity(0)))
        if allowed:
            os.sched_setaffinity(0, allowed)
            return allowed
    except Exception:
        pass
    return None


def shard_streams(n_streams, rank, world_size):
    """Contiguous block of stream ids owned by ``rank`` (SURVEY.md 8e)."""
    base, rem = divmod(n_streams, world_size)
    lo = rank * base + min(rank, rem)
    return list(range(lo, lo + base + (1 if rank < rem else 0)))


class DetectTrackPipeline:
    def __init__(self, model="yolov8s-p2", n_streams=1, frame_hw=(512, 640), imgsz=640, conf=0.15, iou=0.6, max_det=300,
                 max_lost_frames=150, min_hits=1, iou_threshold=0.1, capacity=512, state_dict=None, seed=0, nc=None,
                 nms_mode="exact", overlap_post=False, max_tracks_out=None, tracker="enhanced"):
        """overlap_post: run NMS + tracker of step t on a second CUDA stream while the forward of step t+1 runs on the
        caller's stream (the small latency-bound launches fill the tails of the conv kernels).  The returned device
        tensors are then valid only after ``join()``.
        capacity: track slots per stream.  The reference's track list is unbounded; ``results()`` raises if a detection was
        ever dropped for lack of a slot and grows the bank (x2) once a stream uses more than half of it.
        max_tracks_out: rows per stream of the result block (default: capacity).  The download moves exactly this block,
        so a caller that expects tens of tracks per stream keeps it small; ``results()`` raises if a stream reported more.
        frame_hw: the (h, w) of every stream, or a list of S shapes, one per stream (fixed for the pipeline's life).  Streams that
        all share one shape needing no resize take the frames as [S][h][w][3] and letterbox inside the stem kernel.  Any other
        set of shapes (mixed, or one shape that needs a resize) is the general path: frames are packed back to back
        (``ops.pack_frames``), letterboxed on the GPU into one canvas -- ``auto`` padding for one common shape, the full imgsz
        canvas for mixed shapes, as YOLO.predict does -- and NMS scales each stream's boxes to its own frame.
        tracker: "enhanced" (EnhancedMultiTargetTracker per stream) or "motion_compensated" (MotionCompensatedMultiTracker per
        stream, ``update(dets, frame)``): a mode-1 bank, and the camera-motion detector on the GPU (:class:`GlobalMotionBank`) --
        its flow on the uploaded frames, its decision after NMS, and a reset of the streams it flags before the tracker update.
        ``results()`` then also fills ``host_extra`` [S][max_tracks_out][4] (reset_count, frames_since_reset as int32 bits,
        motion_consistency) and ``host_motion`` [S][8] (``GlobalMotionBank.decide``'s info)."""
        import torch

        if tracker not in ("enhanced", "motion_compensated"):
            raise ValueError(f"tracker={tracker!r}: 'enhanced' or 'motion_compensated'")

        self.device = _lib.require_cuda()
        self.spec = cfg.resolve(model, nc=nc)
        sd = weights.to_numpy_state_dict(state_dict) if state_dict is not None else weights.synthetic_state_dict(self.spec, seed)
        self.S = int(n_streams)
        shapes = [tuple(hw) for hw in frame_hw] if hasattr(frame_hw[0], "__len__") else [tuple(frame_hw)] * self.S
        if len(shapes) != self.S:
            raise ValueError(f"frame_hw lists {len(shapes)} shapes for {self.S} streams")
        self.frame_shapes = [(int(h), int(w)) for h, w in shapes]
        isz = [imgsz, imgsz] if isinstance(imgsz, int) else list(imgsz)
        (self.H, self.W), geom, scale = letterbox_table(self.frame_shapes, isz)
        # identity letterbox (every stream one shape, no resize): the stem kernel pads the frames itself
        self.ragged = len(set(self.frame_shapes)) != 1 or tuple(geom[0, 2:4]) != self.frame_shapes[0]
        self.h0, self.w0 = self.frame_shapes[0]
        self.top, self.left = int(geom[0, 4]), int(geom[0, 5])
        self.conf, self.iou, self.nms_mode = float(conf), float(iou), nms_mode
        self.detect = DetectPipeline(self.spec, sd, self.S, self.H, self.W, max_det)
        self.max_det = int(max_det)
        self.tracker = tracker
        self.bank = TrackerBank(self.S, capacity, max_det, max_lost_frames, min_hits, iou_threshold,
                                max_out=min(int(max_tracks_out), int(capacity)) if max_tracks_out else None,
                                mode=1 if tracker == "motion_compensated" else 0)
        self.motion = GlobalMotionBank(self.S, self.frame_shapes, self.device) if tracker == "motion_compensated" else None
        if self.motion is not None:
            self._tstats = torch.zeros((self.S, 8), dtype=torch.int64, device=self.device)
        self._fixed_out = bool(max_tracks_out)
        self.flops_per_frame = self.detect.engine.flops_per_image
        # double-buffered staging for the host-facing path
        self._copy_stream = torch.cuda.Stream()
        if self.ragged:
            offs, self.packed_bytes = ops.pack_layout(self.frame_shapes)
            self._offsets, self._geom, self._scale = (torch.from_numpy(a).to(self.device) for a in (offs, geom, scale))
            self._dev_frames = [torch.empty((self.packed_bytes,), dtype=torch.uint8, device=self.device) for _ in range(2)]
        else:
            self._dev_frames = [torch.empty((self.S, self.h0, self.w0, 3), dtype=torch.uint8, device=self.device) for _ in range(2)]
        self._ready = [torch.cuda.Event() for _ in range(2)]
        self._consumed = [torch.cuda.Event() for _ in range(2)]
        self._slot = 0
        self._d2h_stream = torch.cuda.Stream()
        self.overlap_post = bool(overlap_post)
        self._post_stream = torch.cuda.Stream()
        self.forward_events = None                     # a list: step_device appends (start, end) events of each forward
        self._cand_done = torch.cuda.Event()
        self._post_done = torch.cuda.Event()
        self._post_done.record()
        self._step_done = torch.cuda.Event()
        self._rows_downloaded = torch.cuda.Event()
        self._rows_downloaded.record()
        self.h2d_bytes_per_step = self._dev_frames[0].numel()
        self._regrow_host = False
        self._alloc_host()

    def _alloc_host(self):
        import torch

        self.host_rows = torch.empty((self.S, self.bank.max_out, _lib.TRACK_COLS), dtype=torch.float32).pin_memory()
        self.host_counts = torch.zeros((self.S,), dtype=torch.int32).pin_memory()
        self.host_stats = torch.zeros((self.S, 8), dtype=torch.int64).pin_memory()
        self.d2h_bytes_per_step = self.host_rows.numel() * 4 + self.host_counts.numel() * 4 + self.host_stats.numel() * 8
        self.host_extra = self.host_motion = None
        if self.motion is not None:
            self.host_extra = torch.empty((self.S, self.bank.max_out, 4), dtype=torch.float32).pin_memory()
            self.host_motion = torch.empty((self.S, 8), dtype=torch.float32).pin_memory()
            self.d2h_bytes_per_step += self.host_extra.numel() * 4 + self.host_motion.numel() * 4

    def _packed(self, frames):
        """The general path's input: ``packed_bytes`` uint8 in the ``ops.pack_frames`` layout (any shape with that many bytes,
        e.g. [S][h][w][3] when every frame is a multiple of 16 bytes)."""
        if frames.dtype.itemsize != 1 or frames.numel() != self.packed_bytes or not frames.is_contiguous():
            raise ValueError(f"expected {self.packed_bytes} contiguous packed frame bytes (ops.pack_frames of shapes {self.frame_shapes}), "
                             f"got {frames.dtype} {tuple(frames.shape)}")
        return frames.view(-1)

    def _motion_flow(self, frames_u8, stream):
        self.motion.flow(frames_u8, self._offsets if self.ragged else None, stream)

    def _motion_reset(self, counts, stream):
        """The decision after NMS and the reset of the flagged streams (MotionCompensatedMultiTracker.update :279-293)."""
        self.bank.stats_async(stream, out=self._tstats)
        flags, _ = self.motion.decide(counts, self._tstats, stream)
        self.bank.reset_streams(flags, stream)

    def step_device(self, frames_u8, with_trajectory=False, stream=None):
        """frames_u8: CUDA uint8 [S][h][w][3] BGR, or on the general path (mixed / resized shapes) the packed frames of
        ``ops.pack_frames``.  Returns (track rows [S][capacity][20], counts [S]) on the GPU."""
        import torch

        cur = stream or torch.cuda.current_stream()
        if not self.overlap_post:
            if self.motion is not None:
                self._motion_flow(frames_u8, stream)
            if self.ragged:
                dets, counts = self.detect.run_ragged(self._packed(frames_u8), self._offsets, self._geom, self._scale, self.conf, self.iou,
                                                      None, False, self.nms_mode, stream)
            else:
                dets, counts = self.detect(frames_u8, self.conf, self.iou, self.top, self.left, (self.h0, self.w0), None, False,
                                           self.nms_mode, stream)
            # the bank's row block is about to be rewritten: a download of the previous step's rows (step_host) must be over
            cur.wait_event(self._rows_downloaded)
            if self.motion is not None:
                self._motion_reset(counts, stream)
            return self.bank.update(dets, counts, with_trajectory=with_trajectory, stream=stream)
        d, ps = self.detect, self._post_stream
        frames_in = frames_u8
        if self.ragged:
            frames_u8 = d.letterbox(self._packed(frames_u8), self._offsets, self._geom, stream)
        if self.forward_events is not None:           # bench.py: CUDA events around the forward graph, on the stream it runs on
            ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
            ev[0].record(cur)
        top, left = (0, 0) if self.ragged else (self.top, self.left)
        d.engine.forward_u8(frames_u8, top, left, stream=stream)
        if self.forward_events is not None:
            ev[1].record(cur)
            self.forward_events.append(ev)
        cur.wait_event(self._post_done)               # NMS of the previous step has read the candidate lists
        if self.motion is not None:                   # ... and its motion decision has read the flow of the previous frame
            self._motion_flow(frames_in, stream)
        d.candidates(self.conf, None, stream)
        self._cand_done.record(cur)
        ps.wait_event(self._cand_done)
        ps.wait_event(self._rows_downloaded)
        if self.ragged:
            dets, counts = d.nms(self.iou, None, False, self.nms_mode, ps, self._scale)
        else:
            dets, counts = d.nms(self.iou, (self.h0, self.w0), False, self.nms_mode, ps)
        if self.motion is not None:
            self._motion_reset(counts, ps)
        out = self.bank.update(dets, counts, with_trajectory=with_trajectory, stream=ps)
        self._post_done.record(ps)
        return out

    def step_host(self, frames_pinned):
        """frames_pinned: pinned host uint8 [S][h][w][3] (general path: the ``ops.pack_frames`` buffer).  Upload on the copy
        stream (overlaps the previous step's compute), run the step, download rows + counts into pinned host buffers on a third stream (overlaps the next
        step).  Returns the host buffers (valid after ``join()`` + ``torch.cuda.current_stream().synchronize()``)."""
        import torch

        cur = torch.cuda.current_stream()
        if self._regrow_host:
            self._alloc_host()
            self._regrow_host = False
        k = self._slot
        self._slot ^= 1
        with torch.cuda.stream(self._copy_stream):
            self._copy_stream.wait_event(self._consumed[k])          # the step that last read this buffer is done
            self._dev_frames[k].copy_(self._packed(frames_pinned) if self.ragged else frames_pinned, non_blocking=True)
            self._ready[k].record(self._copy_stream)
        cur.wait_event(self._ready[k])
        rows, counts = self.step_device(self._dev_frames[k])
        self._consumed[k].record(cur)
        # download on its own stream: it overlaps the next step's forward (which only waits for it before the tracker
        # rewrites the rows, see step_device)
        done = self._post_done if self.overlap_post else self._step_done
        if not self.overlap_post:
            self._step_done.record(cur)
        with torch.cuda.stream(self._d2h_stream):
            self._d2h_stream.wait_event(done)
            self.host_rows.copy_(rows, non_blocking=True)
            self.host_counts.copy_(counts, non_blocking=True)
            self.host_stats.copy_(self.bank.stats_async(self._d2h_stream), non_blocking=True)
            if self.motion is not None:
                self.host_extra.copy_(self.bank.extra, non_blocking=True)
                self.host_motion.copy_(self.motion.info, non_blocking=True)
            self._rows_downloaded.record(self._d2h_stream)
        return self.host_rows, self.host_counts

    def join(self):
        """Make the current stream wait for the last download of step_host and, with overlap_post, for the last step's NMS +
        tracker (host buffers / returned device tensors are valid after it synchronises)."""
        import torch

        torch.cuda.current_stream().wait_event(self._rows_downloaded)
        torch.cuda.current_stream().wait_event(self._post_done)


    def run(self, loader):
        """The driver loop of kalman/aircraft_detection_tracking.py:88-109 for all sources at once: ``loader`` yields
        ``(sources, frames, info)`` with one HWC BGR uint8 frame per stream (``loaders.LoadStreams``, or any iterable of such
        batches).  Yields ``(sources, rows, counts)`` per frame time: numpy copies of the step's track rows [S][max_tracks_out][20]
        and per-stream counts, after the reference-equivalence checks of :meth:`results`."""
        import numpy as np
        import torch

        stage = torch.empty(tuple(self._dev_frames[0].shape), dtype=torch.uint8).pin_memory()
        for sources, frames, _ in loader:
            check_frames(frames, self.frame_shapes)
            if self.ragged:
                ops.pack_frames(frames, out=stage)
            else:
                for k, f in enumerate(frames):
                    stage[k] = torch.from_numpy(np.ascontiguousarray(f))
            self.step_host(stage)
            rows, counts = self.results()                 # synchronises: `stage` may be refilled afterwards
            yield sources, rows.numpy().copy(), counts.numpy().copy()

    def results(self):
        """Synchronise the last ``step_host`` and return its host block (rows [S][max_tracks_out][20], counts [S]) after
        checking that it is the reference's result: no detection was dropped for lack of a track slot (the reference's list
        is unbounded, enhanced_multi_target_tracker.py:92-101) and no stream reported more rows than the block holds.
        Grows the bank ahead of need (a stream above half its capacity doubles it)."""
        self._rows_downloaded.synchronize()
        self._post_done.synchronize()
        check_bank(self.host_stats, self.host_counts, self.bank.capacity, self.bank.max_out)
        out = self.host_rows, self.host_counts
        if int(self.host_stats[:, 2].max()) + 2 * self.max_det > self.bank.capacity and self.bank.capacity < 65535:
            self.bank.grow(min(65535, 2 * self.bank.capacity))
            if not self._fixed_out:
                self._regrow_host = True        # the next step_host reallocates: this step's host block stays valid until then
        return out


def check_frames(frames, shapes):
    """Raises ValueError unless ``frames`` holds one HWC frame per stream, frame k of shape ``shapes[k]`` + (3,)."""
    if len(frames) != len(shapes):
        raise ValueError(f"the loader delivered {len(frames)} frames, the pipeline was built for {len(shapes)} streams")
    for k, (f, hw) in enumerate(zip(frames, shapes)):
        if tuple(f.shape) != (*hw, 3):
            raise ValueError(f"stream {k}: frame shape {tuple(f.shape)}, the pipeline was built for {(*hw, 3)}")


def check_bank(stats, counts, capacity, max_out):
    """stats: [S][8] int64 bank counters, counts: [S] rows reported.  Raises if the bank lost a detection or rows."""
    dropped = int(stats[:, 5].sum())
    if dropped:
        s = int(stats[:, 5].argmax())
        raise RuntimeError(f"track bank overflow: {dropped} detections found no free slot (first in stream {s}, capacity={capacity}); "
                           "the reference never drops a detection -- raise `capacity`")
    over = int(counts.max()) if counts.numel() else 0
    if over > max_out:
        raise RuntimeError(f"result block too small: a stream reported {over} tracks, max_tracks_out={max_out}")


def gather_results(rows, counts, group=None):
    """All-gather fixed-stride per-stream result blocks across ranks (the only collective of the pipeline;
    off the data path).  rows: [S_local][capacity][20], counts: [S_local]; returns lists indexed by rank."""
    import torch
    import torch.distributed as dist

    world = dist.get_world_size(group)
    rows_all = [torch.empty_like(rows) for _ in range(world)]
    counts_all = [torch.empty_like(counts) for _ in range(world)]
    dist.all_gather(rows_all, rows.contiguous(), group=group)
    dist.all_gather(counts_all, counts.contiguous(), group=group)
    return rows_all, counts_all

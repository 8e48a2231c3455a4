"""CUDA-event timing of the ragged-batch LetterBox kernel and of the detect+track step on streams that need it.

  kernel     b2_letterbox_u8 alone on two 256-frame batches: 256 x 1080p (auto canvas 384 x 640) and a mixed 256 (128 x 1080p,
             64 x 720p, 64 x 512x640 -> 640 x 640 canvas).  Noise frames, L2 overwritten before every timed launch.  Bytes are
             the source rows the bilinear taps (or the copy) read, whole rows, plus the canvas written; the share of peak is
             against the 6.5 TB/s copy rate DESIGN.md uses.
  step       DetectTrackPipeline.step_device (yolov8s-p2, 256 streams, NMS + tracker overlapped as in bench.py) on frames already
             in HBM: the unchanged 512 x 640 identity path, 256 x 1080p and the mixed 256, in one process.
  step_host  the host-facing step (pinned packed frames in, track rows out) for 256 x 1080p: 1.6 GB uploaded per step.

Frames of the step rows are synthetic IR videos (8 distinct per shape, 6-frame pool played forth and back, as bench.py).

usage: python tools/letterbox_bench.py [--out profiles/r04_letterbox_bench.jsonl] [--steps 20] [--warmup 3]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch

import b200dt  # noqa: F401
from b200dt import _lib, ops, synth
from b200dt.pipeline import DetectTrackPipeline
from b200dt.predictor import letterbox_table

PEAK_COPY = 6.5e12
P1080, P720, P512 = (1080, 1920), (720, 1280), (512, 640)
UNIFORM = [P1080] * 256
MIXED = [P1080] * 128 + [P720] * 64 + [P512] * 64
POOL = 6


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (q.stdout.strip().splitlines() or ["?, ?"])[0].split(", ")
    return {"gpu": name, "power_limit": power}


def event_ms(fn, iters, before=None):
    """Median device time of ``fn`` over ``iters`` launches (``before`` runs outside the timed window)."""
    ts = []
    for _ in range(iters):
        if before:
            before()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return sorted(ts)[len(ts) // 2]


def touched_bytes(geom, H, W):
    """Source rows the kernel reads (every row of an unresized frame; the rows of the vertical taps otherwise) + canvas bytes."""
    n = 0
    for sh, sw, rh, rw, _, _ in geom.tolist():
        if (rh, rw) == (sh, sw):
            rows = sh
        else:
            f = ((np.arange(rh) + 0.5) * (1.0 / (rh / sh)) - 0.5).astype(np.float32)
            s = np.floor(f).astype(np.int64)
            rows = len(np.unique(np.clip(np.concatenate([s, s + 1]), 0, sh - 1)))
        n += rows * sw * 3
    return n + len(geom) * H * W * 3


def bench_kernel(name, shapes):
    (H, W), geom, _ = letterbox_table(shapes, [640, 640])
    offs, nbytes = ops.pack_layout(shapes)
    packed = torch.randint(0, 256, (nbytes,), dtype=torch.uint8, device="cuda")
    o, g = torch.from_numpy(offs).cuda(), torch.from_numpy(geom).cuda()
    canvas = torch.empty((len(shapes), H, W, 3), dtype=torch.uint8, device="cuda")
    run = lambda: ops.letterbox_u8(packed, o, g, H, W, out=canvas)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    for _ in range(5):
        run()
    ms = event_ms(run, 30, before=lambda: flush.fill_(1))
    nb = touched_bytes(geom, H, W)
    return {"kernel": "b2_letterbox_u8", "batch": name, "images": len(shapes), "canvas": [H, W], "us": ms * 1e3, "bytes": nb,
            "GB_per_s": nb / (ms * 1e-3) / 1e9, "share_of_6.5TBps": nb / (ms * 1e-3) / PEAK_COPY, "l2": "overwritten before each launch"}


def frame_pool(shapes, seed0=2000):
    """POOL steps of packed frames for ``shapes``: 8 distinct IR videos per distinct shape, tiled over the streams."""
    vids = {hw: [synth.IRStream(seed=seed0 + 17 * k + i, h=hw[0], w=hw[1]) for i in range(8)] for k, hw in enumerate(sorted(set(shapes)))}
    steps = []
    for _ in range(POOL):
        fr = {hw: [v.frame() for v in vs] for hw, vs in vids.items()}
        seen = {}
        frames = []
        for hw in shapes:
            i = seen.get(hw, 0)
            seen[hw] = i + 1
            frames.append(fr[hw][i % 8])
        steps.append(frames)
    return steps


def pool_index(i):
    period = 2 * POOL - 2
    k = i % period
    return k if k < POOL else period - k


def timed_steps(pipe, step, steps, warmup):
    for i in range(warmup):
        step(i)
    pipe.join()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        step(warmup + i)
    pipe.join()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def bench_steps(steps, warmup):
    lib = _lib.load()
    for name, shapes in (("512x640 identity", [P512] * 256), ("256 x 1080p", UNIFORM), ("mixed 256", MIXED)):
        pipe = DetectTrackPipeline("yolov8s-p2", 256, shapes if len(set(shapes)) > 1 else shapes[0], 640, 0.15, 0.6, 300, capacity=2048,
                                   overlap_post=True, max_lost_frames=150, min_hits=1, iou_threshold=0.1)
        pool = frame_pool(shapes)
        if pipe.ragged:
            dev = [torch.from_numpy(ops.pack_frames(f)[0]).cuda() for f in pool]
        else:
            dev = [torch.from_numpy(np.stack(f)).cuda() for f in pool]
        l0 = lib.b2_launch_count()
        ms = timed_steps(pipe, lambda i: pipe.step_device(dev[pool_index(i)]), steps, warmup)
        launches = (lib.b2_launch_count() - l0) / (steps + warmup)
        rec = {"step": "step_device", "workload": name, "model": "yolov8s-p2", "streams": 256, "canvas": [pipe.H, pipe.W],
               "ms_per_step": ms, "frames_per_s": 256 / ms * 1e3, "launches_per_step": launches, "steps": steps}
        if name == "256 x 1080p":
            pinned = [torch.from_numpy(ops.pack_frames(f)[0]).pin_memory() for f in pool[:2]]
            ms_h = timed_steps(pipe, lambda i: pipe.step_host(pinned[i % 2]), steps, warmup)
            pipe.results()
            yield rec
            rec = {"step": "step_host", "workload": name, "model": "yolov8s-p2", "streams": 256, "canvas": [pipe.H, pipe.W],
                   "ms_per_step": ms_h, "frames_per_s": 256 / ms_h * 1e3, "h2d_bytes_per_step": pipe.h2d_bytes_per_step,
                   "h2d_GB_per_s_at_this_rate": pipe.h2d_bytes_per_step / (ms_h * 1e-3) / 1e9, "steps": steps}
        yield rec
        del pipe, dev
        torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_letterbox_bench.jsonl"))
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    a = ap.parse_args()
    _lib.require_cuda()
    info = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        def emit(r):
            line = json.dumps(dict(info, **r))
            fh.write(line + "\n")
            fh.flush()
            print(line, flush=True)

        emit(bench_kernel("256 x 1080p", UNIFORM))
        emit(bench_kernel("mixed 256", MIXED))
        for r in bench_steps(a.steps, a.warmup):
            emit(r)


if __name__ == "__main__":
    main()

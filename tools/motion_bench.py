"""CUDA-event timing of the camera-motion kernels (csrc/motion.cu) and of the detect+track step with tracker="motion_compensated".

  kernels    each C entry point alone on 256 streams at 512x640 and at 1080p: the gray pyramid (gray + 3 pyrDown launches), the
             corner response, the corner selection (max + candidates + per-stream select), LK on the selected corners, and the
             whole per-frame bank work (b2_motion_flow + b2_motion_decide).  Textured frames (smooth noise) seen through windows that
             move 1-3 px per frame, one stream in eight by 40 px.  L2 overwritten before every timed launch; median of 20.
             Bytes are computed from the shapes: what each kernel must read and write once.
  step       DetectTrackPipeline.step_device (yolov8s-p2, 256 streams x 512x640, NMS + tracker overlapped as in bench.py) with the
             default tracker and with tracker="motion_compensated", alternated in one process on the same frames in HBM.
  host       the host GlobalMotionDetector (cv2) per 512x640 frame on this machine's CPU, for context.

usage: python tools/motion_bench.py [--out profiles/r05_motion_bench.jsonl] [--steps 20] [--warmup 3] [--rounds 3]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import torch

import b200dt  # noqa: F401
from b200dt import _lib, ops
from b200dt.pipeline import DetectTrackPipeline
from b200dt.tracker import GlobalMotionBank, GlobalMotionDetector

S = 256
SHAPES = {"512x640": (512, 640), "1080p": (1080, 1920)}
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


def textured_frames(hw, n_steps, seed=0):
    """n_steps batches of S uint8 BGR frames [S][h][w][3] (CUDA): windows over a smooth-noise world, 1-3 px steps, a 40 px jolt
    on every eighth stream."""
    h, w = hw
    g = torch.Generator(device="cuda").manual_seed(seed)
    pad = 96
    world = torch.rand((1, 1, (h + 2 * pad) // 8 + 2, (w + 2 * pad) // 8 + 2), generator=g, device="cuda")
    world = torch.nn.functional.interpolate(world, scale_factor=8, mode="bicubic")[0, 0, :h + 2 * pad, :w + 2 * pad]
    world = (world.clamp(0, 1) * 200 + 20).to(torch.uint8)
    rng = np.random.default_rng(seed)
    off = np.full((S, 2), pad)
    out = []
    for t in range(n_steps):
        off = np.clip(off + rng.integers(-3, 4, (S, 2)) + (40 * (np.arange(S) % 8 == 0)[:, None] * (t % 2 * 2 - 1)), 0, 2 * pad)
        fr = torch.stack([world[oy:oy + h, ox:ox + w] for ox, oy in off.tolist()])
        out.append(fr[..., None].expand(S, h, w, 3).contiguous())
    return out


def bench_kernels(name, hw):
    lib = _lib.load()
    frames = textured_frames(hw, 2)
    shapes = [hw] * S
    p0, p1 = ops.GrayPyramid(shapes), ops.GrayPyramid(shapes)
    foff = torch.from_numpy(ops.frame_offsets(frames[0], shapes)).cuda()
    pyr = lambda pyr, fr: _lib.check(lib.b2_gray_pyramid_u8(_lib.ptr(fr), _lib.ptr(foff), S, p0.max_h, p0.max_w, _lib.ptr(pyr.buf),
                                                            _lib.ptr(pyr.off_dev), _lib.ptr(pyr.hw_dev), _lib.stream_ptr()))
    eig = torch.empty((p0.npix,), dtype=torch.float32, device="cuda")
    run_eig = lambda: _lib.check(lib.b2_corner_min_eig(_lib.ptr(p0.buf), _lib.ptr(p0.off_dev), _lib.ptr(p0.hw_dev), _lib.ptr(p0.pix_dev), S,
                                                       p0.max_h, p0.max_w, 7, 3, _lib.ptr(eig), _lib.stream_ptr()))
    wsb = lib.b2_good_features_workspace_bytes(S, p0.npix)
    ws = torch.empty((wsb,), dtype=torch.uint8, device="cuda")
    corners = torch.zeros((S, 200, 2), dtype=torch.float32, device="cuda")
    counts = torch.zeros((S,), dtype=torch.int32, device="cuda")
    run_sel = lambda: _lib.check(lib.b2_good_features(_lib.ptr(eig), _lib.ptr(p0.pix_dev), _lib.ptr(p0.hw_dev), S, p0.max_h, p0.max_w, p0.npix,
                                                      200, 0.01, 15.0, _lib.ptr(ws), wsb, _lib.ptr(corners), _lib.ptr(counts), _lib.stream_ptr()))
    nxt = torch.zeros_like(corners)
    status = torch.zeros((S, 200), dtype=torch.uint8, device="cuda")
    run_lk = lambda: _lib.check(lib.b2_lk_pyr(_lib.ptr(p0.buf), _lib.ptr(p1.buf), _lib.ptr(p0.off_dev), _lib.ptr(p0.hw_dev), S, _lib.ptr(corners),
                                              _lib.ptr(counts), 200, 21, 3, 30, 0.01, _lib.ptr(nxt), _lib.ptr(status), _lib.stream_ptr()))
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    before = lambda: flush.fill_(1)
    h, w = hw
    hwp = h * w
    lvl = p0.level_hw[0]
    lvl_px = int((lvl[:, 0] * lvl[:, 1]).sum())
    pyr(p0, frames[0]), pyr(p1, frames[1]), run_eig(), run_sel(), run_lk()
    torch.cuda.synchronize()
    recs = []
    ms = event_ms(lambda: pyr(p0, frames[0]), 20, before)
    nb = S * (3 * hwp + lvl_px + (lvl_px - int(lvl[3, 0] * lvl[3, 1])))     # frames read, 4 levels written, levels 0-2 read
    recs.append({"kernel": "gray + 3 pyrDown (b2_gray_pyramid_u8, 4 launches)", "bytes": nb, "us": ms * 1e3, "GB_per_s": nb / ms / 1e6})
    ms = event_ms(run_eig, 20, before)
    nb = S * 5 * hwp
    recs.append({"kernel": "eig_kernel (b2_corner_min_eig)", "bytes": nb, "us": ms * 1e3, "GB_per_s": nb / ms / 1e6})
    ms = event_ms(run_sel, 20, before)
    n_cand = int(ws[:S * 8].view(torch.int32)[S:].sum())
    nb = S * 8 * hwp + 16 * n_cand           # response read twice (max, candidates), keys written and read once
    recs.append({"kernel": "corner selection (b2_good_features: max + candidates + select)", "bytes": nb, "candidates_per_stream": n_cand / S,
                 "corners_per_stream": float(counts.float().mean()), "us": ms * 1e3, "GB_per_s": nb / ms / 1e6})
    ms = event_ms(run_lk, 20, before)
    npts = int(counts.sum())
    recs.append({"kernel": "lk_kernel (b2_lk_pyr)", "points": npts, "levels": 4, "tracked": int(status.sum()), "us": ms * 1e3,
                 "points_per_s": npts / ms * 1e3})
    bank = GlobalMotionBank(S, hw)
    dets = torch.full((S,), 20, dtype=torch.int32, device="cuda")
    k = [0]

    def step():
        bank.flow(frames[k[0] % 2])
        bank.decide(dets)
        k[0] += 1

    for _ in range(3):
        step()
    ms = event_ms(step, 20, before)
    recs.append({"kernel": "GlobalMotionBank.flow + decide (per frame, all kernels)", "us": ms * 1e3})
    for r in recs:
        r.update(shape=name, streams=S, l2="overwritten before each launch")
    del bank, p0, p1, frames, eig, ws
    torch.cuda.empty_cache()
    return recs


def bench_steps(steps, warmup, rounds):
    hw = SHAPES["512x640"]
    frames = textured_frames(hw, POOL, seed=1)
    pipes = {t: DetectTrackPipeline("yolov8s-p2", S, hw, 640, 0.15, 0.6, 300, capacity=2048, overlap_post=True, max_lost_frames=150,
                                    min_hits=1, iou_threshold=0.1, tracker=t) for t in ("enhanced", "motion_compensated")}
    lib = _lib.load()
    res = {t: [] for t in pipes}
    launches = {}
    for r in range(rounds):
        for t, pipe in pipes.items():
            for i in range(warmup):
                pipe.step_device(frames[i % POOL])
            pipe.join()
            torch.cuda.synchronize()
            l0 = lib.b2_launch_count()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(steps):
                pipe.step_device(frames[i % POOL])
            pipe.join()
            e1.record()
            torch.cuda.synchronize()
            launches[t] = (lib.b2_launch_count() - l0) / steps
            res[t].append(e0.elapsed_time(e1) / steps)
    for t in pipes:
        ms = sorted(res[t])[len(res[t]) // 2]
        yield {"step": "step_device", "tracker": t, "model": "yolov8s-p2", "streams": S, "frame": list(hw), "ms_per_step": ms,
               "ms_per_step_rounds": res[t], "frames_per_s": S / ms * 1e3, "launches_per_step": launches[t], "steps": steps,
               "alternated": f"{rounds} rounds, trackers alternated in one process, same frames in HBM"}


def bench_host(n=20):
    import cv2

    from golden_common import motion_frames_scene

    frames, _ = motion_frames_scene(n_frames=n + 1, seed=13, hw=(512, 640))
    det = GlobalMotionDetector()
    det.detect_motion(frames[0])
    t0 = time.perf_counter()
    for f in frames[1:]:
        det.detect_motion(f)
    ms = (time.perf_counter() - t0) / n * 1e3
    return {"host": "GlobalMotionDetector.detect_motion (cv2, host)", "frame": [512, 640], "ms_per_frame": ms, "cpu_count": os.cpu_count(),
            "cv2_threads": cv2.getNumThreads(), "ms_for_256_streams_serial": ms * S}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_motion_bench.jsonl"))
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
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

        for name, hw in SHAPES.items():
            for r in bench_kernels(name, hw):
                emit(r)
        for r in bench_steps(a.steps, a.warmup, a.rounds):
            emit(r)
        emit(bench_host())


if __name__ == "__main__":
    main()

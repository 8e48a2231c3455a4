"""CUDA-event timing of the BoT-SORT ReID kernels, and YOLO.track wall time with and without ReID.

  gather   b2_reid_gather at the C4 size: 256 images x 300 kept detections over yolov8s-p2's Detect inputs at 512 x 640
           (levels 128x160x64, 64x80x128, 32x40x256, 16x20x512, s = 64); L2 overwritten before every timed launch.  GB/s counts
           the 2 C_l bytes read and 4 s bytes written per detection.
  cost     b2_botsort_cost + b2_linear_assignment_f64 (D = 64) next to b2_iou_cost + b2_linear_assignment at the same sizes.
  track    YOLO('yolov8n-p2.yaml').track one 512 x 640 synthetic IR frame at a time (persist=True, BoT-SORT, GMC off), host clock
           around each call (its results are on the host, so the call ends synchronised).

usage: python tools/reid_bench.py [--out profiles/r03_reid_bench.jsonl]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch

import b200dt  # noqa: F401
from b200dt import _lib, synth


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


def bench_gather(lib, g):
    B, K, chans, hws = 256, 300, [64, 128, 256, 512], [(128, 160), (64, 80), (32, 40), (16, 20)]
    s = min(chans)
    bufs = [torch.randn((B, h, w, c), device="cuda").bfloat16() for (h, w), c in zip(hws, chans)]
    start = np.cumsum([0] + [h * w for h, w in hws])
    idx = torch.as_tensor(g.integers(0, start[-1], (B, K)).astype(np.int32)).cuda()
    cnt = torch.full((B,), K, dtype=torch.int32, device="cuda")
    out = torch.empty((B, K, s), device="cuda")
    n = len(bufs)
    ints = lambda v: (C.c_int * n)(*v)
    args = ((C.c_void_p * n)(*[b.data_ptr() for b in bufs]), ints([h for h, _ in hws]), ints([w for _, w in hws]), ints(chans),
            ints([0] * n), ints(chans), n)
    run = lambda: _lib.check(lib.b2_reid_gather(*args, _lib.ptr(idx), _lib.ptr(cnt), B, K, s, _lib.ptr(out), _lib.stream_ptr()))
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    for _ in range(5):
        run()
    ms = event_ms(run, 50, before=lambda: flush.fill_(1))
    level = np.searchsorted(start, idx.cpu().numpy(), side="right") - 1
    nbytes = int((2 * np.asarray(chans)[level]).sum()) + B * K * s * 4
    return {"kernel": "b2_reid_gather", "images": B, "dets_per_image": K, "s": s, "us": ms * 1e3, "bytes": nbytes,
            "GB_per_s": nbytes / (ms * 1e-3) / 1e9, "l2": "overwritten before each launch"}


def boxes(g, S, n, span):
    c = g.uniform(0, span, (S, n, 2))
    sz = g.uniform(6, 40, (S, n, 2))
    return np.concatenate([c - sz / 2, c + sz / 2], 2).astype(np.float32)


def bench_cost(lib, g):
    rows = []
    for S, n, m in [(256, 24, 24), (256, 64, 64), (64, 300, 300)]:
        D = 64
        a = boxes(g, S, n, 600)
        b = np.ascontiguousarray(a[:, :m] + g.normal(0, 2, (S, m, 4)).astype(np.float32))
        da, db = torch.as_tensor(a).cuda(), torch.as_tensor(b).cuda()
        sc = torch.rand((S, m), device="cuda")
        fa = torch.nn.functional.normalize(torch.randn((S, n, D), device="cuda"), dim=-1)
        fb = torch.nn.functional.normalize(fa[:, :m] + 0.2 * torch.randn((S, m, D), device="cuda"), dim=-1)
        c32 = torch.empty((S, n, m), device="cuda")
        c64 = torch.empty((S, n, m), dtype=torch.float64, device="cuda")
        x = torch.empty((S, n), dtype=torch.int32, device="cuda")
        y = torch.empty((S, m), dtype=torch.int32, device="cuda")
        iou = lambda: _lib.check(lib.b2_iou_cost(_lib.ptr(da), _lib.ptr(db), _lib.ptr(sc), None, None, S, n, m, _lib.ptr(c32), _lib.stream_ptr()))
        lap32 = lambda: _lib.check(lib.b2_linear_assignment(_lib.ptr(c32), None, None, S, n, m, 0.8, _lib.ptr(x), _lib.ptr(y), _lib.stream_ptr()))
        bot = lambda: _lib.check(lib.b2_botsort_cost(_lib.ptr(da), _lib.ptr(db), _lib.ptr(sc), None, None, _lib.ptr(fa), _lib.ptr(fb), D, S, n, m,
                                                     0.5, 1 - 0.8, _lib.ptr(c64), _lib.stream_ptr()))
        lap64 = lambda: _lib.check(lib.b2_linear_assignment_f64(_lib.ptr(c64), None, None, S, n, m, 0.8, _lib.ptr(x), _lib.ptr(y), _lib.stream_ptr()))
        for fn in (iou, lap32, bot, lap64):
            for _ in range(5):
                fn()
        torch.cuda.synchronize()
        r = {"problems": S, "tracks": n, "detections": m, "D": D}
        for key, fn in (("iou_cost_us", iou), ("lap_f32_us", lap32), ("botsort_cost_us", bot), ("lap_f64_us", lap64)):
            r[key] = event_ms(fn, 50) * 1e3
        r["iou_pair_us"], r["botsort_pair_us"] = r["iou_cost_us"] + r["lap_f32_us"], r["botsort_cost_us"] + r["lap_f64_us"]
        rows.append(r)
    return rows


def bench_track(n_frames=60, warmup=10):
    from b200dt.predictor import YOLO

    vid = synth.IRStream(seed=3, h=512, w=640)
    frames = [vid.frame() for _ in range(n_frames)]
    model = YOLO("yolov8n-p2.yaml")
    out = {}
    for reid in (False, True):
        cfg_ = {"tracker_type": "botsort", "gmc_method": "none", "with_reid": reid}
        model.track(frames[0], tracker=cfg_)
        ts, dets = [], 0
        for i, f in enumerate(frames):
            t0 = time.perf_counter()
            r = model.track(f, tracker=cfg_, persist=True)
            torch.cuda.synchronize()
            if i >= warmup:
                ts.append(time.perf_counter() - t0)
                dets += len(r[0])
        out["reid" if reid else "plain"] = {"ms_per_frame_median": float(np.median(ts)) * 1e3, "ms_per_frame_mean": float(np.mean(ts)) * 1e3,
                                            "frames": len(ts), "tracks_per_frame": dets / len(ts)}
    return {"workload": "YOLO(yolov8n-p2).track, 512x640 synthetic IR stream, BoT-SORT gmc none, conf 0.1", **out}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_reid_bench.jsonl"))
    a = ap.parse_args()
    _lib.require_cuda()
    lib = _lib.load()
    g = np.random.default_rng(0)
    info = gpu_info()
    recs = [dict(info, **bench_gather(lib, g))] + [dict(info, kernel="cost+solver", **r) for r in bench_cost(lib, g)]
    recs.append(dict(info, **bench_track()))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        for r in recs:
            fh.write(json.dumps(r) + "\n")
            print(json.dumps(r), flush=True)


if __name__ == "__main__":
    main()

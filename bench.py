#!/usr/bin/env python
"""Benchmark of the detect+track hot path (BASELINE.json metric: detect+track frames/sec, YOLOv8s-P2 640x512).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path, one rank per GPU
    python bench.py --impl reference --steps K --warmup W    # the reference's CPU path (oracle port) on host cores
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR   # + the last timed step's track rows as .npy files

One "step" = one frame of every resident stream through the whole per-frame path
(uint8 frame -> stem/forward -> DFL decode -> NMS -> Kalman track bank update).
Workload = BASELINE.json configs[3] ("C4"): 256 concurrent synthetic 640x512 IR streams, yolov8s-p2 (nc=80,
seeded synthetic weights), predict conf=0.15 iou=0.6, EnhancedMultiTargetTracker(150, min_hits=1, iou=0.1).
Streams are independent: each rank owns its own 256 streams (weak scaling, no data-path collective); the same line
carries a second record, "strong_scaling": BASELINE config 4 as written, 256 streams in total sharded 256/N per GPU.
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "detect+track frames/sec (YOLOv8s-P2 640x512)"
UNIT = "frames/s"
MODEL = "yolov8s-p2"
FRAME_HW = (512, 640)
CONF, IOU = 0.15, 0.6
TRACKER = dict(max_lost_frames=150, min_hits=1, iou_threshold=0.1)
DISTINCT_STREAMS = 32          # distinct synthetic videos, tiled to the stream count
POOL_FRAMES = 6                # consecutive frames per stream kept resident, played forth and back (0..5,4..1,0..): motion
                               # stays continuous, so tracks persist as they do on a real video
MAX_TRACKS_OUT = 256           # rows per stream of the downloaded result block (asserted sufficient)


def pool_index(i):
    """Ping-pong walk over the resident frame pool."""
    period = 2 * POOL_FRAMES - 2
    k = i % period
    return k if k < POOL_FRAMES else period - k


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--streams", type=int, default=256, help="streams per GPU")
    ap.add_argument("--capacity", type=int, default=2048, help="track slots per stream")
    ap.add_argument("--model", default=MODEL)
    ap.add_argument("--ref-streams", type=int, default=2, help="streams per step of the CPU reference arm")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-profile", default=None, help="write the per-launch table of the forward to this JSON file")
    ap.add_argument("--no-numa-bind", action="store_true", help="do not pin the process to the GPU's local CPU cores")
    ap.add_argument("--no-overlap", action="store_true", help="run NMS + tracker on the forward's stream (no cross-step overlap)")
    ap.add_argument("--no-kernels", action="store_true", help="skip the stand-alone HBM-kernel measurements")
    ap.add_argument("--total-streams", type=int, default=256, help="streams of the strong-scaling record (sharded over the GPUs)")
    ap.add_argument("--no-strong", action="store_true", help="skip the strong-scaling record")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write the track rows and counts of the last timed step (rank 0) as float64 .npy files to DIR")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    return a


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm": d["hbm_gbs"], "tc_burst": d["bf16_tflops"], "tc_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "src": "measured"}
    return {"hbm": 6650.0, "tc_burst": 1590.0, "tc_sustained": 1400.0, "src": "fallback"}


I32_COLS = [0, 6, 7, 8, 9, 10, 11, 12, 16]     # columns of a track row that hold int32 bit patterns (include/b2dt.h)
SLOT_COL = 19                                  # the bank's slot index of the track: implementation-defined
DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, rows, counts):
    """rows: CPU float32 [S][MAX_TRACKS_OUT][20], counts: CPU int32 [S] -> out_dir/{tracks,track_counts,stream_ids}.npy, float64.
    Each stream's reported rows are sorted by track id (the reference's list order; the bank's own row order is an
    implementation detail), int32 columns are converted to their values, the slot column (equally an implementation detail)
    and unused rows are zero.  Streams beyond the
    DUMP_BYTES budget are left out by a fixed-seed sample; stream_ids names the streams kept."""
    import numpy as np

    rows, counts = rows.numpy(), counts.numpy()
    S = rows.shape[0]
    assert int(counts.max()) <= rows.shape[1], "a stream reported more tracks than the result block holds"
    k = min(S, DUMP_BYTES // (rows[0].size * 8 + 16))
    ids = np.arange(S) if k == S else np.sort(np.random.default_rng(0).choice(S, k, replace=False))
    out = np.zeros((k,) + rows.shape[1:], np.float64)
    for j, s in enumerate(ids):
        r = rows[s, :counts[s]]
        v = r.astype(np.float64)
        v[:, I32_COLS] = r.view(np.int32)[:, I32_COLS]
        v[:, SLOT_COL] = 0
        out[j, :len(v)] = v[np.argsort(v[:, 0], kind="stable")]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "tracks.npy"), out)
    np.save(os.path.join(out_dir, "track_counts.npy"), counts[ids].astype(np.float64))
    np.save(os.path.join(out_dir, "stream_ids.npy"), ids.astype(np.float64))


def make_frames(n_streams, n_frames, seed0=1000):
    """uint8 [n_frames][n_streams][h][w][3]: DISTINCT_STREAMS seeded IR videos tiled over the streams."""
    import numpy as np

    from b200dt import synth

    k = min(DISTINCT_STREAMS, n_streams)
    vids = [synth.IRStream(seed=seed0 + s, h=FRAME_HW[0], w=FRAME_HW[1]) for s in range(k)]
    out = np.empty((n_frames, n_streams, FRAME_HW[0], FRAME_HW[1], 3), np.uint8)
    for t in range(n_frames):
        fr = [v.frame() for v in vids]
        for s in range(n_streams):
            out[t, s] = fr[s % k]
    return out


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200", "-i", str(gpu_index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None
        self.t0 = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def mark(self):
        self.t0 = time.time()

    def stop(self):
        t1 = time.time()
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for ts, line in self.rows:
            if self.t0 is not None and not (self.t0 - 0.1 <= ts <= t1 + 0.3):
                continue
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------
# reference arm / CPU baseline: the oracle port of the same per-frame path on host cores
# ---------------------------------------------------------------------------------------------------
class CpuPath:
    def __init__(self, model, n_streams):
        import torch

        from b200dt import cfg, weights
        from oracle import net as onet
        from oracle import tracker as otr

        torch.set_num_threads(os.cpu_count() or 1)
        self.cores = torch.get_num_threads()
        onet.set_conv_backend("aten")       # the conv primitive the reference itself calls on CPU (ATen/oneDNN)
        spec = cfg.resolve(model)
        self.nc = spec["nc"]
        self.net = onet.Net(onet.build_spec(model), weights.synthetic_state_dict(spec, seed=0), "fp32")
        self.trackers = [otr.MultiTracker(TRACKER["max_lost_frames"], TRACKER["min_hits"], TRACKER["iou_threshold"]) for _ in range(n_streams)]

    def step(self, frames):
        """frames: uint8 [n][h][w][3] -> per-stream track dict lists (predict conf/iou as the GPU arm)."""
        from oracle import postprocess as pp

        out = []
        for s, f in enumerate(frames):
            x = pp.preprocess([pp.letterbox_pad_only(f, (640, 640), auto=True, stride=32)])
            y = pp.decode(self.net.forward(x), [4, 8, 16, 32], self.nc)
            d = pp.non_max_suppression(y, CONF, IOU, mode="exact")[0]
            d[:, :4] = pp.scale_boxes(x.shape[2:], d[:, :4], f.shape[:2])
            out.append(self.trackers[s].update([r[:5] for r in d]))
        return out


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import numpy as np  # noqa: F401

    n = a.ref_streams
    frames = make_frames(n, POOL_FRAMES)
    cpu = CpuPath(a.model, n)
    for i in range(a.warmup):
        cpu.step(frames[pool_index(i)])
    t0 = time.perf_counter()
    for i in range(a.steps):
        cpu.step(frames[pool_index(a.warmup + i)])
    dt = time.perf_counter() - t0
    v = n * a.steps / dt
    sample = f"{n} streams x {a.steps} frames of the 256-stream workload, oracle port (numpy + ATen conv, fp32), {cpu.cores} threads"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": dt / a.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": workload_config(a, a.streams),
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cpu.cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def workload_config(a, streams):
    return {"workload": f"C4: {streams} concurrent synthetic 640x512 IR streams per GPU, {a.model} (nc=80, seeded synthetic weights) + "
                        f"Kalman tracker bank, predict conf={CONF} iou={IOU}, tracker(150, min_hits=1, iou=0.1)",
            "streams_per_gpu": streams, "frame": "640x512x3 uint8", "model": a.model,
            "l2": f"inputs larger than L2 ({streams * 640 * 512 * 3 / 1e6:.0f} MB of frames per step, {POOL_FRAMES}-frame resident pool played forth and back)",
            "pipelining": "NMS + tracker of step t on a second stream under the forward of step t+1; all K steps' work, downloads "
                          "included, is joined inside the timed region" if not getattr(a, "no_overlap", False) else "single stream"}


# ---------------------------------------------------------------------------------------------------
# stand-alone HBM-kernel measurements (SURVEY.md 8d): decode at the workload size, Kalman bank at C3 size
# ---------------------------------------------------------------------------------------------------
def time_cuda(fn, iters, flush=None):
    import torch

    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
    for s, e in ev:
        if flush is not None:
            flush()
        s.record()
        fn()
        e.record()
    torch.cuda.synchronize()
    ts = sorted(s.elapsed_time(e) for s, e in ev)
    return ts[len(ts) // 2]


def hbm_kernels(pipe, pk):
    import torch

    # these are kernels timed alone (against the measured copy peak): give the board a moment to leave the power-capped clock the
    # timed steps put it in (tools/fwd_probe.py: ~1590 MHz under the cap, 1965 MHz otherwise) -- on a throttled board the same
    # decode launch measured 0.147 ms instead of 0.121 ms
    torch.cuda.synchronize()
    time.sleep(1.5)
    out = {}
    eng, post = pipe.detect.engine, pipe.detect.post
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    flush = lambda: flush_buf.fill_(1)
    from b200dt import ops

    # DFL decode + confidence filter at C2 size (BASELINE.json configs[1]: batch 64, 640x640, A = 34000, nc = 80):
    # reads (64+nc) bf16 logits per anchor once -- 626.7 MB.  Synthetic logits (the kernel is data-independent except
    # for the candidate writes; N(0,1) class logits at conf 0.15 would flag most anchors, so they are shifted by -6).
    B2, nc2, ls2 = 64, 80, 144
    lh, lw, lst = [160, 80, 40, 20], [160, 80, 40, 20], [4, 8, 16, 32]
    g = torch.Generator(device="cuda").manual_seed(1)
    logits = []
    for h, w in zip(lh, lw):
        t = torch.randn((B2, h * w, ls2), device="cuda", generator=g)
        t[..., 64:] -= 6.0
        logits.append(t.to(torch.bfloat16))
    post2 = ops.DetectPost(B2, lh, lw, lst, nc2, ls2)
    ms = time_cuda(lambda: post2.decode(logits, CONF), 10, flush)
    nbytes = B2 * post2.A * ls2 * 2
    out["decode"] = {"ms": ms, "bytes": nbytes, "achieved_gbs": nbytes / ms / 1e6, "frac_of_hbm_peak": nbytes / ms / 1e6 / pk["hbm"],
                     "size": "C2: 64 x 34000 anchors x 144 bf16 logits", "mean_candidates": float(post2.cand_count.float().mean().item())}
    del logits, post2
    if eng.fused_head:
        # in-pipeline candidate stage of the fused Detect head: the 8-byte {logit, class} record of every anchor is read; the
        # 16-byte distance record is read and a 28-byte candidate written only for anchors that clear conf
        ms = time_cuda(lambda: post.candidates_from_head(eng.head_dist, eng.head_cls, CONF), 10, flush)
        ncand = int(post.cand_count.sum().item())
        nbytes = pipe.S * eng.num_anchors * 8 + ncand * (16 + 28)
        out["head_candidates"] = {"ms": ms, "bytes": nbytes, "achieved_gbs": nbytes / ms / 1e6, "frac_of_hbm_peak": nbytes / ms / 1e6 / pk["hbm"],
                                  "what": f"{pipe.S} x {eng.num_anchors} anchors x 8 B + {ncand} candidates x 44 B"}
    # NMS: latency-bound at realistic candidate counts -- report ms per batch
    ms = time_cuda(lambda: post.nms(IOU), 10, flush)
    out["nms"] = {"ms": ms, "images": pipe.S, "mean_candidates": float(post.cand_count.float().mean().item())}
    # Kalman bank at C3 scale (BASELINE.json configs[2]): 256 streams x 4096 live tracks = 1,048,576 tracks in a bank of
    # 256 x 4608 slots (room for the tracks that clutter detections found), L2 flushed before every timed launch pair
    from b200dt.tracker import TrackerBank

    S, C, L, D = 256, 4608, 4096, 1024
    bank = TrackerBank(S, C, D, 150, 1, 0.1)
    g = torch.Generator(device="cuda").manual_seed(0)
    for r in range(L // D):          # r-th batch of 1024 disjoint boxes per stream -> every box founds a track
        idx = torch.arange(D, device="cuda") + r * D
        x = (idx % 64).float() * 10.0
        y = (idx // 64).float() * 10.0
        boxes = torch.stack([x, y, x + 6, y + 6], 1)[None].repeat(S, 1, 1).contiguous()
        bank.update(boxes, torch.full((S,), D, dtype=torch.int32, device="cuda"), with_trajectory=False)
    torch.cuda.synchronize()
    live = int(bank.export(0)[3][2])
    assert live == L
    pb, ub = TrackerBank.bytes_per_track()
    # (a) a frame without detections: every track coasts -- predict, mark lost, delete test, reported row: the sweep kernel
    zero = torch.zeros((S,), dtype=torch.int32, device="cuda")
    dets = torch.zeros((S, D, 6), device="cuda")
    ms = time_cuda(lambda: bank.update(dets, zero, with_trajectory=False), 10, flush)
    nb = S * live * pb
    out["kalman_sweep_coast"] = {"ms": ms, "tracks": S * live, "bytes_per_track": pb, "achieved_gbs": nb / ms / 1e6,
                                 "frac_of_hbm_peak": nb / ms / 1e6 / pk["hbm"], "tracks_per_s": S * live / ms * 1e3,
                                 "what": "1,048,576 coasting tracks: predict + lifecycle + reported row (sweep_kernel), resolve_kernel idle; "
                                         "L2 flushed before every launch"}
    # (b) the full C3 frame: 10,240 detections per frame = 40 per stream, 70 % drawn from existing tracks (+N(0,1) px),
    # 30 % clutter; predict + IoU candidates + greedy association + update + lifecycle + rows of all 1M tracks
    Dn = 40
    pick = torch.randint(0, L, (S, Dn), device="cuda", generator=g)
    px, py = (pick % 64).float() * 10.0, (pick // 64).float() * 10.0
    clutter = torch.rand((S, Dn), device="cuda", generator=g) < 0.3
    px = torch.where(clutter, torch.rand((S, Dn), device="cuda", generator=g) * 634.0, px + torch.randn((S, Dn), device="cuda", generator=g))
    py = torch.where(clutter, torch.rand((S, Dn), device="cuda", generator=g) * 634.0, py + torch.randn((S, Dn), device="cuda", generator=g))
    dets[:, :Dn, 0], dets[:, :Dn, 1], dets[:, :Dn, 2], dets[:, :Dn, 3], dets[:, :Dn, 4] = px, py, px + 6, py + 6, 0.9
    cnt = torch.full((S,), Dn, dtype=torch.int32, device="cuda")
    ms = time_cuda(lambda: bank.update(dets, cnt, with_trajectory=False), 10, flush)
    live2 = int(bank.stats_async().cpu()[:, 2].sum())
    nb = live2 * pb + S * Dn * (16 + ub)
    out["kalman_frame_c3"] = {"ms": ms, "tracks": live2, "detections": S * Dn, "algorithmic_bytes": nb,
                              "achieved_gbs": nb / ms / 1e6, "frac_of_hbm_peak": nb / ms / 1e6 / pk["hbm"],
                              "tracks_per_s": live2 / ms * 1e3, "dropped": int(bank.stats_async().cpu()[:, 5].sum()),
                              "what": "sweep (predict + IoU candidates + coasting tracks' rows) + resolve (greedy association, Kalman "
                                      "update, motion analysis, new tracks), 256 streams x 4096+ tracks x 40 dets; L2 flushed"}
    # (c) AircraftKalmanTracker.predict alone (x, P, counters, trajectory push: 35 words per track)
    ms = time_cuda(lambda: bank.predict_only(), 10, flush)
    nb = live2 * 35 * 4
    out["kalman_predict_only"] = {"ms": ms, "tracks": live2, "bytes_per_track": 140, "achieved_gbs": nb / ms / 1e6,
                                  "frac_of_hbm_peak": nb / ms / 1e6 / pk["hbm"]}
    del flush_buf
    bank.close()
    # DRAM traffic of the same launches (dram__bytes_read.sum + dram__bytes_write.sum, one `ncu --set full` capture of
    # tools/hbm_probe.py --once, the same sizes and data recipes; committed under profiles/): traffic above the algorithmic bytes
    # means re-reads, below it means the L2 still held written lines when the capture ended
    tp = os.path.join(ROOT, "profiles", "r02_hbm_traffic.json")
    if os.path.exists(tp):
        tk = json.load(open(tp))["kernels"]
        for name, keys in (("decode", ["decode"]), ("head_candidates", ["head_candidates"]), ("nms", ["nms"]),
                           ("kalman_sweep_coast", ["sweep_coast", "resolve_coast"]), ("kalman_frame_c3", ["sweep_frame", "resolve_frame"]),
                           ("kalman_predict_only", ["bank_predict"])):
            if name in out and all(k in tk for k in keys):
                out[name]["traffic"] = sum((tk[k]["dram_read_mb"] + tk[k]["dram_write_mb"]) * 1e6 for k in keys)
                out[name]["ncu_duration_us"] = {k: tk[k]["duration_us"] for k in keys}
                out[name]["traffic_source"] = "profiles/r02_hbm_traffic.json"
    return out


# ---------------------------------------------------------------------------------------------------
def run_b200(a):
    import numpy as np
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    # stdout carries exactly ONE JSON line: libraries that print there (NCCL prints its version banner on the first
    # communicator) are diverted to stderr until the line is written
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    import b200dt  # noqa: F401
    from b200dt import _lib
    from b200dt.pipeline import DetectTrackPipeline, bind_host_to_gpu, gather_results, shard_streams

    affinity0 = os.sched_getaffinity(0)
    if not a.no_numa_bind:
        bind_host_to_gpu(local)          # before any pinned allocation

    pk = peaks()
    S = a.streams
    pipe = DetectTrackPipeline(a.model, S, FRAME_HW, 640, CONF, IOU, 300, capacity=a.capacity, overlap_post=not a.no_overlap,
                               max_tracks_out=MAX_TRACKS_OUT, **TRACKER)
    main_pipe = pipe
    host = torch.from_numpy(make_frames(S, POOL_FRAMES, seed0=1000 + 97 * rank)).pin_memory()
    dev = host.cuda()
    lib = _lib.load()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(step_fn, steps, pipe=None):
        pipe = pipe or main_pipe
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            step_fn(i)
        pipe.join()                 # the last step's download (own stream) is inside the timed region
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    # ---- device-resident: inputs already in HBM -------------------------------------------------
    for i in range(a.warmup):
        pipe.step_device(dev[pool_index(i)])
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.mark()
    l0 = lib.b2_launch_count()
    pipe.forward_events = [] if not a.no_overlap else None
    ms_dev = timed(lambda i: pipe.step_device(dev[pool_index(a.warmup + i)]), a.steps)
    fwd_ms_insitu = None
    if pipe.forward_events:
        fwd_ms_insitu = sum(e0.elapsed_time(e1) for e0, e1 in pipe.forward_events) / len(pipe.forward_events)
    pipe.forward_events = None
    launches = lib.b2_launch_count() - l0
    # step_device returns views of the bank's result block: take the last timed step's copy before the host-facing steps
    # below overwrite it
    last_out = (pipe.bank.rows.cpu(), pipe.bank.counts.cpu()) if a.dump_outputs and rank == 0 else None
    clocks = sampler.stop() if sampler else None
    value = S * world * a.steps / ms_dev * 1e3

    # ---- end to end through the host-facing call: pinned host frames in, track rows out --------------
    for i in range(a.warmup):
        pipe.step_host(host[pool_index(a.warmup + a.steps + i)])
    ms_e2e = timed(lambda i: pipe.step_host(host[pool_index(2 * a.warmup + a.steps + i)]), a.steps)
    e2e = S * world * a.steps / ms_e2e * 1e3
    # the host block of the last step, after the checks that make it the reference's result: no detection was dropped for
    # lack of a track slot (the reference's track list is unbounded) and no stream reported more rows than were downloaded
    rows, counts = pipe.results()
    stats = pipe.host_stats.numpy().copy()
    st = pipe.bank.export(0)[3]
    assert int(stats[:, 5].sum()) == 0 and int(st[7]) == 0, "the track bank dropped detections: not the reference's computation"
    n_dets = pipe.detect.post.out_count.float()

    # ---- BASELINE config 4 as written: 256 streams in total, sharded 256 / N per GPU (strong scaling) ----
    strong = None
    if not a.no_strong:
        total = a.total_streams
        if world == 1 and S == total:
            strong = {"streams_total": total, "streams_per_gpu": S, "value": value, "ms_per_step": ms_dev / a.steps,
                      "e2e": e2e, "e2e_ms_per_step": ms_e2e / a.steps, "note": "same run as the weak-scaling record at N=1"}
        else:
            mine = shard_streams(total, rank, world)
            Ss = len(mine)
            sp = DetectTrackPipeline(a.model, Ss, FRAME_HW, 640, CONF, IOU, 300, capacity=a.capacity, overlap_post=not a.no_overlap,
                                     max_tracks_out=MAX_TRACKS_OUT, **TRACKER)
            sdev = dev[:, :Ss].contiguous()
            shost = host[:, :Ss].contiguous().pin_memory()
            for i in range(a.warmup):
                sp.step_device(sdev[pool_index(i)])
            ms_s = timed(lambda i: sp.step_device(sdev[pool_index(a.warmup + i)]), a.steps, sp)
            for i in range(a.warmup):
                sp.step_host(shost[pool_index(a.warmup + a.steps + i)])
            ms_se = timed(lambda i: sp.step_host(shost[pool_index(2 * a.warmup + a.steps + i)]), a.steps, sp)
            sp.results()
            strong = {"streams_total": total, "streams_per_gpu": Ss, "value": total * a.steps / ms_s * 1e3, "ms_per_step": ms_s / a.steps,
                      "e2e": total * a.steps / ms_se * 1e3, "e2e_ms_per_step": ms_se / a.steps,
                      "note": "256 streams sharded contiguously over the ranks (pipeline.shard_streams); max over ranks"}
            del sp, sdev, shost

    # the only collective: gather per-stream result blocks (off the data path; not in the timed region)
    if world > 1:
        gather_results(pipe.bank.rows[:, :64].contiguous(), pipe.bank.counts)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (tcgen05 implicit-GEMM conv), per-launch CUDA events ----------
    # (eager launches with an event between consecutive launches; per launch the median of five passes after one warm-up pass:
    #  a single pass varies by several per cent under the power cap)
    pipe.detect.engine.profile_u8(dev[0], pipe.top, pipe.left)
    passes = [pipe.detect.engine.profile_u8(dev[1 + i % (POOL_FRAMES - 1)], pipe.top, pipe.left) for i in range(5)]
    prof = [dict(p0, ms=sorted(pp_[i]["ms"] for pp_ in passes)[2]) for i, p0 in enumerate(passes[0])]
    if a.dump_profile:
        json.dump(prof, open(a.dump_profile, "w"), indent=0)
    conv = [p for p in prof if p["op"] == "conv"]
    conv_ms, conv_fl = sum(p["ms"] for p in conv), sum(p["flops"] for p in conv)
    all_ms = sum(p["ms"] for p in prof)
    ms_step = ms_dev / a.steps
    # The kernel's launch durations inside the timed region: CUDA events around every forward of the K timed steps (one CUDA
    # graph: stem, the conv launches with programmatic dependent launch between them, SPPF pool; recorded on the stream it runs
    # on), times the conv launches' share of the forward from the eager per-launch passes below.  Why not the eager sums
    # themselves: the board is power capped (tools/fwd_probe.py: ~1000 W, SM clock 1965 -> ~1590 MHz once forwards run back to
    # back for > 0.2 s), and the eager passes -- an event between consecutive launches -- run at the unthrottled clock: 10.5 ms
    # against 11.4 ms for the same launches inside the step.  The sustained cuBLAS peak is the denominator that belongs to
    # the in-step time (MEASURED_PEAKS: burst for a kernel timed alone, sustained inside a long step); the eager reading against
    # the burst peak is reported beside it (frac_alone_vs_burst), and K back-to-back forwards without the rest of the step too.
    conv_share = conv_ms / all_ms
    conv_ms_eager = conv_ms
    eng = pipe.detect.engine
    for i in range(a.warmup):
        eng.forward_u8(dev[pool_index(i)], pipe.top, pipe.left)
    torch.cuda.synchronize()
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g0.record()
    for i in range(a.steps):
        eng.forward_u8(dev[pool_index(a.warmup + i)], pipe.top, pipe.left)
    g1.record()
    torch.cuda.synchronize()
    fwd_ms_graph = g0.elapsed_time(g1) / a.steps
    conv_ms = (fwd_ms_insitu if fwd_ms_insitu is not None else fwd_ms_graph) * conv_share
    achieved = conv_fl / conv_ms / 1e9
    # DRAM traffic per launch of the same kernel: dram__bytes_read.sum + dram__bytes_write.sum over the conv launches of one
    # forward of this workload, from the committed ncu capture (profiles/; per-launch list beside it), averaged per launch
    traffic, traffic_src = None, None
    for tp_name in ("r02_conv_traffic.json", "r01_conv_traffic_v38.json"):
        tp = os.path.join(ROOT, "profiles", tp_name)
        if os.path.exists(tp) and S == 256 and a.model == MODEL:
            tj = json.load(open(tp))
            if tj["conv_launches"] != len(conv):
                continue                 # captured on a different launch plan (e.g. before the chained launches): not this build
            traffic, traffic_src = tj["conv_dram_bytes_per_launch"], "profiles/%s (ncu, %d launches)" % (tp_name, tj["conv_launches"])
            break
    conv_bytes = sum(p["bytes"] for p in conv)
    roofline = {"bound": "tensor", "kernel": f"conv_tc_kernel (tcgen05 implicit GEMM, {len(conv)} launches/step)", "achieved": achieved,
                "peak": pk["tc_sustained"], "peak_kind": f"bf16 dense sustained, {pk['src']}", "unit": "TFLOP/s",
                "frac": achieved / pk["tc_sustained"], "traffic": traffic, "traffic_source": traffic_src,
                "algorithmic_bytes_per_launch": conv_bytes / len(conv), "avg_launch_ms": conv_ms / len(conv),
                "algorithmic_flops_per_step": conv_fl, "share_of_forward": conv_share, "share_of_step": conv_ms / ms_step,
                "timing": "CUDA events around each forward graph of the K timed steps x the conv launches' share of the forward (eager per-launch events)",
                "frac_alone_vs_burst": conv_fl / conv_ms_eager / 1e9 / pk["tc_burst"], "achieved_alone": conv_fl / conv_ms_eager / 1e9,
                "forward_ms_graph": fwd_ms_graph, "forward_ms_timed_region": fwd_ms_insitu, "forward_ms_eager_events": all_ms, "avg_launch_ms_eager": conv_ms_eager / len(conv), "end_to_end_tensor_frac": pipe.flops_per_frame * S / (ms_step * 1e-3) / 1e12 / pk["tc_sustained"]}
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": workload_config(a, S), "clocks": clocks,
        "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": pipe.h2d_bytes_per_step, "d2h_bytes_per_step": pipe.d2h_bytes_per_step,
                "ms_per_step": ms_e2e / a.steps},
        "gpu_launches": int(launches), "roofline": roofline, "strong_scaling": strong,
        "tracks": {"active_stream0": int(st[2]), "created_stream0": int(st[0]), "dropped_no_slot_all_streams": int(stats[:, 5].sum()),
                   "active_max_over_streams": int(stats[:, 2].max()), "recoveries_stream0": int(st[4]),
                   "mean_emitted_per_stream": float(counts.float().mean().item()), "max_emitted_per_stream": int(counts.max().item()),
                   "rows_downloaded_per_stream": MAX_TRACKS_OUT,
                   "mean_detections_per_frame": float(n_dets.mean().item()), "max_detections_per_frame": int(n_dets.max().item()),
                   "frames_per_stream": int(st[5])},
    }
    if world == 1 and not a.no_kernels:
        line["hbm_kernels"] = hbm_kernels(pipe, pk)
    if world == 1 and not a.no_cpu_baseline:
        os.sched_setaffinity(0, affinity0)       # the CPU leg may use every core the process started with
        n = a.ref_streams
        cpu = CpuPath(a.model, n)
        fr = host[:, :n].numpy()
        cpu.step(fr[0])
        t0, k = time.perf_counter(), 0
        while k < 6 or (time.perf_counter() - t0 < 12.0 and k < 200):
            cpu.step(fr[k % POOL_FRAMES])
            k += 1
        dt = time.perf_counter() - t0
        line["cpu_baseline"] = {"value": n * k / dt, "unit": UNIT, "cores": cpu.cores, "kind": "port",
                                "sample": f"{n} streams x {k} frames of the same workload (oracle port: numpy + ATen conv fp32, exact NMS, float64 tracker)"}
    if last_out is not None:
        dump_outputs(a.dump_outputs, *last_out)
    sys.stdout.flush()
    os.dup2(saved_stdout, 1)
    print(json.dumps(line), flush=True)
    os.dup2(2, 1)
    if world > 1:
        dist.destroy_process_group()


def main():
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)


if __name__ == "__main__":
    main()

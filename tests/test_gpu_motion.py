"""Global camera motion on the GPU (csrc/motion.cu): the batched gray pyramid, corner response, corner selection and pyramidal LK
against OpenCV, GlobalMotionBank against the host GlobalMotionDetector, the per-stream tracker reset, and
DetectTrackPipeline(tracker="motion_compensated") against YOLO.predict + a host MotionCompensatedMultiTracker per stream."""
import numpy as np
import pytest

from golden_common import motion_frames_scene

cv2 = pytest.importorskip("cv2")

SHAPES = [(256, 320), (512, 640)]
MIXED = [(256, 320), (257, 321), (199, 263), (512, 640), (120, 160), (60, 81)]     # the last two: LK from level 2 / level 1


def select_corners(eig, max_corners=200, quality=0.01, min_distance=15):
    """goodFeaturesToTrack's selection on a response, restated: keep > quality * max (threshold in float32 of the float64
    product), 3x3 local maxima off the one-pixel border, order by (value, linear index) descending, greedy at d^2 >= min_distance^2."""
    H, W = eig.shape
    thr = np.float32(float(eig.max()) * quality)
    e = np.where(eig > thr, eig, np.float32(0)).astype(np.float32)
    dil = cv2.dilate(e, None)
    ys, xs = np.nonzero((e != 0) & (e == dil))
    keep = (ys > 0) & (ys < H - 1) & (xs > 0) & (xs < W - 1)
    ys, xs = ys[keep], xs[keep]
    order = np.lexsort((-(ys * W + xs), -e[ys, xs]))
    out = []
    for k in order:
        x, y = int(xs[k]), int(ys[k])
        if all((x - a) ** 2 + (y - b) ** 2 >= min_distance ** 2 for a, b in out):
            out.append((x, y))
            if len(out) == max_corners:
                break
    return np.asarray(out, np.float32).reshape(-1, 2)


def _cv2_gftt(gray):
    c = cv2.goodFeaturesToTrack(gray, maxCorners=200, qualityLevel=0.01, minDistance=15, blockSize=7)
    return np.zeros((0, 2), np.float32) if c is None else c.reshape(-1, 2)


def _color_noise(seed, h, w):
    g = np.random.default_rng(seed)
    base = cv2.GaussianBlur(g.integers(0, 256, (h, w, 3), dtype=np.uint8), (0, 0), 2.0)
    return np.ascontiguousarray(base)


# ------------------------------------------------------------------------------------------------------------------------------
# CPU
# ------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("f", [0, 12, 25, 41])
def test_selection_rule_is_cv2_good_features_on_its_own_response(f):
    frames, _ = motion_frames_scene()
    gray = cv2.cvtColor(frames[f], cv2.COLOR_BGR2GRAY)
    got = select_corners(cv2.cornerMinEigenVal(gray, 7, 3))
    np.testing.assert_array_equal(got, _cv2_gftt(gray))


# ------------------------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------------------------
def _batches():
    """(frames list, packed?) batches: two seeds at each uniform shape, and a mixed-resolution packed batch with odd sizes."""
    out = []
    for hw in SHAPES:
        fs = [motion_frames_scene(n_frames=3, seed=s, hw=hw)[0] for s in (13, 21)]
        out.append(([f[t] for f in fs for t in (0, 2)], False))
    out.append(([_scene_crop(30 + k, hw) if k % 2 else _color_noise(k, *hw) for k, hw in enumerate(MIXED)], True))
    return out


def _scene_crop(seed, hw, n_frames=1):
    """Frames of the jolting scene at (h, w): a crop of the 256x320 scene for smaller shapes."""
    h, w = hw
    frames, _ = motion_frames_scene(n_frames=n_frames, seed=seed, hw=(max(h, 256), max(w, 320)))
    crops = [np.ascontiguousarray(f[:h, :w]) for f in frames]
    return crops[0] if n_frames == 1 else crops


def _pyramid(frames, packed):
    import torch

    from b200dt import ops

    if packed:
        dev = torch.from_numpy(ops.pack_frames(frames)[0]).cuda()
        return ops.gray_pyramid_u8(dev, [f.shape[:2] for f in frames])
    return ops.gray_pyramid_u8(torch.from_numpy(np.stack(frames)).cuda())


@pytest.mark.gpu
def test_gray_pyramid_is_bit_exact():
    for frames, packed in _batches():
        pyr = _pyramid(frames, packed)
        for s, f in enumerate(frames):
            want = cv2.cvtColor(f, cv2.COLOR_BGR2GRAY)
            for lvl in range(4):
                np.testing.assert_array_equal(pyr.level(s, lvl).cpu().numpy(), want, err_msg=f"stream {s} level {lvl} {f.shape}")
                want = cv2.pyrDown(want)


@pytest.mark.gpu
def test_corner_response_and_selection():
    from b200dt import ops

    for frames, packed in _batches():
        pyr = _pyramid(frames, packed)
        eig = ops.corner_min_eig(pyr)
        corners, counts = ops.good_features_to_track(pyr, eig=eig)
        corners, counts = corners.cpu().numpy(), counts.cpu().numpy()
        for s, f in enumerate(frames):
            gray = cv2.cvtColor(f, cv2.COLOR_BGR2GRAY)
            ref = cv2.cornerMinEigenVal(gray, 7, 3)
            mine = pyr.plane(eig, s).cpu().numpy()
            assert np.abs(mine - ref).max() <= 1e-5 * ref.max(), (s, f.shape)
            got = corners[s, :counts[s]]
            np.testing.assert_array_equal(got, select_corners(mine))      # exact on the kernel's own response
            cv = _cv2_gftt(gray)
            common = len(set(map(tuple, got.tolist())) & set(map(tuple, cv.tolist())))
            assert common >= min(197, len(cv)) and abs(len(got) - len(cv)) <= 3, (s, common, len(got), len(cv))


@pytest.mark.gpu
def test_pyr_lk_matches_cv2_on_cv2_corners():
    import torch

    from b200dt import ops

    status_eq = n_pts = n_both = n_close = 0
    worst = 0.0
    for hw in SHAPES + [(120, 160), (60, 81)]:
        frames = _scene_crop(13, hw, n_frames=30)
        for t in (1, 12, 24, 25, 29):
            prev, nxt = frames[t - 1], frames[t]
            g0, g1 = (cv2.cvtColor(f, cv2.COLOR_BGR2GRAY) for f in (prev, nxt))
            pts = _cv2_gftt(g0)
            ref, st, _ = cv2.calcOpticalFlowPyrLK(g0, g1, pts.reshape(-1, 1, 2), None, winSize=(21, 21), maxLevel=3,
                                                  criteria=(cv2.TERM_CRITERIA_EPS | cv2.TERM_CRITERIA_COUNT, 30, 0.01))
            ref, st = ref.reshape(-1, 2), st.reshape(-1)
            p0, p1 = _pyramid([prev], False), _pyramid([nxt], False)
            got, gst = ops.optical_flow_pyr_lk(p0, p1, torch.from_numpy(pts[None].copy()).cuda())
            got, gst = got[0].cpu().numpy(), gst[0].cpu().numpy()
            status_eq += int((gst == st).sum())
            n_pts += len(st)
            both = (gst == 1) & (st == 1)
            d = np.abs(got[both] - ref[both]).max(1)
            n_both += int(both.sum())
            n_close += int((d <= 0.01).sum())
            worst = max(worst, float(d.max()) if len(d) else 0.0)
    assert status_eq >= 0.99 * n_pts, (status_eq, n_pts)
    assert n_close >= 0.995 * n_both, (n_close, n_both)
    assert worst <= 0.5, worst


def _scene_streams(S, n_frames=60, hw=(256, 320)):
    return [motion_frames_scene(n_frames=n_frames, seed=13 + s, hw=hw) for s in range(S)]


def _why_flow_differs(prev, cur):
    """Which input of the motion vector differs between this library and cv2 on one frame pair: 'corners' (the selected set),
    'lk status' or 'lk position' (> 0.01 px, LK run by both on cv2's corners); None if all agree."""
    import torch

    from b200dt import ops

    g0, g1 = (cv2.cvtColor(f, cv2.COLOR_BGR2GRAY) for f in (prev, cur))
    p0, p1 = _pyramid([prev], False), _pyramid([cur], False)
    corners, counts = ops.good_features_to_track(p0)
    mine = corners[0, :int(counts[0])].cpu().numpy()
    ref = _cv2_gftt(g0)
    if len(mine) != len(ref) or set(map(tuple, mine.tolist())) != set(map(tuple, ref.tolist())):
        return "corners"
    nxt, st, _ = cv2.calcOpticalFlowPyrLK(g0, g1, ref.reshape(-1, 1, 2), None, winSize=(21, 21), maxLevel=3,
                                          criteria=(cv2.TERM_CRITERIA_EPS | cv2.TERM_CRITERIA_COUNT, 30, 0.01))
    got, gst = ops.optical_flow_pyr_lk(p0, p1, torch.from_numpy(ref[None].copy()).cuda())
    got, gst = got[0].cpu().numpy(), gst[0].cpu().numpy()
    if not np.array_equal(gst, st.reshape(-1)):
        return "lk status"
    both = gst == 1
    if (np.abs(got[both] - nxt.reshape(-1, 2)[both]) > 0.01).any():
        return "lk position"
    return None


@pytest.mark.gpu
def test_global_motion_bank_matches_host_detector_per_stream():
    import torch

    from b200dt.tracker import GlobalMotionBank, MotionCompensatedMultiTracker

    S, T = 8, 60
    scenes = _scene_streams(S, T)
    bank = GlobalMotionBank(S, (256, 320))
    host = [MotionCompensatedMultiTracker() for _ in range(S)]
    resets = close = 0
    worst = 0.0
    off = []
    for t in range(T):
        frames = torch.from_numpy(np.stack([sc[0][t] for sc in scenes])).cuda()
        counts = torch.tensor([len(sc[1][t]) for sc in scenes], dtype=torch.int32, device="cuda")
        bank.flow(frames)
        flags, info = bank.decide(counts)
        info, flags = info.cpu().numpy(), flags.cpu().numpy()
        for s in range(S):
            h = host[s]
            before = h.stats["global_resets"]
            h.update(scenes[s][1][t], scenes[s][0][t])
            fi = h.frame_motion_info
            d = max(abs(info[s, 0] - fi["magnitude"]), *np.abs(info[s, 1:3] - np.asarray(fi["vector"])))
            close += d <= 0.02
            worst = max(worst, float(d))
            assert bool(info[s, 3]) == fi["is_motion"] and bool(info[s, 4]) == fi["should_reset"], (t, s, info[s], fi)
            g = h.stats["global_resets"] > before
            assert bool(flags[s]) == g == bool(info[s, 5]), (t, s)
            resets += g
            if d > 0.02:
                off.append((t, s, float(d), _why_flow_differs(scenes[s][0][t - 1], scenes[s][0][t])))
    print(f"motion vector within 0.02 px of the host detector on {close} of {S * T} stream-frames, worst {worst:.4f} px: {off}")
    # measured on a B200: 478 of 480 within 0.02 px, worst 1.12 px; the decisions above are exact on every frame.  Where the vector
    # differs, the inputs of the mean differ: a corner the two selections break differently (a near-tie of the response), or an
    # LK status / position cv2's float sums put on the other side of a threshold
    assert close >= 478 and worst <= 1.12, (close, worst, off)
    assert all(why is not None for *_, why in off), off
    assert resets > 0
    for s, st in enumerate(bank.stats()):
        md = host[s].motion_detector.stats
        for k in ("total_detections", "motion_events", "reset_triggers"):
            assert st[k] == md[k], (s, k)
        assert abs(st["avg_motion_magnitude"] - md["avg_motion_magnitude"]) <= 0.02
        assert st["global_motion_events"] == host[s].stats["global_motion_events"]
        assert st["global_resets"] == host[s].stats["global_resets"]


@pytest.mark.gpu
def test_tracker_reset_streams():
    import torch

    from b200dt.tracker import TrackerBank

    scenes = _scene_streams(4, 6)
    S = 4

    def dets_of(t):
        d = torch.zeros((S, 300, 4), dtype=torch.float32)
        c = torch.zeros((S,), dtype=torch.int32)
        for s in range(S):
            rows = np.asarray(scenes[s][1][t], np.float32).reshape(-1, 5)[:, :4]
            d[s, :len(rows)] = torch.from_numpy(rows)
            c[s] = len(rows)
        return d.cuda(), c.cuda()

    bank = TrackerBank(S, 64, 300, 150, 1, 0.1, mode=1)
    for t in range(4):
        bank.update(*dets_of(t))
    before = {s: (bank.export(s), bank.export_reset(s)) for s in range(S)}
    bank.reset_streams(torch.tensor([1, 0, 1, 0], dtype=torch.int32, device="cuda"))
    fresh = TrackerBank(S, 64, 300, 150, 1, 0.1, mode=1)
    for s in range(S):
        got = bank.export(s)
        want = fresh.export(s) if s in (0, 2) else before[s][0]
        for a, b in zip(got, want):
            np.testing.assert_array_equal(a, b)
        if s in (1, 3):
            np.testing.assert_array_equal(bank.export_reset(s), before[s][1])
    # the next frame on a reset stream is the first frame of a fresh bank
    d, c = dets_of(4)
    r1, c1 = (x.cpu().numpy().copy() for x in bank.update(d, c))
    r2, c2 = (x.cpu().numpy().copy() for x in fresh.update(d, c))
    for s in (0, 2):
        assert c1[s] == c2[s]
        np.testing.assert_array_equal(r1[s, :c1[s]].view(np.int32), r2[s, :c2[s]].view(np.int32))



def _pipe(shapes, imgsz, capacity=1024, **kw):
    from b200dt.pipeline import DetectTrackPipeline

    return DetectTrackPipeline("yolov8n-p2", len(shapes), shapes, imgsz, 0.15, 0.6, 300, capacity=capacity, tracker="motion_compensated", **kw)


def _mixed_scene(shapes, T):
    sc = [motion_frames_scene(n_frames=T, seed=13 + s, hw=hw) for s, hw in enumerate(shapes)]
    return [[sc[s][0][t] for s in range(len(shapes))] for t in range(T)]


def _check_pipeline(shapes, imgsz, T, packed):
    import torch

    from b200dt import ops
    from b200dt.predictor import YOLO
    from b200dt.tracker import MotionCompensatedMultiTracker, rows_to_dicts

    frames = _mixed_scene(shapes, T)
    pipe = _pipe(shapes, imgsz)
    model = YOLO("yolov8n-p2.yaml")
    host = [MotionCompensatedMultiTracker(150, 1, 0.1, capacity=1024) for _ in shapes]
    n = resets = 0
    for t, fr in enumerate(frames):
        buf = ops.pack_frames(fr)[0] if packed else np.stack(fr)
        pipe.step_host(torch.from_numpy(buf).pin_memory())
        rows, counts = pipe.results()
        rows, counts, extra, motion = rows.numpy(), counts.numpy(), pipe.host_extra.numpy(), pipe.host_motion.numpy()
        res = model.predict(fr, conf=0.15, iou=0.6, imgsz=imgsz)
        for s in range(len(shapes)):
            h = host[s]
            before = h.stats["global_resets"]
            want = h.update([[*r[:4], r[4]] for r in res[s].boxes.data.cpu().numpy()], fr[s])
            assert bool(motion[s, 5]) == (h.stats["global_resets"] > before), (t, s)
            resets += h.stats["global_resets"] > before
            r = rows[s, :counts[s]]
            got = rows_to_dicts(r)
            assert [g["track_id"] for g in got] == [w["track_id"] for w in want], (t, s)
            order = np.argsort(r.view(np.int32)[:, 0], kind="stable")
            ex = extra[s, :counts[s]][order]
            for g, w, e in zip(got, want, ex):
                np.testing.assert_allclose(g["bbox"], w["bbox"], rtol=1e-5, atol=1e-3)
                for k in ("age", "hits", "hit_streak", "time_since_update", "lost_frames", "is_lost"):
                    assert g[k] == w[k], (t, s, k)
                assert int(e[:2].view(np.int32)[0]) == w["reset_count"] and int(e[:2].view(np.int32)[1]) == w["frames_since_reset"]
                assert np.float32(e[2]) == np.float32(w["motion_consistency"])
            n += len(got)
    assert n > 0 and resets > 0
    return pipe


@pytest.mark.gpu
def test_motion_pipeline_uniform_equals_predict_plus_host_tracker():
    pipe = _check_pipeline([(256, 320)] * 3, 320, 30, packed=False)
    assert not pipe.ragged and pipe.bank.mode == 1


@pytest.mark.gpu
def test_motion_pipeline_mixed_equals_predict_plus_host_tracker():
    pipe = _check_pipeline([(256, 320), (288, 352), (256, 320)], 320, 30, packed=True)
    assert pipe.ragged


@pytest.mark.gpu
def test_motion_pipeline_entry_points_agree():
    import torch

    from b200dt import ops

    for shapes, packed in (([(256, 320)] * 3, False), ([(256, 320), (288, 352), (256, 320)], True)):
        frames = _mixed_scene(shapes, 14)         # a jolt (global reset) at frame 12; no bank grows at this capacity
        bufs = [ops.pack_frames(f)[0] if packed else np.stack(f) for f in frames]
        plain, over, host = _pipe(shapes, 320, 8192), _pipe(shapes, 320, 8192, overlap_post=True), _pipe(shapes, 320, 8192)
        for t, b in enumerate(bufs):
            dev = torch.from_numpy(b).cuda()
            r0, c0 = (x.cpu().numpy().copy() for x in plain.step_device(dev))
            rows, counts = over.step_device(dev)
            over.join()
            r1, c1 = (x.cpu().numpy().copy() for x in (rows, counts))
            host.step_host(torch.from_numpy(b).pin_memory())
            r2, c2 = (x.numpy() for x in host.results())
            np.testing.assert_array_equal(c0, c1)
            np.testing.assert_array_equal(c0, c2)
            for s in range(len(shapes)):
                np.testing.assert_array_equal(r0[s, :c0[s]].view(np.int32), r1[s, :c1[s]].view(np.int32))
                np.testing.assert_array_equal(r0[s, :c0[s]].view(np.int32), r2[s, :c2[s]].view(np.int32))
            np.testing.assert_array_equal(plain.motion.info.cpu().numpy(), host.host_motion.numpy())


@pytest.mark.gpu
def test_default_pipeline_launches_what_it_launched_before():
    """tracker="enhanced" (the default) builds no motion bank and launches the forward, the candidate stage, NMS and the tracker."""
    import torch

    from b200dt import _lib
    from b200dt.pipeline import DetectTrackPipeline

    lib = _lib.load()
    shapes = [(96, 128)] * 3
    frames = [torch.from_numpy(np.stack(f)).cuda() for f in (_mixed_scene([(256, 320)] * 3, 2))]
    frames = [f[:, :96, :128].contiguous() for f in frames]
    pipe, probe = (DetectTrackPipeline("yolov8n-p2", 3, shapes, 128, 0.15, 0.6, 300, capacity=1024) for _ in range(2))
    assert pipe.motion is None and pipe.bank.mode == 0 and pipe.host_extra is None
    pipe.step_device(frames[0])
    probe.step_device(frames[0])
    torch.cuda.synchronize()

    def delta(fn):
        n0 = lib.b2_launch_count()
        r = fn()
        torch.cuda.synchronize()
        return lib.b2_launch_count() - n0, r

    n_fwd, _ = delta(lambda: probe.detect.engine.forward_u8(frames[1], probe.top, probe.left))
    n_cand, _ = delta(lambda: probe.detect.candidates(0.15))
    n_nms, (dets, counts) = delta(lambda: probe.detect.nms(0.6, (96, 128)))
    n_trk, _ = delta(lambda: probe.bank.update(dets, counts, with_trajectory=False))
    n_step, _ = delta(lambda: pipe.step_device(frames[1]))
    assert n_step == n_fwd + n_cand + n_nms + n_trk


@pytest.mark.gpu
def test_unsupported_parameters_are_rejected():
    import torch

    from b200dt import ops

    pyr = ops.gray_pyramid_u8(torch.zeros((1, 256, 320, 3), dtype=torch.uint8, device="cuda"))
    with pytest.raises(NotImplementedError):
        ops.good_features_to_track(pyr, max_corners=100)
    with pytest.raises(NotImplementedError):
        ops.corner_min_eig(pyr, block_size=5)
    pts = torch.zeros((1, 4, 2), dtype=torch.float32, device="cuda")
    with pytest.raises(NotImplementedError):
        ops.optical_flow_pyr_lk(pyr, pyr, pts, max_level=2)


@pytest.mark.gpu
def test_results_of_the_step_that_grows_the_bank():
    """results() on the step after which the bank grows returns that step's rows (the host block is reallocated at the next
    step_host), and the grown pipeline goes on equal to one that never grew."""
    import torch

    from b200dt.pipeline import DetectTrackPipeline

    shapes = [(256, 320)] * 3
    frames = _mixed_scene(shapes, 3)
    # max_det 100: a frame never overflows 256 slots, and 56 live tracks are enough for results() to grow the bank
    small, big = (DetectTrackPipeline("yolov8n-p2", 3, shapes, 320, 0.15, 0.6, 100, capacity=c) for c in (256, 8192))
    grew = False
    for fr in frames:
        buf = np.stack(fr)
        cap = small.bank.capacity
        small.step_host(torch.from_numpy(buf).pin_memory())
        rows, counts = (x.numpy().copy() for x in small.results())
        grew |= small.bank.capacity > cap
        r2, c2 = (x.cpu().numpy() for x in big.step_device(torch.from_numpy(buf).cuda()))
        np.testing.assert_array_equal(counts, c2)
        for s in range(3):                    # row order follows slots, which depend on the capacity: compare in id order
            a, b = rows[s, :counts[s]].view(np.int32), r2[s, :c2[s]].view(np.int32)
            a, b = a[np.argsort(a[:, 0], kind="stable")], b[np.argsort(b[:, 0], kind="stable")]
            np.testing.assert_array_equal(a[:, :19], b[:, :19])      # column 19 is the slot
    assert grew

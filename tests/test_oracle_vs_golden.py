"""Pin the CPU oracle against outputs of the reference itself (tests/golden/*.npz, produced by
tests/golden/make_golden.py running the unmodified reference in the build container)."""
import os

import numpy as np
import pytest

import b200dt  # noqa: F401
from b200dt import cfg, synth, weights
from oracle import kalman_filter as okf
from oracle import net as onet
from oracle import postprocess as pp
from oracle import tracker as otr

from golden_common import pack_tracks, synth_pred

G = os.path.join(os.path.dirname(__file__), "golden")


def _load(name):
    return np.load(os.path.join(G, name), allow_pickle=False)


# ----------------------------------------------------------------------------- tracker
def _run_oracle_tracker(seed, n_frames, params, python_floats, **seq_kw):
    seq = synth.DetectionSequence(seed=seed, **seq_kw)
    trk = otr.MultiTracker(int(params[0]), int(params[1]), float(params[2]))
    outs, states = [], []
    for _ in range(n_frames):
        d = seq.step()
        dd = [[float(v) for v in r] for r in d] if python_floats else [r for r in d]
        outs.append(trk.update(dd))
        states.append([(int(t.track_id[1:]), t.x.copy(), t.P.copy(), t.lost_frames, t.is_lost) for t in trk.trackers])
    return trk, outs, states


@pytest.mark.parametrize("tag,pyf", [("f32", False), ("f64", True)])
def test_tracker_sequence_matches_reference(tag, pyf):
    g = dict(_load(f"tracker_seq_{tag}.npz"), states=_load(f"tracker_seq_{tag}_states.npz")["states"])
    trk, outs, states = _run_oracle_tracker(int(g["seed"]), int(g["n_frames"]), g["params"], pyf, n_targets=8)
    rows, cols, tl, tr = pack_tracks(outs)
    assert rows.shape == g["rows"].shape
    ci = {c: i for i, c in enumerate(cols)}
    exact = [ci[c] for c in ("frame", "id", "predicted", "age", "hits", "hit_streak", "time_since_update",
                             "lost_frames", "is_lost", "is_stable_motion")]
    np.testing.assert_array_equal(rows[:, exact], g["rows"][:, exact])      # track ids / lifecycle: bit-exact
    np.testing.assert_allclose(rows, g["rows"], rtol=1e-9, atol=1e-9)
    np.testing.assert_array_equal(tl, g["traj_len"])
    np.testing.assert_allclose(tr, g["traj"], rtol=1e-5, atol=1e-3)
    st = np.asarray([np.r_[f, tid, x, P.reshape(-1), lf, float(il)] for f, s in enumerate(states) for tid, x, P, lf, il in s])
    np.testing.assert_allclose(st, g["states"], rtol=1e-9, atol=1e-9)
    s = trk.get_statistics()
    got = [s[k] for k in ("total_tracks_created", "total_tracks_terminated", "current_active_tracks",
                          "long_term_predictions", "successful_recoveries", "frame_count")]
    np.testing.assert_array_equal(got, g["stats"])
    assert trk.last_min_iou_gap > 1e-7      # fixture stays away from IoU near-ties (SURVEY H4)


def test_tracker_second_parameterisation():
    g = _load("tracker_seq_default.npz")
    trk, outs, _ = _run_oracle_tracker(int(g["seed"]), int(g["n_frames"]), g["params"], False,
                                       n_targets=12, p_detect=0.7, clutter=0.5, burst=(50, 110))
    rows, cols, tl, tr = pack_tracks(outs)
    np.testing.assert_allclose(rows, g["rows"], rtol=1e-9, atol=1e-9)
    np.testing.assert_array_equal(tl, g["traj_len"])
    got = [trk.stats[k] for k in ("total_tracks_created", "total_tracks_terminated", "current_active_tracks",
                                  "long_term_predictions", "successful_recoveries")] + [trk.frame_count]
    np.testing.assert_array_equal(got, g["stats"])


def test_tracker_known_answer():
    """SURVEY.md 8c: 3-frame hand case (double predict on the first lost frame, K_pos = 150.1/160.1)."""
    g = _load("tracker_kat.npz")
    trk = otr.MultiTracker(150, 1, 0.1)
    kat = [[[10, 10, 20, 20, .9], [100, 100, 110, 112, .5]], [[11, 11, 21, 21, .9]], [[12, 12, 22, 22, .9]]]
    outs = [trk.update(d) for d in kat]
    rows, *_ = pack_tracks(outs)
    np.testing.assert_allclose(rows, g["rows"], rtol=1e-12, atol=1e-12)
    t1, t2 = trk.trackers
    np.testing.assert_allclose(t1.x, g["x_T001"], rtol=1e-12)
    np.testing.assert_allclose(t1.P, g["P_T001"], rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(t2.P, g["P_T002"], rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(t1.x[:2], [16.9370963082, 16.9370963082], rtol=1e-10)
    np.testing.assert_allclose([t1.P[0, 0], t1.P[0, 4], t1.P[4, 4]], [8.563355054998, 6.304735633999, 10.070621104413], rtol=1e-10)
    assert (t2.age, t2.time_since_update, t2.lost_frames) == (3, 3, 2)
    np.testing.assert_allclose([t2.P[0, 0], t2.P[0, 4], t2.P[4, 4]], [950.8, 300.3, 100.3], rtol=1e-12)
    # structural fact used by the CUDA bank: P[i,j] != 0 only when i == j (mod 4)
    mask = (np.arange(8)[:, None] - np.arange(8)[None]) % 4 != 0
    assert np.all(t1.P[mask] == 0)


# ----------------------------------------------------------------------------- Ultralytics KF
@pytest.mark.parametrize("kind", ["xyah", "xywh"])
def test_ultralytics_kf(kind):
    g = _load("kf_ultra.npz")
    z0, meas, hit = g[f"{kind}_z0"], g[f"{kind}_meas"], g[f"{kind}_hit"]
    mc = [okf.initiate(kind, z) for z in z0]
    means, covs = np.array([m for m, _ in mc]), np.array([c for _, c in mc])
    np.testing.assert_allclose(means, g[f"{kind}_init_mean"], rtol=1e-12)
    np.testing.assert_allclose(covs, g[f"{kind}_init_cov"], rtol=1e-12)
    for t in range(meas.shape[0]):
        means, covs = okf.predict(kind, means, covs)
        gd = np.stack([okf.gating_distance(kind, means[i], covs[i], meas[t]) for i in range(len(z0))])
        gp = np.stack([okf.gating_distance(kind, means[i], covs[i], meas[t], only_position=True) for i in range(len(z0))])
        np.testing.assert_allclose(gd, g[f"{kind}_gating"][t, 0], rtol=1e-8)
        np.testing.assert_allclose(gp, g[f"{kind}_gating"][t, 1], rtol=1e-8)
        for i in range(len(z0)):
            if hit[t, i]:
                means[i], covs[i] = okf.update(kind, means[i], covs[i], meas[t, i])
        np.testing.assert_allclose(means, g[f"{kind}_means"][t], rtol=1e-9, atol=1e-12)
        np.testing.assert_allclose(covs, g[f"{kind}_covs"][t], rtol=1e-8, atol=1e-12)


def test_ultralytics_kf_known_answer():
    g = _load("kf_ultra.npz")
    m, c = okf.initiate("xywh", [100., 50, 20, 40])
    np.testing.assert_allclose(np.diag(c), [4, 16, 4, 16, 1.5625, 6.25, 1.5625, 6.25])
    m, c = okf.predict("xywh", m, c)
    m2, c2 = okf.update("xywh", m, c, [102., 51, 21, 41])
    np.testing.assert_allclose(m2, g["kat_xywh_mean"], rtol=1e-12)
    np.testing.assert_allclose(np.diag(c2), g["kat_xywh_diag"], rtol=1e-12)
    np.testing.assert_allclose(okf.gating_distance("xywh", m, c, np.array([[102., 51, 21, 41], [107., 56, 26, 46]])),
                               [0.7272727273, 13.6198347107], rtol=1e-9)


# ----------------------------------------------------------------------------- NMS
def test_nms_hand_cases():
    b = np.array([[0, 0, 10, 10], [1, 1, 11, 11], [20, 20, 30, 30], [0, 0, 10, 10]], np.float32)
    s = np.array([.9, .8, .7, .6], np.float32)
    assert pp.nms_exact(b, s, 0.6).tolist() == [0, 2] and pp.nms_legacy(b, s, 0.6).tolist() == [0, 2]
    g = _load("nms_cases.npz")
    b = np.array([[200., 200, 210, 210], [0, 0, 10, 10], [0, 0, 10, 10.5]], np.float32)
    s = np.array([.9, .8, .7], np.float32)
    assert pp.nms_legacy(b, s, 0.6).tolist() == g["hand_div_legacy"].tolist() == [0, 1, 2]
    assert pp.nms_exact(b, s, 0.6).tolist() == g["hand_div_exact"].tolist() == [0, 1]


@pytest.mark.parametrize("ci", range(6))
@pytest.mark.parametrize("mode", ["exact", "legacy"])
def test_nms_matches_reference(ci, mode):
    g = _load("nms_cases.npz")
    seed, B, nc, A, conf, iou, max_det, agn = g[f"c{ci}_cfg"]
    frac = 0.05 if ci == 0 else 0.15
    pred = synth_pred(int(seed), int(B), int(nc), int(A), frac=frac)
    classes = g[f"c{ci}_classes"].tolist() if f"c{ci}_classes" in g.files else None
    out = pp.non_max_suppression(pred, float(conf), float(iou), classes=classes, agnostic=bool(agn),
                                 max_det=int(max_det), mode=mode)
    for b in range(int(B)):
        ref = g[f"c{ci}_{mode}_{b}"]
        assert out[b].shape == ref.shape
        np.testing.assert_array_equal(out[b], ref)          # fp32 arithmetic in the same order: bit-exact


# ----------------------------------------------------------------------------- network
def _model(name="yolov8n-p2"):
    spec, ospec = cfg.resolve(name), onet.build_spec(name)
    return spec, ospec, weights.synthetic_state_dict(spec, seed=0)


def test_spec_matches_between_host_and_oracle():
    for name in ("yolov8n-p2", "yolov8s-p2", "yolov8x-p2", "yolov8-small"):
        a, b = cfg.resolve(name), onet.build_spec(name)
        key = lambda L: (L["type"], L.get("c1"), L.get("c2"), L.get("n"), L.get("ch"), L["f"])
        assert [key(x) for x in a["layers"]] == [key(x) for x in b["layers"]]
    # SURVEY.md 8d algorithmic FLOPs
    assert abs(cfg.conv_flops(cfg.resolve("yolov8n-p2"), 512, 640) / 1e9 - 13.782) < 0.01
    assert abs(cfg.conv_flops(cfg.resolve("yolov8s-p2"), 512, 640) / 1e9 - 31.477) < 0.01
    assert abs(cfg.conv_flops(cfg.resolve("yolov8s-p2"), 640, 640) / 1e9 - 39.346) < 0.01
    assert abs(cfg.conv_flops(cfg.resolve("yolov8x-p2"), 1280, 1280) / 1e9 - 1267.7) < 0.1
    assert abs(onet.conv_flops(onet.build_spec("yolov8s-p2"), 640, 640) - cfg.conv_flops(cfg.resolve("yolov8s-p2"), 640, 640)) == 0


def test_net_forward_matches_reference():
    g = _load("net_n_p2_small.npz")
    spec, ospec, sd = _model()
    x = np.random.default_rng(0).random((1, 3, 64, 96), dtype=np.float32)
    net = onet.Net(ospec, sd, "fp32")
    heads = net.forward(x, record=True)
    for i, h in enumerate(heads):
        np.testing.assert_allclose(h, g[f"head{i}"], rtol=1e-4, atol=1e-3)
    for i in (0, 2, 9, 18, 27):
        np.testing.assert_allclose(net.trace[f"layer.{i}" if i else "model.0"], g[f"layer{i}"], rtol=1e-4, atol=1e-3)
    y = pp.decode(heads, [4, 8, 16, 32], 80)
    np.testing.assert_allclose(y, g["y"], rtol=1e-4, atol=5e-3)
    # decode fed with the reference's own head maps: isolates the DFL/anchor arithmetic
    y2 = pp.decode([g[f"head{i}"] for i in range(4)], [4, 8, 16, 32], 80)
    np.testing.assert_allclose(y2, g["y"], rtol=1e-5, atol=1e-4)


@pytest.mark.parametrize("tag,hw", [("512x640", (512, 640)), ("500x640", (500, 640))])
@pytest.mark.parametrize("mode", ["exact", "legacy"])
def test_predict_end_to_end_matches_reference(tag, hw, mode):
    """Full predict(): letterbox -> forward -> decode -> NMS -> scale_boxes vs YOLO(...).predict of the reference."""
    g = _load("predict_n_p2.npz")
    spec, ospec, sd = _model()
    frames = [synth.IRStream(seed=7, h=hw[0], w=hw[1]).frame(), synth.IRStream(seed=8, h=hw[0], w=hw[1]).frame()]
    lb = [pp.letterbox_pad_only(f, (640, 640), auto=True, stride=32) for f in frames]
    x = pp.preprocess(lb)
    heads = onet.Net(ospec, sd, "fp32").forward(x)
    y = pp.decode(heads, [4, 8, 16, 32], 80)
    dets = pp.non_max_suppression(y, 0.15, 0.6, mode=mode)
    for b, d in enumerate(dets):
        ref = g[f"{tag}_{mode}_{b}"]
        d = d.copy()
        d[:, :4] = pp.scale_boxes(x.shape[2:], d[:, :4], hw)
        # fp32 conv summation order differs (oneDNN vs numpy): allow a few borderline rows to differ
        assert abs(len(d) - len(ref)) <= 3
        # match rows by (cls, nearest box)
        matched = 0
        for r in ref:
            c = d[d[:, 5] == r[5]]
            if len(c) and np.min(np.abs(c[:, :4] - r[:4]).max(1) + np.abs(c[:, 4] - r[4])) < 5e-2:
                matched += 1
        assert matched >= len(ref) - 3


# ----------------------------------------------------------------------------- N1: motion-reset tracker (SURVEY.md 8f)
def test_motion_reset_track_matches_reference():
    """oracle.motion_reset.MotionResetTrack against camera_motion_compensation/motion_reset_kalman_tracker.py driven
    frame by frame (predict; update or mark_as_lost; get_track_info) over a script with jumps, a size change and gaps."""
    from oracle.motion_reset import MotionResetTrack

    g = _load("motion_reset.npz")
    dets, rows = g["dets"], g["rows"]
    trk = MotionResetTrack([float(v) for v in dets[0]], "T001", 150)
    assert int(rows[-1, 4 + 8 + 64 + 4 + 1]) >= 3                      # the script does trigger resets
    for t in range(1, len(dets)):
        pb = np.asarray(trk.predict(), np.float64)
        if np.isnan(dets[t][0]):
            trk.mark_lost()
        else:
            trk.update([float(v) for v in dets[t]])
        info = trk.info()
        r = rows[t - 1]
        np.testing.assert_allclose(pb, r[0:4], rtol=1e-12, atol=1e-9, err_msg=f"predict() frame {t}")
        np.testing.assert_allclose(trk.x, r[4:12], rtol=1e-12, atol=1e-9, err_msg=f"x frame {t}")
        np.testing.assert_allclose(trk.P.ravel(), r[12:76], rtol=1e-11, atol=1e-9, err_msg=f"P frame {t}")
        np.testing.assert_allclose(np.asarray(info["bbox"], np.float64), r[76:80], rtol=1e-12, atol=1e-9, err_msg=f"bbox frame {t}")
        got = [info["confidence"], trk.reset_count, trk.last_reset_frame, trk.age, trk.hits, trk.hit_streak, trk.time_since_update,
               float(trk.is_lost), trk.lost_frames, trk.motion_consistency, len(trk.position_history), len(trk.motion_scores),
               info["frames_since_reset"]]
        np.testing.assert_allclose(got, r[80:93], rtol=1e-12, atol=1e-12, err_msg=f"scalars frame {t}")


def test_motion_compensated_multi_tracker_matches_reference():
    """oracle.motion_reset.MotionCompensatedMultiTracker against camera_motion_compensation/motion_compensated_multi_tracker.py
    (update without a frame) on 160 frames of multi-target detections with camera shakes: same number of live tracks every
    frame, same per-track state in list order (the reference's ids are random uuids), same reset / recovery counters."""
    from oracle.motion_reset import MotionCompensatedMultiTracker

    g = _load("motion_multi.npz")
    dets, ndets, rows, counts, stats = g["dets"], g["ndets"], g["rows"], g["counts"], g["stats"]
    assert stats[1] >= 5                                                    # the script triggers individual resets
    trk = MotionCompensatedMultiTracker(150, 1, 0.1)
    k = 0
    for f in range(len(ndets)):
        d = [[float(v) for v in dets[f, 5 * i:5 * i + 5]] for i in range(int(ndets[f]))]
        res = trk.update(d)
        assert len(res) == counts[f], f"frame {f}"
        for info, t in zip(res, trk.trackers):
            got = np.concatenate([np.asarray(info["bbox"], np.float64), t.x, [info["confidence"], t.reset_count, t.age, t.hits, t.hit_streak,
                                  t.time_since_update, float(t.is_lost), t.lost_frames, t.motion_consistency, info["frames_since_reset"]]])
            np.testing.assert_allclose(got, rows[k], rtol=1e-11, atol=1e-8, err_msg=f"frame {f} track {t.track_id}")
            k += 1
    assert k == len(rows)
    assert [trk.stats["total_frames"], trk.stats["individual_resets"], trk.stats["tracking_recoveries"]] == list(stats[:3])


def test_resize_oracle_is_cv2():
    """The oracle's fixed-point bilinear is cv2.resize(INTER_LINEAR) on uint8, byte for byte (the letterbox resize of
    data/augment.py:1718); cv2 is the third-party implementation the reference calls, present in both containers."""
    cv2 = pytest.importorskip("cv2")
    g = np.random.default_rng(4)
    for (sh, sw), (dh, dw) in [((512, 640), (1024, 1280)), ((480, 640), (384, 512)), ((100, 130), (197, 256)), ((512, 640), (640, 800)),
                               ((720, 1280), (360, 640)), ((333, 517), (640, 640)), ((1080, 1920), (384, 640)), ((50, 60), (640, 512))]:
        img = g.integers(0, 256, (sh, sw, 3), dtype=np.uint8)
        np.testing.assert_array_equal(pp.resize_bilinear_u8(img, dh, dw), cv2.resize(img, (dw, dh), interpolation=cv2.INTER_LINEAR))
    # LetterBox in full against the reference's geometry + cv2
    img = g.integers(0, 256, (480, 640, 3), dtype=np.uint8)
    out = pp.letterbox(img, (1280, 1280), auto=True, stride=32)
    assert out.shape == (960, 1280, 3)
    np.testing.assert_array_equal(out, cv2.resize(img, (1280, 960), interpolation=cv2.INTER_LINEAR))


@pytest.mark.parametrize("name,gfile", [("yolov8n-p2", "predict_n_p2.npz"), ("yolov8s-p2", "predict_s_p2.npz"), ("yolov8-small", "predict_small.npz")])
def test_bf16_rounding_points_keep_the_reference_detection_set(name, gfile):
    """The oracle evaluated at the engine's rounding points (bf16 stored activations, fp32 accumulate) returns the SAME
    detection set as the fp32 reference's predict(), boxes within 1e-2 relative, outside the stated exclusion band
    (golden_common.detection_set_report).  This is the north_star tolerance, and the floor the CUDA engine is held to in
    tests/test_gpu_detect.py."""
    from golden_common import detection_set_report

    g = _load(gfile)
    spec, ospec, sd = _model(name)
    hw = (512, 640)
    f3 = synth.IRStream(seed=1001, h=hw[0], w=hw[1])
    frames = [synth.IRStream(seed=7, h=hw[0], w=hw[1]).frame(), synth.IRStream(seed=8, h=hw[0], w=hw[1]).frame(),
              [f3.frame() for _ in range(4)][-1]]
    onet.set_conv_backend("aten")
    try:
        y = pp.decode(onet.Net(ospec, sd, "bf16").forward(pp.preprocess(frames)), [4, 8, 16, 32], spec["nc"])
    finally:
        onet.set_conv_backend("numpy")
    dets = pp.non_max_suppression(y, 0.15, 0.6, mode="exact")
    strict = total = 0
    for b, d in enumerate(dets):
        d = d.copy()
        d[:, :4] = pp.scale_boxes(hw, d[:, :4], hw)
        rep = detection_set_report(d, g[f"512x640_exact_{b}"], g[f"512x640_cand_{b}"], 0.15, 0.6, frame_hw=hw)
        assert not rep["errors"], (b, rep)
        strict += rep["n_ref_strict"]; total += rep["n_ref"]
    assert strict >= 0.6 * total, (strict, total)            # the band must not swallow the comparison


BYTE_PARAMS = {"default": {}, "nofuse": dict(track_high_thresh=0.4, track_low_thresh=0.15, new_track_thresh=0.5, track_buffer=8,
                                             match_thresh=0.7, fuse_score=False)}


def _xywh(d):
    return np.stack([(d[:, 0] + d[:, 2]) / 2, (d[:, 1] + d[:, 3]) / 2, d[:, 2] - d[:, 0], d[:, 3] - d[:, 1]], 1).astype(np.float32)


@pytest.mark.parametrize("tag", ["default", "nofuse"])
def test_bytetrack_oracle_matches_reference(tag):
    """oracle.byte_tracker.BYTETracker against the reference's BYTETracker.update (ultralytics/trackers/byte_tracker.py) over the
    scripted 90-frame scene (misses, low-score boxes, clutter, crossings): the same rows every frame -- track id, score, class
    and detection index bit-exact, boxes to float32 rounding -- and the same filter state for every tracked / lost track."""
    from golden_common import bytetrack_script
    from oracle import byte_tracker as obt

    g = _load("bytetrack.npz")
    t = obt.BYTETracker(**BYTE_PARAMS[tag])
    off = so = 0
    assert g[f"{tag}_rows"][:, 4].max() > 30 and (g[f"{tag}_state"] == obt.LOST).sum() > 50         # the script exercises lost / re-found tracks
    for f, d in enumerate(bytetrack_script()):
        r = t.update(_xywh(d), d[:, 4], d[:, 5]).reshape(-1, 8)
        n = int(g[f"{tag}_counts"][f])
        ref = g[f"{tag}_rows"][off:off + n]
        off += n
        assert len(r) == n, (f, len(r), n)
        assert np.array_equal(r[:, 4:], ref[:, 4:]), f
        np.testing.assert_allclose(r[:, :4], ref[:, :4], rtol=0, atol=1e-4)
        st = sorted(((q.track_id, q.state, q.mean, np.diag(q.covariance)) for q in t.tracked_stracks + t.lost_stracks), key=lambda q: q[0])
        ns = int(g[f"{tag}_nstate"][f])
        assert [q[0] for q in st] == list(g[f"{tag}_ids"][so:so + ns]) and [q[1] for q in st] == list(g[f"{tag}_state"][so:so + ns]), f
        if ns:
            np.testing.assert_allclose(np.array([q[2] for q in st]), g[f"{tag}_mean"][so:so + ns], rtol=1e-8, atol=1e-5)
            np.testing.assert_allclose(np.array([q[3] for q in st]), g[f"{tag}_cov_diag"][so:so + ns], rtol=1e-7, atol=1e-9)
        so += ns


def test_linear_assignment_oracle_cases():
    """matching.linear_assignment(cost, thresh) through the reference module (its default lap branch, `lap` = the restated
    extended-matrix problem) on rectangular random costs; every match respects the limit and the restated optimum is not beaten by
    a brute-force search on the small case."""
    import itertools

    from oracle import byte_tracker as obt

    g = _load("bytetrack.npz")
    for k in range(5):
        c, x, th = g[f"lap{k}_cost"], g[f"lap{k}_x"], float(g[f"lap{k}_thresh"])
        _, x2, _ = obt.lapjv(c, extend_cost=True, cost_limit=th)
        assert np.array_equal(x, x2)
        assert all(c[i, j] <= th for i, j in enumerate(x) if j >= 0)
    c, x, th = g["lap0_cost"], g["lap0_x"], float(g["lap0_thresh"])         # 5 x 7: brute force over partial matchings
    n, m = c.shape
    best = min(sum((c[i, j] - th) for i, j in enumerate(p) if j >= 0)
               for p in itertools.product(range(-1, m), repeat=n) if len({j for j in p if j >= 0}) == sum(j >= 0 for j in p))
    got = sum((c[i, j] - th) for i, j in enumerate(x) if j >= 0)
    assert abs(got - best) < 1e-9


@pytest.mark.parametrize("tag,use_img", [("botsort", True), ("botsort_nogmc", False)])
def test_botsort_oracle_matches_reference(tag, use_img):
    """oracle.byte_tracker.BOTSORT (bot_sort.py without ReID: XYWH filter, sparse-optical-flow GMC through the same OpenCV calls)
    against the reference's BOTSORT.update over the shaking-camera scene, with and without the frames."""
    from golden_common import botsort_scene
    from oracle import byte_tracker as obt

    g = _load("bytetrack.npz")
    frames, dets = botsort_scene()
    t = obt.BOTSORT()
    off = 0
    assert not np.array_equal(g["botsort_counts"], g["botsort_nogmc_counts"])          # the compensation changes the outcome
    for f, d in enumerate(dets):
        r = t.update(_xywh(d), d[:, 4], d[:, 5], frames[f] if use_img else None).reshape(-1, 8)
        n = int(g[f"{tag}_counts"][f])
        ref = g[f"{tag}_rows"][off:off + n]
        off += n
        assert len(r) == n and np.array_equal(r[:, 4:], ref[:, 4:]), f
        np.testing.assert_allclose(r[:, :4], ref[:, :4], rtol=0, atol=1e-4)


def test_motion_tracker_with_frames_matches_reference():
    """oracle.motion_reset.MotionCompensatedMultiTracker.update(detections, frame) -- the restated GlobalMotionDetector (optical
    flow through the same OpenCV calls) and global-reset rules -- against the reference on the drifting / jolting camera scene:
    motion magnitude, global resets, track counts and per-track state every frame."""
    pytest.importorskip("cv2")
    from golden_common import motion_frames_scene
    from oracle.motion_reset import MotionCompensatedMultiTracker

    g = _load("motion_frames.npz")
    rows, counts, stats = g["rows"], g["counts"], g["stats"]
    assert stats[3] >= 2 and stats[4] > stats[3]
    frames, script = motion_frames_scene()
    trk = MotionCompensatedMultiTracker(150, 1, 0.1)
    k = 0
    for f, dets in enumerate(script):
        res = trk.update([list(r) for r in dets], frames[f])
        assert len(res) == counts[f], f"frame {f}"
        assert abs((trk.frame_motion_info["magnitude"] if trk.frame_motion_info else 0.0) - g["magnitude"][f]) < 1e-9
        assert trk.stats["global_resets"] == g["global_resets"][f]
        for info, t in zip(res, trk.trackers):
            got = np.concatenate([np.asarray(info["bbox"], np.float64), t.x, [info["confidence"], t.reset_count, t.age, t.hits, t.hit_streak,
                                  t.time_since_update, float(t.is_lost), t.lost_frames, t.motion_consistency, info["frames_since_reset"]]])
            np.testing.assert_allclose(got, rows[k], rtol=1e-11, atol=1e-8, err_msg=f"frame {f}")
            k += 1
    assert k == len(rows)
    assert [trk.stats[n] for n in ("total_frames", "individual_resets", "tracking_recoveries", "global_resets", "global_motion_events")] == [int(v) for v in stats]

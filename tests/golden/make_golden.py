"""Generate the golden vectors in this directory by running the UNMODIFIED reference in-process.

Runs only where /root/reference exists (the build container):
    python tests/golden/make_golden.py
Inputs are seeded numpy data from the package's own recipes (``synth``, ``weights``), so the tests can
regenerate them anywhere; only the reference's OUTPUTS are stored (small .npz files).

Files written:
  tracker_seq_f32.npz / tracker_seq_f64.npz   EnhancedMultiTargetTracker over a 260-frame multi-target
                                              sequence (float32 resp. python-float detections); the per-frame
                                              Kalman states (x, P) in tracker_seq_{f32,f64}_states.npz
  tracker_kat.npz                             the 3-frame known-answer case of SURVEY.md 8c
  kf_ultra.npz                                KalmanFilterXYAH / XYWH initiate/predict/update/gating
  nms_cases.npz                               non_max_suppression, both branches (TorchNMS.nms / torchvision)
  net_n_p2_small.npz                          yolov8n-p2 head maps + decoded tensor on a 64x96 input
  bytetrack.npz                               BYTETracker.update over a scripted 90-frame scene (two parameterisations) + linear_assignment cases
  overlay.npz                                 TrajectoryVisualizer.draw_tracks over a scripted 14-frame scene (annotated frames)
  predict_n_p2.npz / predict_s_p2.npz         YOLO(cfg).predict on 512x640 (and 500x640) frames + the NMS candidate lists
  results_exports.npz                         Results.summary / save_txt / plot digests (golden_common.results_exports)
"""
import contextlib
import importlib.util
import io
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = "/root/reference"
sys.path.insert(0, ROOT)
sys.path.insert(0, REF)
os.environ.setdefault("YOLO_CONFIG_DIR", "/tmp/ycfg")
os.environ.setdefault("OMP_NUM_THREADS", "8")

import numpy as np
import torch

import b200dt  # noqa: F401
from b200dt import cfg, synth, weights

sys.path.insert(0, os.path.dirname(HERE))
from golden_common import pack_tracks, synth_pred  # noqa: E402

def run_tracker(dets_per_frame, as_python_floats, params):
    from kalman.enhanced_multi_target_tracker import EnhancedMultiTargetTracker

    with contextlib.redirect_stdout(io.StringIO()):
        trk = EnhancedMultiTargetTracker(*params)
        outs, states = [], []
        for d in dets_per_frame:
            dd = [[float(v) for v in row] for row in d] if as_python_floats else [row for row in d]
            res = trk.update(dd)
            # deep-copy what get_track_info returned (velocity is a view of x)
            outs.append([{**t, "bbox": np.array(t["bbox"]), "velocity": np.array(t["velocity"])} for t in res])
            states.append([(int(t.track_id[1:]), t.x.copy(), t.P.copy(), t.lost_frames, t.is_lost) for t in trk.trackers])
    return trk, outs, states


def gold_tracker():
    params = (150, 1, 0.1)
    seq = synth.DetectionSequence(seed=3, n_targets=8)
    dets = [seq.step() for _ in range(260)]
    for tag, pyf in (("f32", False), ("f64", True)):
        trk, outs, states = run_tracker(dets, pyf, params)
        rows, cols, tl, tr = pack_tracks(outs)
        st_rows = []
        for f, st in enumerate(states):
            for tid, x, P, lf, il in st:
                st_rows.append(np.r_[f, tid, x, P.reshape(-1), lf, float(il)])
        stats = trk.get_statistics()
        # the per-frame Kalman states go to a file of their own: together with the rows they exceed 1 MB
        np.savez_compressed(os.path.join(HERE, f"tracker_seq_{tag}_states.npz"), states=np.asarray(st_rows))
        np.savez_compressed(os.path.join(HERE, f"tracker_seq_{tag}.npz"), rows=rows, cols=np.array(cols), traj_len=tl,
                            traj=tr.astype(np.float32),
                            stats=np.array([stats[k] for k in ("total_tracks_created", "total_tracks_terminated",
                                                               "current_active_tracks", "long_term_predictions",
                                                               "successful_recoveries", "frame_count")]),
                            params=np.array(params), seed=3, n_frames=260)
        print("tracker", tag, rows.shape, "tracks created", stats["total_tracks_created"], "terminated", stats["total_tracks_terminated"],
              "recoveries", stats["successful_recoveries"], "ltp", stats["long_term_predictions"])
    # second parameterisation: (40, 3, 0.3): min_hits gating, deletions after 40 lost frames
    seq = synth.DetectionSequence(seed=11, n_targets=12, p_detect=0.7, clutter=0.5, burst=(50, 110))
    dets = [seq.step() for _ in range(200)]
    trk, outs, states = run_tracker(dets, False, (40, 3, 0.3))
    rows, cols, tl, tr = pack_tracks(outs)
    np.savez_compressed(os.path.join(HERE, "tracker_seq_default.npz"), rows=rows, cols=np.array(cols), traj_len=tl,
                        traj=tr.astype(np.float32), params=np.array((40, 3, 0.3)), seed=11, n_frames=200,
                        stats=np.array([trk.stats[k] for k in ("total_tracks_created", "total_tracks_terminated",
                                                               "current_active_tracks", "long_term_predictions",
                                                               "successful_recoveries")] + [trk.frame_count]))
    print("tracker default", rows.shape, trk.stats)
    # known-answer (SURVEY 8c)
    kat = [[[10, 10, 20, 20, .9], [100, 100, 110, 112, .5]], [[11, 11, 21, 21, .9]], [[12, 12, 22, 22, .9]]]
    trk, outs, states = run_tracker(kat, True, (150, 1, 0.1))
    rows, cols, tl, tr = pack_tracks(outs)
    st = states[-1]
    np.savez_compressed(os.path.join(HERE, "tracker_kat.npz"), rows=rows, cols=np.array(cols),
                        x_T001=st[0][1], P_T001=st[0][2], x_T002=st[1][1], P_T002=st[1][2])
    print("kat T001 x", st[0][1])


def gold_kf():
    spec = importlib.util.spec_from_file_location("ref_kf", os.path.join(REF, "ultralytics/trackers/utils/kalman_filter.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    g = np.random.default_rng(5)
    out = {}
    for kind, cls in (("xyah", mod.KalmanFilterXYAH), ("xywh", mod.KalmanFilterXYWH)):
        kf = cls()
        N, T = 16, 12
        if kind == "xyah":
            z0 = np.stack([g.uniform(50, 600, N), g.uniform(50, 400, N), g.uniform(0.3, 2.0, N), g.uniform(10, 120, N)], 1)
        else:
            z0 = np.stack([g.uniform(50, 600, N), g.uniform(50, 400, N), g.uniform(8, 90, N), g.uniform(10, 120, N)], 1)
        meas = z0[None] + np.cumsum(g.normal(0, 1.0, (T, N, 4)) * np.array([2, 2, 0.01 if kind == "xyah" else 1, 1]), 0)
        hit = g.random((T, N)) < 0.75
        means, covs = zip(*[kf.initiate(z) for z in z0])
        means, covs = np.array(means), np.array(covs)
        out[f"{kind}_z0"], out[f"{kind}_meas"], out[f"{kind}_hit"] = z0, meas, hit
        out[f"{kind}_init_mean"], out[f"{kind}_init_cov"] = means.copy(), covs.copy()
        mh, ch, gh = [], [], []
        for t in range(T):
            pm, pc = kf.multi_predict(means, covs)
            # per-track predict must agree with multi_predict (reference property)
            for i in range(N):
                a, b = kf.predict(means[i], covs[i])
                assert np.allclose(a, pm[i]) and np.allclose(b, pc[i])
            means, covs = pm.copy(), pc.copy()
            gd = np.stack([kf.gating_distance(means[i], covs[i], meas[t]) for i in range(N)])
            gd_pos = np.stack([kf.gating_distance(means[i], covs[i], meas[t], only_position=True) for i in range(N)])
            for i in range(N):
                if hit[t, i]:
                    means[i], covs[i] = kf.update(means[i], covs[i], meas[t, i])
            mh.append(means.copy()); ch.append(covs.copy()); gh.append(np.stack([gd, gd_pos]))
        out[f"{kind}_means"], out[f"{kind}_covs"], out[f"{kind}_gating"] = np.array(mh), np.array(ch), np.array(gh)
    # survey known answers
    kf = mod.KalmanFilterXYWH()
    m, c = kf.initiate(np.array([100., 50, 20, 40])); m, c = kf.predict(m, c); m2, c2 = kf.update(m, c, np.array([102., 51, 21, 41]))
    out["kat_xywh_mean"], out["kat_xywh_diag"] = m2, np.diag(c2)
    out["kat_xywh_gate"] = kf.gating_distance(m, c, np.array([[102., 51, 21, 41], [107., 56, 26, 46]]))
    np.savez_compressed(os.path.join(HERE, "kf_ultra.npz"), **out)
    print("kf", {k: v.shape for k, v in out.items() if "means" in k}, out["kat_xywh_gate"])


def _nms_both(pred, conf, iou, **kw):
    from ultralytics.utils.nms import non_max_suppression

    res = {}
    tv = sys.modules.pop("torchvision", None)
    try:
        assert "torchvision" not in sys.modules
        res["legacy"] = non_max_suppression(pred.clone(), conf, iou, **kw)
    finally:
        if tv is not None:
            sys.modules["torchvision"] = tv
    import torchvision  # noqa: F401

    res["exact"] = non_max_suppression(pred.clone(), conf, iou, **kw)
    return res


def gold_nms():
    out = {}
    cases = [dict(seed=0, B=2, nc=80, A=800, conf=0.15, iou=0.6, frac=0.05), dict(seed=1, B=1, nc=1, A=1200, conf=0.15, iou=0.6),
             dict(seed=2, B=3, nc=4, A=600, conf=0.25, iou=0.45), dict(seed=3, B=1, nc=2, A=3000, conf=0.05, iou=0.7, max_det=50),
             dict(seed=4, B=1, nc=80, A=500, conf=0.15, iou=0.6, agnostic=True),
             dict(seed=5, B=1, nc=80, A=500, conf=0.15, iou=0.6, classes=[0, 3, 7])]
    for ci, c in enumerate(cases):
        pred = synth_pred(c["seed"], c["B"], c["nc"], c["A"], frac=c.get("frac", 0.15))
        kw = {k: c[k] for k in ("max_det", "agnostic", "classes") if k in c}
        res = _nms_both(torch.from_numpy(pred), c["conf"], c["iou"], **kw)
        for mode, lst in res.items():
            for b, det in enumerate(lst):
                out[f"c{ci}_{mode}_{b}"] = det.numpy()
        out[f"c{ci}_cfg"] = np.array([c["seed"], c["B"], c["nc"], c["A"], c["conf"], c["iou"], c.get("max_det", 300),
                                      float(c.get("agnostic", False))])
        if "classes" in c:
            out[f"c{ci}_classes"] = np.array(c["classes"])
        print("nms case", ci, {m: [len(d) for d in l] for m, l in res.items()})
    # SURVEY 8c hand cases through TorchNMS.nms / torchvision.ops.nms directly
    from ultralytics.utils.nms import TorchNMS
    import torchvision
    b = torch.tensor([[200., 200, 210, 210], [0, 0, 10, 10], [0, 0, 10, 10.5]]); s = torch.tensor([.9, .8, .7])
    out["hand_div_legacy"] = TorchNMS.nms(b, s, 0.6).numpy(); out["hand_div_exact"] = torchvision.ops.nms(b, s, 0.6).numpy()
    np.savez_compressed(os.path.join(HERE, "nms_cases.npz"), **out)
    print("hand", out["hand_div_legacy"], out["hand_div_exact"])


def _ref_model(name, seed=0):
    from ultralytics.nn.tasks import DetectionModel

    spec = cfg.resolve(name)
    sd = weights.synthetic_state_dict(spec, seed=seed)
    m = DetectionModel(name + ".yaml", ch=3, nc=spec["nc"], verbose=False).eval()
    m.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in sd.items()})
    return spec, sd, m


def gold_net():
    spec, sd, m = _ref_model("yolov8n-p2")
    x = np.random.default_rng(0).random((1, 3, 64, 96), dtype=np.float32)
    m.fuse()   # the predict path always runs the BN-folded graph (AutoBackend(fuse=True))
    feats = {}
    hooks = [m.model[i].register_forward_hook(lambda mod, inp, out, i=i: feats.__setitem__(i, out.detach().numpy().copy()))
             for i in (0, 2, 9, 18, 27)]
    with torch.no_grad():
        y, heads = m(torch.from_numpy(x))
    for h in hooks:
        h.remove()
    np.savez_compressed(os.path.join(HERE, "net_n_p2_small.npz"), y=y.numpy(), **{f"head{i}": h.numpy() for i, h in enumerate(heads)},
                        **{f"layer{i}": v for i, v in feats.items()})
    print("net", y.shape, [h.shape for h in heads])


def gold_predict(names=("yolov8n-p2", "yolov8s-p2", "yolov8-small")):
    """YOLO(cfg).predict of the unmodified reference (fp32, CPU) on synthetic IR frames, both NMS branches, plus the
    candidate list the NMS saw (every anchor with best-class score > conf, boxes in original-frame pixels): the tests
    derive their exclusion band (near-ties an fp32-vs-bf16 comparison cannot decide) from it."""
    from ultralytics import YOLO
    from ultralytics.utils import ops as uops

    for name in names:
        spec = cfg.resolve(name)
        sd = weights.synthetic_state_dict(spec, seed=0)
        out = {}
        shapes = (("512x640", (512, 640)), ("500x640", (500, 640))) if name == "yolov8n-p2" else (("512x640", (512, 640)),)
        for tag, (h, w) in shapes:
            frames = [synth.IRStream(seed=7, h=h, w=w).frame(), synth.IRStream(seed=8, h=h, w=w).frame()]
            f3 = synth.IRStream(seed=1001, h=h, w=w)            # a later frame of a third stream
            frames.append([f3.frame() for _ in range(4)][-1])
            for mode in ("legacy", "exact"):
                tv = sys.modules.pop("torchvision", None) if mode == "legacy" else None
                try:
                    if mode == "exact":
                        import torchvision  # noqa: F401
                    yolo = YOLO(name + ".yaml", verbose=False)
                    yolo.model.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in sd.items()})
                    res = yolo.predict(frames, conf=0.15, iou=0.6, device="cpu", verbose=False)
                finally:
                    if tv is not None:
                        sys.modules["torchvision"] = tv
                for b, r in enumerate(res):
                    out[f"{tag}_{mode}_{b}"] = r.boxes.data.numpy()
                    assert r.orig_shape == (h, w)
                print("predict", name, tag, mode, [len(r.boxes) for r in res])
            # candidates of the fp32 reference (the predictor's own preprocess + inference, then nms.py:74-113 by hand)
            pr = yolo.predictor
            im = pr.preprocess([f.copy() for f in frames])
            with torch.no_grad():
                preds = pr.inference(im)
            y = preds[0] if isinstance(preds, (list, tuple)) else preds
            for b in range(len(frames)):
                yb = y[b].T                                       # (A, 4 + nc)
                sc, cl = yb[:, 4:].max(1)
                keep = sc > 0.15
                box = uops.xywh2xyxy(yb[keep, :4])
                # NMS runs on the letterboxed, UNCLIPPED boxes (clip_boxes comes after it, ops.py:105-138): the candidates are
                # stored in original-frame coordinates without the clip; these frames need no resize (gain 1)
                gain = min(im.shape[2] / h, im.shape[3] / w)
                assert gain == 1.0
                pad_x, pad_y = round((im.shape[3] - w) / 2 - 0.1), round((im.shape[2] - h) / 2 - 0.1)
                box = box - torch.tensor([pad_x, pad_y, pad_x, pad_y], dtype=box.dtype)
                out[f"{tag}_cand_{b}"] = torch.cat([box, sc[keep, None], cl[keep, None].float()], 1).numpy()
        np.savez_compressed(os.path.join(HERE, f"predict_{name[6:].strip('-').replace('-', '_')}.npz"), **out)


def motion_reset_script(n=140, seed=11):
    """One target: smooth drift, a 70 px jump (camera shake), a second jump inside the cooldown, a size jump, two detection
    gaps (one of them right after a reset), noise of 0.5 px.  Returns a list of bbox-or-None per frame."""
    rng = np.random.default_rng(seed)
    cx, cy, w, h = 120.0, 90.0, 14.0, 10.0
    out = []
    for t in range(n):
        cx += 1.5; cy += 0.7
        if t == 30: cx += 70.0                       # position jump
        if t == 36: cy -= 55.0                       # inside the cooldown of the first reset
        if t == 60: w *= 1.6; h *= 1.5               # size jump
        if t == 85: cx -= 48.0; cy += 30.0           # jump + velocity change
        if t == 110: cx += 200.0                     # large jump (factor capped at 2)
        miss = (44 <= t < 49) or (86 <= t < 90) or (t % 23 == 22)
        n4 = rng.normal(0.0, 0.5, 4)
        out.append(None if miss else [float(cx - w / 2 + n4[0]), float(cy - h / 2 + n4[1]), float(cx + w / 2 + n4[2]), float(cy + h / 2 + n4[3])])
    return out


def gold_motion_reset():
    """camera_motion_compensation/motion_reset_kalman_tracker.py driven frame by frame the way the multi-tracker drives a
    track: predict(); update(det) or mark_as_lost(); get_track_info()."""
    sys.path.insert(0, REF)
    from camera_motion_compensation.motion_reset_kalman_tracker import MotionResetKalmanTracker

    script = motion_reset_script()
    rows = []
    with contextlib.redirect_stdout(io.StringIO()):
        trk = MotionResetKalmanTracker(script[0], track_id="T001", max_lost_frames=150)
        for det in script[1:]:
            pb = np.asarray(trk.predict(), np.float64)
            if det is not None:
                trk.update(det)
            else:
                trk.mark_as_lost()
            info = trk.get_track_info()
            rows.append(np.concatenate([pb, trk.x, trk.P.ravel(), np.asarray(info["bbox"], np.float64),
                                        [info["confidence"], trk.reset_count, trk.last_reset_frame, trk.age, trk.hits, trk.hit_streak,
                                         trk.time_since_update, float(trk.is_lost), trk.lost_frames, trk.motion_consistency,
                                         len(trk.position_history), len(trk.motion_scores), info["frames_since_reset"]]]))
    rows = np.array(rows)
    np.savez_compressed(os.path.join(HERE, "motion_reset.npz"), rows=rows,
                        dets=np.array([d if d is not None else [np.nan] * 4 for d in script]))
    print("motion_reset", rows.shape, "resets", int(rows[-1, 4 + 8 + 64 + 4 + 1]))


def motion_multi_script(n=160, seed=21):
    """Multi-target detections (synth.DetectionSequence) with camera shakes: at a few frames every detection of the frame and of
    all later frames is shifted by a common offset (what a panning / shaking camera does), python floats."""
    seq = synth.DetectionSequence(seed=seed, n_targets=6, p_detect=0.9, clutter=0.15, burst=(70, 85))
    # boxes are blown up 3x (12..72 px) so that a 45 px shake still overlaps the predicted box (IoU > 0.1: the track is matched
    # and its jump detector fires) while smaller ones lose the association and found new tracks
    shakes = {25: (45.0, 0.0), 26: (10.0, -8.0), 60: (-32.0, 34.0), 95: (0.0, 44.0), 130: (-43.0, -10.0), 132: (-6.0, 2.0)}
    off = np.zeros(2)
    out = []
    for t in range(n):
        if t in shakes:
            off = off + np.array(shakes[t])
        d = seq.step().astype(np.float64)
        if len(d):
            cx, cy = (d[:, 0] + d[:, 2]) / 2, (d[:, 1] + d[:, 3]) / 2
            hw, hh = 1.5 * (d[:, 2] - d[:, 0]), 1.5 * (d[:, 3] - d[:, 1])
            if t == 100:
                hw, hh = hw * 1.5, hh * 1.5                      # zoom: size-change detector
            d[:, 0], d[:, 2] = cx - hw + off[0], cx + hw + off[0]
            d[:, 1], d[:, 3] = cy - hh + off[1], cy + hh + off[1]
        out.append([[float(v) for v in r] for r in d])
    return out


def gold_motion_multi():
    """camera_motion_compensation/motion_compensated_multi_tracker.py, update(detections) without a frame."""
    sys.path.insert(0, REF)
    from camera_motion_compensation.motion_compensated_multi_tracker import MotionCompensatedMultiTracker

    script = motion_multi_script()
    rows, counts = [], []
    with contextlib.redirect_stdout(io.StringIO()):
        trk = MotionCompensatedMultiTracker(150, 1, 0.1)
        for dets in script:
            res = trk.update([list(r) for r in dets])
            assert len(res) == len(trk.trackers)
            counts.append(len(res))
            for info, t in zip(res, trk.trackers):
                rows.append(np.concatenate([np.asarray(info["bbox"], np.float64), t.x, [info["confidence"], t.reset_count, t.age, t.hits,
                                            t.hit_streak, t.time_since_update, float(t.is_lost), t.lost_frames, t.motion_consistency,
                                            info["frames_since_reset"]]]))
    stats = [trk.stats["total_frames"], trk.stats["individual_resets"], trk.stats["tracking_recoveries"], trk.stats["global_resets"]]
    flat = np.array([[v for r in dets for v in r] + [np.nan] * (5 * 16 - 5 * len(dets)) for dets in script])
    np.savez_compressed(os.path.join(HERE, "motion_multi.npz"), rows=np.array(rows), counts=np.array(counts), stats=np.array(stats),
                        dets=flat, ndets=np.array([len(d) for d in script]))
    print("motion_multi", np.array(rows).shape, "stats", stats, "max tracks", max(counts))


def gold_motion_frames():
    """camera_motion_compensation/motion_compensated_multi_tracker.py, update(detections, frame): the GlobalMotionDetector (optical
    flow, OpenCV) on a shaking / jolting camera scene, global resets included."""
    sys.path.insert(0, REF)
    from camera_motion_compensation.motion_compensated_multi_tracker import MotionCompensatedMultiTracker

    from golden_common import motion_frames_scene

    frames, script = motion_frames_scene()
    rows, counts, mags, resets = [], [], [], []
    with contextlib.redirect_stdout(io.StringIO()):
        trk = MotionCompensatedMultiTracker(150, 1, 0.1)
        for f, dets in enumerate(script):
            res = trk.update([list(r) for r in dets], frames[f])
            assert len(res) == len(trk.trackers)
            counts.append(len(res))
            mags.append(trk.frame_motion_info["magnitude"] if trk.frame_motion_info else 0.0)
            resets.append(trk.stats["global_resets"])
            for info, t in zip(res, trk.trackers):
                rows.append(np.concatenate([np.asarray(info["bbox"], np.float64), t.x, [info["confidence"], t.reset_count, t.age, t.hits,
                                            t.hit_streak, t.time_since_update, float(t.is_lost), t.lost_frames, t.motion_consistency,
                                            info["frames_since_reset"]]]))
    stats = [trk.stats["total_frames"], trk.stats["individual_resets"], trk.stats["tracking_recoveries"], trk.stats["global_resets"],
             trk.stats["global_motion_events"]]
    np.savez_compressed(os.path.join(HERE, "motion_frames.npz"), rows=np.array(rows), counts=np.array(counts), stats=np.array(stats),
                        magnitude=np.array(mags), global_resets=np.array(resets))
    print("motion_frames", np.array(rows).shape, "stats", stats, "max magnitude", max(mags))


def gold_bytetrack():
    """The reference's BYTETracker (ultralytics/trackers/byte_tracker.py) over the scripted scene, default bytetrack.yaml values and a
    second parameterisation (no score fusion, short buffer).  `lap` (gatagat/lap) is not installed here: matching.py's import
    is satisfied by a module whose lapjv is oracle.byte_tracker.lapjv (the restated extended-matrix problem solved by scipy)."""
    import types

    from golden_common import bytetrack_script
    from oracle import byte_tracker as obt

    lap = types.ModuleType("lap")
    lap.__version__ = "0.5.12"
    lap.lapjv = obt.lapjv
    sys.modules["lap"] = lap
    from ultralytics.engine.results import Boxes
    from ultralytics.trackers.byte_tracker import BYTETracker
    from ultralytics.utils import IterableSimpleNamespace

    out = {}
    frames = bytetrack_script()
    for tag, args in (("default", dict(track_high_thresh=0.25, track_low_thresh=0.1, new_track_thresh=0.25, track_buffer=30, match_thresh=0.8, fuse_score=True)),
                      ("nofuse", dict(track_high_thresh=0.4, track_low_thresh=0.15, new_track_thresh=0.5, track_buffer=8, match_thresh=0.7, fuse_score=False))):
        trk = BYTETracker(IterableSimpleNamespace(tracker_type="bytetrack", **args), frame_rate=30)
        rows, counts, states = [], [], []
        for f, d in enumerate(frames):
            r = trk.update(Boxes(d, (512, 640)).numpy())
            r = np.asarray(r, dtype=np.float32).reshape(-1, 8)
            rows.append(r); counts.append(len(r))
            # filter state of every live track, by id (means / covariances are float64 in the reference)
            st = sorted(((t.track_id, t.state, t.mean, t.covariance) for t in trk.tracked_stracks + trk.lost_stracks), key=lambda q: q[0])
            states.append((np.array([q[0] for q in st]), np.array([q[1] for q in st]), np.array([q[2] for q in st], dtype=np.float64).reshape(-1, 8),
                           np.array([q[3] for q in st], dtype=np.float64).reshape(-1, 8, 8)))
        out[f"{tag}_rows"] = np.concatenate(rows) if rows else np.zeros((0, 8), np.float32)
        out[f"{tag}_counts"] = np.array(counts)
        out[f"{tag}_ids"] = np.concatenate([s[0] for s in states]); out[f"{tag}_nstate"] = np.array([len(s[0]) for s in states])
        out[f"{tag}_state"] = np.concatenate([s[1] for s in states]); out[f"{tag}_mean"] = np.concatenate([s[2] for s in states])
        out[f"{tag}_cov_diag"] = np.concatenate([np.diagonal(s[3], axis1=1, axis2=2) for s in states])
    # linear_assignment known answers on random rectangular costs (the default lap branch through the same module)
    from ultralytics.trackers.utils import matching

    g = np.random.default_rng(3)
    for k, (n, m, th) in enumerate([(5, 7, 0.8), (12, 9, 0.5), (1, 6, 0.7), (20, 20, 0.9), (30, 4, 0.6)]):
        c = g.uniform(0, 1, (n, m)).astype(np.float32)
        mt, ua, ub = matching.linear_assignment(c, th)
        x = np.full(n, -1); 
        for i, j in mt:
            x[i] = j
        out[f"lap{k}_cost"] = c; out[f"lap{k}_x"] = x; out[f"lap{k}_thresh"] = np.float32(th)
    # BoT-SORT (bot_sort.py) without ReID, botsort.yaml defaults: XYWH filter + sparse-optical-flow GMC driven by the frames
    from golden_common import botsort_scene
    from ultralytics.trackers.bot_sort import BOTSORT

    frames_b, dets_b = botsort_scene()
    bargs = dict(tracker_type="botsort", track_high_thresh=0.25, track_low_thresh=0.1, new_track_thresh=0.25, track_buffer=30, match_thresh=0.8,
                 fuse_score=True, gmc_method="sparseOptFlow", proximity_thresh=0.5, appearance_thresh=0.8, with_reid=False, model="auto")
    for tag, use_img in (("botsort", True), ("botsort_nogmc", False)):
        trk = BOTSORT(IterableSimpleNamespace(**bargs), frame_rate=30)
        rows, counts, warps = [], [], []
        for f, d in enumerate(dets_b):
            r = np.asarray(trk.update(Boxes(d, frames_b[f].shape[:2]).numpy(), frames_b[f] if use_img else None), dtype=np.float32).reshape(-1, 8)
            rows.append(r); counts.append(len(r))
        out[f"{tag}_rows"] = np.concatenate(rows); out[f"{tag}_counts"] = np.array(counts)
    np.savez_compressed(os.path.join(HERE, "bytetrack.npz"), **out)


def gold_overlay():
    """kalman/trajectory_visualizer.py TrajectoryVisualizer.draw_tracks over the scripted scene: the pixels of every frame."""
    from golden_common import overlay_scene
    spec = importlib.util.spec_from_file_location("ref_trajectory_visualizer", os.path.join(REF, "kalman", "trajectory_visualizer.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    vis = mod.TrajectoryVisualizer()
    out = []
    for image, tracks, dets, info in overlay_scene():
        keep = image.copy()
        out.append(vis.draw_tracks(image, tracks, dets, info))
        assert np.array_equal(image, keep)
    import hashlib
    digests = np.array([hashlib.sha256(np.ascontiguousarray(o).tobytes()).hexdigest() for o in out])
    full = [0, 5, 8]                # whole frames for three of them (a failing digest can then be looked at), digests for all
    np.savez_compressed(os.path.join(HERE, "overlay.npz"), digests=digests, full_index=np.array(full), full=np.stack([out[i] for i in full]))


def gold_results_exports():
    """ultralytics/engine/results.py Results.summary / save_txt / plot over the fixed boxes of golden_common.results_exports."""
    from golden_common import results_exports
    from ultralytics.engine.results import Results

    out = results_exports(lambda img, path, names, data: Results(img, path, names, boxes=torch.as_tensor(data)))
    np.savez_compressed(os.path.join(HERE, "results_exports.npz"), **{k: np.array(v) for k, v in out.items()})


if __name__ == "__main__":
    which = sys.argv[1:] or ["tracker", "kf", "nms", "net", "predict"]
    for w in which:
        globals()["gold_" + w]()
    for f in sorted(os.listdir(HERE)):
        if f.endswith(".npz"):
            print(f, os.path.getsize(os.path.join(HERE, f)) // 1024, "KiB")

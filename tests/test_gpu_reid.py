"""GPU parity of BoT-SORT ReID on the detector's own features (botsort.yaml ``with_reid: True``, ``model: auto``): the embedding
gather against get_obj_feats, the combined BoT-SORT cost against its float64 restatement, the float64 assignment solver against
lapjv, BOTSORT(with_reid=True) against the oracle tracker on a scripted crossing scene, and YOLO.track end to end."""
import numpy as np
import pytest

import b200dt  # noqa: F401
from b200dt import cfg, synth, weights
from oracle import byte_tracker as obt
from oracle import net as onet
from oracle import postprocess as pp
from oracle import reid as oreid

pytestmark = pytest.mark.gpu


def _torch():
    import torch

    return torch


def _gather(levels, idx, counts, s):
    """b2_reid_gather over ``levels`` ((ptr, h, w, cstride, coff, C) per level) into a NaN-filled [B][K][s] tensor."""
    import ctypes as C

    from b200dt import _lib

    torch = _torch()
    B, K = idx.shape
    out = torch.full((B, K, s), float("nan"), device="cuda")
    n = len(levels)
    arr = lambda k: (C.c_int * n)(*[lv[k] for lv in levels])
    di = torch.as_tensor(np.ascontiguousarray(idx, np.int32)).cuda()
    dc = torch.as_tensor(np.ascontiguousarray(counts, np.int32)).cuda()
    _lib.check(_lib.load().b2_reid_gather((C.c_void_p * n)(*[lv[0] for lv in levels]), arr(1), arr(2), arr(3), arr(4), arr(5), n,
                                          _lib.ptr(di), _lib.ptr(dc), B, K, s, _lib.ptr(out), _lib.stream_ptr()))
    return out.cpu().numpy()


def _maps(levels, B):
    """NCHW float32 copies of the Detect-input slices the levels describe (bf16 values)."""
    from b200dt.engine import _view_bf16

    return [_view_bf16(p, (B, h, w, cs))[..., co:co + c].float().permute(0, 3, 1, 2).cpu().numpy() for p, h, w, cs, co, c in levels]


def _check_rows(got, ref, counts):
    """Rows below the count equal the group means within 1e-6 of the row's magnitude; rows past it are untouched (NaN)."""
    for b, n in enumerate(counts):
        assert np.isnan(got[b, n:]).all(), b
        if n:
            r = np.asarray(ref[b], np.float32)
            scale = np.abs(r).max(axis=1, keepdims=True) + 1e-30
            assert (np.abs(got[b, :n] - r) <= 1e-6 * scale).all(), (b, float((np.abs(got[b, :n] - r) / scale).max()))


@pytest.mark.parametrize("name,B,H,W,fuse_head", [("yolov8n-p2", 3, 512, 640, True), ("yolov8s-p2", 3, 512, 640, True),
                                                  ("yolov8-small", 3, 512, 640, True), ("yolov8x-p2", 3, 320, 384, True),
                                                  ("yolov8n-p2", 3, 512, 640, False)])
def test_gather_equals_get_obj_feats_on_engine_buffers(name, B, H, W, fuse_head):
    """DetectPipeline.embed after one detect step == get_obj_feats over the engine's own bf16 Detect inputs, for the rows NMS kept
    (image 1's count forced to 0, image 2's cut short); then the kernel with hand-picked anchor ids: first and last of every level.
    yolov8-small's P2 level is 24 channels of a 32-wide padded buffer: the padding is never averaged in."""
    from b200dt.predictor import DetectPipeline

    torch = _torch()
    spec = cfg.resolve(name)
    sd = weights.synthetic_state_dict(spec, seed=0)
    pipe = DetectPipeline(spec, sd, B, H, W, max_det=300, fuse_head=fuse_head)
    frames = np.stack([synth.IRStream(seed=60 + b, h=H, w=W, n_targets=8).frame() for b in range(B)])
    pipe(torch.from_numpy(frames).cuda(), 0.05, 0.7)
    nms_counts = pipe.post.out_count.cpu().numpy()
    assert nms_counts.sum() > 0
    counts = np.array([nms_counts[0], 0, min(int(nms_counts[2]), 5)], np.int32)
    pipe.post.out_count.copy_(torch.as_tensor(counts))
    pipe.embed()
    pipe.feats.fill_(float("nan"))
    got = pipe.embed().cpu().numpy()
    levels = pipe.engine.detect_inputs()
    det = spec["layers"][-1]
    s = min(det["ch"])
    assert got.shape == (B, 300, s) and [lv[5] for lv in levels] == list(det["ch"])
    if name == "yolov8-small":
        assert any(lv[3] > lv[5] for lv in levels)                 # a padded buffer
    maps = _maps(levels, B)
    idx = pipe.post.out_idx.cpu().numpy()
    ref = oreid.get_obj_feats(maps, [idx[b, :counts[b]] for b in range(B)])
    assert isinstance(ref[1], list) and ref[1] == []
    _check_rows(got, ref, counts)
    # hand-picked anchors: the first and the last anchor of every level, in Detect order
    start = np.cumsum([0] + [h * w for _, h, w, *_ in levels])
    ids = np.array([[start[l], start[l + 1] - 1][e] for l in range(len(levels)) for e in (0, 1)], np.int32)
    K = len(ids)
    hand = np.stack([ids, ids[::-1], ids])
    hcounts = np.array([K, 0, K - 1], np.int32)
    got = _gather(levels, hand, hcounts, s)
    _check_rows(got, oreid.get_obj_feats(maps, [hand[b, :hcounts[b]] for b in range(B)]), hcounts)


@pytest.mark.parametrize("name,coff", [("yolov8n-p2", 8), ("yolov8-small", 4)])
def test_gather_on_oracle_fp32_detect_inputs(name, coff):
    """The gather fed oracle/net.py's fp32 Detect inputs (stored as bf16 slices [coff, coff + C) of wider buffers; coff = 4 breaks
    the 16-byte alignment and takes the scalar path) against get_obj_feats on the fp32 maps: rel-L2 <= 4e-3, the gate of the
    per-layer conv parity (one bf16 rounding of the input)."""
    torch = _torch()
    B, H, W = 2, 64, 96
    spec = cfg.resolve(name)
    sd = weights.synthetic_state_dict(spec, seed=0)
    net = onet.Net(onet.build_spec(name), sd, "fp32")
    net.forward(pp.preprocess([synth.IRStream(seed=70 + b, h=H, w=W, n_targets=4).frame() for b in range(B)]), record=True)
    det = spec["layers"][-1]
    maps = [net.trace[f"layer.{f}"] for f in det["f"]]
    assert [m.shape[1] for m in maps] == list(det["ch"])
    keep, levels = [], []
    for m in maps:
        c = m.shape[1]
        buf = torch.zeros((B, m.shape[2], m.shape[3], c + 16), dtype=torch.bfloat16, device="cuda")
        buf[..., coff:coff + c] = torch.from_numpy(np.ascontiguousarray(m.transpose(0, 2, 3, 1))).cuda().bfloat16()
        keep.append(buf)
        levels.append((buf.data_ptr(), m.shape[2], m.shape[3], c + 16, coff, c))
    A = sum(m.shape[2] * m.shape[3] for m in maps)
    g = np.random.default_rng(2)
    idx = np.stack([np.r_[0, A - 1, g.choice(A, 40, replace=False)] for _ in range(B)]).astype(np.int32)
    counts = np.array([42, 17], np.int32)
    s = min(det["ch"])
    got = _gather(levels, idx, counts, s)
    ref = oreid.get_obj_feats(maps, [idx[b, :counts[b]] for b in range(B)])
    for b in range(B):
        err = float(np.linalg.norm(got[b, :counts[b]] - ref[b]) / np.linalg.norm(ref[b]))
        assert err <= 4e-3, (b, err)
        assert np.isnan(got[b, counts[b]:]).all()


def test_botsort_cost_matches_float64_restatement():
    """b2_botsort_cost against get_dists restated with numpy / scipy (iou_distance, fuse_score in float32, the proximity mask in
    float32, cdist cosine in float64, the appearance gate in float64, minimum in float64) on ragged batched problems: the fused
    IoU term bit-exact, the gates exact, the embedding term within 1e-12, entries outside each problem's corner untouched.  Edge
    cases: identical / orthogonal / opposite features (cosine distance 0 / 1 / 2), an IoU distance of exactly 0.5 (the proximity
    limit), embedding costs 2e-6 either side of the appearance limit."""
    from scipy.spatial.distance import cdist

    from b200dt import _lib

    torch = _torch()
    g = np.random.default_rng(5)
    S, N, M, D = 4, 20, 30, 100
    na, nb = np.array([20, 0, 7, 13], np.int32), np.array([30, 5, 1, 29], np.int32)
    A = np.zeros((S, N, 4), np.float32)
    Bx = np.zeros((S, M, 4), np.float32)
    for s in range(S):
        c = g.uniform(50, 150, (N, 2)).astype(np.float32)
        A[s] = np.concatenate([c, c + g.uniform(20, 40, (N, 2)).astype(np.float32)], 1)
        j = g.integers(0, N, M)
        Bx[s] = A[s, j] + g.normal(0, 6, (M, 4)).astype(np.float32)
    FA = g.standard_normal((S, N, D)).astype(np.float32)
    FB = g.standard_normal((S, M, D)).astype(np.float32)
    FB[0, :N] = FA[0] + np.float32(0.3) * g.standard_normal((N, D)).astype(np.float32)      # mostly similar pairs
    # edge cases in problem 0
    A[0, 0], Bx[0, 0] = [0, 0, 10, 10], [0, 0, 10, 5]           # IoU distance exactly 0.5 in float32
    FB[0, 0] = FA[0, 0]                                          # identical -> cosine distance 0
    A[0, 1], Bx[0, 1] = [200, 200, 240, 240], [202, 201, 242, 241]
    e = np.eye(D, dtype=np.float32)
    FA[0, 1], FB[0, 1], FB[0, 2] = e[0], e[1], -e[0]              # orthogonal (1), opposite (2)
    A[0, 2], Bx[0, 3], Bx[0, 4] = [300, 300, 340, 340], [308, 300, 348, 340], [300, 308, 340, 348]     # IoU 2/3: d = 1/3
    FA[0, 2] = e[0]
    for col, off in ((3, 2e-6), (4, -2e-6)):                     # emb = (1 - cos) / 2 = 0.2 +- 2e-6
        t = np.arccos(1 - 2 * (0.2 + off))
        FB[0, col] = np.cos(t) * e[0] + np.sin(t) * e[1]
    sc = g.uniform(0.3, 1, (S, M)).astype(np.float32)
    out = {}
    for fuse in (True, False):
        cost = torch.full((S, N, M), -7.0, dtype=torch.float64, device="cuda")
        dev = lambda a: torch.as_tensor(np.ascontiguousarray(a)).cuda()
        dA, dB, dFA, dFB, dS, dna, dnb = dev(A), dev(Bx), dev(FA), dev(FB), dev(sc), dev(na), dev(nb)
        _lib.check(_lib.load().b2_botsort_cost(_lib.ptr(dA), _lib.ptr(dB), _lib.ptr(dS) if fuse else None, _lib.ptr(dna), _lib.ptr(dnb),
                                               _lib.ptr(dFA), _lib.ptr(dFB), D, S, N, M, float(np.float32(1 - 0.5)), 1 - 0.8,
                                               _lib.ptr(cost), _lib.stream_ptr()))
        out[fuse] = cost.cpu().numpy()
    for fuse, got in out.items():
        for s in range(S):
            n, m = na[s], nb[s]
            assert (got[s, n:] == -7.0).all() and (got[s, :, m:] == -7.0).all()
            if not (n and m):
                continue
            d = 1 - obt.bbox_iou_f32(A[s, :n], Bx[s, :m])
            mask = d > (1 - 0.5)
            if fuse:
                d = 1 - (1 - d) * sc[s, :m][None].repeat(n, 0)
            assert d.dtype == np.float32
            raw = np.maximum(0.0, cdist(FA[s, :n], FB[s, :m], "cosine")) / 2.0
            emb = raw.copy()
            emb[emb > (1 - 0.8)] = 1.0
            emb[mask] = 1.0
            ref = np.minimum(d, emb)
            assert ref.dtype == np.float64
            g_ = got[s, :n, :m]
            iou_side = ref == d.astype(np.float64)
            assert np.array_equal(g_[iou_side], ref[iou_side]), s          # the IoU / fused term and every gate, bit for bit
            assert np.abs(g_ - ref).max() <= 1e-12, (s, np.abs(g_ - ref).max())
        c0 = got[0]
        assert c0[0, 0] <= 1e-12 and 1 - obt.bbox_iou_f32(A[0, :1], Bx[0, :1])[0, 0] == np.float32(0.5)   # not masked at exactly 0.5
        assert c0[2, 3] > 0.3 and abs(c0[2, 4] - (0.2 - 2e-6)) < 1e-7                                     # straddling the gate


def test_linear_assignment_f64_matches_lapjv():
    """b2_linear_assignment_f64 == the restated lapjv on float64 costs, including entries 1e-10 from the threshold that the float32
    entry point rounds onto it (and so cannot separate); random rectangular problems and a ragged batch."""
    from b200dt import byte_tracker as bt

    torch = _torch()
    th = 0.8
    c = np.ones((3, 3))
    c[0, 0], c[1, 1], c[2, 2] = th - 1e-10, th + 1e-10, th - 5e-10
    m_, _, _ = bt.linear_assignment(c, th)
    assert sorted(map(tuple, m_)) == [(0, 0), (2, 2)]
    assert obt.linear_assignment(c, th)[0] == [[0, 0], [2, 2]]
    m32, _, _ = bt.linear_assignment(c.astype(np.float32), th)
    assert len(m32) == 0                                              # float32 cannot tell th - 1e-10 from th
    g = np.random.default_rng(9)
    for n, m in [(1, 7), (24, 24), (40, 17), (64, 64), (150, 300)]:
        c = g.uniform(0, 1, (n, m))
        near = g.random((n, m)) < 0.1
        c[near] = th + g.choice([-1, 1], near.sum()) * g.uniform(1e-11, 1e-9, near.sum())
        x, y = bt.linear_assignment_device(torch.as_tensor(c).cuda()[None], th)
        _, xo, yo = obt.lapjv(c, extend_cost=True, cost_limit=th)
        assert np.array_equal(x[0].cpu().numpy(), xo) and np.array_equal(y[0].cpu().numpy(), yo), (n, m)
    S, N, M = 5, 20, 30
    C = g.uniform(0, 1, (S, N, M))
    na, nb = np.array([20, 0, 5, 20, 13], np.int32), np.array([30, 7, 0, 2, 13], np.int32)
    x, y = bt.linear_assignment_device(torch.as_tensor(C).cuda(), 0.7, torch.as_tensor(na).cuda(), torch.as_tensor(nb).cuda())
    x, y = x.cpu().numpy(), y.cpu().numpy()
    for s in range(S):
        assert (x[s, na[s]:] == -1).all() and (y[s, nb[s]:] == -1).all()
        if na[s] and nb[s]:
            _, xo, yo = obt.lapjv(C[s, :na[s], :nb[s]], extend_cost=True, cost_limit=0.7)
            assert np.array_equal(x[s, :na[s]], xo) and np.array_equal(y[s, :nb[s]], yo)
        else:
            assert (x[s] == -1).all() and (y[s] == -1).all()


def reid_scene(D=32, n_frames=44, seed=1):
    """Scripted BoT-SORT scene, per frame (dets (n, 6) [x1, y1, x2, y2, conf, cls], feats (n, D) float32, target of each row).
    Targets A and B (40 x 40, 4 px apart vertically) approach each other at 4 px / frame, meet at frame 30 and bounce back: the
    Kalman prediction carries each box onto the other target with IoU above the proximity gate, so without appearance the ids
    swap.  C is occluded for frames 25-29 (lost, then re-activated), D is a low-score box in frames 10-12 and every box is
    low-score in frames 38-39 (stage 2, features smoothed there), a clutter box lives for one frame (8: an unconfirmed track that
    is removed) and another for two (14-15: confirmed in stage 3).  Features: a seeded vector per target plus noise."""
    g = np.random.default_rng(seed)
    ident = g.standard_normal((6, D)).astype(np.float32)
    T = {0: [100, 200, 4, 0, 40, 40], 1: [340, 204, -4, 0, 40, 40], 2: [80, 400, 3, -1, 30, 50], 3: [500, 80, -2, 2, 36, 30]}
    pos = {k: np.array(v[:2], np.float64) for k, v in T.items()}
    vel = {k: np.array(v[2:4], np.float64) for k, v in T.items()}
    out = []
    for f in range(n_frames):
        if f == 31:
            vel[0], vel[1] = -vel[0], -vel[1]
        rows, fe, who = [], [], []
        for k, v in T.items():
            pos[k] = pos[k] + vel[k] if f else pos[k]
            if k == 2 and 25 <= f < 30:
                continue
            conf = 0.2 if ((k == 3 and 10 <= f <= 12) or f in (38, 39)) else 0.85 - 0.01 * k
            x, y = pos[k] + g.normal(0, 0.3, 2)
            rows.append([x, y, x + v[4], y + v[5], conf, 0])
            fe.append(ident[k] + 0.15 * g.standard_normal(D))
            who.append(k)
        if f == 8 or f in (14, 15):
            x, y = (560, 450) if f == 8 else (300, 60)
            rows.append([x, y, x + 20, y + 20, 0.7, 0])
            fe.append(ident[4 if f == 8 else 5] + 0.15 * g.standard_normal(D))
            who.append(4 if f == 8 else 5)
        out.append((np.asarray(rows, np.float32), np.asarray(fe, np.float32), np.asarray(who)))
    return out


def _xywh(d):
    return np.stack([(d[:, 0] + d[:, 2]) / 2, (d[:, 1] + d[:, 3]) / 2, d[:, 2] - d[:, 0], d[:, 3] - d[:, 1]], 1).astype(np.float32)


def _targets(rows, d, who):
    """target -> track id of a frame's output rows (``idx`` counts inside the high- or low-score subset, as in the reference)."""
    conf = d[:, 4]
    high, low = conf >= 0.25, (conf > 0.1) & (conf < 0.25)
    return {int(who[np.flatnonzero(high if r[5] >= 0.25 else low)[int(r[7])]]): int(r[4]) for r in rows}


def test_botsort_reid_matches_oracle_on_crossing_scene():
    """BOTSORT(with_reid=True) against the oracle BOTSORT fed the same boxes and host-made features: every frame ids / scores /
    classes / idx bit-exact, boxes within 2e-3 px, every live track's smooth_feat within 1e-5; the oracle's decisions are far from
    any floating-point tie; the same scene without ReID swaps A's and B's ids, with ReID it does not."""
    from b200dt import byte_tracker as bt
    from b200dt.predictor import Boxes

    scene = reid_scene()
    args = dict(tracker_type="botsort", gmc_method="none", with_reid=True)
    trk, ora = bt.BOTSORT(args), oreid.BOTSORT(gmc_method="none")
    worst_box = worst_feat = 0.0
    first = last = None
    for f, (d, fe, who) in enumerate(scene):
        r = np.asarray(trk.update(Boxes(d, (512, 640)), None, fe), dtype=np.float32).reshape(-1, 8)
        o = ora.update(_xywh(d), d[:, 4], d[:, 5], None, fe).reshape(-1, 8)
        assert r.shape == o.shape, (f, r.shape, o.shape)
        assert np.array_equal(r[:, 4:], o[:, 4:]), f
        if len(r):
            worst_box = max(worst_box, float(np.abs(r[:, :4] - o[:, :4]).max()))
        live = {t.track_id: t for t in ora.tracked_stracks + ora.lost_stracks}
        mine = {t.track_id: t for t in trk.tracked_stracks + trk.lost_stracks}
        assert sorted(live) == sorted(mine), f
        for k, t in mine.items():
            assert t.smooth_feat.shape == (32,) and len(t.features) == len(live[k].features)
            worst_feat = max(worst_feat, float(np.abs(t.smooth_feat.cpu().numpy() - live[k].smooth_feat).max()))
            worst_feat = max(worst_feat, float(np.abs(t.curr_feat.cpu().numpy() - live[k].curr_feat).max()))
        if f == 25:
            first = _targets(r, d, who)
        last = _targets(r, d, who)
    assert worst_box < 2e-3, worst_box
    assert worst_feat < 1e-5, worst_feat
    # decision gaps of the oracle: GPU boxes (2e-3 px) and features (1e-5) move a cost by well under 1e-3
    assert ora.gaps["match"] > 5e-3 and ora.gaps["appearance"] > 0.1 and ora.gaps["competing"] > 0.1, ora.gaps
    assert (first[0], first[1]) == (last[0], last[1])                             # ReID keeps A and B apart
    plain = bt.BOTSORT(dict(tracker_type="botsort", gmc_method="none"))
    for f, (d, fe, who) in enumerate(scene):
        r = np.asarray(plain.update(Boxes(d, (512, 640))), dtype=np.float32).reshape(-1, 8)
        if f == 25:
            p_first = _targets(r, d, who)
    p_last = _targets(r, d, who)
    assert (p_first[0], p_first[1]) == (p_last[1], p_last[0])                    # IoU alone swaps them at the bounce
    with pytest.raises(ValueError):
        bt.BOTSORT(args).update(Boxes(scene[0][0], (512, 640)))                   # ReID without features
    with pytest.raises(NotImplementedError):
        bt.BOTSORT(dict(args, model="yolo11n-cls.pt"))


def test_yolo_track_with_reid_end_to_end(tmp_path, monkeypatch):
    """YOLO.track with BoT-SORT ReID through a dict and through a YAML file: Results carry ids, the tracker receives (n, 32) feats
    with n the frame's NMS count of a plain predict, a classifier ReID model raises; a directory of PNGs run with batch=2 hands
    the tracker the same feats as one in-memory call (the gather runs before the next forward reuses the arena); predict without
    the switch sets no feats."""
    import cv2

    from b200dt import byte_tracker as bt
    from b200dt.predictor import YOLO

    torch = _torch()
    vid = synth.IRStream(seed=11, h=512, w=640)
    frames = [vid.frame() for _ in range(5)]
    model = YOLO("yolov8n-p2.yaml")
    plain = model.predict(frames, conf=0.1)
    assert all(not hasattr(r, "feats") for r in plain)
    seen = []
    orig = bt.BOTSORT.update

    def spy(self, results, img=None, feats=None):
        seen.append(None if feats is None else feats.clone())
        return orig(self, results, img, feats)

    monkeypatch.setattr(bt.BOTSORT, "update", spy)
    res = model.track(frames, tracker={"tracker_type": "botsort", "with_reid": True, "gmc_method": "none"})
    mem = list(seen)
    yml = tmp_path / "reid.yaml"
    yml.write_text("tracker_type: botsort\nwith_reid: True\nmodel: auto\ngmc_method: none\n")
    seen.clear()
    res_y = model.track(frames, tracker=str(yml))
    from_yaml = list(seen)
    d = tmp_path / "frames"
    d.mkdir()
    for i, f in enumerate(frames):
        cv2.imwrite(str(d / f"f{i}.png"), f)
    seen.clear()
    list(model.track(str(d), tracker=str(yml), batch=2))
    from_dir = list(seen)
    assert len(mem) == len(from_yaml) == len(from_dir) == len(frames)
    for i, (p, fm, fy, fd) in enumerate(zip(plain, mem, from_yaml, from_dir)):
        assert fm.is_cuda and fm.dtype == torch.float32 and tuple(fm.shape) == (len(p), 32), (i, tuple(fm.shape), len(p))
        assert torch.equal(fm, fy) and torch.equal(fm, fd), i
    assert any(len(r) and r.boxes.is_track for r in res) and any(len(r) and r.boxes.is_track for r in res_y)
    yml.write_text("tracker_type: botsort\nwith_reid: True\nmodel: yolo11n-cls.pt\n")
    with pytest.raises(NotImplementedError):
        model.track(frames[:1], tracker=str(yml))
    yml.write_text("tracker_type: deepsort\n")
    with pytest.raises(AssertionError):
        model.track(frames[:1], tracker=str(yml))
    r = model.predict(frames[:2], conf=0.1, _feats=True)
    assert [tuple(x.feats.shape) for x in r] == [(len(p), 32) for p in plain[:2]]

"""GPU parity of the detect path (engine forward, DFL decode, NMS, predict) against the oracle and the
reference-generated golden vectors."""
import os

import numpy as np
import pytest

import b200dt  # noqa: F401
from b200dt import cfg, synth, weights
from oracle import net as onet
from oracle import postprocess as pp

from golden_common import synth_pred

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(__file__), "golden")


def _torch():
    import torch

    return torch


def _rel_l2(a, b):
    return float(np.linalg.norm(a - b) / (np.linalg.norm(b) + 1e-12))


@pytest.fixture(scope="module")
def n_p2():
    spec = cfg.resolve("yolov8n-p2")
    return spec, onet.build_spec("yolov8n-p2"), weights.synthetic_state_dict(spec, seed=0)


def _diag(msg):
    d = os.path.join(os.path.dirname(os.path.dirname(__file__)), "gpurun_out")
    if os.path.isdir(d):
        with open(os.path.join(d, "parity_diag.txt"), "a") as fh:
            fh.write(msg + "\n")


@pytest.mark.parametrize("head", ["unfused", "fused", "fused-chain15"])
@pytest.mark.parametrize("name,B,H,W", [("yolov8n-p2", 2, 64, 96), ("yolov8s-p2", 1, 96, 64), ("yolov8x-p2", 1, 64, 64), ("yolov8s-p2", 3, 128, 160),
                                        ("yolov8-small", 2, 64, 96)])      # the project's own model: widths 12 / 24 padded to 16 / 32
def test_engine_every_layer_matches_oracle_on_identical_inputs(name, B, H, W, head, monkeypatch):
    """Primary kernel gate (SURVEY.md H1 (i)): after one engine forward, EVERY launch of the plan is re-evaluated in float64
    on the engine's own input buffer (bf16 values, bf16 weights) and must agree with the engine's output buffer to about one
    bf16 rounding (tests/plan_ref.py).  ``fused``: the Detect head as DetectPipeline builds it, with the DFL and class-max
    epilogues; ``fused-chain15`` (B2_CHAIN=15) also chains the class tail (conv_tc_kernel<2, 2, 2, 16, 1>)."""
    from b200dt.engine import Engine

    import plan_ref

    if head == "fused-chain15":
        monkeypatch.setenv("B2_CHAIN", "15")
    torch = _torch()
    spec = cfg.resolve(name)
    sd = weights.synthetic_state_dict(spec, seed=0)
    x = pp.preprocess([synth.IRStream(seed=40 + b, h=H, w=W, n_targets=4).frame() for b in range(B)])
    eng = Engine(spec, sd, B, H, W, fuse_head=head != "unfused")
    xt = torch.from_numpy(x).cuda()
    eng.forward_tensor(xt)
    torch.cuda.synchronize()
    rep = []
    worst = plan_ref.check_plan(eng, xt, report=rep)
    kinds = sorted({k for _, k, _ in rep})
    assert ("dfl" in kinds and "cls" in kinds) == (head != "unfused"), kinds
    _diag(f"per-layer parity {name} {B}x{H}x{W} {head}: {len(eng.plan.ops)} launches ({', '.join(kinds)}), worst conv rel-L2 {worst:.2e}")
    eng.close()


def test_engine_graph_and_end_to_end_drift(n_p2):
    """End-to-end against the oracle evaluated with the engine's rounding points.  Two different summation orders
    decorrelate through ~25 random layers, so this bound is loose; the tight gate is the per-layer test above."""
    from b200dt.engine import Engine

    torch = _torch()
    spec, ospec, sd = n_p2
    B, H, W = 2, 64, 96
    x = pp.preprocess([synth.IRStream(seed=40 + b, h=H, w=W, n_targets=4).frame() for b in range(B)])
    eng = Engine(spec, sd, B, H, W)
    eng.forward_tensor(torch.from_numpy(x).cuda())
    torch.cuda.synchronize()
    net = onet.Net(ospec, sd, "bf16")
    heads = net.forward(x, record=True)
    errs = {}
    for name, ref in net.trace.items():
        if name.startswith("layer.") or name not in eng.plan.named:
            continue                      # chained launches keep their intermediate tile in shared memory: no buffer to read
        got = eng.activation(name).cpu().numpy()
        assert got.shape == ref.shape, name
        errs[name] = _rel_l2(got, ref)
    _diag("engine vs bf16 oracle, rel-L2: model.0 %.2e, model.9.cv2 %.2e, model.27.cv2 %.2e, worst %.2e (%s)" % (
        errs["model.0"], errs["model.9.cv2"], errs["model.27.cv2"], max(errs.values()), max(errs, key=errs.get)))
    assert errs["model.0"] < 4e-3 and max(errs.values()) < 0.12, errs
    for l, hd in enumerate(heads):
        got = eng.level_logits(l).float().cpu().numpy()[..., :64 + spec["nc"]]
        ref = hd.reshape(B, hd.shape[1], -1).transpose(0, 2, 1)
        assert _rel_l2(got, ref) < 5e-2, (l, _rel_l2(got, ref))
    # CUDA graph replay gives the same bits as the first (capturing) run, and as eager launches
    first = [eng.level_logits(l).clone() for l in range(eng.n_levels)]
    eng.forward_tensor(torch.from_numpy(x).cuda())
    torch.cuda.synchronize()
    for l in range(eng.n_levels):
        assert torch.equal(first[l], eng.level_logits(l))
    eng.use_graph(False)
    eng.forward_tensor(torch.from_numpy(x).cuda())
    torch.cuda.synchronize()
    for l in range(eng.n_levels):
        assert torch.equal(first[l], eng.level_logits(l))


@pytest.mark.parametrize("chain", ["default", "15", "0"])
@pytest.mark.parametrize("name,nc", [("yolov8n-p2", 80), ("yolov8n-p2", 1), ("yolov8s-p2", 80)])
def test_fused_head_equals_unfused_decode(name, nc, chain, monkeypatch):
    """DFL + class max inside the conv epilogue (fused head) vs plain logits + decode kernel: same candidates, same bits --
    with the default chained launches, with every chain pattern on (B2_CHAIN=15: the class tail too) and with none."""
    if chain != "default":
        monkeypatch.setenv("B2_CHAIN", chain)
    from b200dt import ops
    from b200dt.engine import Engine

    torch = _torch()
    spec = cfg.resolve(name, nc=nc)
    sd = weights.synthetic_state_dict(spec, seed=0)
    B, H, W = 2, 96, 160
    frames = torch.from_numpy(np.stack([synth.IRStream(seed=60 + b, h=H, w=W, n_targets=5).frame() for b in range(B)])).cuda()
    res = []
    conf = None
    for fused in (False, True):
        eng = Engine(spec, sd, B, H, W, fuse_head=fused)
        eng.forward_u8(frames)
        post = ops.DetectPost(B, eng.level_h, eng.level_w, eng.level_stride, eng.nc, eng.lstride)
        for c in ([0.15, 0.02, 1e-3, 1e-5] if conf is None else [conf]):      # first threshold that leaves candidates (nc = 1 scores are low)
            if fused:
                post.candidates_from_head(eng.head_dist, eng.head_cls, c)
            else:
                post.decode(eng.level_ptrs, c)
            torch.cuda.synchronize()
            cnt = post.cand_count.cpu().numpy()
            if cnt.min() > 0:
                conf = c
                break
        out = []
        for b in range(B):
            idx = post.cand_idx[b, :cnt[b]].cpu().numpy()
            rows = post.cand[b, :cnt[b]].cpu().numpy()
            o = np.argsort(idx)
            out.append((idx[o], rows[o]))
        res.append(out)
    for b in range(B):
        assert len(res[0][b][0]) > 0
        np.testing.assert_array_equal(res[0][b][0], res[1][b][0])
        np.testing.assert_array_equal(res[0][b][1], res[1][b][1])


def test_engine_vs_reference_fp32_golden(n_p2):
    """bf16 engine vs the reference's own fp32 forward (tests/golden/net_n_p2_small.npz, uniform-noise input).

    A random-weight net amplifies bf16 rounding (SURVEY.md H1), so the gate has two parts: (i) the engine agrees
    tightly with the oracle evaluated at the engine's rounding points, and (ii) its distance to the fp32
    reference is no larger than the distance of that bf16 oracle to the fp32 reference (the bf16 noise floor)."""
    from b200dt import ops
    from b200dt.engine import Engine

    torch = _torch()
    spec, ospec, sd = n_p2
    g = np.load(os.path.join(G, "net_n_p2_small.npz"))
    x = np.random.default_rng(0).random((1, 3, 64, 96), dtype=np.float32)
    eng = Engine(spec, sd, 1, 64, 96)
    eng.forward_tensor(torch.from_numpy(x).cuda())
    post = ops.DetectPost(1, eng.level_h, eng.level_w, eng.level_stride, eng.nc, eng.lstride)
    dense = torch.zeros((1, 4 + eng.nc, eng.num_anchors), dtype=torch.float32, device="cuda")
    post.decode(eng.level_ptrs, 0.15, dense_out=dense)
    y = dense.cpu().numpy()
    ref = g["y"]
    yb = pp.decode(onet.Net(ospec, sd, "bf16").forward(x), [4, 8, 16, 32], 80)

    def box_err(a, b):
        return np.abs(a[:, :4] - b[:, :4]).max(1) / np.maximum(b[:, 2:4].max(1), 1.0)

    e_gpu, e_floor = box_err(y, ref), box_err(yb, ref)
    _diag(f"noise input 64x96: box err / box size vs fp32 reference: engine median {np.median(e_gpu):.3e}, bf16-oracle floor {np.median(e_floor):.3e}")
    assert np.median(e_gpu) < 1.25 * np.median(e_floor) + 1e-3, (np.median(e_gpu), np.median(e_floor))
    assert np.abs(y[:, 4:] - ref[:, 4:]).max() < np.abs(yb[:, 4:] - ref[:, 4:]).max() + 0.1


def test_decode_matches_oracle_on_same_logits():
    """DFL + anchors + sigmoid + candidate filter on given bf16 logits: exact arithmetic restatement."""
    from b200dt import ops

    torch = _torch()
    g = np.random.default_rng(1)
    B, nc = 3, 80
    hs, ws, st = [16, 8, 4, 2], [24, 12, 6, 3], [4, 8, 16, 32]
    lstride = 144
    maps, bufs = [], []
    for h, w in zip(hs, ws):
        m = onet.bf16_round((g.standard_normal((B, 64 + nc, h, w)) * 2.0).astype(np.float32))
        m[:, 64:] -= 3.0
        m = onet.bf16_round(m)
        maps.append(m)
        bufs.append(torch.from_numpy(np.ascontiguousarray(m.reshape(B, 64 + nc, h * w).transpose(0, 2, 1))).cuda().to(torch.bfloat16).contiguous())
    ref = pp.decode(maps, st, nc)                                       # (B, 84, A)
    post = ops.DetectPost(B, hs, ws, st, nc, lstride)
    dense = torch.zeros((B, 4 + nc, post.A), dtype=torch.float32, device="cuda")
    conf = 0.15
    post.decode(bufs, conf, dense_out=dense)
    y = dense.cpu().numpy()
    np.testing.assert_allclose(y[:, :4], ref[:, :4], rtol=2e-5, atol=2e-4)
    np.testing.assert_allclose(y[:, 4:], ref[:, 4:], rtol=2e-5, atol=1e-6)
    # candidate set == anchors whose best score > conf, outside a tiny band around the threshold
    cnt = post.cand_count.cpu().numpy()
    cand = post.cand.cpu().numpy()
    cidx = post.cand_idx.cpu().numpy()
    for b in range(B):
        best = ref[b, 4:].max(0)
        sure = set(np.nonzero(best > conf + 1e-5)[0].tolist())
        maybe = set(np.nonzero(best > conf - 1e-5)[0].tolist())
        got = set(cidx[b, :cnt[b]].tolist())
        assert sure <= got <= maybe
        order = np.argsort(cidx[b, :cnt[b]])
        rows = cand[b, :cnt[b]][order]
        a = cidx[b, :cnt[b]][order]
        xyxy = pp.xywh2xyxy(ref[b, :4].T[a])
        np.testing.assert_allclose(rows[:, :4], xyxy, rtol=2e-5, atol=3e-4)
        np.testing.assert_array_equal(rows[:, 5].astype(int), ref[b, 4:].argmax(0)[a])


@pytest.mark.parametrize("ci", range(6))
@pytest.mark.parametrize("mode", ["exact", "legacy"])
def test_nms_bit_exact_vs_reference(ci, mode):
    """non_max_suppression (candidate filter, class offsets, greedy NMS, max_det) vs the reference's outputs."""
    from b200dt import ops

    torch = _torch()
    g = np.load(os.path.join(G, "nms_cases.npz"))
    seed, B, nc, A, conf, iou, max_det, agn = g[f"c{ci}_cfg"]
    pred = synth_pred(int(seed), int(B), int(nc), int(A), frac=0.05 if ci == 0 else 0.15)
    classes = g[f"c{ci}_classes"].tolist() if f"c{ci}_classes" in g.files else None
    out = ops.non_max_suppression(torch.from_numpy(pred).cuda(), float(conf), float(iou), classes=classes, agnostic=bool(agn),
                                  max_det=int(max_det), mode=mode)
    for b in range(int(B)):
        ref = g[f"c{ci}_{mode}_{b}"]
        got = out[b].cpu().numpy()
        assert got.shape == ref.shape
        np.testing.assert_array_equal(got, ref)


def test_nms_edge_cases():
    from b200dt import ops

    torch = _torch()
    # no candidates at all
    pred = torch.zeros((2, 6, 50), device="cuda")
    out = ops.non_max_suppression(pred, 0.25, 0.45)
    assert [tuple(o.shape) for o in out] == [(0, 6), (0, 6)]
    # SURVEY 8c hand case: legacy early exit keeps all, exact suppresses the duplicate
    boxes = np.array([[200, 200, 210, 210], [0, 0, 10, 10], [0, 0, 10, 10.5]], np.float32)
    xywh = np.stack([(boxes[:, 0] + boxes[:, 2]) / 2, (boxes[:, 1] + boxes[:, 3]) / 2, boxes[:, 2] - boxes[:, 0], boxes[:, 3] - boxes[:, 1]], 0)
    pred = np.concatenate([xywh, np.array([[.9, .8, .7]], np.float32)], 0)[None]
    ex = ops.non_max_suppression(torch.from_numpy(pred).cuda(), 0.25, 0.6, mode="exact")[0]
    lg = ops.non_max_suppression(torch.from_numpy(pred).cuda(), 0.25, 0.6, mode="legacy")[0]
    assert len(ex) == 2 and len(lg) == 3
    with pytest.raises(AssertionError):
        ops.non_max_suppression(torch.from_numpy(pred).cuda(), 1.5, 0.6)
    # many candidates (global-memory sort path) against the oracle, bit-exact
    big = synth_pred(9, 1, 3, 6000, frac=0.3)
    got = ops.non_max_suppression(torch.from_numpy(big).cuda(), 0.05, 0.5, max_det=300)[0].cpu().numpy()
    ref = pp.non_max_suppression(big, 0.05, 0.5, max_det=300, mode="exact")[0]
    np.testing.assert_array_equal(got, ref)
    # several NMS blocks with a long kept list (blocked exact path: members are tested against earlier blocks' kept boxes)
    big2 = synth_pred(11, 2, 2, 9000, frac=0.4)
    got2 = ops.non_max_suppression(torch.from_numpy(big2).cuda(), 0.05, 0.3, max_det=1000)
    ref2 = pp.non_max_suppression(big2, 0.05, 0.3, max_det=1000, mode="exact")
    for b in range(2):
        np.testing.assert_array_equal(got2[b].cpu().numpy(), ref2[b])


def _golden_frames(hw):
    f3 = synth.IRStream(seed=1001, h=hw[0], w=hw[1])
    return [synth.IRStream(seed=7, h=hw[0], w=hw[1]).frame(), synth.IRStream(seed=8, h=hw[0], w=hw[1]).frame(),
            [f3.frame() for _ in range(4)][-1]]


@pytest.mark.parametrize("name,gfile,tag,hw", [("yolov8n-p2", "predict_n_p2.npz", "512x640", (512, 640)),
                                               ("yolov8n-p2", "predict_n_p2.npz", "500x640", (500, 640)),
                                               ("yolov8s-p2", "predict_s_p2.npz", "512x640", (512, 640)),
                                               ("yolov8-small", "predict_small.npz", "512x640", (512, 640))])
def test_predict_matches_reference_golden(name, gfile, tag, hw):
    """North-star gate: YOLO(cfg).predict on uint8 frames returns the SAME detection set as the reference's predict()
    (fp32, CPU; tests/golden/predict_*.npz) at conf 0.15 / iou 0.6 -- every decided reference detection present with its box
    within 1e-2 relative and its score within 5e-2, nothing the reference decidedly suppresses -- outside the stated
    exclusion band (golden_common.detection_set_report: candidates whose NMS fate flips when the reference's own logits
    move by +-0.12 and its boxes by +-0.1 px, the measured reach of bf16 activation storage)."""
    from b200dt.predictor import YOLO

    from golden_common import detection_set_report

    g = np.load(os.path.join(G, gfile))
    frames = _golden_frames(hw)
    model = YOLO(name + ".yaml")
    res = model.predict(frames, conf=0.15, iou=0.6, verbose=False)
    assert len(res) == 3
    strict = total = band = matched = 0
    for b, r in enumerate(res):
        ref, cand = g[f"{tag}_exact_{b}"], g[f"{tag}_cand_{b}"]
        d = r.boxes.data.cpu().numpy()
        assert r.orig_shape == hw and d.shape[1] == 6
        assert np.all(np.diff(d[:, 4]) <= 0)                              # sorted by descending confidence
        assert d[:, [0, 2]].min() >= 0 and d[:, [0, 2]].max() <= hw[1] and d[:, [1, 3]].max() <= hw[0]
        rep = detection_set_report(d, ref, cand, 0.15, 0.6, frame_hw=hw)
        _diag(f"predict {name} {tag} frame {b}: reference {rep['n_ref']} detections ({rep['n_ref_strict']} decided, {rep['n_ref_in_band']} in the "
              f"band), engine {rep['n_det']} ({rep['n_ref_matched']} of the reference rows, {rep['n_det_not_in_ref']} others), violations {len(rep['errors'])}")
        assert not rep["errors"], (b, rep["errors"][:5])
        # outside the band: the same set -- every decided reference row is there, and every engine row is either a decided
        # reference row or a band candidate
        strict += rep["n_ref_strict"]; total += rep["n_ref"]; band += rep["n_ref_in_band"]; matched += rep["n_ref_matched"]
    if tag == "512x640":
        assert strict >= 0.6 * total, (strict, total)        # the band must not swallow the comparison
    # band or not: how many of the reference's rows the engine reports with the box within 1e-2 (measured: 512x640 207 of 212,
    # 500x640 -- 200 to 225 detections per frame, most of them clutter at the confidence threshold -- 530 of 633)
    assert matched >= (0.93 if tag == "512x640" else 0.78) * total, (matched, total)
    # the reference API surface
    r = res[0]
    assert r.boxes.xyxy.shape[1] == 4 and r.boxes.conf.ndim == 1 and r.boxes.cls.ndim == 1 and r.boxes.id is None
    xy = r.boxes.xyxy.cpu().numpy()
    assert xy.dtype == np.float32


def test_predict_engine_agrees_with_bf16_oracle(n_p2):
    """The engine against the oracle evaluated at the same rounding points: the two differ only by summation order and the
    fast SiLU / exp, an order of magnitude below the bf16 storage noise, so outside a band a quarter as wide the sets are
    identical."""
    import golden_common as gc
    from b200dt.predictor import YOLO

    spec, ospec, sd = n_p2
    hw = (512, 640)
    frames = _golden_frames(hw)
    res = YOLO("yolov8n-p2.yaml").predict(frames, conf=0.15, iou=0.6)
    yb = pp.decode(onet.Net(ospec, sd, "bf16").forward(pp.preprocess(frames)), [4, 8, 16, 32], 80)
    ob = pp.non_max_suppression(yb, 0.15, 0.6, mode="exact")
    saved = gc.BAND_LOGIT, gc.BAND_BOX
    gc.BAND_LOGIT, gc.BAND_BOX = 0.03, 0.03
    try:
        for b in range(3):
            t = yb[b].T
            sc, cl = t[:, 4:].max(1), t[:, 4:].argmax(1)
            k = sc > 0.15
            xy = np.stack([t[k, 0] - t[k, 2] / 2, t[k, 1] - t[k, 3] / 2, t[k, 0] + t[k, 2] / 2, t[k, 1] + t[k, 3] / 2], 1)
            cand = np.concatenate([xy, sc[k, None], cl[k, None]], 1)                 # unclipped: what NMS sees (no padding at 512x640)
            o = ob[b].copy()
            o[:, :4] = pp.scale_boxes(hw, o[:, :4], hw)
            rep = gc.detection_set_report(res[b].boxes.data.cpu().numpy(), o, cand, 0.15, 0.6, frame_hw=hw)
            _diag(f"engine vs bf16 oracle frame {b}: oracle {rep['n_ref']} ({rep['n_ref_strict']} decided), engine {rep['n_det']}, violations {len(rep['errors'])}")
            assert not rep["errors"], (b, rep["errors"][:5])
            assert rep["n_ref_strict"] >= 0.8 * rep["n_ref"]
    finally:
        gc.BAND_LOGIT, gc.BAND_BOX = saved

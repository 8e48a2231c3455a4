"""Frames of any size through the detect path: the batched LetterBox kernel (b2_letterbox_u8) against cv2 and the oracle, NMS with a
per-image scale_boxes table (b2_nms_scaled), YOLO.predict on a list of frames of different shapes as one forward, and
DetectTrackPipeline over streams of mixed resolutions or of one resolution that needs a resize.  The CPU tests at the end cover
the packing, the per-image geometry and the input checks."""
import numpy as np
import pytest

import b200dt  # noqa: F401
from b200dt import ops, pipeline, predictor
from oracle import postprocess as pp

KW = dict(max_lost_frames=150, min_hits=1, iou_threshold=0.1)
MIXED = [(96, 128), (120, 160), (128, 96), (200, 128)]


def _noise(seed, h, w):
    return np.random.default_rng(seed).integers(0, 256, (h, w, 3), dtype=np.uint8)


def _upload(*arrs):
    import torch

    return [torch.from_numpy(a).cuda() for a in arrs]


def _letterbox_gpu(frames, imgsz):
    (H, W), geom, _ = predictor.letterbox_table([f.shape[:2] for f in frames], [imgsz, imgsz])
    packed, offs = ops.pack_frames(frames)
    p, o, g = _upload(packed, offs, geom)
    return ops.letterbox_u8(p, o, g, H, W).cpu().numpy(), geom


def _cv2_letterbox(img, g, H, W):
    """LetterBox as the reference writes it with cv2 (the oracle comparison alone where cv2 is not installed)."""
    try:
        import cv2
    except ImportError:
        return None
    _, _, rh, rw, top, left = (int(v) for v in g)
    r = img if (rh, rw) == img.shape[:2] else cv2.resize(img, (rw, rh), interpolation=cv2.INTER_LINEAR)
    return cv2.copyMakeBorder(r, top, H - rh - top, left, W - rw - left, cv2.BORDER_CONSTANT, value=(114, 114, 114))


@pytest.mark.gpu
def test_letterbox_kernel_matches_cv2_and_oracle_ragged():
    """Downscales up to 6x, exact 2x, identity (aligned and at an odd column), odd sizes, upscale and portrait in one batch."""
    shapes = [(1080, 1920), (720, 1280), (2160, 3840), (1024, 1280), (512, 640), (333, 517), (50, 60), (1280, 200), (640, 500)]
    frames = [_noise(10 + i, h, w) for i, (h, w) in enumerate(shapes)]
    got, geom = _letterbox_gpu(frames, 640)
    assert got.shape == (len(frames), 640, 640, 3)
    for b, img in enumerate(frames):
        ref = _cv2_letterbox(img, geom[b], 640, 640)
        if ref is not None:
            np.testing.assert_array_equal(got[b], ref, err_msg=str(shapes[b]))
        np.testing.assert_array_equal(got[b], pp.letterbox(img, (640, 640), auto=False), err_msg=str(shapes[b]))


@pytest.mark.gpu
def test_letterbox_kernel_matches_cv2_uniform_auto():
    frames = [_noise(30 + i, 1080, 1920) for i in range(3)]
    got, geom = _letterbox_gpu(frames, 640)
    assert got.shape == (3, 384, 640, 3)
    for b, img in enumerate(frames):
        ref = _cv2_letterbox(img, geom[b], 384, 640)
        if ref is not None:
            np.testing.assert_array_equal(got[b], ref)
        np.testing.assert_array_equal(got[b], pp.letterbox(img, (640, 640), auto=True))


@pytest.mark.gpu
def test_nms_scaled_equals_nms_per_image():
    import torch

    B, cap = 5, 256
    g = np.random.default_rng(7)
    post = ops.DetectPost(B, [16], [16], [8], 4, 64)
    assert post.cand_cap == cap
    xy = g.uniform(0, 600, (B, cap, 2)).astype(np.float32)
    wh = g.uniform(4, 60, (B, cap, 2)).astype(np.float32)
    cand = np.concatenate([xy, xy + wh, g.uniform(0.2, 1, (B, cap, 1)), g.integers(0, 4, (B, cap, 1))], -1).astype(np.float32)
    counts = np.array([0, 3, 40, 256, 120], np.int32)
    shapes = [(1080, 1920), (720, 1280), (50, 60), (1280, 200), (512, 640)]
    _, _, scale = predictor.letterbox_table(shapes, [640, 640])
    post.cand.copy_(torch.from_numpy(cand))
    post.cand_idx.copy_(torch.arange(cap, dtype=torch.int32).repeat(B, 1))
    post.cand_count.copy_(torch.from_numpy(counts))
    out, cnt = post.nms(0.5, scale=_upload(scale)[0])
    out, cnt, idx = out.clone(), cnt.clone(), post.out_idx.clone()
    one = ops.DetectPost(1, [16], [16], [8], 4, 64)
    for b in range(B):
        one.cand.copy_(post.cand[b:b + 1]); one.cand_idx.copy_(post.cand_idx[b:b + 1]); one.cand_count.copy_(post.cand_count[b:b + 1])
        o1, c1 = one.nms(0.5, scale=tuple(float(v) for v in scale[b]))
        n = int(c1[0])
        assert n == int(cnt[b])
        assert torch.equal(o1[0, :n], out[b, :n]) and torch.equal(one.out_idx[0, :n], idx[b, :n])
    assert int(cnt.sum()) > 0


def _per_frame_reference(model, frames, imgsz, feats=False):
    """The path a mixed list took one frame at a time: its own auto=False geometry, a batch-1 pipeline, the stem-fused pad."""
    import torch

    from b200dt.predictor import DetectPipeline, letterbox_geometry

    out = []
    for f in frames:
        h0, w0 = f.shape[:2]
        (rh, rw), (H, W), top, left = letterbox_geometry(h0, w0, [imgsz, imgsz], auto=False)
        u8 = torch.from_numpy(f[None].copy()).cuda()
        if (rh, rw) != (h0, w0):
            u8 = ops.resize_bilinear_u8(u8, rh, rw)
        pipe = DetectPipeline(model.spec, model.state_dict, 1, H, W, 300)
        d, c = pipe(u8, 0.15, 0.6, top, left, (h0, w0))
        n = int(c[0])
        out.append((d[0, :n].clone(), pipe.embed()[0, :n].clone() if feats else None))
    return out


@pytest.mark.gpu
def test_predict_mixed_list_is_one_forward_equal_to_per_frame():
    """Bit equality: every output pixel's accumulation order is independent of the batch size, and the canvas the kernel
    builds is byte-identical to the resize + stem-fused pad of the per-frame path."""
    import torch

    from b200dt import synth
    from b200dt.predictor import YOLO

    frames = [synth.IRStream(seed=90 + i, h=h, w=w, n_targets=4).frame() for i, (h, w) in enumerate(MIXED + [(50, 60)])]
    model = YOLO("yolov8n-p2.yaml")
    res = model.predict(frames, conf=0.15, iou=0.6, imgsz=128, _feats=True)
    assert list(model._pipes) == [(len(frames), 128, 128, 300)]             # one forward, no batch-1 pipeline
    ref = _per_frame_reference(model, frames, 128, feats=True)
    assert sum(len(r) for r in res) > 0
    for i, (r, f, (d, ft)) in enumerate(zip(res, frames, ref)):
        assert r.orig_shape == f.shape[:2] and r.path == f"image{i}.jpg"
        assert torch.equal(r.boxes.data, d), i
        assert torch.equal(r.feats, ft), i


def _streams(shapes, T, seed=40):
    from b200dt import synth

    vids = [synth.IRStream(seed=seed + s, h=h, w=w, n_targets=4) for s, (h, w) in enumerate(shapes)]
    return [[v.frame() for v in vids] for _ in range(T)]


def _pipe(shapes, **kw):
    from b200dt.pipeline import DetectTrackPipeline

    return DetectTrackPipeline("yolov8n-p2", len(shapes), shapes, 128, 0.15, 0.6, 300, capacity=1024, **KW, **kw)


def _snap(rows, counts):
    c = counts.cpu().numpy().copy()
    r = rows.cpu().numpy().copy()
    return [r[s, :c[s]].view(np.int32).copy() for s in range(len(c))]


def _check_against_predict_and_tracker(shapes, frames, pipe, step):
    from b200dt.predictor import YOLO
    from b200dt.tracker import EnhancedMultiTargetTracker, rows_to_dicts

    model = YOLO("yolov8n-p2.yaml")
    trks = [EnhancedMultiTargetTracker(150, 1, 0.1, capacity=1024, max_dets=300) for _ in shapes]
    n = 0
    for t, fr in enumerate(frames):
        rows, counts = step(pipe, fr)
        c = counts.cpu().numpy()
        res = model.predict(fr, conf=0.15, iou=0.6, imgsz=128)
        for s in range(len(shapes)):
            want = trks[s].update([[*r[:4], r[4]] for r in res[s].boxes.data.cpu().numpy()])
            got = rows_to_dicts(rows[s, :c[s]].cpu().numpy())
            assert [g["track_id"] for g in got] == [w["track_id"] for w in want], (t, s)
            for g, w in zip(got, want):
                np.testing.assert_allclose(g["bbox"], w["bbox"], rtol=1e-5, atol=1e-3)
            n += len(got)
    assert n > 0


def _step_packed(pipe, frames):
    import torch

    return pipe.step_device(torch.from_numpy(ops.pack_frames(frames)[0]).cuda())


@pytest.mark.gpu
def test_mixed_resolution_pipeline_equals_predict_plus_tracker():
    frames = _streams(MIXED, 6)
    pipe = _pipe(MIXED)
    assert pipe.ragged and (pipe.H, pipe.W) == (128, 128)
    assert pipe.h2d_bytes_per_step == ops.pack_layout(MIXED)[1]
    _check_against_predict_and_tracker(MIXED, frames, pipe, _step_packed)


@pytest.mark.gpu
def test_mixed_resolution_pipeline_entry_points_agree():
    import torch

    frames = _streams(MIXED, 6, seed=50)
    packed = [ops.pack_frames(f)[0] for f in frames]
    plain, over, host = _pipe(MIXED), _pipe(MIXED, overlap_post=True), _pipe(MIXED, overlap_post=True)
    pinned = [torch.from_numpy(p).pin_memory() for p in packed]
    for t in range(len(frames)):
        dev = torch.from_numpy(packed[t]).cuda()
        ref = _snap(*plain.step_device(dev))
        rows, counts = over.step_device(dev)
        over.join()
        got = _snap(rows, counts)
        hr, hc = host.step_host(pinned[t])
        host.join()
        torch.cuda.synchronize()
        c = hc.numpy()
        for s in range(len(MIXED)):
            np.testing.assert_array_equal(got[s], ref[s])
            np.testing.assert_array_equal(hr.numpy()[s, :c[s]].view(np.int32), ref[s])
    with pytest.raises(ValueError, match="packed frame bytes"):
        plain.step_device(torch.zeros((len(MIXED), 96, 128, 3), dtype=torch.uint8, device="cuda"))


@pytest.mark.gpu
def test_uniform_shape_that_needs_a_resize():
    import torch

    shapes = [(192, 256)] * 3
    frames = _streams(shapes, 6, seed=60)
    pipe = _pipe(shapes)
    assert pipe.ragged and (pipe.H, pipe.W) == (96, 128)
    # [S][h][w][3] is the packed layout when every frame is a multiple of 16 bytes
    _check_against_predict_and_tracker(shapes, frames, pipe, lambda p, fr: p.step_device(torch.from_numpy(np.stack(fr)).cuda()))


@pytest.mark.gpu
def test_pipeline_run_over_mixed_stream_loader_equals_stepping(tmp_path):
    cv2 = pytest.importorskip("cv2")
    import torch

    from b200dt import synth
    from b200dt.loaders import LoadStreams

    shapes = [(96, 128), (120, 160), (96, 128)]
    clips = []
    for k, (h, w) in enumerate(shapes):
        vid = synth.IRStream(seed=80 + k, h=h, w=w, n_targets=4)
        path = str(tmp_path / f"s{k}.avi")
        wr = cv2.VideoWriter(path, cv2.VideoWriter_fourcc(*"MJPG"), 25, (w, h))
        for _ in range(6):
            wr.write(vid.frame())
        wr.release()
        clips.append(path)
    (tmp_path / "s.streams").write_text("\n".join(clips))
    a, b = _pipe(shapes), _pipe(shapes)
    got = list(a.run(LoadStreams(str(tmp_path / "s.streams"), buffer=True)))
    assert len(got) == 6
    for (src, rows, counts), (_, frames, _) in zip(got, LoadStreams(str(tmp_path / "s.streams"), buffer=True)):
        r2, c2 = _step_packed(b, frames)
        torch.cuda.synchronize()
        c2 = c2.cpu().numpy()
        assert np.array_equal(counts, c2)
        for s in range(len(shapes)):
            assert np.array_equal(rows[s, :counts[s]], r2[s, :c2[s]].cpu().numpy())
    assert sum(int(c.sum()) for _, _, c in got) > 0
    with pytest.raises(ValueError, match="stream 1"):
        next(a.run([(None, [np.zeros((96, 128, 3), np.uint8)] * 3, None)]))


@pytest.mark.gpu
def test_identity_path_launches_what_it_launched_before(monkeypatch):
    """Streams of one shape that needs no resize keep the stem-fused pad: per step the forward, the candidate stage, NMS and the
    tracker, and no letterbox launch."""
    import torch

    from b200dt import _lib

    lib = _lib.load()
    shapes = [(96, 128)] * 3
    frames = [torch.from_numpy(np.stack(f)).cuda() for f in _streams(shapes, 3, seed=70)]

    def boom(*a, **k):
        raise AssertionError("letterbox_u8 called on the identity path")

    monkeypatch.setattr(ops, "letterbox_u8", boom)
    pipe, probe = _pipe(shapes), _pipe(shapes)
    assert not pipe.ragged and pipe.h2d_bytes_per_step == 3 * 96 * 128 * 3
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
    assert pipe.detect.canvas is None


# ------------------------------------------------------------------------------------------------------------------------------
# CPU
# ------------------------------------------------------------------------------------------------------------------------------
def test_pack_frames_offsets_are_16_byte_aligned():
    shapes = [(5, 7), (16, 16), (3, 3), (333, 517), (1, 1)]
    frames = [_noise(i, h, w) for i, (h, w) in enumerate(shapes)]
    packed, offs = ops.pack_frames(frames)
    want, n = ops.pack_layout(shapes)
    assert offs.dtype == np.int64 and list(offs) == list(want) and packed.shape == (n,)
    assert all(o % 16 == 0 for o in offs) and n % 16 == 0
    for o, f, nxt in zip(offs, frames, list(offs[1:]) + [n]):
        assert o + f.size <= nxt and nxt - (o + f.size) < 16
        np.testing.assert_array_equal(packed[o:o + f.size].reshape(f.shape), f)
    with pytest.raises(ValueError, match="packed buffer"):
        ops.pack_frames(frames, out=np.empty((n - 16,), np.uint8))


@pytest.mark.parametrize("shapes,imgsz", [([(1080, 1920), (720, 1280), (512, 640), (50, 60), (1280, 200)], 640),
                                          ([(1080, 1920)] * 3, 640), ([(512, 640)] * 2, 640), (MIXED, 128), ([(192, 256)] * 3, 128)])
def test_letterbox_table_is_letterbox_geometry_per_image(shapes, imgsz):
    auto = len(set(shapes)) == 1
    (H, W), geom, scale = predictor.letterbox_table(shapes, [imgsz, imgsz])
    assert geom.dtype == np.int32 and geom.shape == (len(shapes), 6) and scale.dtype == np.float32 and scale.shape == (len(shapes), 5)
    for (h0, w0), g, sc in zip(shapes, geom, scale):
        (rh, rw), hw, top, left = predictor.letterbox_geometry(h0, w0, [imgsz, imgsz], auto)
        assert hw == (H, W) and tuple(g) == (h0, w0, rh, rw, top, left)
        np.testing.assert_array_equal(sc, np.asarray(predictor.scale_params((H, W), (h0, w0)), np.float32))
        r, new_unpad, t, b, l, rr = pp.letterbox_geometry(h0, w0, (imgsz, imgsz), auto, 32)
        assert (rw, rh) == new_unpad and (top, left) == (t, l)
    if not auto:
        assert (H, W) == (imgsz, imgsz)


def test_check_frames_names_the_stream():
    shapes = [(96, 128), (120, 160)]
    pipeline.check_frames([np.zeros((96, 128, 3), np.uint8), np.zeros((120, 160, 3), np.uint8)], shapes)
    with pytest.raises(ValueError, match="stream 1"):
        pipeline.check_frames([np.zeros((96, 128, 3), np.uint8)] * 2, shapes)
    with pytest.raises(ValueError, match="3 frames"):
        pipeline.check_frames([np.zeros((96, 128, 3), np.uint8)] * 3, shapes)


def test_ultralytics_plugin_mixed_shapes_reach_the_device(tmp_path, monkeypatch):
    """The plug-in's mixed-shape branch builds its tables and then needs the GPU (no CPU fallback, no per-image loop)."""
    import torch

    if torch.cuda.is_available():
        pytest.skip("CPU-container test")
    monkeypatch.setenv("YOLO_CONFIG_DIR", str(tmp_path))
    pytest.importorskip("ultralytics")
    from b200dt import ultra_plugin

    cls = ultra_plugin.predictor_class()
    p = cls.__new__(cls)
    p.imgsz = 128
    with pytest.raises(RuntimeError, match="CUDA device"):
        p.preprocess([np.zeros((96, 128, 3), np.uint8), np.zeros((120, 160, 3), np.uint8)])

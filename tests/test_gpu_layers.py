"""GPU parity of the layer kernels (through the C ABI) against the numpy oracle on seeded inputs."""
import numpy as np
import pytest

import b200dt  # noqa: F401
from b200dt import weights
from oracle import net as onet
from oracle import postprocess as pp

pytestmark = pytest.mark.gpu


def _t():
    import torch

    return torch


def _bf16_tensor(a):
    """numpy fp32 (already bf16-representable) NHWC -> CUDA bf16 tensor."""
    torch = _t()
    return torch.from_numpy(np.ascontiguousarray(a)).cuda().to(torch.bfloat16)


def _rand_bf16(g, shape, scale=1.0):
    return onet.bf16_round((g.standard_normal(shape) * scale).astype(np.float32))


CONV_CASES = [
    # B, H, W, Cin, Cout, k, s, act, residual
    (1, 16, 16, 16, 16, 1, 1, True, False),
    (2, 24, 40, 32, 64, 3, 1, True, False),
    (1, 20, 12, 64, 80, 3, 1, True, True),
    (2, 17, 23, 48, 32, 3, 1, True, False),       # ragged spatial size, BK=16 chunks
    (1, 32, 48, 64, 128, 3, 2, True, False),      # stride 2, even size
    (2, 15, 21, 32, 48, 3, 2, True, False),       # stride 2, odd size
    (1, 8, 8, 256, 512, 1, 1, True, False),       # two N tiles
    (1, 12, 20, 128, 64, 1, 1, False, False),     # plain conv (Detect output), no activation
    (1, 10, 10, 80, 1, 1, 1, False, False),       # nc = 1 output
    (3, 6, 10, 96, 144, 1, 1, True, False),
    (1, 40, 40, 16, 32, 3, 1, True, True),
    (1, 64, 64, 192, 96, 1, 1, True, False),      # K = 3 chunks of 64
    (4, 5, 7, 160, 160, 3, 1, True, False),       # x-scale widths, tiny maps, several images per tile
    # more tiles than the 2 x 148 CTA slots: every CTA runs several tiles (accumulator ring, alternate MMA warps, bias reload)
    (4, 128, 160, 32, 32, 3, 1, True, False),     # 3x3 stride 1, 81920 output pixels
    (3, 256, 320, 32, 64, 3, 2, True, False),     # stride 2, 61440 output pixels
    (4, 64, 96, 64, 512, 1, 1, True, False),      # Cout 512: two N tiles per pixel tile, 24576 pixels
]


# the 3x3 shapes, run under both input-staging plans by test_conv_kernel_variants_match_oracle
STAGING_CASES = [c for c in CONV_CASES if c[5] == 3] + [
    (2, 33, 19, 128, 64, 3, 1, True, True),       # tap mode (map below the halo tile-efficiency cut), two images per tile, shortcut
    (1, 48, 24, 80, 80, 3, 1, True, False),       # K segments 64 + 16; default: single halo box, two MMA warps
    (2, 16, 32, 256, 80, 3, 1, True, False),      # three-box halo mode with streamed weights (too large to stay resident)
    (1, 31, 45, 32, 128, 3, 2, True, False),      # stride 2, odd-sized input
    (5, 8, 8, 64, 64, 3, 1, False, True),         # several images per tile, no activation, shortcut
    (3, 64, 48, 96, 64, 3, 2, True, False),       # stride 2, K segments 64 + 32; default: parity boxes, two MMA warps
    (2, 34, 62, 16, 32, 3, 2, True, False),       # stride 2 tap mode, ragged 17 x 31 output, several images per tile, 32-byte rows
]


CHAIN_CASES = [
    # B, H, W, Cin, Cout, stride, residual, Cx (extra source), Cout2, act2
    (2, 64, 96, 32, 64, 2, False, 0, 64, True),          # Conv(k3 s2) -> C2f.cv1 (P2 of yolov8s-p2)
    (2, 32, 48, 32, 32, 1, True, 64, 64, True),          # Bottleneck.cv2 + shortcut -> C2f.cv2 over cat(y0, y1 | m)
    (1, 40, 24, 32, 32, 1, False, 64, 64, True),         # head C2f (no shortcut)
    (2, 33, 47, 64, 64, 1, False, 0, 64, False),         # Detect box tail (plain 1x1, no activation), ragged map
    (1, 48, 32, 80, 80, 1, False, 0, 80, False),         # Detect class tail: K blocks 64 + 16
    (3, 16, 24, 16, 16, 1, True, 32, 32, True),          # yolov8n widths: 32-byte rows, extra source of 32
    (1, 130, 70, 32, 64, 2, False, 0, 64, True),         # stride 2, ragged 65 x 35 output, many tiles per CTA
    (2, 24, 24, 48, 48, 1, True, 96, 96, True),          # K blocks 64 + 32 (extra) and 32 + 16 (main)
    (4, 256, 320, 32, 64, 2, False, 0, 64, True),        # 81920 output pixels: the look-ahead loads and double buffers of many tiles per CTA
]


@pytest.mark.parametrize("case", CHAIN_CASES)
def test_chained_conv_matches_oracle(case):
    """conv3x3 (+ shortcut) -> bf16 -> [extra | .] -> conv1x1 in one launch vs the oracle evaluating the two convs with the
    intermediate rounded to bf16 (exactly what the unchained path stores)."""
    from b200dt import ops

    torch = _t()
    B, H, W, cin, cout, stride, has_res, cx, cout2, act2 = case
    g = np.random.default_rng(hash(case) % (2 ** 31))
    if not ops.conv_chain_plan_ok(H, W, cin, cout, 3, stride, has_res, cx, cout2, B=B):
        pytest.skip("pair not taken by the chained kernel's plan")
    Ho, Wo = (H - 1) // stride + 1, (W - 1) // stride + 1
    x = _rand_bf16(g, (B, H, W, cin))
    w = _rand_bf16(g, (cout, 3, 3, cin), 1.0 / np.sqrt(9 * cin * 0.36))
    b = g.standard_normal(cout).astype(np.float32) * 0.1
    res = _rand_bf16(g, (B, Ho, Wo, cout)) if has_res else None
    ex = _rand_bf16(g, (B, Ho, Wo, cx)) if cx else None
    w2 = _rand_bf16(g, (cout2, cx + cout), 1.0 / np.sqrt((cx + cout) * 0.36))
    b2 = g.standard_normal(cout2).astype(np.float32) * 0.1
    got = ops.conv2d_chain_bf16(_bf16_tensor(x), _bf16_tensor(w), torch.from_numpy(b).cuda(), stride, _bf16_tensor(w2), torch.from_numpy(b2).cuda(), act=True, act2=act2,
                                residual=None if res is None else _bf16_tensor(res), extra=None if ex is None else _bf16_tensor(ex)).float().cpu().numpy()
    mid = onet.silu(onet.conv2d(x.transpose(0, 3, 1, 2), np.ascontiguousarray(w.transpose(0, 3, 1, 2)), b, stride, 1))
    if has_res:
        mid = mid + res.transpose(0, 3, 1, 2)
    mid = onet.bf16_round(mid)
    if cx:
        mid = np.concatenate([ex.transpose(0, 3, 1, 2), mid], 1)
    ref = onet.conv2d(mid, w2.reshape(cout2, cx + cout, 1, 1), b2, 1, 0)
    if act2:
        ref = onet.silu(ref)
    ref = ref.transpose(0, 2, 3, 1)
    assert got.shape == ref.shape
    err = float(np.linalg.norm(got - ref) / np.linalg.norm(ref))
    assert err < 4e-3, err
    np.testing.assert_allclose(got, ref, rtol=1e-2, atol=1e-2 * max(1.0, float(np.abs(ref).max()) / 16))


@pytest.mark.parametrize("mode", ["0", "2"])
@pytest.mark.parametrize("case", STAGING_CASES)
def test_conv_kernel_variants_match_oracle(case, mode, monkeypatch):
    """The 3x3 shapes under two input-staging plans of conv_tc_kernel.  mode = B2_CONV_HALO2: "2" is the default plan (one
    (TW+2) x (TH+2) box per K chunk for resident-weight stride-1 layers, parity boxes for stride 2 where they fit); "0" turns
    both single-box modes off (B2_CONV_S2BOX=0 too), so the same shapes stage one box per kw (halo 1) or one per filter tap."""
    monkeypatch.setenv("B2_CONV_HALO2", mode)
    monkeypatch.setenv("B2_CONV_S2BOX", "1" if mode == "2" else "0")
    test_conv_matches_oracle(case)


@pytest.mark.parametrize("case", CONV_CASES)
def test_conv_matches_oracle(case):
    from b200dt import ops

    torch = _t()
    B, H, W, Cin, Cout, k, s, act, res = case
    g = np.random.default_rng(hash(case) % (2 ** 31))
    x = _rand_bf16(g, (B, H, W, Cin))
    w = _rand_bf16(g, (Cout, Cin, k, k), 1.0 / np.sqrt(Cin * k * k))
    b = g.standard_normal(Cout).astype(np.float32) * 0.1
    ref = onet.conv2d(x.transpose(0, 3, 1, 2), w, b, s, k // 2)
    if act:
        ref = onet.silu(ref)
    r = None
    if res:
        r = _rand_bf16(g, ref.transpose(0, 2, 3, 1).shape)
        ref = ref + r.transpose(0, 3, 1, 2)
    out = None
    if Cout % 8:      # channel strides must be multiples of 8: write into a wider buffer (as the engine does for nc=1)
        out = torch.zeros((B, ref.shape[2], ref.shape[3], 8), dtype=torch.bfloat16, device="cuda")
    y = ops.conv2d_bf16(_bf16_tensor(x), _bf16_tensor(weights.pack_ohwi(w)), torch.from_numpy(b).cuda(), k, s, act,
                        out=out, residual=_bf16_tensor(r) if res else None)
    torch.cuda.synchronize()
    got = y.float().cpu().numpy().transpose(0, 3, 1, 2)[:, :Cout]
    assert got.shape == ref.shape
    # one bf16 rounding of the output (2^-9 relative) + fp32 accumulation-order noise
    np.testing.assert_allclose(got, ref, rtol=6e-3, atol=6e-3)


def test_conv_channel_slices_and_strides():
    """Concat-by-offset: read a channel slice of a wider buffer, write into a slice of another, residual from a third."""
    from b200dt import ops

    torch = _t()
    g = np.random.default_rng(5)
    B, H, W = 2, 12, 20
    xin = _rand_bf16(g, (B, H, W, 96))
    w = _rand_bf16(g, (32, 32, 3, 3), 1 / 17.0)
    b = g.standard_normal(32).astype(np.float32) * 0.1
    out = _bf16_tensor(np.full((B, H, W, 128), 7.0, np.float32))
    ops.conv2d_bf16(_bf16_tensor(xin), _bf16_tensor(weights.pack_ohwi(w)), torch.from_numpy(b).cuda(), 3, 1, True,
                    out=out, out_coff=64, in_coff=32, cin=32, residual=_bf16_tensor(xin), res_coff=64)
    torch.cuda.synchronize()
    got = out.float().cpu().numpy()
    ref = onet.silu(onet.conv2d(xin[..., 32:64].transpose(0, 3, 1, 2), w, b, 1, 1)) + xin[..., 64:96].transpose(0, 3, 1, 2)
    np.testing.assert_allclose(got[..., 64:96].transpose(0, 3, 1, 2), ref, rtol=6e-3, atol=6e-3)
    assert np.all(got[..., :64] == 7.0) and np.all(got[..., 96:] == 7.0)      # neighbours untouched


UPCAT_CASES = [(2, 16, 24, 64, 32, 48), (1, 32, 40, 128, 64, 96), (3, 8, 8, 32, 80, 64), (1, 6, 10, 256, 128, 128)]     # B, H, W, C0, C1, Cout


@pytest.mark.parametrize("shape", UPCAT_CASES)
def test_conv_over_upsample_concat_matches_oracle(shape):
    """C2f.cv1 over Concat([Upsample(x_lo), skip]) (yolov8-p2.yaml:33-36) with the upsample and the concat folded
    into the conv's TMA loads (zero-stride tensor-map dimensions replicate each low-resolution pixel 2x2)."""
    from b200dt import ops

    torch = _t()
    B, H, W, C0, C1, Cout = shape
    g = np.random.default_rng(sum(shape))
    lo = _rand_bf16(g, (B, H // 2, W // 2, C0))
    skip = _rand_bf16(g, (B, H, W, C1))
    w = _rand_bf16(g, (Cout, C0 + C1, 1, 1), 1.0 / np.sqrt(C0 + C1))
    b = g.standard_normal(Cout).astype(np.float32) * 0.1
    cat = np.concatenate([lo.repeat(2, 1).repeat(2, 2), skip], -1)
    ref = onet.silu(onet.conv2d(cat.transpose(0, 3, 1, 2), w, b, 1, 0))
    y = ops.conv2d_cat_bf16(_bf16_tensor(lo), _bf16_tensor(skip), _bf16_tensor(weights.pack_ohwi(w)), torch.from_numpy(b).cuda(), up0=2)
    torch.cuda.synchronize()
    np.testing.assert_allclose(y.float().cpu().numpy().transpose(0, 3, 1, 2), ref, rtol=6e-3, atol=6e-3)
    # plain two-source concat (no upsample), 3x3
    a0, a1 = _rand_bf16(g, (B, H, W, C0)), _rand_bf16(g, (B, H, W, C1))
    w3 = _rand_bf16(g, (Cout, C0 + C1, 3, 3), 1.0 / np.sqrt(9 * (C0 + C1)))
    ref = onet.silu(onet.conv2d(np.concatenate([a0, a1], -1).transpose(0, 3, 1, 2), w3, b, 1, 1))
    y = ops.conv2d_cat_bf16(_bf16_tensor(a0), _bf16_tensor(a1), _bf16_tensor(weights.pack_ohwi(w3)), torch.from_numpy(b).cuda(), ksize=3)
    torch.cuda.synchronize()
    np.testing.assert_allclose(y.float().cpu().numpy().transpose(0, 3, 1, 2), ref, rtol=6e-3, atol=6e-3)


def test_conv_rejects_bad_arguments():
    from b200dt import ops

    torch = _t()
    x = torch.zeros((1, 8, 8, 24), dtype=torch.bfloat16, device="cuda")
    w = torch.zeros((16, 1, 1, 24), dtype=torch.bfloat16, device="cuda")
    with pytest.raises(ValueError):
        ops.conv2d_bf16(x, w, torch.zeros(16, device="cuda"), 1)            # Cin % 16 != 0
    x = torch.zeros((1, 8, 8, 32), dtype=torch.bfloat16, device="cuda")
    w = torch.zeros((16, 5, 5, 32), dtype=torch.bfloat16, device="cuda")
    with pytest.raises(ValueError):
        ops.conv2d_bf16(x, w, torch.zeros(16, device="cuda"), 5)            # k = 5 unsupported


STEM_CASES = [
    # B, canvas, frame, (pad top, pad left), C0
    (2, (64, 96), (64, 96), (0, 0), 16),
    (2, (64, 96), (52, 96), (6, 0), 16),
    (2, (32, 64), (32, 50), (0, 7), 16),
    # several tiles per CTA (16 x 8 output pixels per tile, up to 8 CTAs per SM): the next-patch prefetch and the mixed-radix
    # tile advance with the grid stride above the tiles per image (160) ...
    (16, (256, 320), (256, 320), (0, 0), 16),
    (16, (256, 320), (256, 320), (0, 0), 32),
    # ... and below them (3200 tiles per image)
    (1, (1280, 1280), (1280, 1280), (0, 0), 32),
    # many small padded images (12 tiles per image), the x-scale stem width
    (128, (64, 96), (52, 96), (6, 0), 80),
    (128, (64, 96), (64, 90), (0, 3), 32),
]


@pytest.mark.parametrize("B,hw,src,pad,C0", STEM_CASES, ids=[f"hw{i}-src{i}-pad{i}" for i in range(len(STEM_CASES))])
def test_stem_u8_matches_oracle(B, hw, src, pad, C0):
    """Letterbox pad (114) + BGR->RGB + /255 + Conv(3->C0, k3, s2) + SiLU on raw uint8 frames."""
    from b200dt import ops

    torch = _t()
    g = np.random.default_rng(2)
    H, W = hw
    frames = g.integers(0, 256, (B, src[0], src[1], 3), dtype=np.uint8)
    w = (g.standard_normal((C0, 3, 3, 3)) / 3.0).astype(np.float32)
    b = (0.1 * g.standard_normal(C0)).astype(np.float32)
    canvas = np.full((B, H, W, 3), 114, np.uint8)
    canvas[:, pad[0]:pad[0] + src[0], pad[1]:pad[1] + src[1]] = frames
    x = pp.preprocess(list(canvas))
    ref = onet.bf16_round(onet.silu(onet.conv2d(x, onet.bf16_round(w), b, 2, 1)))     # bf16 weights, exact uint8 inputs
    wp = torch.from_numpy(weights.pack_stem(w).view(np.int16)).cuda().view(torch.bfloat16)
    y = ops.stem_u8(torch.from_numpy(frames).cuda(), wp, torch.from_numpy(b).cuda(), H, W, pad[0], pad[1])
    got = y.float().cpu().numpy().transpose(0, 3, 1, 2)
    np.testing.assert_allclose(got, ref, rtol=8e-3, atol=2e-3)
    # stand-alone preprocess (BasePredictor.preprocess): exact
    p = ops.preprocess_u8(torch.from_numpy(frames).cuda(), H, W, pad[0], pad[1]).cpu().numpy()
    np.testing.assert_allclose(p, x, rtol=0, atol=1e-7)


def test_sppf_pool_and_upsample_exact():
    from b200dt import ops

    g = np.random.default_rng(3)
    B, H, W, C = 2, 9, 13, 16
    x = _rand_bf16(g, (B, H, W, C))
    buf = np.zeros((B, H, W, 4 * C), np.float32)
    buf[..., :C] = x
    t = ops.sppf_pool(_bf16_tensor(buf), 0, C)
    got = t.float().cpu().numpy()
    y = x.transpose(0, 3, 1, 2)
    for j in range(1, 4):
        y = onet.maxpool5(y)
        np.testing.assert_array_equal(got[..., j * C:(j + 1) * C].transpose(0, 3, 1, 2), y)
    out = _bf16_tensor(np.zeros((B, 2 * H, 2 * W, 48), np.float32))
    ops.upsample_slice(_bf16_tensor(x), out, 2, out_coff=32)
    o = out.float().cpu().numpy()
    np.testing.assert_array_equal(o[..., 32:].transpose(0, 3, 1, 2), onet.upsample2(x.transpose(0, 3, 1, 2)))
    assert np.all(o[..., :32] == 0)


def test_resize_matches_cv2():
    cv2 = pytest.importorskip("cv2")
    from b200dt import ops

    torch = _t()
    g = np.random.default_rng(4)
    for (sh, sw), (dh, dw) in [((512, 640), (1024, 1280)), ((480, 640), (384, 512)), ((100, 130), (197, 256)), ((512, 640), (640, 800)),
                               ((720, 1280), (360, 640)), ((333, 517), (640, 640))]:
        img = g.integers(0, 256, (sh, sw, 3), dtype=np.uint8)
        ref = cv2.resize(img, (dw, dh), interpolation=cv2.INTER_LINEAR)
        got = ops.resize_bilinear_u8(torch.from_numpy(img[None]).cuda(), dh, dw)[0].cpu().numpy()
        np.testing.assert_array_equal(got, ref)          # byte work: bit-exact (cv2's 11-bit fixed-point bilinear)

"""The persistent tile loop of the conv, chained-conv, fused-head and stem kernels with many tiles per CTA.

Every CTA of conv_tc_kernel / stem_tc_kernel loops over ``tile = blockIdx.x; tile < total_tiles; tile += gridDim.x`` with a
grid of at most (SMs x CTAs per SM).  State that only matters from a CTA's second tile on -- the accumulator ring and its
phase, the two MMA warps taking alternate tiles, the chained kernel's look-ahead loads and double buffers, the class-head
epilogue's key double buffer, the per-tile bias reload with several N tiles, the stem's next-patch prefetch -- is checked
three ways:

* ``B2_CONV_GRID`` caps the conv grid at 1, 2, 3, 7 and 37 CTAs.  The plan does not depend on the grid, so every output must
  be bit-identical to the default grid; at grid 3 the layer tests' oracles run as well.
* Shapes with more tiles than CTA slots at the default grid (test_gpu_layers.py, the last cases of each list).
* The full-size plans the product builds (through DetectPipeline), every launch checked in float64 at sampled pixels.
"""
import numpy as np
import pytest

import b200dt  # noqa: F401
from b200dt import cfg, synth, weights
from b200dt import engine as eng_mod
from oracle import postprocess as pp

import plan_ref
import test_gpu_layers as layers

pytestmark = pytest.mark.gpu
GRIDS = [1, 2, 3, 7, 37]


def _torch():
    import torch

    return torch


def _diag(msg):
    print(msg)                  # shown with pytest -rP


def _t(a):
    return layers._bf16_tensor(a)


def _conv_out(case):
    from b200dt import ops

    torch = _torch()
    B, H, W, cin, cout, k, s, act, res = case
    g = np.random.default_rng(hash(case) % (2 ** 31))
    x = layers._rand_bf16(g, (B, H, W, cin))
    w = layers._rand_bf16(g, (cout, k, k, cin), 1.0 / np.sqrt(cin * k * k))
    b = torch.from_numpy(g.standard_normal(cout).astype(np.float32) * 0.1).cuda()
    Ho, Wo = (H - 1) // s + 1, (W - 1) // s + 1
    r = _t(layers._rand_bf16(g, (B, Ho, Wo, cout))) if res else None
    out = torch.zeros((B, Ho, Wo, 8), dtype=torch.bfloat16, device="cuda") if cout % 8 else None
    return ops.conv2d_bf16(_t(x), _t(w), b, k, s, act, out=out, residual=r)


def _chain_out(case):
    from b200dt import ops

    torch = _torch()
    B, H, W, cin, cout, stride, has_res, cx, cout2, act2 = case
    if not ops.conv_chain_plan_ok(H, W, cin, cout, 3, stride, has_res, cx, cout2, B=B):
        return None
    g = np.random.default_rng(hash(case) % (2 ** 31))
    Ho, Wo = (H - 1) // stride + 1, (W - 1) // stride + 1
    x = layers._rand_bf16(g, (B, H, W, cin))
    w = layers._rand_bf16(g, (cout, 3, 3, cin), 1.0 / np.sqrt(9 * cin * 0.36))
    b = torch.from_numpy(g.standard_normal(cout).astype(np.float32) * 0.1).cuda()
    res = _t(layers._rand_bf16(g, (B, Ho, Wo, cout))) if has_res else None
    ex = _t(layers._rand_bf16(g, (B, Ho, Wo, cx))) if cx else None
    w2 = layers._rand_bf16(g, (cout2, cx + cout), 1.0 / np.sqrt((cx + cout) * 0.36))
    b2 = torch.from_numpy(g.standard_normal(cout2).astype(np.float32) * 0.1).cuda()
    return ops.conv2d_chain_bf16(_t(x), _t(w), b, stride, _t(w2), b2, act=True, act2=act2, residual=res, extra=ex)


def _upcat_out(shape):
    from b200dt import ops

    torch = _torch()
    B, H, W, C0, C1, cout = shape
    g = np.random.default_rng(sum(shape))
    lo, skip = layers._rand_bf16(g, (B, H // 2, W // 2, C0)), layers._rand_bf16(g, (B, H, W, C1))
    w = layers._rand_bf16(g, (cout, 1, 1, C0 + C1), 1.0 / np.sqrt(C0 + C1))
    w3 = layers._rand_bf16(g, (cout, 3, 3, C0 + C1), 1.0 / np.sqrt(9 * (C0 + C1)))
    b = torch.from_numpy(g.standard_normal(cout).astype(np.float32) * 0.1).cuda()
    a1 = layers._rand_bf16(g, (B, H, W, C0))
    return (ops.conv2d_cat_bf16(_t(lo), _t(skip), _t(w), b, up0=2), ops.conv2d_cat_bf16(_t(a1), _t(skip), _t(w3), b, ksize=3))


def _all_outputs(monkeypatch):
    """Every conv / chained / upsample-concat shape of test_gpu_layers.py; the 3x3 shapes under both input-staging plans."""
    torch = _torch()
    outs = {}
    seen = set()
    for case in layers.CONV_CASES + layers.STAGING_CASES:
        if case in seen:
            continue
        seen.add(case)
        for mode in (("2", "0") if case[5] == 3 else ("2",)):
            monkeypatch.setenv("B2_CONV_HALO2", mode)
            monkeypatch.setenv("B2_CONV_S2BOX", "1" if mode == "2" else "0")
            outs[("conv", mode, case)] = _conv_out(case)
    monkeypatch.delenv("B2_CONV_HALO2", raising=False)
    monkeypatch.delenv("B2_CONV_S2BOX", raising=False)
    for case in layers.CHAIN_CASES:
        outs[("chain", case)] = _chain_out(case)
    for shape in layers.UPCAT_CASES:
        outs[("upcat", shape)] = _upcat_out(shape)
    torch.cuda.synchronize()
    return outs


@pytest.fixture(scope="module")
def default_grid_outputs():
    mp = pytest.MonkeyPatch()
    mp.delenv("B2_CONV_GRID", raising=False)
    try:
        yield _all_outputs(mp)
    finally:
        mp.undo()


@pytest.mark.parametrize("grid", GRIDS)
def test_conv_outputs_bit_identical_under_forced_grid(grid, default_grid_outputs, monkeypatch):
    """CONV_CASES, STAGING_CASES (both staging plans), CHAIN_CASES and the upsample/concat convs with the grid capped at
    ``grid`` CTAs: the same bits as the default grid."""
    torch = _torch()
    monkeypatch.setenv("B2_CONV_GRID", str(grid))
    outs = _all_outputs(monkeypatch)
    assert outs.keys() == default_grid_outputs.keys()
    for key, ref in default_grid_outputs.items():
        got = outs[key]
        if ref is None:
            assert got is None, key
            continue
        for a, b in zip(got if isinstance(got, tuple) else (got,), ref if isinstance(ref, tuple) else (ref,)):
            assert torch.equal(a.view(torch.int16), b.view(torch.int16)), (grid, key, int((a != b).sum()))


def test_conv_kernels_match_oracle_at_grid_3(monkeypatch):
    """The layer tests' float oracles with every conv launch on three CTAs."""
    from b200dt import ops

    monkeypatch.setenv("B2_CONV_GRID", "3")
    for case in layers.CONV_CASES:
        layers.test_conv_matches_oracle(case)
    for case in layers.STAGING_CASES:
        for mode in ("0", "2"):
            layers.test_conv_kernel_variants_match_oracle(case, mode, monkeypatch)
    monkeypatch.delenv("B2_CONV_HALO2")
    monkeypatch.delenv("B2_CONV_S2BOX")
    for case in layers.CHAIN_CASES:
        if ops.conv_chain_plan_ok(*case[1:3], case[3], case[4], 3, case[5], case[6], case[7], case[8], B=case[0]):
            layers.test_chained_conv_matches_oracle(case)
    for shape in layers.UPCAT_CASES:
        layers.test_conv_over_upsample_concat_matches_oracle(shape)


def _engine_buffers(eng):
    """Every buffer's bits (int16: the head buffers hold fp32 records, whose halves can read as bf16 NaNs)."""
    import torch

    return [eng.buffer(i).view(torch.int16).clone() for i in range(len(eng.plan.bufs))]


@pytest.mark.parametrize("chain", ["default", "15"])
@pytest.mark.parametrize("name", ["yolov8n-p2", "yolov8s-p2"])
def test_fused_head_engine_bit_identical_under_forced_grid(name, chain, monkeypatch):
    """A fused-head engine (DFL and class-max epilogues; B2_CHAIN=15 chains the class tail too) at 2 x 128 x 160: every
    buffer of the forward is the same bits at every forced grid as at the default grid, and at grid 3 every launch matches
    the float64 per-op reference."""
    from b200dt.engine import Engine

    torch = _torch()
    if chain != "default":
        monkeypatch.setenv("B2_CHAIN", chain)
    monkeypatch.delenv("B2_CONV_GRID", raising=False)
    spec = cfg.resolve(name)
    sd = weights.synthetic_state_dict(spec, seed=0)
    B, H, W = 2, 128, 160
    frames = torch.from_numpy(np.stack([synth.IRStream(seed=70 + b, h=H, w=W, n_targets=5).frame() for b in range(B)])).cuda()

    def run():
        eng = Engine(spec, sd, B, H, W, fuse_head=True)
        eng.forward_u8(frames)
        torch.cuda.synchronize()
        return eng

    eng = run()
    ref = _engine_buffers(eng)
    eng.close()
    for grid in GRIDS:
        monkeypatch.setenv("B2_CONV_GRID", str(grid))
        eng = run()
        for i, (a, b) in enumerate(zip(_engine_buffers(eng), ref)):
            assert torch.equal(a, b), (grid, i, int((a != b).sum()))
        if grid == 3:
            rep = []
            worst = plan_ref.check_plan(eng, plan_ref.canvas_u8(frames, H, W), report=rep)
            assert {"dfl", "cls"} <= {k for _, k, _ in rep}
            _diag(f"grid 3 {name} chain {chain} {B}x{H}x{W}: {len(rep)} launches, worst conv rel-L2 {worst:.2e}")
        eng.close()


# The plans the product runs: C4 (256 streams x 512x640 uint8), the `auto` canvas of 1080p streams (1080x1920 -> 360x640,
# padded to 384x640), C2 (64 x 640^2 fp32 tensors), C5 (32 x 1280^2 bf16 tensors), and the project's own padded-width model.
FULL_SIZE = {
    "c4-yolov8s-p2-u8": ("yolov8s-p2", 256, (512, 640), "u8", (512, 640), 0),
    "canvas1080p-yolov8s-p2-u8": ("yolov8s-p2", 256, (384, 640), "u8", (360, 640), 12),
    "c2-yolov8s-p2-f32": ("yolov8s-p2", 64, (640, 640), "f32", None, 0),
    "c5-yolov8x-p2-bf16": ("yolov8x-p2", 32, (1280, 1280), "bf16", None, 0),
    "yolov8-small-512x640-u8": ("yolov8-small", 64, (512, 640), "u8", (512, 640), 0),
}


@pytest.mark.parametrize("config", list(FULL_SIZE))
def test_full_size_plan_every_launch_at_sampled_pixels(config):
    """One forward of the plan DetectPipeline builds, then every launch against the float64 per-op reference at ~1400
    pixels of its output: the tile / image border rows and columns crossed in images 0, 1, B/2, B-1, and 1000 random ones.
    Convs within the per-layer gate's tolerances, pool and upsample exact, the head records within their bounds.  The check
    itself is shown to fail when one sampled output element is off by 2 %."""
    from b200dt.predictor import DetectPipeline

    torch = _torch()
    name, B, (H, W), kind, src, pad = FULL_SIZE[config]
    spec = cfg.resolve(name)
    sd = weights.synthetic_state_dict(spec, seed=0)
    hw = src or (H, W)
    base = [synth.IRStream(seed=300 + i, h=hw[0], w=hw[1], n_targets=6).frame() for i in range(8)]
    pipe = DetectPipeline(spec, sd, B, H, W)
    try:
        if kind == "u8":
            frames = torch.from_numpy(np.stack([base[b % 8] for b in range(B)])).cuda()
            pipe(frames, 0.25, 0.7, pad_top=pad)
            x_in = plan_ref.canvas_u8(frames, H, W, pad)
        else:
            x8 = torch.from_numpy(pp.preprocess(base)).cuda()
            x = x8[torch.arange(B, device="cuda") % 8].contiguous()
            if kind == "bf16":
                x = x.to(torch.bfloat16)
            pipe.run_tensor(x, 0.25, 0.7)
            x_in = x.float()
        torch.cuda.synchronize()
        eng = pipe.engine
        pix_fn = lambda b, h, w: plan_ref.sample_pixels(b, h, w, 1000, seed=h * 7 + w)      # noqa: E731
        rep = []
        worst = plan_ref.check_plan(eng, x_in, pix_fn=pix_fn, report=rep)
        kinds = {k for _, k, _ in rep}
        assert {"stem", "conv", "pool", "dfl", "cls"} <= kinds, kinds
        wi, wk, _ = max(rep, key=lambda t: t[2])
        _diag(f"full size {config}: {len(rep)} launches, worst conv rel-L2 {worst:.2e} (op {wi}, {wk}: {eng.plan.ops[wi][:10]})")

        # self-test: the sampled check fails on a 2 % error in one element
        pl = plan_ref.Plan(eng)
        op = next(o for o in eng.plan.ops if o[0] == eng_mod.OP_CONV and not o[19])
        r = plan_ref.evaluate(pl, op, x_in, pix_fn(B, *pl.out_hw(op)))
        plan_ref.check(r)
        i = np.unravel_index(np.abs(r["got"]).argmax(), r["got"].shape)
        assert abs(r["got"][i]) > 1.0
        r["got"][i] *= 1.02
        with pytest.raises(AssertionError):
            plan_ref.check(r)
    finally:
        pipe.engine.close()

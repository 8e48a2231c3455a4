"""Per-op reference of an engine launch plan (engine.py ``Plan.ops``), evaluated on the engine's own input buffers.

For one op after an engine forward, :func:`evaluate` reads the op's inputs from the engine arena (bf16 values, so the
reference starts from exactly what the kernel read), evaluates the op in float64 on the CPU with the plan's bf16 weights
and fp32 biases, and reads what the kernel wrote.  ``pix`` selects output pixels ``(b, h, w)``: only the input patches those
pixels need are gathered on the GPU and copied, so the full-size plans (256 x 512 x 640 and up) can be checked launch by
launch.  Without ``pix`` the whole output map is evaluated.  :func:`check` applies the tolerances of each op kind.

Op kinds: the stem (``x_in``: the canvas it convolves, [B][3][H][W] RGB in [0, 1] on the GPU), convs (two sources with a
nearest-2x upsample folded into the loads, shortcut, chained 1x1 conv with an extra K source), the SPPF pool, upsample /
slice copies, and the fused Detect-head epilogues (``op[19]`` 1: four DFL distances, 2: {class logit, class} as fp32
records in the op's output buffer).
"""
import numpy as np

from b200dt import engine as eng_mod
from b200dt import weights
from oracle import net as onet

U_BF16 = 2.0 ** -8           # unit roundoff of bf16 (8 significand bits): one rounding moves a value by at most U |v|
CHUNK = 1 << 22              # gathered elements per chunk


def _torch():
    import torch

    return torch


def rel_l2(a, b):
    return float(np.linalg.norm(a - b) / (np.linalg.norm(b) + 1e-12))


def all_pixels(B, Ho, Wo):
    b, h, w = np.meshgrid(np.arange(B), np.arange(Ho), np.arange(Wo), indexing="ij")
    return b.ravel(), h.ravel(), w.ravel()


def sample_pixels(B, Ho, Wo, n_random=1000, seed=0):
    """Rows and columns {0, 1, 7, 8, 15, 16, 17, mid, last-1, last} crossed, in images {0, 1, B/2, B-1}, plus ``n_random``
    uniform pixels: the tile and image borders of every tile shape the planner picks, and the bulk."""
    def edges(n):
        return sorted({v for v in (0, 1, 7, 8, 15, 16, 17, n // 2, n - 2, n - 1) if 0 <= v < n})

    imgs = sorted({0, 1 % B, B // 2, B - 1})
    b, h, w = np.meshgrid(imgs, edges(Ho), edges(Wo), indexing="ij")
    g = np.random.default_rng(seed)
    r = (g.integers(0, B, n_random), g.integers(0, Ho, n_random), g.integers(0, Wo, n_random))
    key = np.unique(np.concatenate([(b.ravel() * Ho + h.ravel()) * Wo + w.ravel(), (r[0] * Ho + r[1]) * Wo + r[2]]))
    return key // (Ho * Wo), key // Wo % Ho, key % Wo


def canvas_u8(frames, H, W, pad_top=0, pad_left=0):
    """What the stem convolves for uint8 BGR ``frames`` [B][h][w][3] (CUDA) letterboxed at (pad_top, pad_left) into H x W:
    border 114, RGB, / 255, as float32 [B][3][H][W]."""
    torch = _torch()
    B, h, w, _ = frames.shape
    c = torch.full((B, H, W, 3), 114, dtype=torch.uint8, device=frames.device)
    c[:, pad_top:pad_top + h, pad_left:pad_left + w] = frames
    return c.flip(-1).permute(0, 3, 1, 2).float() / 255.0


def _gather(t, b, y, x, c0, c1, up=1, Hv=None, Wv=None, fill=0.0):
    """t: [B][h][w][C] CUDA tensor; b, y, x: CUDA int64 of one shape (coordinates at the virtual resolution h*up x w*up).
    Returns float32 [..., c1 - c0] on the GPU, ``fill`` outside the map."""
    Hv = t.shape[1] * up if Hv is None else Hv
    Wv = t.shape[2] * up if Wv is None else Wv
    ok = (y >= 0) & (y < Hv) & (x >= 0) & (x < Wv)
    v = t[b, (y.clamp(0, Hv - 1) // up), (x.clamp(0, Wv - 1) // up), c0:c1].float()
    v[~ok] = fill
    return v


def _silu(x):
    return x / (1.0 + np.exp(-x))


def _bf16_round64(a):
    return onet.bf16_round(a.astype(np.float32)).astype(np.float64)


def _blob_bf16(blob, off, n):
    return weights.bf16_bits_to_f32(np.frombuffer(blob, np.uint16, count=n, offset=off)).astype(np.float64)


def _blob_f32(blob, off, n):
    return np.frombuffer(blob, np.float32, count=n, offset=off).astype(np.float64)


class Plan:
    """The engine's plan with the weight blob read once and the buffers as CUDA views."""

    def __init__(self, eng):
        self.eng, self.P, self.blob = eng, eng.plan, eng.plan.blob.bytes()
        self.B = eng.B
        self._views = {}

    def buf(self, i):
        if i not in self._views:
            self._views[i] = self.eng.buffer(i)
        return self._views[i]

    def out_hw(self, op):
        if op[0] == eng_mod.OP_POOL:
            return self.P.bufs[op[1]][:2]
        if op[0] == eng_mod.OP_STEM:
            return self.P.bufs[op[1]][:2]
        if op[0] == eng_mod.OP_UP:
            return self.P.bufs[op[5]][:2]
        return self.P.bufs[op[4]][:2]


def _chunks(n, per_pixel):
    step = max(1, CHUNK // max(1, per_pixel))
    for s in range(0, n, step):
        yield slice(s, min(n, s + step))


def _conv(pl, op, b, h, w):
    """Reference and kernel output of an OP_CONV at pixels (b, h, w) (CUDA int64).  Returns dict(ref, absdot, got)."""
    torch = _torch()
    _, ib, ioff, cin, ob, ooff, cout, k, s, act, rb, roff, woff, boff = op[:14]
    ib2, ioff2, cin2, up0, up1, epi = op[14:20]
    up0 = 2 if up0 == 2 else 1
    up1 = 2 if up1 == 2 else 1
    x0 = pl.buf(ib)
    Hv, Wv = x0.shape[1] * up0, x0.shape[2] * up0
    ct = cin + (cin2 if ib2 >= 0 else 0)
    wm = _blob_bf16(pl.blob, woff, cout * k * k * ct).reshape(cout, k * k * ct).T           # [k*k*ct][cout], K order (kh, kw, c)
    bias = _blob_f32(pl.blob, boff, cout)
    chained = bool(op[20])
    if chained:
        w2off, b2off, cout2, act2, xb, xoff, xc = op[21:28]
        xc = xc if xb >= 0 else 0
        w2 = _blob_bf16(pl.blob, w2off, cout2 * (xc + cout)).reshape(cout2, xc + cout).T
        b2 = _blob_f32(pl.blob, b2off, cout2)
    p = k // 2
    dy = torch.arange(k, device=b.device)
    refs, absd = [], []
    for sl in _chunks(len(b), k * k * ct):
        bb, hh, ww = b[sl], h[sl], w[sl]
        bk, yy, xx = torch.broadcast_tensors(bb[:, None, None], (hh * s - p)[:, None, None] + dy[None, :, None],
                                             (ww * s - p)[:, None, None] + dy[None, None, :])
        a = _gather(x0, bk, yy, xx, ioff, ioff + cin, up0, Hv, Wv)
        if ib2 >= 0:
            a = torch.cat([a, _gather(pl.buf(ib2), bk, yy, xx, ioff2, ioff2 + cin2, up1, Hv, Wv)], -1)
        a = a.reshape(len(bb), k * k * ct).cpu().numpy().astype(np.float64)
        z = a @ wm + bias
        ad = np.abs(a) @ np.abs(wm) + np.abs(bias)
        if act:
            z = _silu(z)
        if rb >= 0:
            r = _gather(pl.buf(rb), bb, hh, ww, roff, roff + cout).cpu().numpy().astype(np.float64)
            z = z + r
            ad = ad + np.abs(r)
        if chained:
            # the main conv's tile is rounded to bf16 (as the unchained path stores it) and read behind the extra source
            mid = _bf16_round64(z)
            if xc:
                mid = np.concatenate([_gather(pl.buf(xb), bb, hh, ww, xoff, xoff + xc).cpu().numpy().astype(np.float64), mid], 1)
            z = mid @ w2 + b2
            ad = np.abs(mid) @ np.abs(w2) + np.abs(b2)
            if act2:
                z = _silu(z)
        refs.append(z)
        absd.append(ad)
    ref, absdot = np.concatenate(refs), np.concatenate(absd)
    cf = cout2 if chained else cout
    if epi:
        rec = pl.buf(ob).view(torch.float32)                       # fp32 records: 4 distances, or {logit, class}
        got = rec[b, h, w].cpu().numpy().astype(np.float64)
    else:
        got = pl.buf(ob)[b, h, w, ooff:ooff + cf].float().cpu().numpy().astype(np.float64)
    return dict(kind={0: "conv", 1: "dfl", 2: "cls"}[epi], ref=ref, absdot=absdot, got=got)


def _stem(pl, op, x_in, b, h, w):
    torch = _torch()
    _, ob, ooff, c0, woff, boff = op[:6]
    wm = _blob_bf16(pl.blob, woff, c0 * 32).reshape(c0, 32)[:, :27].T                 # K = (kh, kw, rgb)
    bias = _blob_f32(pl.blob, boff, c0)
    xs = x_in.permute(0, 2, 3, 1)                                                      # NHWC view of the canvas
    d = torch.arange(3, device=b.device)
    bk, yy, xx = torch.broadcast_tensors(b[:, None, None], (2 * h - 1)[:, None, None] + d[None, :, None], (2 * w - 1)[:, None, None] + d[None, None, :])
    a = _gather(xs, bk, yy, xx, 0, 3).reshape(len(b), 27).cpu().numpy().astype(np.float64)
    ref = _silu(a @ wm + bias)
    got = pl.buf(ob)[b, h, w, ooff:ooff + c0].float().cpu().numpy().astype(np.float64)
    return dict(kind="stem", ref=ref, got=got)


def _pool(pl, op, b, h, w):
    """SPPF: slice j (1..3) is slice 0 max-pooled three times by 5x5 with -inf padding == the max over the (4j+1)^2 window
    clipped to the map.  Maxima of bf16 values are exact, so the reference is taken on the GPU."""
    torch = _torch()
    _, bi, off, c = op[:4]
    t = pl.buf(bi)
    refs, gots = [], []
    for j in (1, 2, 3):
        r = 2 * j
        d = torch.arange(-r, r + 1, device=b.device)
        out = []
        for sl in _chunks(len(b), (2 * r + 1) ** 2 * c):
            bk, yy, xx = torch.broadcast_tensors(b[sl][:, None, None], h[sl][:, None, None] + d[None, :, None], w[sl][:, None, None] + d[None, None, :])
            v = _gather(t, bk, yy, xx, off, off + c, fill=-np.inf)
            out.append(v.amax(dim=(1, 2)).cpu().numpy())
        refs.append(np.concatenate(out))
        gots.append(t[b, h, w, off + j * c:off + (j + 1) * c].float().cpu().numpy())
    return dict(kind="pool", ref=np.concatenate(refs, 1), got=np.concatenate(gots, 1))


def _up(pl, op, b, h, w):
    _, ib, ioff, c, scale, ob, ooff = op[:7]
    ref = pl.buf(ib)[b, h // scale, w // scale, ioff:ioff + c].float().cpu().numpy()
    got = pl.buf(ob)[b, h, w, ooff:ooff + c].float().cpu().numpy()
    return dict(kind="up", ref=ref, got=got)


def evaluate(pl, op, x_in=None, pix=None):
    """Reference and kernel output of one plan op.  ``pl``: :class:`Plan`; ``x_in``: the stem's canvas (OP_STEM only);
    ``pix``: (b, h, w) integer arrays of output pixels, or None for the whole map."""
    torch = _torch()
    if pix is None:
        pix = all_pixels(pl.B, *pl.out_hw(op))
    dev = pl.buf(op[1]).device
    b, h, w = (torch.as_tensor(np.asarray(v, np.int64), device=dev) for v in pix)
    if op[0] == eng_mod.OP_CONV:
        return _conv(pl, op, b, h, w)
    if op[0] == eng_mod.OP_STEM:
        return _stem(pl, op, x_in, b, h, w)
    if op[0] == eng_mod.OP_POOL:
        return _pool(pl, op, b, h, w)
    if op[0] == eng_mod.OP_UP:
        return _up(pl, op, b, h, w)
    raise ValueError(f"opcode {op[0]}")


def head_logit_tol(z, absdot):
    """How far a kernel logit may sit from the float64 reference: one bf16 rounding of the logit (U |z|) plus the fp32
    accumulation noise and, in the chained head, a bf16 rounding of the intermediate tile that lands on the other side of a
    tie (2^-10 of sum |w x|)."""
    return U_BF16 * np.abs(z) + 2.0 ** -10 * absdot + 1e-6


def check(r, what=""):
    """Assert the kernel output of one :func:`evaluate` result against its reference.  Returns the rel-L2 error (convs, stem)
    or 0 for the exact and record kinds.

    * conv / stem: rel-L2 < 4e-3 and |got - ref| <= 1e-2 |ref| + 1e-2 max(1, max|ref| / 16) (about one bf16 rounding of the
      output plus fp32 accumulation-order noise);
    * pool / upsample: bit-exact;
    * DFL records: each distance within sum_i p_i |i - d| dz_i (the first-order effect of moving each of the 16 logits by
      its tolerance dz_i from :func:`head_logit_tol`), times 1.5, plus 2e-4 for the fp32 softmax;
    * class records: the logit within two roundings (one bf16 ulp) of the reference maximum; the class is the reference
      arg-max (lowest index on ties), or a class whose reference logit is within that tolerance of the maximum."""
    kind, got, ref = r["kind"], r["got"], r["ref"]
    if kind in ("pool", "up"):
        np.testing.assert_array_equal(got, ref, err_msg=what)
        return 0.0
    if kind in ("conv", "stem"):
        assert got.shape == ref.shape, (what, got.shape, ref.shape)
        err = rel_l2(got, ref)
        assert err < 4e-3, (what, err)
        np.testing.assert_allclose(got, ref, rtol=1e-2, atol=1e-2 * max(1.0, float(np.abs(ref).max()) / 16), err_msg=what)
        return err
    z, ad = r["ref"], r["absdot"]
    tol = head_logit_tol(z, ad)
    if kind == "dfl":
        z4 = z.reshape(-1, 4, 16)
        t4 = tol.reshape(-1, 4, 16)
        e = np.exp(z4 - z4.max(-1, keepdims=True))
        pr = e / e.sum(-1, keepdims=True)
        bins = np.arange(16.0)
        d = (pr * bins).sum(-1)
        bound = 1.5 * (pr * np.abs(bins - d[..., None]) * t4).sum(-1) + 2e-4
        dev = np.abs(got - d)
        bad = np.argwhere(~(dev <= bound))
        assert len(bad) == 0, (what, "DFL distance outside its bound", len(bad), [(tuple(i), got[tuple(i)], d[tuple(i)], bound[tuple(i)]) for i in bad[:5]])
        return 0.0
    # class records
    nc = z.shape[1]
    zmax = z.max(1)
    tmax = 2 * U_BF16 * np.abs(zmax) + tol.max(1)
    logit, cls = got[:, 0], got[:, 1]
    assert np.all(cls == np.round(cls)) and np.all((cls >= 0) & (cls < nc)), (what, "class index out of range")
    bad = np.nonzero(~(np.abs(logit - zmax) <= tmax))[0]
    assert len(bad) == 0, (what, "class logit", len(bad), [(i, logit[i], zmax[i], tmax[i]) for i in bad[:5]])
    arg = z.argmax(1)
    ci = cls.astype(np.int64)
    zc = z[np.arange(len(z)), ci]
    bad = np.nonzero((ci != arg) & ~(zc >= zmax - 2 * tmax))[0]
    assert len(bad) == 0, (what, "class arg-max", len(bad), [(i, ci[i], arg[i], zc[i], zmax[i]) for i in bad[:5]])
    return 0.0


def check_plan(eng, x_in, pix_fn=None, report=None):
    """Check every op of ``eng``'s plan after a forward.  ``pix_fn(B, Ho, Wo)`` picks the output pixels of each op (None:
    whole maps).  Returns the worst conv / stem rel-L2; ``report``, if a list, collects (op index, kind, rel-L2)."""
    pl = Plan(eng)
    worst = 0.0
    for i, op in enumerate(pl.P.ops):
        pix = pix_fn(pl.B, *pl.out_hw(op)) if pix_fn else None
        r = evaluate(pl, op, x_in, pix)
        err = check(r, f"op {i} {r['kind']} {op}")
        worst = max(worst, err)
        if report is not None:
            report.append((i, r["kind"], err))
    return worst

"""Lowering of the resolved YOLOv8-P2 graph to the launch plan executed by ``b2_engine_*`` (csrc/engine.cu).

Host-side counterpart of ``BaseModel._predict_once`` (ultralytics/nn/tasks.py:159-188) plus
``BaseModel.fuse`` (:224-254): the layer list of :func:`cfg.resolve` is flattened into a program over NHWC
bf16 buffers in which every ``torch.cat`` / ``chunk`` of C2f (block.py:315-319), SPPF (:237-241),
``Concat`` (conv.py:673-683) and Detect (head.py:116-121) is a channel offset:

  * a ``Concat`` layer owns one buffer; its producers write straight into their channel slice
    (``nn.Upsample`` becomes the slice-writing copy kernel);
  * a ``C2f`` owns a (2+n)*c buffer: ``cv1`` fills [0, 2c), bottleneck j reads slice 1+j and writes slice 2+j
    (residual read from slice 1+j), ``cv2`` reads the whole buffer;
  * ``SPPF`` owns a 4*c_ buffer filled by ``cv1`` and the pooling kernel;
  * each Detect level owns a ``[B][h*w][64 + ceil8(nc)]`` logits buffer filled by ``cv2[l][2]`` / ``cv3[l][2]``.

Plan layout (int32 words): ``[magic, n_bufs, n_ops, n_levels, nc, lstride]``, ``n_bufs x (h, w, c)``,
``n_levels x (buf, stride)``, ``n_ops x 28`` (opcode + 27 arguments, see ``OP_*`` below and csrc/engine.cu).

Chained launches (``chain=True``, default): a 3x3 conv whose output is read only by a following 1x1 conv runs WITH that 1x1
conv in one launch -- the intermediate tile stays in shared memory (csrc/conv_tc.cu, ``ConvParams::chain``).  Three places:
``Conv(k3, s2) -> C2f.cv1``, ``Bottleneck[n-1].cv2 (+ shortcut) -> C2f.cv2`` (the other channels of the C2f buffer are the 1x1
conv's extra K source) and the Detect tails ``cv2[l][1] -> cv2[l][2]`` / ``cv3[l][1] -> cv3[l][2]``.  Each is taken only when
``b2_conv_chain_plan_ok`` says the pair fits the chained kernel; otherwise the two convs stay separate launches.

``Concat([Upsample(a), b])`` feeding a C2f is *virtual*: its ``cv1`` 1x1 conv takes both tensors as inputs and the
nearest-2x upsample is folded into the conv's TMA loads (zero-stride tensor-map dimensions), so neither the upsampled
tensor nor the concatenation is ever written.
"""
from __future__ import annotations

import os

import ctypes as C

import numpy as np

from . import _lib, cfg, weights

MAGIC = 0xB2D7
OP_STEM, OP_CONV, OP_POOL, OP_UP = 1, 2, 3, 4
OP_WORDS = 28
ACT_NONE, ACT_SILU = 0, 1


class _Blob:
    """Weight blob builder: 256-byte aligned sections."""

    def __init__(self):
        self.parts, self.size = [], 0

    def add(self, arr):
        raw = np.ascontiguousarray(arr).tobytes()
        off = self.size
        pad = (-len(raw)) % 256
        self.parts.append(raw + b"\0" * pad)
        self.size += len(raw) + pad
        return off

    def bytes(self):
        return b"".join(self.parts)


class Plan:
    """Result of :func:`lower`: the int32 program, the weight blob and where every tensor lives."""

    def __init__(self):
        self.bufs = []          # (h, w, c)
        self.ops = []           # lists of OP_WORDS ints
        self.levels = []        # (buf, stride, dist_buf, cls_buf); the last two are -1 without the fused head
        self.loc = {}           # layer index -> (buf, coff, C)
        self.named = {}         # module path (e.g. 'model.2.m.0.cv1') -> (buf, coff, C)
        self.blob = _Blob()
        self.nc = 0
        self.lstride = 0
        self.flops = 0

    def new_buf(self, h, w, c):
        self.bufs.append((int(h), int(w), int(c)))
        return len(self.bufs) - 1

    def words(self):
        head = [MAGIC, len(self.bufs), len(self.ops), len(self.levels), self.nc, self.lstride]
        flat = head + [v for b in self.bufs for v in b] + [v for l in self.levels for v in l] + [v for o in self.ops for v in o]
        return np.asarray(flat, dtype=np.int32)


def _shapes(spec, H, W):
    """(h, w) of every layer output for an H x W input."""
    hw, cur = {}, (H, W)
    for L in spec["layers"]:
        f = L["f"]
        f0 = f[0] if isinstance(f, tuple) else f
        h, w = cur if f0 == -1 else hw[f0]
        if L["type"] == "Conv":
            p = L["k"] // 2
            h, w = (h + 2 * p - L["k"]) // L["s"] + 1, (w + 2 * p - L["k"]) // L["s"] + 1
        elif L["type"] == "Upsample":
            h, w = 2 * h, 2 * w
        hw[L["i"]] = (h, w)
        cur = (h, w)
    return hw


def _chain_ok(H, W, cin, cout, k, s, has_res, xc, cout2):
    """Would the chained kernel take this (3x3 conv at input resolution H x W) -> (1x1 conv) pair?  Pure planning in the library."""
    try:
        lib = _lib.load()
    except Exception:
        return False
    return bool(lib.b2_conv_chain_plan_ok(1, int(H), int(W), int(cin), int(cout), int(k), int(s), int(bool(has_res)), int(xc), int(cout2)))


CHAIN_CONV_CV1, CHAIN_C2F_TAIL, CHAIN_DETECT_BOX, CHAIN_DETECT_CLS = 1, 2, 4, 8
# measured on the bench workload (tools/ab_chain.py, one process, per-launch CUDA events; conv time of one forward 10.33 ms unchained):
# CONV_CV1 -0.07 ms, C2F_TAIL -0.11 ms, DETECT_BOX -0.10 ms, DETECT_CLS +0.19 ms (its class-max epilogue on 8 warps is slower than
# the stand-alone tail kernel's 16) -> the class tail stays a launch of its own
CHAIN_DEFAULT = CHAIN_CONV_CV1 | CHAIN_C2F_TAIL | CHAIN_DETECT_BOX


def lower(spec, state_dict, H, W, fuse_head=False, merge_head=True, chain=True):
    """Lower ``spec`` (from :func:`cfg.resolve`) with weights ``state_dict`` for an ``H x W`` letterboxed input.

    ``fuse_head``: run DFL (softmax expectation) and the class max inside the epilogue of each Detect level's last
    two convs (head.py:152-187 fused into head.py:93-96): the ``64 + nc`` logits are never written; the engine then
    exposes ``b2_engine_head`` buffers instead of ``b2_engine_levels`` logits."""
    if H % 32 or W % 32:
        raise ValueError(f"input size {H}x{W} must be a multiple of the maximum stride 32")
    chain = CHAIN_DEFAULT if chain is True else int(chain or 0)      # bit mask of the CHAIN_* patterns to take
    sd = state_dict
    layers = spec["layers"]
    hw = _shapes(spec, H, W)
    P = Plan()
    nc = spec["nc"]
    P.nc = nc
    P.lstride = 64 + ((nc + 7) // 8) * 8

    def src(i, f):
        return i - 1 if f == -1 else f

    # ---- placement: which concat slice does each layer write into? ----
    placement = {}
    extra_copies = []                     # (layer, concat buffer slice) when a layer feeds a second Concat
    consumers = {}
    for L in layers:
        fs = L["f"] if isinstance(L["f"], tuple) else (L["f"],)
        for f in fs:
            consumers.setdefault(src(L["i"], f), []).append(L["i"])
    virtual = {}                          # concat layer -> [(source layer, up)], upsample layers folded away
    for L in layers:
        if L["type"] != "Concat" or len(L["f"]) != 2:
            continue
        i = L["i"]
        a, b = (src(i, f) for f in L["f"])
        cons = consumers.get(i, [])
        if (layers[a]["type"] == "Upsample" and consumers.get(a) == [i] and len(cons) == 1 and layers[cons[0]]["type"] == "C2f"
                and layers[b]["type"] != "Upsample"):
            virtual[i] = [(src(a, layers[a]["f"]), 2), (b, 1)]
    for L in layers:
        if L["type"] != "Concat" or L["i"] in virtual:
            continue
        i = L["i"]
        h, w = hw[i]
        buf = P.new_buf(h, w, L["c_out"])
        off = 0
        for f in L["f"]:
            s = src(i, f)
            c = layers[s]["c_out"]
            if s in placement:
                extra_copies.append((s, (buf, off, c)))
            else:
                placement[s] = (buf, off, c)
            off += c
        P.loc[i] = (buf, 0, L["c_out"])

    def out_loc(L):
        i = L["i"]
        if i in placement:
            return placement[i]
        h, w = hw[i]
        return (P.new_buf(h, w, L["c_out"]), 0, L["c_out"])

    def check_c(c, what):
        if c % 16:
            raise NotImplementedError(f"{what}: {c} channels -- the tcgen05 conv path needs multiples of 16")

    def emit_conv(prefix, inp, out, k, s, bn, res=None, inp2=None, ups=(1, 1), epi=0, chain2=None):
        """inp/out/res/inp2: (buf, coff, C).  inp2: second input of a folded Concat; ups: resolution factors of the inputs.
        chain2: dict(prefix, bn, x) -- the 1x1 conv ``prefix`` chained onto this conv (x: (buf, coff, C) extra K source or None);
        ``out`` and ``epi`` then describe the chained conv's output.
        prefix: one module name, or a tuple of modules that read the same input -- their filters are stacked along Cout and run
        as ONE GEMM (the input tile is fetched once, and a wider N uses the tensor pipe better: N = 144 runs at the pipe's
        N/2 cycles per MMA where N = 64 and N = 80 are bound by the operand fetch); ``out`` then covers all their channels."""
        if isinstance(prefix, tuple):
            ws, bs = zip(*(weights.folded(sd, q, bn) for q in prefix))
            w, b = np.concatenate(ws, 0), np.concatenate(bs, 0)
            c0 = out[1]
            for q, wq in zip(prefix, ws):
                P.named[q] = (out[0], c0, wq.shape[0])
                c0 += wq.shape[0]
            prefix = "+".join(prefix)
        else:
            w, b = weights.folded(sd, prefix, bn)
        cout, cin = w.shape[0], w.shape[1]
        assert cin == inp[2] + (inp2[2] if inp2 else 0) and (epi or chain2 or cout == out[2]), (prefix, w.shape, inp, inp2, out)
        check_c(inp[2], prefix + " input")
        if inp2:
            check_c(inp2[2], prefix + " second input")
        woff = P.blob.add(weights.f32_to_bf16_bits(weights.pack_ohwi(w)))
        boff = P.blob.add(b.astype(np.float32))
        hb, wb, _ = P.bufs[out[0]]
        P.flops += 2 * hb * wb * cout * cin * k * k
        tail = [0] * 8
        if chain2:
            w2, b2 = weights.folded(sd, chain2["prefix"], chain2["bn"])
            x = chain2.get("x")
            cout2, k2 = w2.shape[0], w2.shape[1]
            assert w2.shape[2:] == (1, 1) and k2 == cout + (x[2] if x else 0) and (epi or cout2 == out[2]), (chain2["prefix"], w2.shape, out)
            w2off = P.blob.add(weights.f32_to_bf16_bits(w2.reshape(cout2, k2)))
            b2off = P.blob.add(b2.astype(np.float32))
            P.flops += 2 * hb * wb * cout2 * k2
            tail = [1, w2off, b2off, cout2, ACT_SILU if chain2["bn"] else ACT_NONE, x[0] if x else -1, x[1] if x else 0, x[2] if x else 0]
            P.named[chain2["prefix"]] = out
        P.ops.append([OP_CONV, inp[0], inp[1], inp[2], out[0], out[1], cout, k, s, ACT_SILU if bn else ACT_NONE,
                      res[0] if res else -1, res[1] if res else 0, woff, boff,
                      inp2[0] if inp2 else -1, inp2[1] if inp2 else 0, inp2[2] if inp2 else 0, ups[0], ups[1], epi] + tail)
        if not chain2:
            P.named[prefix] = out

    pending = {}                          # Conv layers chained into the cv1 of the C2f that follows them
    for L in layers:
        i, t = L["i"], L["type"]
        p = f"model.{i}"
        h, w = hw[i]
        if t == "Conv":
            out = None
            if i == 0:
                out = out_loc(L)
                if L["k"] != 3 or L["s"] != 2 or L["c1"] != 3:
                    raise NotImplementedError("stem must be Conv(3 -> C0, k=3, s=2)")
                wf, bf = weights.fold_conv_bn(sd, p)
                woff = P.blob.add(weights.pack_stem(wf))                       # [C0][32] bf16, K = (kh,kw,rgb) padded
                boff = P.blob.add(bf.astype(np.float32))
                P.flops += 2 * h * w * L["c2"] * 27
                P.ops.append([OP_STEM, out[0], out[1], L["c2"], woff, boff] + [0] * (OP_WORDS - 6))
                P.named[p] = out
            else:
                nxt = consumers.get(i, [])
                Lc = layers[nxt[0]] if len(nxt) == 1 else None
                hi_, wi_ = hw[src(i, L["f"])]
                if ((chain & CHAIN_CONV_CV1) and Lc is not None and Lc["type"] == "C2f" and not isinstance(Lc["f"], tuple) and src(Lc["i"], Lc["f"]) == i
                        and i not in placement and L["k"] == 3 and _chain_ok(hi_, wi_, L["c1"], L["c2"], 3, L["s"], False, 0, 2 * Lc["c"])):
                    pending[i] = (p, P.loc[src(i, L["f"])], L)          # emitted together with the C2f's cv1
                    P.loc[i] = None
                    continue
                out = out_loc(L)
                emit_conv(p, P.loc[src(i, L["f"])], out, L["k"], L["s"], True)
            P.loc[i] = out
        elif t == "C2f":
            c, n = L["c"], L["n"]
            check_c(c, p + " hidden")
            s_in = src(i, L["f"])
            cat = P.new_buf(h, w, (2 + n) * c)
            if s_in in virtual:                                   # Concat([Upsample(a), b]) folded into cv1
                (la, ua), (lb, ub) = virtual[s_in]
                emit_conv(p + ".cv1", P.loc[la], (cat, 0, 2 * c), 1, 1, True, inp2=P.loc[lb], ups=(ua, ub))
            elif s_in in pending:                                 # Conv(k3) -> cv1 in one launch
                pp, pin, Lp = pending.pop(s_in)
                emit_conv(pp, pin, (cat, 0, 2 * c), Lp["k"], Lp["s"], True, chain2=dict(prefix=p + ".cv1", bn=True, x=None))
            else:
                emit_conv(p + ".cv1", P.loc[s_in], (cat, 0, 2 * c), 1, 1, True)
            out = out_loc(L)
            for j in range(n):
                a = (cat, (1 + j) * c, c)
                tmp = P.new_buf(h, w, c)
                emit_conv(f"{p}.m.{j}.cv1", a, (tmp, 0, c), 3, 1, True)
                res = a if L["shortcut"] else None
                if (chain & CHAIN_C2F_TAIL) and j == n - 1 and _chain_ok(h, w, c, c, 3, 1, res is not None, (1 + n) * c, L["c2"]):
                    # last bottleneck conv + cv2 in one launch: cv2's other inputs (y0, y1, m_1..m_n-1) are the first (1+n)c
                    # channels of the C2f buffer, its last c input channels never leave the SM
                    emit_conv(f"{p}.m.{j}.cv2", (tmp, 0, c), out, 3, 1, True, res=res,
                              chain2=dict(prefix=p + ".cv2", bn=True, x=(cat, 0, (1 + n) * c)))
                    break
                emit_conv(f"{p}.m.{j}.cv2", (tmp, 0, c), (cat, (2 + j) * c, c), 3, 1, True, res=res)
            else:
                emit_conv(p + ".cv2", (cat, 0, (2 + n) * c), out, 1, 1, True)
            P.loc[i] = out
        elif t == "SPPF":
            if L["k"] != 5:
                raise NotImplementedError("SPPF: only k=5")
            c_ = L["c1"] // 2
            inp = P.loc[src(i, L["f"])]
            cat = P.new_buf(h, w, 4 * c_)
            emit_conv(p + ".cv1", inp, (cat, 0, c_), 1, 1, True)
            P.ops.append([OP_POOL, cat, 0, c_] + [0] * (OP_WORDS - 4))
            out = out_loc(L)
            emit_conv(p + ".cv2", (cat, 0, 4 * c_), out, 1, 1, True)
            P.loc[i] = out
        elif t == "Upsample":
            if any(i == src(c_, layers[c_]["f"][0]) for c_ in virtual):
                continue                              # folded into the consumer conv's loads
            inp = P.loc[src(i, L["f"])]
            out = out_loc(L)
            P.ops.append([OP_UP, inp[0], inp[1], inp[2], 2, out[0], out[1]] + [0] * (OP_WORDS - 7))
            P.loc[i] = out
        elif t == "Concat":
            pass                                  # producers already wrote their slices
        elif t == "Detect":
            cb, cc = L["c2_box"], L["c3_cls"]
            for l, f in enumerate(L["f"]):
                inp = P.loc[f]
                hh, ww = hw[f]
                if merge_head and (cb + cc) <= 256 and cb % 8 == 0:
                    # the first conv of the box branch and of the class branch read the same feature map: one conv, Cout = cb + cc
                    tu = P.new_buf(hh, ww, cb + cc)
                    emit_conv((f"{p}.cv2.{l}.0", f"{p}.cv3.{l}.0"), inp, (tu, 0, cb + cc), 3, 1, True)
                    t1_loc, u1_loc = (tu, 0, cb), (tu, cb, cc)
                else:
                    t1, u1 = P.new_buf(hh, ww, cb), P.new_buf(hh, ww, cc)
                    emit_conv(f"{p}.cv2.{l}.0", inp, (t1, 0, cb), 3, 1, True)
                    emit_conv(f"{p}.cv3.{l}.0", inp, (u1, 0, cc), 3, 1, True)
                    t1_loc, u1_loc = (t1, 0, cb), (u1, 0, cc)
                if fuse_head and nc <= 256:
                    dist = P.new_buf(hh, ww, 8)                       # 4 fp32 per pixel
                    clsb = P.new_buf(hh, ww, 4)                       # 2 fp32 per pixel
                    for q, a_loc, c_, o_loc, e_, n2 in ((f"{p}.cv2.{l}", t1_loc, cb, (dist, 0, 8), 1, 64),
                                                    (f"{p}.cv3.{l}", u1_loc, cc, (clsb, 0, 4), 2, nc)):
                        if (chain & (CHAIN_DETECT_BOX if e_ == 1 else CHAIN_DETECT_CLS)) and _chain_ok(hh, ww, c_, c_, 3, 1, False, 0, n2):
                            # 3x3 conv + the branch's final 1x1 conv + DFL / class-max epilogue in one launch
                            emit_conv(q + ".1", a_loc, o_loc, 3, 1, True, epi=e_, chain2=dict(prefix=q + ".2", bn=False, x=None))
                        else:
                            t_loc = (P.new_buf(hh, ww, c_), 0, c_)
                            emit_conv(q + ".1", a_loc, t_loc, 3, 1, True)
                            emit_conv(q + ".2", t_loc, o_loc, 1, 1, False, epi=e_)
                    P.levels.append((-1, H // hh, dist, clsb))
                else:
                    t2, u2 = P.new_buf(hh, ww, cb), P.new_buf(hh, ww, cc)
                    emit_conv(f"{p}.cv2.{l}.1", t1_loc, (t2, 0, cb), 3, 1, True)
                    emit_conv(f"{p}.cv3.{l}.1", u1_loc, (u2, 0, cc), 3, 1, True)
                    logits = P.new_buf(hh, ww, P.lstride)
                    emit_conv(f"{p}.cv2.{l}.2", (t2, 0, cb), (logits, 0, 64), 1, 1, False)
                    emit_conv(f"{p}.cv3.{l}.2", (u2, 0, cc), (logits, 64, nc), 1, 1, False)
                    P.levels.append((logits, H // hh, -1, -1))
        else:
            raise NotImplementedError(t)
        # a layer that feeds more than one Concat: copy its slice into the others
        for s_, dst in extra_copies:
            if s_ == i:
                o = P.loc[i]
                P.ops.append([OP_UP, o[0], o[1], o[2], 1, dst[0], dst[1]] + [0] * (OP_WORDS - 7))
    for o in P.ops:
        assert len(o) == OP_WORDS, o
    return P


class Engine:
    """One compiled forward for a fixed (batch, H, W): owns the device arena, weights and CUDA graph.

    Stands where ``AutoBackend(model=nn.Module, fuse=True)`` stands in the reference
    (ultralytics/nn/autobackend.py:196-219, :608-637).
    """

    def __init__(self, spec, state_dict, batch, H, W, fuse_head=False):
        _lib.require_cuda()
        self.lib = _lib.load()
        self.spec, self.B, self.H, self.W = spec, int(batch), int(H), int(W)
        self.lowered_spec = spec
        if weights.needs_padding(spec):
            # widths that are not multiples of 16 (yolov8-small.yaml at its default scale: 12 / 24): the same function with the
            # hidden widths rounded up and zero weights in the padding (weights.pad_channels)
            self.lowered_spec, state_dict = weights.pad_channels(spec, state_dict)
        # B2_MERGE_HEAD=0: keep Detect's first box / class convs as two launches (A/B experiments)
        self.plan = lower(self.lowered_spec, state_dict, H, W, fuse_head=fuse_head, merge_head=os.environ.get("B2_MERGE_HEAD", "1") != "0",
                          chain=int(os.environ.get("B2_CHAIN", str(CHAIN_DEFAULT))))      # B2_CHAIN: bit mask of CHAIN_* (0: every conv its own launch)
        self.fused_head = self.plan.levels[0][0] < 0
        words = self.plan.words()
        blob = self.plan.blob.bytes()
        self._h = C.c_void_p()
        rc = self.lib.b2_engine_create(words.ctypes.data_as(C.c_void_p), len(words), blob, len(blob),
                                       self.B, self.H, self.W, C.byref(self._h))
        _lib.check(rc)
        n = C.c_int()
        ptrs = (C.c_void_p * 8)()
        hs, ws, ss = (C.c_int * 8)(), (C.c_int * 8)(), (C.c_int * 8)()
        ls = C.c_int()
        _lib.check(self.lib.b2_engine_levels(self._h, C.byref(n), ptrs, hs, ws, ss, C.byref(ls)))   # logits pointers are NULL with the fused head
        self.n_levels, self.lstride, self.nc = n.value, ls.value, spec["nc"]
        self.level_ptrs = [ptrs[i] for i in range(n.value)]
        self.level_h = [hs[i] for i in range(n.value)]
        self.level_w = [ws[i] for i in range(n.value)]
        self.level_stride = [ss[i] for i in range(n.value)]
        self.num_anchors = sum(h * w for h, w in zip(self.level_h, self.level_w))
        self.head_dist = self.head_cls = None
        if self.fused_head:
            dp, cp = (C.c_void_p * 8)(), (C.c_void_p * 8)()
            _lib.check(self.lib.b2_engine_head(self._h, dp, cp))
            self.head_dist = [dp[i] for i in range(n.value)]
            self.head_cls = [cp[i] for i in range(n.value)]
        self.flops_per_image = cfg.conv_flops(spec, H, W)          # algorithmic FLOPs of the model as given (padding channels are not work)
        self.stride = max(self.level_stride)
        self.names = spec["names"]

    def close(self):
        if getattr(self, "_h", None):
            self.lib.b2_engine_destroy(self._h)
            self._h = None

    __del__ = close

    @property
    def arena_bytes(self):
        return self.lib.b2_engine_arena_bytes(self._h)

    @property
    def launches_per_forward(self):
        return self.lib.b2_engine_num_launches(self._h)

    def use_graph(self, on):
        _lib.check(self.lib.b2_engine_use_graph(self._h, int(bool(on))))

    def forward_u8(self, frames, pad_top=0, pad_left=0, stream=None):
        """frames: CUDA uint8 tensor [B][h][w][3] BGR; letterboxed (border 114) into the H x W canvas."""
        assert frames.is_cuda and frames.dtype.itemsize == 1 and frames.is_contiguous()
        b, sh, sw, ch = frames.shape
        if b != self.B or ch != 3:
            raise ValueError(f"expected {self.B} BGR frames, got {tuple(frames.shape)}")
        _lib.check(self.lib.b2_engine_forward_u8(self._h, _lib.ptr(frames), sh, sw, pad_top, pad_left, _lib.stream_ptr(stream)))

    def profile_u8(self, frames, pad_top=0, pad_left=0, stream=None):
        """Per-launch device milliseconds of one eager forward (CUDA events on the launch stream) and the
        algorithmic FLOPs of each launch: list of dicts {op, ms, flops, desc}."""
        n = self.launches_per_forward
        ms = (C.c_float * n)()
        b, sh, sw, _ = frames.shape
        _lib.check(self.lib.b2_engine_profile_u8(self._h, _lib.ptr(frames), sh, sw, pad_top, pad_left, ms, _lib.stream_ptr(stream)))
        out = []
        for i, op in enumerate(self.plan.ops):
            kind = {OP_STEM: "stem", OP_CONV: "conv", OP_POOL: "pool", OP_UP: "upsample"}[op[0]]
            fl, desc, nbytes = 0, "", 0
            if op[0] == OP_CONV:
                _, ib, ioff, cin, ob, ooff, cout, k, s, act, rb = op[:11]
                ib2, cin2 = op[14], op[16]
                h, w, _c = self.plan.bufs[ob]
                hi, wi, _ci = self.plan.bufs[ib]
                in_elems = hi * wi * cin
                if ib2 >= 0:
                    h2, w2, _c2 = self.plan.bufs[ib2]
                    in_elems += h2 * w2 * cin2
                ct = cin + (cin2 if ib2 >= 0 else 0)
                fl = 2 * h * w * cout * ct * k * k * self.B
                nbytes = (in_elems + h * w * cout * (2 if rb >= 0 else 1)) * 2 * self.B + cout * ct * k * k * 2
                desc = f"{ct}->{cout} k{k} s{s} @{h}x{w}" + ("  [up2|cat]" if ib2 >= 0 else "")
                if op[20]:          # chained 1x1 conv: its flops, its extra source, its output instead of the main conv's
                    cout2, xc = op[23], op[27]
                    fl += 2 * h * w * cout2 * (cout + xc) * self.B
                    nbytes = (in_elems + h * w * (xc + cout2 + (cout if rb >= 0 else 0))) * 2 * self.B + (cout * ct * k * k + cout2 * (cout + xc)) * 2
                    desc += f"  -> 1x1 {cout + xc}->{cout2}"
                if op[19]:
                    nbytes = (in_elems * 2 + h * w * (16 if op[19] == 1 else 8)) * self.B + cout * ct * 2
                    desc += "  [DFL]" if op[19] == 1 else "  [cls max]"
            elif op[0] == OP_STEM:
                h, w, _c = self.plan.bufs[op[1]]
                fl = 2 * h * w * op[3] * 27 * self.B
                nbytes = (self.H * self.W * 3 + h * w * op[3] * 2) * self.B
                desc = f"3->{op[3]} k3 s2 @{h}x{w}"
            elif op[0] == OP_POOL:
                h, w, _c = self.plan.bufs[op[1]]
                nbytes = h * w * op[3] * 4 * 2 * self.B
            elif op[0] == OP_UP:
                h, w, _c = self.plan.bufs[op[1]]
                nbytes = h * w * op[3] * 2 * (1 + op[4] * op[4]) * self.B
            out.append({"op": kind, "ms": float(ms[i]), "flops": fl, "bytes": nbytes, "desc": desc})
        return out

    def forward_tensor(self, x, stream=None):
        """x: CUDA float32 / bfloat16 tensor [B][3][H][W] RGB in [0, 1] (data/loaders.py:566-638 LoadTensor)."""
        import torch

        assert x.is_cuda and x.is_contiguous()
        if tuple(x.shape) != (self.B, 3, self.H, self.W):
            raise ValueError(f"expected {(self.B, 3, self.H, self.W)}, got {tuple(x.shape)}")
        dt = {torch.float32: 0, torch.bfloat16: 1}.get(x.dtype)
        if dt is None:
            raise NotImplementedError(f"dtype {x.dtype}")
        _lib.check(self.lib.b2_engine_forward_f32(self._h, _lib.ptr(x), dt, _lib.stream_ptr(stream)))

    def buffer(self, buf):
        """Debug/parity view of activation buffer ``buf`` as a torch bf16 tensor [B][h][w][c] (no copy)."""
        p, h, w, c = C.c_void_p(), C.c_int(), C.c_int(), C.c_int()
        _lib.check(self.lib.b2_engine_buffer(self._h, buf, C.byref(p), C.byref(h), C.byref(w), C.byref(c)))
        return _view_bf16(p.value, (self.B, h.value, w.value, c.value))

    def activation(self, name):
        """NCHW float32 copy of a named module output (e.g. ``'model.2.m.0.cv1'``) or layer index."""
        buf, off, c = self.plan.named[name] if isinstance(name, str) else self.plan.loc[name]
        return self.buffer(buf)[..., off:off + c].float().permute(0, 3, 1, 2).contiguous()

    def detect_inputs(self):
        """The feature maps that feed Detect (its ``f`` layers, in ``f`` order) as they stand after the last forward: one
        (device pointer, h, w, buffer channel stride, channel offset, C) per level.  C is Detect's own input width (``ch``), so
        the zero channels a padded plan adds after it are not part of the slice.  These are the maps the reference's ReID
        hook reads (trackers/track.py on_predict_start, ``model: auto``); they stay valid until the next forward."""
        det = self.spec["layers"][-1]
        s = min(det["ch"])
        if any(c % s for c in det["ch"]):
            raise NotImplementedError(f"Detect input widths {det['ch']}: get_obj_feats needs every width to be a multiple of {s}")
        out = []
        for f, c in zip(det["f"], det["ch"]):
            buf, coff, _ = self.plan.loc[f]
            h, w, cstride = self.plan.bufs[buf]
            p, hh, ww, cc = C.c_void_p(), C.c_int(), C.c_int(), C.c_int()
            _lib.check(self.lib.b2_engine_buffer(self._h, buf, C.byref(p), C.byref(hh), C.byref(ww), C.byref(cc)))
            out.append((p.value, h, w, cstride, coff, c))
        return out

    def level_logits(self, l):
        """[B][h*w][lstride] bf16 view of Detect level ``l`` (64 DFL bins, then nc class logits)."""
        return _view_bf16(self.level_ptrs[l], (self.B, self.level_h[l] * self.level_w[l], self.lstride))


def _view_bf16(ptr, shape):
    """Wrap library-owned device memory as a torch tensor via ``__cuda_array_interface__`` (uint16 -> bf16 view)."""
    import torch

    class _Mem:
        pass

    m = _Mem()
    n = int(np.prod(shape))
    m.__cuda_array_interface__ = {"shape": (n,), "typestr": "<u2", "data": (int(ptr), False), "version": 2}
    t = torch.as_tensor(m, device="cuda")
    return t.view(torch.bfloat16).view(*shape)

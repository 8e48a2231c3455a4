"""Functional wrappers over the C ABI (``include/b2dt.h``), mirroring the reference's operator names.

  conv2d_bf16            Conv.forward_fuse (ultralytics/nn/modules/conv.py:83-93) on NHWC bf16 tensors
  sppf_pool, upsample_slice, stem_u8, preprocess_u8, resize_bilinear_u8
  letterbox_u8           LetterBox (data/augment.py:1692-1733) of a ragged batch packed by ``pack_frames``
  decode                 Detect._inference (ultralytics/nn/modules/head.py:152-187) + candidate filter
  nms                    tail of non_max_suppression (ultralytics/utils/nms.py:129-160) + scale_boxes
  non_max_suppression    the reference signature (ultralytics/utils/nms.py:13-167) on a (B, 4+nc, A) tensor
  gray_pyramid_u8        cv2.cvtColor(BGR2GRAY) + three cv2.pyrDown levels of S frames (bit-exact), as a :class:`GrayPyramid`
  corner_min_eig         cv2.cornerMinEigenVal(gray, 7, 3)
  good_features_to_track cv2.goodFeaturesToTrack(maxCorners=200, qualityLevel=0.01, minDistance=15, blockSize=7) per stream
  optical_flow_pyr_lk    cv2.calcOpticalFlowPyrLK(winSize=(21, 21), maxLevel=3, criteria=(COUNT|EPS, 30, 0.01)) per stream

Every function needs a CUDA device and raises if the library is missing: there is no CPU fallback.
torch is used for device memory and streams only.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib

MAX_WH = 7680.0      # ultralytics/utils/nms.py:26
MAX_NMS = 30000      # ultralytics/utils/nms.py:25


def _torch():
    import torch

    return torch


def conv2d_bf16(x, w, bias, ksize, stride=1, act=True, out=None, out_coff=0, in_coff=0, cin=None, residual=None,
                res_coff=0, stream=None):
    """x: [B][H][W][Cs] bf16 CUDA (channels [in_coff, in_coff+cin) are the input); w: [Cout][k][k][cin] bf16;
    bias: [Cout] fp32.  Returns (or fills a channel slice of) ``out`` [B][Ho][Wo][Co_s] bf16."""
    torch = _torch()
    lib = _lib.load()
    B, H, W, cs = x.shape
    cin = cs - in_coff if cin is None else cin
    cout = w.shape[0]
    pad = ksize // 2
    Ho, Wo = (H + 2 * pad - ksize) // stride + 1, (W + 2 * pad - ksize) // stride + 1
    if out is None:
        out = torch.empty((B, Ho, Wo, cout), dtype=torch.bfloat16, device=x.device)
    assert x.is_contiguous() and w.is_contiguous() and out.is_contiguous()
    assert x.dtype == torch.bfloat16 and w.dtype == torch.bfloat16 and bias.dtype == torch.float32
    _lib.check(lib.b2_conv2d_bf16(_lib.ptr(x), B, H, W, cs, in_coff, cin, _lib.ptr(w), _lib.ptr(bias), cout, ksize, stride,
                                  1 if act else 0, _lib.ptr(out), out.shape[3], out_coff,
                                  _lib.ptr(residual), residual.shape[3] if residual is not None else 0, res_coff,
                                  _lib.stream_ptr(stream)))
    return out


def conv_chain_plan_ok(H, W, cin, cout, ksize, stride, has_residual, xc, cout2, B=1):
    """Does ``conv2d_chain_bf16`` take this pair?  (Pure planning in the library; works without a GPU.)"""
    return bool(_lib.load().b2_conv_chain_plan_ok(B, H, W, cin, cout, ksize, stride, int(bool(has_residual)), xc, cout2))


def conv2d_chain_bf16(x, w, bias, stride, w2, bias2, act=True, act2=True, residual=None, extra=None, out=None, out_coff=0, stream=None):
    """SiLU(conv3x3(x) + b) (+ residual), rounded to bf16, concatenated BEHIND ``extra`` along channels and fed to the 1x1 conv
    ``w2`` [Cout2][Cx + Cout] (+ SiLU if ``act2``), in one launch (csrc/conv_tc.cu, ConvParams::chain).
    x: [B][H][W][Cin] bf16, w: [Cout][3][3][Cin], extra: [B][Ho][Wo][Cx] bf16 or None.  Returns [B][Ho][Wo][Cout2] bf16.
    Raises NotImplementedError when the pair does not fit the chained kernel."""
    torch = _torch()
    lib = _lib.load()
    B, H, W, cin = x.shape
    cout, cout2 = w.shape[0], w2.shape[0]
    Ho, Wo = (H + 2 - 3) // stride + 1, (W + 2 - 3) // stride + 1
    if out is None:
        out = torch.empty((B, Ho, Wo, cout2), dtype=torch.bfloat16, device=x.device)
    xc = extra.shape[3] if extra is not None else 0
    assert tuple(w2.shape) == (cout2, xc + cout) and x.is_contiguous() and w.is_contiguous() and w2.is_contiguous()
    _lib.check(lib.b2_conv2d_chain_bf16(_lib.ptr(x), B, H, W, cin, 0, cin, _lib.ptr(w), _lib.ptr(bias), cout, 3, stride, 1 if act else 0,
                                        _lib.ptr(residual), residual.shape[3] if residual is not None else 0, 0,
                                        _lib.ptr(extra), xc, 0, xc, _lib.ptr(w2), _lib.ptr(bias2), cout2, 1 if act2 else 0,
                                        _lib.ptr(out), out.shape[3], out_coff, _lib.stream_ptr(stream)))
    return out


def conv2d_cat_bf16(x0, x1, w, bias, ksize=1, stride=1, act=True, up0=1, up1=1, out=None, out_coff=0, stream=None):
    """Conv over cat([up(x0), up(x1)], channel) without materialising the upsample or the concat.
    x0, x1: [B][h][w][C] bf16 (full NHWC tensors; up_i = 2 means stored at half the conv resolution)."""
    torch = _torch()
    lib = _lib.load()
    B = x0.shape[0]
    H, W = x0.shape[1] * up0, x0.shape[2] * up0
    cout = w.shape[0]
    pad = ksize // 2
    Ho, Wo = (H + 2 * pad - ksize) // stride + 1, (W + 2 * pad - ksize) // stride + 1
    if out is None:
        out = torch.empty((B, Ho, Wo, cout), dtype=torch.bfloat16, device=x0.device)
    _lib.check(lib.b2_conv2d_cat_bf16(_lib.ptr(x0), x0.shape[3], 0, x0.shape[3], up0,
                                      _lib.ptr(x1), x1.shape[3] if x1 is not None else 0, 0, x1.shape[3] if x1 is not None else 0, up1,
                                      B, H, W, _lib.ptr(w), _lib.ptr(bias), cout, ksize, stride, 1 if act else 0,
                                      _lib.ptr(out), out.shape[3], out_coff, _lib.stream_ptr(stream)))
    return out


def stem_u8(frames, w, bias, H, W, pad_top=0, pad_left=0, stream=None):
    """frames [B][h][w][3] uint8 BGR -> SiLU(conv3x3 s2(letterbox(frames)/255)) as [B][H/2][W/2][C0] bf16.
    w: [C0][32] bf16 from ``weights.pack_stem`` (CUDA tensor)."""
    torch = _torch()
    lib = _lib.load()
    B, sh, sw, _ = frames.shape
    c0 = w.shape[0]
    out = torch.empty((B, H // 2, W // 2, c0), dtype=torch.bfloat16, device=frames.device)
    _lib.check(lib.b2_stem_u8(_lib.ptr(frames), B, sh, sw, H, W, pad_top, pad_left, _lib.ptr(w), _lib.ptr(bias), c0,
                              _lib.ptr(out), c0, 0, _lib.stream_ptr(stream)))
    return out


def preprocess_u8(frames, H, W, pad_top=0, pad_left=0, stream=None):
    """BasePredictor.preprocess (engine/predictor.py:152-175) for same-shape uint8 BGR frames that need no
    resize: letterbox pad (114), BGR->RGB, HWC->CHW, /255.  Returns [B][3][H][W] float32."""
    torch = _torch()
    lib = _lib.load()
    B, sh, sw, _ = frames.shape
    out = torch.empty((B, 3, H, W), dtype=torch.float32, device=frames.device)
    _lib.check(lib.b2_preprocess_u8(_lib.ptr(frames), B, sh, sw, H, W, pad_top, pad_left, _lib.ptr(out), _lib.stream_ptr(stream)))
    return out


def resize_bilinear_u8(frames, dh, dw, stream=None):
    """cv2.resize(..., interpolation=cv2.INTER_LINEAR) on uint8 HWC frames (data/augment.py:1718)."""
    torch = _torch()
    lib = _lib.load()
    B, sh, sw, _ = frames.shape
    out = torch.empty((B, dh, dw, 3), dtype=torch.uint8, device=frames.device)
    _lib.check(lib.b2_resize_bilinear_u8(_lib.ptr(frames), B, sh, sw, _lib.ptr(out), dh, dw, _lib.stream_ptr(stream)))
    return out


def pack_layout(shapes):
    """Byte offsets (int64 [B], each a multiple of 16) of HWC uint8 frames of ``shapes`` [(h, w), ...] packed back to back, and the
    packed size.  16-byte offsets let ``letterbox_u8`` copy unresized frames with vector loads."""
    offs, n = [], 0
    for h, w in shapes:
        offs.append(n)
        n += -(-int(h) * int(w) * 3 // 16) * 16
    return np.asarray(offs, np.int64), n


def pack_frames(frames, out=None):
    """Pack HWC BGR uint8 frames at the offsets of :func:`pack_layout` into ``out`` (a 1-D uint8 numpy array or CPU tensor,
    e.g. pinned; a new array when None).  Returns (packed, offsets)."""
    offs, n = pack_layout([f.shape[:2] for f in frames])
    if out is None:
        out = np.empty((n,), np.uint8)
    buf = out.numpy() if hasattr(out, "numpy") else out
    if buf.ndim != 1 or buf.dtype != np.uint8 or buf.shape[0] != n:
        raise ValueError(f"packed buffer: need {n} uint8 bytes, got {buf.dtype} {tuple(buf.shape)}")
    for f, o in zip(frames, offs):
        if not (f.ndim == 3 and f.shape[2] == 3 and f.dtype == np.uint8):
            raise TypeError("frames must be HWC BGR uint8 arrays")
        buf[o:o + f.size] = np.ascontiguousarray(f).reshape(-1)
    return out, offs


def letterbox_u8(packed, offsets, geom, H, W, out=None, stream=None):
    """LetterBox of a ragged batch: ``packed`` CUDA uint8 (frames at ``offsets``, CUDA int64 [B]), ``geom`` CUDA int32 [B][6]
    {src_h, src_w, rh, rw, top, left} (``predictor.letterbox_table``).  Returns (or fills) the canvas [B][H][W][3] uint8."""
    torch = _torch()
    lib = _lib.load()
    B = geom.shape[0]
    if out is None:
        out = torch.empty((B, H, W, 3), dtype=torch.uint8, device=packed.device)
    assert tuple(out.shape) == (B, H, W, 3) and out.is_contiguous() and packed.is_contiguous()
    assert offsets.dtype == torch.int64 and geom.dtype == torch.int32 and offsets.shape[0] == B and tuple(geom.shape) == (B, 6)
    _lib.check(lib.b2_letterbox_u8(_lib.ptr(packed), _lib.ptr(offsets), _lib.ptr(geom), B, H, W, _lib.ptr(out), _lib.stream_ptr(stream)))
    return out


def pyramid_layout(shapes):
    """Layout of the gray pyramids of frames of ``shapes`` [(h, w), ...] (host only): level byte offsets int64 [S][4], level shapes
    int32 [S][4][2], level-0 pixel offsets int64 [S], total bytes, total level-0 pixels."""
    lib = _lib.load()
    S = len(shapes)
    sh = np.ascontiguousarray(np.asarray(shapes, np.int32).reshape(S, 2))
    off, hw, pix, tot = np.zeros((S, 4), np.int64), np.zeros((S, 4, 2), np.int32), np.zeros((S,), np.int64), np.zeros((2,), np.int64)
    _lib.check(lib.b2_pyramid_layout(S, sh.ctypes.data_as(C.c_void_p), off.ctypes.data_as(C.c_void_p), hw.ctypes.data_as(C.c_void_p),
                                     pix.ctypes.data_as(C.c_void_p), tot.ctypes.data_as(C.c_void_p)))
    return off, hw, pix, int(tot[0]), int(tot[1])


class GrayPyramid:
    """The 4-level gray pyramids of S frames in one CUDA uint8 buffer (``pyramid_layout``); ``level(s, l)`` is a [h][w] view."""

    def __init__(self, shapes, device=None):
        torch = _torch()
        dev = device or _lib.require_cuda()
        self.shapes = [(int(h), int(w)) for h, w in shapes]
        self.S = len(self.shapes)
        self.level_off, self.level_hw, self.pix_off, nbytes, self.npix = pyramid_layout(self.shapes)
        self.max_h, self.max_w = max(h for h, _ in self.shapes), max(w for _, w in self.shapes)
        self.buf = torch.empty((nbytes,), dtype=torch.uint8, device=dev)
        self.off_dev, self.hw_dev, self.pix_dev = (torch.from_numpy(a).to(dev) for a in (self.level_off, self.level_hw, self.pix_off))

    def level(self, s, l):
        h, w = (int(v) for v in self.level_hw[s, l])
        o = int(self.level_off[s, l])
        return self.buf[o:o + h * w].view(h, w)

    def plane(self, flat, s):
        """Stream ``s``'s [h][w] view of a level-0-sized per-pixel buffer (``corner_min_eig``)."""
        h, w = self.shapes[s]
        o = int(self.pix_off[s])
        return flat[o:o + h * w].view(h, w)


def frame_offsets(frames, shapes):
    """Byte offsets (int64 numpy [S]) of the frames in ``frames``: a CUDA uint8 [S][h][w][3] batch, or the 1-D ``pack_frames`` layout."""
    if frames.dim() == 4:
        S, h, w, _ = frames.shape
        return np.arange(S, dtype=np.int64) * (h * w * 3)
    offs, n = pack_layout(shapes)
    if frames.numel() != n:
        raise ValueError(f"packed frames: expected {n} bytes for shapes {shapes}, got {frames.numel()}")
    return offs


def gray_pyramid_u8(frames, shapes=None, out=None, stream=None):
    """cv2.cvtColor(COLOR_BGR2GRAY) + three cv2.pyrDown levels of S HWC BGR uint8 frames, bit-exact.  frames: CUDA uint8
    [S][h][w][3], or 1-D packed by ``pack_frames`` with their ``shapes``.  Returns (or fills) a :class:`GrayPyramid`."""
    torch = _torch()
    lib = _lib.load()
    assert frames.is_cuda and frames.dtype == torch.uint8 and frames.is_contiguous()
    if shapes is None:
        shapes = [tuple(frames.shape[1:3])] * frames.shape[0]
    pyr = out or GrayPyramid(shapes, frames.device)
    offs = torch.from_numpy(frame_offsets(frames, shapes)).to(frames.device)
    _lib.check(lib.b2_gray_pyramid_u8(_lib.ptr(frames), _lib.ptr(offs), pyr.S, pyr.max_h, pyr.max_w, _lib.ptr(pyr.buf), _lib.ptr(pyr.off_dev),
                                      _lib.ptr(pyr.hw_dev), _lib.stream_ptr(stream)))
    return pyr


def corner_min_eig(pyr, block_size=7, ksize=3, stream=None):
    """cv2.cornerMinEigenVal(level 0, blockSize, ksize) of every stream of a :class:`GrayPyramid`: float32 CUDA [npix]
    (``pyr.plane(out, s)`` is stream s).  Only blockSize=7, ksize=3 (the reference's) are provided."""
    torch = _torch()
    out = torch.empty((pyr.npix,), dtype=torch.float32, device=pyr.buf.device)
    _lib.check(_lib.load().b2_corner_min_eig(_lib.ptr(pyr.buf), _lib.ptr(pyr.off_dev), _lib.ptr(pyr.hw_dev), _lib.ptr(pyr.pix_dev), pyr.S,
                                             pyr.max_h, pyr.max_w, int(block_size), int(ksize), _lib.ptr(out), _lib.stream_ptr(stream)))
    return out


def good_features_to_track(pyr, max_corners=200, quality_level=0.01, min_distance=15, block_size=7, eig=None, stream=None):
    """cv2.goodFeaturesToTrack(level 0, maxCorners, qualityLevel, minDistance, blockSize=blockSize) for every stream of a
    :class:`GrayPyramid`; ``eig`` (``corner_min_eig``'s output) is computed when None.  Returns (corners float32 CUDA
    [S][200][2] (x, y), counts int32 CUDA [S]); rows past a stream's count are not written."""
    torch = _torch()
    lib = _lib.load()
    if eig is None:
        eig = corner_min_eig(pyr, block_size, 3, stream)
    elif block_size != 7:
        raise NotImplementedError("good_features_to_track: only blockSize=7")
    dev = pyr.buf.device
    wsb = lib.b2_good_features_workspace_bytes(pyr.S, pyr.npix)
    ws = torch.empty((wsb,), dtype=torch.uint8, device=dev)
    corners = torch.zeros((pyr.S, int(max_corners), 2), dtype=torch.float32, device=dev)
    counts = torch.zeros((pyr.S,), dtype=torch.int32, device=dev)
    _lib.check(lib.b2_good_features(_lib.ptr(eig), _lib.ptr(pyr.pix_dev), _lib.ptr(pyr.hw_dev), pyr.S, pyr.max_h, pyr.max_w, pyr.npix,
                                    int(max_corners), float(quality_level), float(min_distance), _lib.ptr(ws), wsb, _lib.ptr(corners),
                                    _lib.ptr(counts), _lib.stream_ptr(stream)))
    return corners, counts


def optical_flow_pyr_lk(prev, nxt, pts, counts=None, win_size=(21, 21), max_level=3, criteria=(3, 30, 0.01), stream=None):
    """cv2.calcOpticalFlowPyrLK(prev, next, pts, None, winSize, maxLevel, criteria) per stream between two :class:`GrayPyramid`
    of the same shapes.  pts: CUDA float32 [S][P][2]; counts: CUDA int32 [S] (None: P each).  Returns (next points float32
    [S][P][2], status uint8 [S][P]); rows past a count are not written.  criteria must include COUNT and EPS (type 3)."""
    torch = _torch()
    assert prev.shapes == nxt.shapes and pts.is_cuda and pts.dtype == torch.float32 and pts.is_contiguous() and pts.shape[0] == prev.S
    if int(criteria[0]) != 3 or tuple(win_size) != (21, 21):
        raise NotImplementedError("optical_flow_pyr_lk: only winSize=(21, 21), criteria type COUNT|EPS")
    P = pts.shape[1]
    if counts is None:
        counts = torch.full((prev.S,), P, dtype=torch.int32, device=pts.device)
    out = torch.zeros_like(pts)
    status = torch.zeros((prev.S, P), dtype=torch.uint8, device=pts.device)
    _lib.check(_lib.load().b2_lk_pyr(_lib.ptr(prev.buf), _lib.ptr(nxt.buf), _lib.ptr(prev.off_dev), _lib.ptr(prev.hw_dev), prev.S,
                                     _lib.ptr(pts), _lib.ptr(counts), P, int(win_size[0]), int(max_level), int(criteria[1]),
                                     float(criteria[2]), _lib.ptr(out), _lib.ptr(status), _lib.stream_ptr(stream)))
    return out, status


def sppf_pool(buf, coff, c, stream=None):
    lib = _lib.load()
    B, H, W, cs = buf.shape
    _lib.check(lib.b2_sppf_pool(_lib.ptr(buf), B, H, W, cs, coff, c, _lib.stream_ptr(stream)))
    return buf


def upsample_slice(x, out, scale=2, in_coff=0, c=None, out_coff=0, stream=None):
    lib = _lib.load()
    B, H, W, cs = x.shape
    c = cs - in_coff if c is None else c
    _lib.check(lib.b2_upsample_slice(_lib.ptr(x), B, H, W, cs, in_coff, c, scale, _lib.ptr(out), out.shape[3], out_coff,
                                     _lib.stream_ptr(stream)))
    return out


class DetectPost:
    """Pre-allocated decode + NMS pipeline for a fixed (batch, levels) geometry."""

    def __init__(self, batch, level_h, level_w, level_stride, nc, lstride, cand_cap=None, max_det=300, device=None):
        torch = _torch()
        self.lib = _lib.load()
        dev = device or _lib.require_cuda()
        self.B, self.nc, self.lstride = batch, nc, lstride
        self.n_levels = len(level_h)
        self.h = (C.c_int * self.n_levels)(*level_h)
        self.w = (C.c_int * self.n_levels)(*level_w)
        self.s = (C.c_int * self.n_levels)(*level_stride)
        self.A = sum(a * b for a, b in zip(level_h, level_w))
        # one slot per anchor by default: the conf filter cannot overflow, so results never depend on append order
        self.cand_cap = int(cand_cap or self.A)
        self.max_det = max_det
        self.cand = torch.empty((batch, self.cand_cap, 6), dtype=torch.float32, device=dev)
        self.cand_idx = torch.empty((batch, self.cand_cap), dtype=torch.int32, device=dev)
        self.cand_count = torch.zeros((batch,), dtype=torch.int32, device=dev)
        self.ws_bytes = self.lib.b2_nms_workspace_bytes(batch, self.cand_cap)
        self.ws = torch.empty((self.ws_bytes,), dtype=torch.uint8, device=dev)
        self.out = torch.zeros((batch, max_det, 6), dtype=torch.float32, device=dev)
        self.out_count = torch.zeros((batch,), dtype=torch.int32, device=dev)
        self.out_idx = torch.zeros((batch, max_det), dtype=torch.int32, device=dev)

    def decode(self, level_ptrs, conf, classes_mask=None, dense_out=None, stream=None):
        ptrs = (C.c_void_p * self.n_levels)(*[p if isinstance(p, int) or p is None else p.data_ptr() for p in level_ptrs])
        _lib.check(self.lib.b2_decode(ptrs, self.h, self.w, self.s, self.n_levels, self.B, self.nc, self.lstride, float(conf),
                                      _lib.ptr(classes_mask), _lib.ptr(self.cand), _lib.ptr(self.cand_idx), _lib.ptr(self.cand_count),
                                      self.cand_cap, _lib.ptr(dense_out), _lib.stream_ptr(stream)))

    def candidates_from_head(self, dist_ptrs, cls_ptrs, conf, classes_mask=None, stream=None):
        """Candidate stage on the fused Detect-head outputs of an ``Engine(fuse_head=True)``."""
        dp = (C.c_void_p * self.n_levels)(*dist_ptrs)
        cp = (C.c_void_p * self.n_levels)(*cls_ptrs)
        _lib.check(self.lib.b2_candidates_from_head(dp, cp, self.h, self.w, self.s, self.n_levels, self.B, float(conf), _lib.ptr(classes_mask),
                                                    _lib.ptr(self.cand), _lib.ptr(self.cand_idx), _lib.ptr(self.cand_count), self.cand_cap,
                                                    _lib.stream_ptr(stream)))

    def nms(self, iou, agnostic=False, mode="exact", max_nms=MAX_NMS, scale=None, stream=None):
        """scale: None or (gain, pad_x, pad_y, orig_w, orig_h) for the fused scale_boxes/clip_boxes epilogue, or a CUDA float32
        [B][5] tensor of those per image (frames of different original shapes)."""
        torch = _torch()
        if isinstance(scale, torch.Tensor):
            assert scale.is_cuda and scale.dtype == torch.float32 and tuple(scale.shape) == (self.B, 5) and scale.is_contiguous()
            _lib.check(self.lib.b2_nms_scaled(_lib.ptr(self.cand), _lib.ptr(self.cand_idx), _lib.ptr(self.cand_count), self.cand_cap, self.B,
                                              float(iou), self.max_det, int(max_nms), int(bool(agnostic)), MAX_WH, {"exact": 0, "legacy": 1}[mode],
                                              _lib.ptr(scale), _lib.ptr(self.out), _lib.ptr(self.out_count), _lib.ptr(self.out_idx),
                                              _lib.ptr(self.ws), self.ws_bytes, _lib.stream_ptr(stream)))
            return self.out, self.out_count
        g = scale or (1.0, 0.0, 0.0, 0.0, 0.0)
        _lib.check(self.lib.b2_nms(_lib.ptr(self.cand), _lib.ptr(self.cand_idx), _lib.ptr(self.cand_count), self.cand_cap, self.B,
                                   float(iou), self.max_det, int(max_nms), int(bool(agnostic)), MAX_WH, {"exact": 0, "legacy": 1}[mode],
                                   float(g[0]), float(g[1]), float(g[2]), float(g[3]), float(g[4]), 0 if scale is None else 1,
                                   _lib.ptr(self.out), _lib.ptr(self.out_count), _lib.ptr(self.out_idx), _lib.ptr(self.ws), self.ws_bytes,
                                   _lib.stream_ptr(stream)))
        return self.out, self.out_count


def _classes_mask(classes, nc, device):
    torch = _torch()
    if classes is None:
        return None
    m = torch.zeros((nc,), dtype=torch.uint8)
    for c in (classes if hasattr(classes, "__iter__") else [classes]):
        if 0 <= int(c) < nc:
            m[int(c)] = 1
    return m.to(device)


def non_max_suppression(prediction, conf_thres=0.25, iou_thres=0.45, classes=None, agnostic=False, multi_label=False,
                        labels=(), max_det=300, nc=0, max_time_img=0.05, max_nms=MAX_NMS, max_wh=MAX_WH, in_place=True,
                        rotated=False, end2end=False, return_idxs=False, mode="exact"):
    """Drop-in for ``ultralytics.utils.nms.non_max_suppression`` (utils/nms.py:13-167) on the detect path.

    ``prediction``: CUDA float tensor (B, 4+nc, A) [cx, cy, w, h, class scores...] (or a list/tuple whose first
    element is that tensor, nms.py:64-65).  Returns a list of B tensors (n_i, 6) [x1, y1, x2, y2, conf, cls].
    ``mode``: "exact" == torchvision.ops.nms branch, "legacy" == TorchNMS.nms branch (nms.py:152-157).
    The input is not modified (the reference mutates it in place, nms.py:85-87).
    """
    torch = _torch()
    assert 0 <= conf_thres <= 1, f"Invalid Confidence threshold {conf_thres}, valid values are between 0.0 and 1.0"
    assert 0 <= iou_thres <= 1, f"Invalid IoU {iou_thres}, valid values are between 0.0 and 1.0"
    if isinstance(prediction, (list, tuple)):
        prediction = prediction[0]
    if multi_label or rotated or end2end or len(labels):
        raise NotImplementedError("multi_label / rotated / end2end / labels are outside the detect hot path")
    if max_wh != MAX_WH:
        raise NotImplementedError("max_wh is fixed at 7680 as in the reference default")
    lib = _lib.load()
    pred = prediction.float().contiguous()
    B, no, A = pred.shape
    nc = nc or no - 4
    dev = pred.device
    cap = A
    cand = torch.empty((B, cap, 6), dtype=torch.float32, device=dev)
    cidx = torch.empty((B, cap), dtype=torch.int32, device=dev)
    ccnt = torch.zeros((B,), dtype=torch.int32, device=dev)
    _lib.check(lib.b2_candidates_from_dense(_lib.ptr(pred), B, nc, no, A, float(conf_thres), _lib.ptr(_classes_mask(classes, nc, dev)),
                                            _lib.ptr(cand), _lib.ptr(cidx), _lib.ptr(ccnt), cap, _lib.stream_ptr()))
    md = int(max_det)
    out = torch.zeros((B, md, 6), dtype=torch.float32, device=dev)
    ocnt = torch.zeros((B,), dtype=torch.int32, device=dev)
    oidx = torch.zeros((B, md), dtype=torch.int32, device=dev)
    wsb = lib.b2_nms_workspace_bytes(B, cap)
    ws = torch.empty((wsb,), dtype=torch.uint8, device=dev)
    _lib.check(lib.b2_nms(_lib.ptr(cand), _lib.ptr(cidx), _lib.ptr(ccnt), cap, B, float(iou_thres), md, int(max_nms),
                          int(bool(agnostic)), MAX_WH, {"exact": 0, "legacy": 1}[mode], 1.0, 0.0, 0.0, 0.0, 0.0, 0,
                          _lib.ptr(out), _lib.ptr(ocnt), _lib.ptr(oidx), _lib.ptr(ws), wsb, _lib.stream_ptr()))
    counts = ocnt.cpu().tolist()
    res = [out[b, :counts[b]].clone() for b in range(B)]
    if return_idxs:
        return res, [oidx[b, :counts[b]].long() for b in range(B)]
    return res


def to_numpy(t):
    return t.detach().cpu().numpy() if hasattr(t, "detach") else np.asarray(t)

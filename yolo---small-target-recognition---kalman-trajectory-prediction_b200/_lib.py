"""ctypes binding of ``libb2dt.so`` (the C ABI declared in ``include/b2dt.h``).

There is no CPU fallback: if the CUDA library is missing and cannot be built, importing any compute
entry point raises.  PyTorch is used only for device memory (``tensor.data_ptr()``) and streams.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.environ.get("B2DT_LIB") or os.path.join(_HERE, "libb2dt.so")     # B2DT_LIB: an experiment build (tools/build_variant.sh)
_lib = None

c_void_p, c_int, c_float, c_size_t = C.c_void_p, C.c_int, C.c_float, C.c_size_t
_P = c_void_p

# name -> (restype, argtypes); mirrors include/b2dt.h one to one
SIGNATURES = {
    "b2_last_error": (C.c_char_p, []),
    "b2_version": (c_int, []),
    "b2_launch_count": (C.c_longlong, []),
    "b2_conv2d_bf16": (c_int, [_P, c_int, c_int, c_int, c_int, c_int, c_int, _P, _P, c_int, c_int, c_int, c_int,
                               _P, c_int, c_int, _P, c_int, c_int, _P]),
    "b2_conv2d_cat_bf16": (c_int, [_P, c_int, c_int, c_int, c_int, _P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, _P, _P,
                                   c_int, c_int, c_int, c_int, _P, c_int, c_int, _P]),
    "b2_conv2d_chain_bf16": (c_int, [_P, c_int, c_int, c_int, c_int, c_int, c_int, _P, _P, c_int, c_int, c_int, c_int, _P, c_int, c_int,
                                     _P, c_int, c_int, c_int, _P, _P, c_int, c_int, _P, c_int, c_int, _P]),
    "b2_conv_chain_plan_ok": (c_int, [c_int] * 10),
    "b2_stem_u8": (c_int, [_P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, _P, _P, c_int, _P, c_int, c_int, _P]),
    "b2_stem_f32": (c_int, [_P, c_int, c_int, c_int, c_int, _P, _P, c_int, _P, c_int, c_int, _P]),
    "b2_preprocess_u8": (c_int, [_P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, _P, _P]),
    "b2_resize_bilinear_u8": (c_int, [_P, c_int, c_int, c_int, _P, c_int, c_int, _P]),
    "b2_letterbox_u8": (c_int, [_P, _P, _P, c_int, c_int, c_int, _P, _P]),
    "b2_sppf_pool": (c_int, [_P, c_int, c_int, c_int, c_int, c_int, c_int, _P]),
    "b2_upsample_slice": (c_int, [_P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, _P, c_int, c_int, _P]),
    "b2_decode": (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, c_int, c_float, _P, _P, _P, _P, c_int, _P, _P]),
    "b2_candidates_from_head": (c_int, [_P, _P, _P, _P, _P, c_int, c_int, c_float, _P, _P, _P, _P, c_int, _P]),
    "b2_candidates_from_dense": (c_int, [_P, c_int, c_int, c_int, c_int, c_float, _P, _P, _P, _P, c_int, _P]),
    "b2_nms": (c_int, [_P, _P, _P, c_int, c_int, c_float, c_int, c_int, c_int, c_float, c_int,
                       c_float, c_float, c_float, c_float, c_float, c_int, _P, _P, _P, _P, c_size_t, _P]),
    "b2_nms_scaled": (c_int, [_P, _P, _P, c_int, c_int, c_float, c_int, c_int, c_int, c_float, c_int, _P,
                              _P, _P, _P, _P, c_size_t, _P]),
    "b2_nms_workspace_bytes": (c_size_t, [c_int, c_int]),
    "b2_engine_create": (c_int, [_P, c_int, _P, c_size_t, c_int, c_int, c_int, C.POINTER(_P)]),
    "b2_engine_destroy": (c_int, [_P]),
    "b2_engine_forward_u8": (c_int, [_P, _P, c_int, c_int, c_int, c_int, _P]),
    "b2_engine_profile_u8": (c_int, [_P, _P, c_int, c_int, c_int, c_int, _P, _P]),
    "b2_engine_forward_f32": (c_int, [_P, _P, c_int, _P]),
    "b2_engine_levels": (c_int, [_P, C.POINTER(c_int), C.POINTER(_P), C.POINTER(c_int), C.POINTER(c_int),
                                 C.POINTER(c_int), C.POINTER(c_int)]),
    "b2_engine_head": (c_int, [_P, C.POINTER(_P), C.POINTER(_P)]),
    "b2_engine_buffer": (c_int, [_P, c_int, C.POINTER(_P), C.POINTER(c_int), C.POINTER(c_int), C.POINTER(c_int)]),
    "b2_engine_arena_bytes": (c_size_t, [_P]),
    "b2_engine_num_launches": (c_int, [_P]),
    "b2_engine_use_graph": (c_int, [_P, c_int]),
    "b2_tracker_create": (c_int, [c_int, c_int, c_int, c_int, c_int, c_float, C.POINTER(_P)]),
    "b2_tracker_create_ex": (c_int, [c_int, c_int, c_int, c_int, c_int, c_float, c_int, C.POINTER(_P)]),
    "b2_tracker_destroy": (c_int, [_P]),
    "b2_tracker_reset": (c_int, [_P, _P]),
    "b2_tracker_reset_streams": (c_int, [_P, _P, _P]),
    "b2_tracker_capacity": (c_int, [_P]),
    "b2_tracker_grow": (c_int, [_P, c_int, _P]),
    "b2_tracker_stats": (c_int, [_P, _P, _P]),
    "b2_tracker_update": (c_int, [_P, _P, c_int, _P, _P, _P, _P, _P, c_int, _P]),
    "b2_tracker_update_ex": (c_int, [_P, _P, c_int, _P, _P, _P, _P, _P, _P, c_int, _P]),
    "b2_tracker_export_reset": (c_int, [_P, c_int, _P, _P]),
    "b2_tracker_export": (c_int, [_P, c_int, _P, _P, _P, _P, _P]),
    "b2_tracker_export_motion": (c_int, [_P, c_int, _P, _P]),
    "b2_tracker_bytes_per_track": (c_int, [C.POINTER(c_int), C.POINTER(c_int)]),
    "b2_tracker_bank_predict": (c_int, [_P, _P]),
    "b2_tracker_seed": (c_int, [_P, _P, _P, c_int, _P]),
    "b2_kf_initiate": (c_int, [c_int, _P, _P, _P, c_int, _P]),
    "b2_kf_predict": (c_int, [c_int, _P, _P, c_int, _P]),
    "b2_kf_project": (c_int, [c_int, _P, _P, _P, _P, c_int, _P]),
    "b2_kf_update": (c_int, [c_int, _P, _P, _P, _P, c_int, _P]),
    "b2_kf_gating": (c_int, [c_int, _P, _P, c_int, _P, c_int, c_int, c_int, _P, _P]),
    "b2_iou_cost": (c_int, [_P, _P, _P, _P, _P, c_int, c_int, c_int, _P, _P]),
    "b2_linear_assignment": (c_int, [_P, _P, _P, c_int, c_int, c_int, c_float, _P, _P, _P]),
    "b2_linear_assignment_f64": (c_int, [_P, _P, _P, c_int, c_int, c_int, C.c_double, _P, _P, _P]),
    "b2_botsort_cost": (c_int, [_P, _P, _P, _P, _P, _P, _P, c_int, c_int, c_int, c_int, c_float, C.c_double, _P, _P]),
    "b2_reid_gather": (c_int, [_P, _P, _P, _P, _P, _P, c_int, _P, _P, c_int, c_int, c_int, _P, _P]),
    "b2_reid_update": (c_int, [_P, _P, _P, c_int, c_int, _P]),
    "b2_pyramid_layout": (c_int, [c_int, _P, _P, _P, _P, _P]),
    "b2_gray_pyramid_u8": (c_int, [_P, _P, c_int, c_int, c_int, _P, _P, _P, _P]),
    "b2_corner_min_eig": (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, c_int, c_int, _P, _P]),
    "b2_good_features_workspace_bytes": (c_size_t, [c_int, C.c_longlong]),
    "b2_good_features": (c_int, [_P, _P, _P, c_int, c_int, c_int, C.c_longlong, c_int, C.c_double, C.c_double, _P, c_size_t, _P, _P, _P]),
    "b2_lk_pyr": (c_int, [_P, _P, _P, _P, c_int, _P, _P, c_int, c_int, c_int, c_int, C.c_double, _P, _P, _P]),
    "b2_motion_create": (c_int, [c_int, _P, C.POINTER(_P)]),
    "b2_motion_flow": (c_int, [_P, _P, _P, _P]),
    "b2_motion_decide": (c_int, [_P, _P, _P, _P, _P, _P]),
    "b2_motion_stats": (c_int, [_P, _P, _P]),
    "b2_motion_reset": (c_int, [_P, _P]),
    "b2_motion_destroy": (c_int, [_P]),
}

B2_OK, B2_ERR_ARG, B2_ERR_CUDA, B2_ERR_STATE, B2_ERR_UNSUPPORTED = 0, -1, -2, -3, -4
TRACK_COLS, TRAJ_LEN = 20, 30


def lib_path():
    return _LIB_PATH


def load(build_if_missing=True):
    """Load (building first if needed and possible) and return the ctypes library handle."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_LIB_PATH):
        if not build_if_missing:
            raise RuntimeError(f"{_LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'`")
        from .build import build

        build()
    lib = C.CDLL(_LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)       # AttributeError here == header and library out of sync
        fn.restype, fn.argtypes = res, args
    _lib = lib
    return lib


def last_error():
    return load().b2_last_error().decode("utf-8", "replace")


def check(rc):
    """Map a C status to the exception the reference would raise for the same mistake."""
    if rc == B2_OK:
        return
    msg = last_error()
    if rc == B2_ERR_ARG:
        raise ValueError(msg)
    if rc == B2_ERR_UNSUPPORTED:
        raise NotImplementedError(msg)
    raise RuntimeError(f"b2dt error {rc}: {msg}")


def ptr(t):
    """Device/host pointer of a torch tensor (or None)."""
    return None if t is None else C.c_void_p(t.data_ptr())


def stream_ptr(stream=None):
    import torch

    s = torch.cuda.current_stream() if stream is None else stream
    return C.c_void_p(s.cuda_stream)


def require_cuda():
    import torch

    if not torch.cuda.is_available():
        raise RuntimeError("b2dt needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device())

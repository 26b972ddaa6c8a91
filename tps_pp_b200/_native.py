"""ctypes binding of libtpspp.so (C ABI declared in include/tpspp.h).

There is deliberately no fallback: if the shared library is missing or a call fails, a
``RuntimeError`` is raised -- the product path never routes through PyTorch/CPU code.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, Structure, c_char_p, c_float, c_int, c_int32, c_size_t, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("TPSPP_LIB", os.path.join(_HERE, "libtpspp.so"))

OK = 0
F32, BF16, SRC0_BF16 = 0, 1, 2
MODE_ATTENTION, MODE_CLASSICAL = 0, 1
VARIANT_AUTO, VARIANT_GENERIC, VARIANT_STAGED, VARIANT_TILED = 0, 1, 2, 3


class WarpCfg(Structure):
    """Mirror of ``tpspp_warp_cfg`` (include/tpspp.h)."""
    _fields_ = [
        ("batch", c_int32), ("channels0", c_int32), ("src0_h", c_int32), ("src0_w", c_int32),
        ("channels1", c_int32), ("src1_h", c_int32), ("src1_w", c_int32),
        ("out_h", c_int32), ("out_w", c_int32), ("num_fiducial", c_int32), ("mode", c_int32),
        ("theta", c_float), ("feat_dtype", c_int32), ("variant", c_int32),
    ]


class HeadCfg(Structure):
    """Mirror of ``tpspp_head_cfg`` (include/tpspp.h)."""
    _fields_ = [
        ("batch", c_int32), ("height", c_int32), ("width", c_int32), ("point_h", c_int32), ("point_w", c_int32),
        ("p_stride", c_int32), ("precision", c_int32), ("flags", c_int32),
    ]


class StageCfg(Structure):
    """Mirror of ``tpspp_stage_cfg`` (include/tpspp.h)."""
    _fields_ = [("batch", c_int32), ("height", c_int32), ("width", c_int32), ("precision", c_int32), ("flags", c_int32)]


class ConvCfg(Structure):
    """Mirror of ``tpspp_conv_cfg`` (include/tpspp.h)."""
    _fields_ = [("batch", c_int32), ("cin", c_int32), ("height", c_int32), ("width", c_int32), ("ksize", c_int32),
                ("stride_h", c_int32), ("stride_w", c_int32), ("relu", c_int32), ("nsrc", c_int32),
                ("up_h", c_int32 * 3), ("up_w", c_int32 * 3)]


class LocnetCfg(Structure):
    """Mirror of ``tpspp_locnet_cfg`` (include/tpspp.h)."""
    _fields_ = [("batch", c_int32), ("channels", c_int32), ("height", c_int32), ("width", c_int32), ("num_fiducial", c_int32),
                ("flags", c_int32)]


LP_COUNT = 24


class AttnCfg(Structure):
    """Mirror of ``tpspp_attn_cfg`` (include/tpspp.h)."""
    _fields_ = [("batch", c_int32), ("heads", c_int32), ("head_dim", c_int32), ("kv_len", c_int32), ("kv_capacity", c_int32),
                ("temperature", c_float), ("q_stride", c_int32), ("new_stride", c_int32), ("kv_head_major", c_int32)]


class AttnEncodeCfg(Structure):
    """Mirror of ``tpspp_attn_encode_cfg`` (include/tpspp.h)."""
    _fields_ = [("batch", c_int32), ("heads", c_int32), ("head_dim", c_int32), ("seq_len", c_int32), ("temperature", c_float),
                ("row_stride", c_int32)]


class OcrPrepCfg(Structure):
    """Mirror of ``tpspp_ocr_prep_cfg`` (include/tpspp.h)."""
    _fields_ = [("n", c_int32), ("out_h", c_int32), ("out_w", c_int32), ("mean", c_float * 3), ("std", c_float * 3),
                ("pad_value", c_int32), ("flags", c_int32), ("packed_bytes", ctypes.c_int64)]


class LinearCfg(Structure):
    """Mirror of ``tpspp_linear_cfg`` (include/tpspp.h)."""
    _fields_ = [("rows", ctypes.c_int64), ("in_features", c_int32), ("out_features", c_int32), ("weight_batches", c_int32),
                ("flags", c_int32)]


SP_COUNT = 81
HEAD_FP32, HEAD_TC, HEAD_BF16 = 0, 1, 2
HEAD_FLAG_WEIGHTS_CACHED = 1
HEAD_FLAG_UNFUSED_DOWN = 2
HEAD_FLAG_UNFUSED_SCORE = 4
HEAD_FLAG_TF32X3_CONV = 8
HEAD_FLAG_FEATGRID_BF16 = 16
LINEAR_FLAG_WEIGHTS_CACHED = 1
ACT_NONE, ACT_GELU = 0, 1
ABI_VERSION = 2
P_COUNT = 58
WS_NAMES = ("f0", "f1", "f2", "a0", "a1", "e0", "e1", "e2", "e3", "cbam", "d0", "d1", "d2", "de", "x1", "v", "de2", "p1", "wprep", "t1", "fs", "hid", "p1img")

_SIGNATURES = {
    "tpspp_version": (c_int, []),
    "tpspp_last_error": (c_char_p, []),
    "tpspp_last_launch_count": (c_int, []),
    "tpspp_launch_profile": (c_int, [c_int]),
    "tpspp_launch_profile_read": (c_int, [POINTER(ctypes.c_float), c_int, POINTER(c_int)]),
    "tpspp_device_info": (c_int, [POINTER(c_int), POINTER(c_int), POINTER(c_int)]),
    "tpspp_warp_workspace_bytes": (c_size_t, [POINTER(WarpCfg)]),
    "tpspp_warp_fwd_workspace_bytes": (c_size_t, [POINTER(WarpCfg)]),
    "tpspp_warp_fwd": (c_int, [POINTER(WarpCfg)] + [c_void_p] * 12),
    "tpspp_sample_fwd": (c_int, [POINTER(WarpCfg)] + [c_void_p] * 6),
    "tpspp_warp_bwd": (c_int, [POINTER(WarpCfg)] + [c_void_p] * 15),
    "tpspp_head_workspace_bytes": (c_size_t, [POINTER(HeadCfg)]),
    "tpspp_head_workspace_offsets": (c_int, [POINTER(HeadCfg), POINTER(c_size_t)]),
    "tpspp_head_fwd": (c_int, [POINTER(HeadCfg), c_void_p, c_void_p, c_void_p, POINTER(c_void_p),
                               c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "tpspp_conv_workspace_bytes": (c_size_t, [POINTER(ConvCfg)]),
    "tpspp_conv_fwd": (c_int, [POINTER(ConvCfg)] + [c_void_p] * 6),
    "tpspp_conv_bwd": (c_int, [POINTER(ConvCfg)] + [c_void_p] * 9),
    "tpspp_convcat_fwd": (c_int, [POINTER(ConvCfg), POINTER(c_void_p)] + [c_void_p] * 5),
    "tpspp_convcat_bwd": (c_int, [POINTER(ConvCfg), POINTER(c_void_p)] + [c_void_p] * 3 + [POINTER(c_void_p)] + [c_void_p] * 4),
    "tpspp_locnet_workspace_bytes": (c_size_t, [POINTER(LocnetCfg)]),
    "tpspp_locnet_fwd": (c_int, [POINTER(LocnetCfg), c_void_p, POINTER(c_void_p), c_void_p, c_void_p, c_void_p]),
    "tpspp_attn_decode": (c_int, [POINTER(AttnCfg)] + [c_void_p] * 8),
    "tpspp_attn_encode": (c_int, [POINTER(AttnEncodeCfg)] + [c_void_p] * 6),
    "tpspp_ocr_prep": (c_int, [POINTER(OcrPrepCfg)] + [c_void_p] * 4),
    "tpspp_linear_fwd_ex": (c_int, [POINTER(LinearCfg)] + [c_void_p] * 4 + [c_int32] + [c_void_p] * 3),
    "tpspp_linear_ln_fwd": (c_int, [POINTER(LinearCfg)] + [c_void_p] * 4 + [c_int32] + [c_void_p] * 3 + [ctypes.c_float] + [c_void_p] * 3),
    "tpspp_linear_workspace_bytes": (c_size_t, [POINTER(LinearCfg)]),
    "tpspp_linear_fwd": (c_int, [POINTER(LinearCfg)] + [c_void_p] * 6),
    "tpspp_linear_bwd": (c_int, [POINTER(LinearCfg)] + [c_void_p] * 8),
    "tpspp_stage_workspace_bytes": (c_size_t, [POINTER(StageCfg)]),
    "tpspp_stage_fwd": (c_int, [POINTER(StageCfg), c_void_p, POINTER(c_void_p), c_void_p, c_void_p, c_void_p, c_void_p,
                                c_void_p]),
}
_OPTIONAL = {}

_lib = None


def exported_symbols():
    """Names every build of the library must export (tests check this without a GPU)."""
    return sorted(_SIGNATURES)


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"libtpspp.so not found at {LIB_PATH}: build it with `python -m tps_pp_b200.build` "
                "(there is no CPU/PyTorch fallback for the TPS++ hot path)")
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in {**_SIGNATURES, **_OPTIONAL}.items():
            try:
                fn = getattr(handle, name)
            except AttributeError:
                if name in _OPTIONAL:
                    continue
                raise RuntimeError(f"{LIB_PATH} does not export {name}; rebuild it")
            fn.restype = res
            fn.argtypes = args
        if handle.tpspp_version() != ABI_VERSION:
            raise RuntimeError("libtpspp ABI version mismatch; rebuild it")
        _lib = handle
    return _lib


def last_error() -> str:
    return lib().tpspp_last_error().decode("utf-8", "replace")


def check(rc: int, what: str) -> None:
    if rc != OK:
        raise RuntimeError(f"{what} failed (code {rc}): {last_error()}")


def last_launch_count() -> int:
    return int(lib().tpspp_last_launch_count())


def device_info():
    sm, maj, mi = c_int(0), c_int(0), c_int(0)
    check(lib().tpspp_device_info(ctypes.byref(sm), ctypes.byref(maj), ctypes.byref(mi)), "tpspp_device_info")
    return sm.value, maj.value, mi.value

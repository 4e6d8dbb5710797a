"""ctypes binding of libgfla_warp.so (the C ABI in include/gfla_warp.h).

There is deliberately NO fallback: if the CUDA library is missing or cannot be
loaded, importing the ops raises.  The CPU oracle under oracle/ is test
infrastructure and is never imported from here.
"""
from __future__ import annotations

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("GFLA_LIB") or os.path.join(_HERE, "lib", "libgfla_warp.so")   # GFLA_LIB: A/B testing of builds

GFLA_F32, GFLA_F64, GFLA_BF16, GFLA_F16 = 0, 1, 2, 3
GFLA_NCHW, GFLA_NHWC = 0, 1
ABI_VERSION = 1

_vp, _i = ctypes.c_void_p, ctypes.c_int

# name -> argtypes; mirrors include/gfla_warp.h one to one (tests/test_abi.py checks the header against this table)
SIGNATURES = {
    "gfla_abi_version": [],
    "gfla_device_check": [],
    "gfla_debug_launch_count": [],
    "gfla_debug_set_buffer": [_vp],
    "gfla_debug_wait_profile": [_i, _i, _vp],
    "gfla_relayout": [_vp, _vp] + [_i] * 6 + [_vp],
    "gfla_block_extract_fwd": [_vp, _vp, _vp] + [_i] * 9 + [_vp],
    "gfla_block_extract_bwd": [_vp] * 5 + [_i] * 11 + [_vp],
    "gfla_convert": [_vp, _i, _vp, _i, ctypes.c_longlong, _vp],
    "gfla_attn_reshape_fwd": [_vp, _vp] + [_i] * 5 + [_vp],
    "gfla_attn_reshape_bwd": [_vp, _vp] + [_i] * 6 + [_vp],
    "gfla_resample2d_fwd": [_vp] * 3 + [_i] * 9 + [_vp],
    "gfla_resample2d_bwd": [_vp] * 5 + [_i] * 10 + [_vp],
    "gfla_resample2d_cosine_fwd": [_vp] * 5 + [_i] * 8 + [ctypes.c_double, _i, _vp],
    "gfla_resample2d_cosine_bwd": [_vp] * 9 + [_i] * 8 + [ctypes.c_double, _i, _i, _vp],
    "gfla_resample2d_fwd_nhwc": [_vp] * 3 + [_i] * 9 + [_vp],
    "gfla_resample2d_bwd_nhwc": [_vp] * 5 + [_i] * 11 + [_vp],
    "gfla_resample2d_cosine_fwd_nhwc": [_vp] * 5 + [_i] * 8 + [ctypes.c_double, _i, _vp],
    "gfla_resample2d_cosine_bwd_nhwc": [_vp] * 9 + [_i] * 8 + [ctypes.c_double, _i, _i, _i, _vp],
    "gfla_local_attn_fwd": [_vp] * 5 + [_i] * 11 + [_vp],
    "gfla_local_attn_blend_fwd": [_vp] * 6 + [_i] * 11 + [_vp],
    "gfla_local_attn_bwd": [_vp] * 7 + [_i] * 12 + [_vp],
    "gfla_local_attn_bwd_workspace_bytes": [_i],
    "gfla_local_attn_bwd_ws": [_vp] * 7 + [_i] * 12 + [_vp, ctypes.c_longlong, _vp],
}

_lib = None


class GflaError(RuntimeError):
    pass


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise GflaError(
                f"{LIB_PATH} is not built. Run `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a). There is no CPU / PyTorch fallback for these ops.")
        l = ctypes.CDLL(LIB_PATH)
        for name, argtypes in SIGNATURES.items():
            fn = getattr(l, name)          # AttributeError if the .so lacks a declared symbol
            fn.argtypes = argtypes
            fn.restype = _i
        l.gfla_debug_launch_count.restype = ctypes.c_ulonglong
        l.gfla_local_attn_bwd_workspace_bytes.restype = ctypes.c_longlong
        l.gfla_error_string.argtypes = [_i]
        l.gfla_error_string.restype = ctypes.c_char_p
        if l.gfla_abi_version() != ABI_VERSION:
            raise GflaError(f"libgfla_warp.so ABI {l.gfla_abi_version()} != binding {ABI_VERSION}: rebuild")
        _lib = l
    return _lib


def check(code: int, what: str) -> None:
    if code != 0:
        msg = lib().gfla_error_string(code).decode()
        raise GflaError(f"{what} failed with code {code}: {msg}")

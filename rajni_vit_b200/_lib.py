"""ctypes binding of librajni_b200.so (the C ABI in include/rajni_b200.h).

There is no CPU path and no fallback: if the library is missing, cannot be
loaded, or the device is not sm_100, every entry point raises.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, Structure, c_char_p, c_float, c_int, c_longlong, c_size_t, c_uint64, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "librajni_b200.so")

RAJNI_OK, RAJNI_EINVAL, RAJNI_ECUDA, RAJNI_EARCH, RAJNI_ERANGE = 0, -1, -2, -3, -4
ATTN_AUTO, ATTN_PIPE, ATTN_TC, ATTN_LONG = 0, 1, 2, 3
EPI_BIAS, EPI_GELU, EPI_RESIDUAL, EPI_OUT_F32, EPI_LN_FOLD, EPI_ROW_STATS, HINT_REVERSE_M = 1, 2, 4, 8, 16, 32, 64
ABI_VERSION = 12


class GemmArgs(Structure):
    """struct rajni_gemm_args (include/rajni_b200.h)"""
    _fields_ = [("A", c_void_p), ("W", c_void_p), ("bias", c_void_p), ("D", c_void_p),
                ("M", c_int), ("N", c_int), ("K", c_int), ("flags", c_int),
                ("residual", c_void_p), ("ldres", c_longlong), ("res_row_map", c_void_p),
                ("ldd", c_longlong), ("out_row_map", c_void_p),
                ("ln_stats", c_void_p), ("ln_stats_ld", c_longlong), ("ln_slots", c_int),
                ("ln_wsum", c_void_p), ("ln_eps", c_float),
                ("row_stats", c_void_p), ("row_stats_ld", c_longlong)]



# symbol -> (restype, argtypes); mirrors include/rajni_b200.h one to one
SIGNATURES = {
    "rajni_abi_version": (c_int, []),
    "rajni_last_error": (c_char_p, []),
    "rajni_device_check": (c_int, []),
    "rajni_launch_count": (c_uint64, []),
    "rajni_select_prefix": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "rajni_score_select_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_int]),
    "rajni_score_select_needs_workspace": (c_int, [c_int, c_int]),
    "rajni_score_select_prefix": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_float,
                                          c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "rajni_gather_rows": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "rajni_layernorm_strided": (c_int, [c_void_p, c_longlong, c_void_p, c_void_p, c_float, c_void_p, c_longlong, c_int, c_int,
                                        c_void_p]),
    "rajni_layernorm_strided_f32": (c_int, [c_void_p, c_longlong, c_void_p, c_void_p, c_float, c_void_p, c_longlong, c_int, c_int,
                                            c_void_p]),
    "rajni_layernorm_row_stats": (c_int, [c_void_p, c_longlong, c_void_p, c_void_p, c_float, c_void_p, c_longlong, c_int, c_int,
                                          c_void_p, c_longlong, c_int, c_void_p]),
    "rajni_mean_pool_layernorm": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_float, c_void_p, c_longlong,
                                          c_void_p]),
    "rajni_mean_pool_layernorm_f32": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_float, c_void_p,
                                              c_longlong, c_void_p]),
    "rajni_gemm_bf16_ex": (c_int, [POINTER(GemmArgs), c_void_p]),
    "rajni_gemm_row_stats_slots": (c_int, [c_int]),
    "rajni_attention_fwd_ex": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_float, c_int, c_int, c_void_p]),
    "rajni_resize_workspace_bytes": (c_size_t, [c_int, c_int]),
    "rajni_resize_center_crop_u8": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_size_t, c_void_p]),
    "rajni_resize_status": (c_int, [c_void_p, c_int, c_int, c_void_p]),
    "rajni_patch_im2col_prefix": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_void_p, c_int,
                                          c_void_p, c_longlong, c_int, c_void_p, c_void_p, c_void_p]),
}

_lib = None


class RajniError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(message)
        self.code = code


def load() -> ctypes.CDLL:
    """Load the library (once). Raises if it has not been built — there is no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -m rajni_vit_b200.csrc.build` "
            "(or __graft_entry__.build()). rajni_vit_b200 has no CPU or eager fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the .so is stale
        fn.restype = res
        fn.argtypes = args
    if lib.rajni_abi_version() != ABI_VERSION:
        raise RuntimeError(f"librajni_b200.so ABI {lib.rajni_abi_version()} != expected {ABI_VERSION}; rebuild")
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != RAJNI_OK:
        msg = load().rajni_last_error().decode("utf-8", "replace")
        raise RajniError(rc, msg)


def launch_count() -> int:
    return int(load().rajni_launch_count())

"""ctypes binding of the C ABI in ``include/b200lev.h`` (``libb200lev.so``).

This is the whole boundary between the Python host code and the hand-written sm_100a
kernels: plain pointers, sizes and a stream handle.  There is no CPU implementation
behind it -- if the shared library has not been built, or no CUDA device is present,
the first call raises.
"""
from __future__ import annotations

import ctypes
import os
from typing import Optional

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libb200lev.so")

OK = 0
FLAG_REF_NO_EOS, FLAG_HYP_NO_EOS, FLAG_EMPTY_REF, FLAG_WIDE_TOKENS, FLAG_BAD_TARGET = 1, 2, 4, 8, 16
F32, F16, BF16, F64 = 0, 1, 2, 3
REDUCE = {"none": 0, "mean": 1, "sum": 2}

c_i32, c_i64, c_f32, c_vp, c_sz = (ctypes.c_int32, ctypes.c_int64, ctypes.c_float,
                                   ctypes.c_void_p, ctypes.c_size_t)


class Tokens(ctypes.Structure):
    """``b200lev_tokens_t``: a borrowed strided (T, N) token view."""

    _fields_ = [("data", c_vp), ("elem_bytes", c_i32), ("T", c_i64), ("N", c_i64),
                ("stride_t", c_i64), ("stride_n", c_i64)]


class Opts(ctypes.Structure):
    """``b200lev_opts_t``: the knobs of ``_string_matching`` (_string.py:146-163)."""

    _fields_ = [("has_eos", c_i32), ("eos", c_i64), ("include_eos", c_i32),
                ("ins_cost", c_f32), ("del_cost", c_f32), ("sub_cost", c_f32),
                ("norm", c_i32), ("exclude_last", c_i32), ("padding", c_i64),
                ("return_mistakes", c_i32), ("ref_group", c_i32)]


_PT, _PO = ctypes.POINTER(Tokens), ctypes.POINTER(Opts)

# name -> (restype, argtypes); every symbol include/b200lev.h declares
SIGNATURES = {
    "b200lev_abi_version": (ctypes.c_int, []),
    "b200lev_last_error": (ctypes.c_char_p, []),
    "b200lev_device_count": (ctypes.c_int, []),
    "b200lev_workspace_bytes": (c_sz, [_PT, _PT, c_i32, c_i32]),
    "b200lev_final": (ctypes.c_int, [_PT, _PT, _PO, c_vp, c_vp, c_sz, c_vp, c_vp]),
    "b200lev_prefix": (ctypes.c_int, [_PT, _PT, _PO, c_vp, c_i64, c_i64, c_vp, c_sz, c_vp, c_vp]),
    "b200lev_completion_count": (ctypes.c_int, [_PT, _PT, _PO, c_vp, c_sz, c_vp, c_vp, c_vp]),
    "b200lev_completion_fill": (ctypes.c_int, [_PT, _PT, _PO, c_vp, c_sz, c_i64, c_vp, c_i64,
                                               c_i64, c_vp]),
    "b200lev_ocd_forward": (ctypes.c_int, [c_vp, c_i32, c_i64, c_i64, c_i64, c_i64, c_i64, c_vp,
                                           c_i64, c_i64, c_i64, c_vp, c_i64, c_i32, c_i32, c_vp,
                                           c_vp, c_vp, c_vp, c_vp, c_vp]),
    "b200lev_ocd_backward": (ctypes.c_int, [c_vp, c_i32, c_i64, c_i64, c_i64, c_i64, c_i64, c_vp,
                                            c_i64, c_i64, c_i64, c_vp, c_i64, c_i32, c_i32, c_vp,
                                            c_vp, c_vp, c_vp, c_vp]),
    "b200lev_mwer_forward": (ctypes.c_int, [c_vp, c_vp, c_i32, c_i64, c_i64, c_i64, c_i64, c_i32,
                                            c_i32, c_vp, c_vp, c_vp]),
    "b200lev_mwer_backward": (ctypes.c_int, [c_vp, c_vp, c_i32, c_i64, c_i64, c_i64, c_i64, c_i32,
                                             c_i32, c_vp, c_vp, c_vp]),
    "b200lev_final_sums": (ctypes.c_int, [_PT, _PT, _PO, c_vp, c_vp, c_sz, c_vp, c_vp, c_vp]),
    "b200lev_final_cross_workspace_bytes": (c_sz, [_PT, _PT, c_i64, c_i64, _PO]),
    "b200lev_final_cross": (ctypes.c_int, [_PT, _PT, c_i64, c_i64, _PO, c_vp, c_vp, c_sz, c_vp, c_vp]),
    "b200lev_mbr": (ctypes.c_int, [c_vp, c_vp, c_i32, c_i64, c_i64, c_i64, c_i64, c_vp, c_vp, c_vp]),
    "b200lev_error_counts": (ctypes.c_int, [_PT, _PT, _PO, c_vp, c_vp, c_sz, c_vp, c_vp]),
    "b200lev_error_alignment": (ctypes.c_int, [_PT, _PT, _PO, c_vp, c_i64, c_i64, c_vp, c_sz, c_vp, c_vp]),
    "b200lev_infix": (ctypes.c_int, [_PT, _PT, _PO, c_vp, c_vp, c_vp, c_vp, c_sz, c_vp, c_vp]),
    "b200lev_after_eos_mask": (ctypes.c_int, [c_vp, c_i64, c_i64, c_i64, c_i64, c_vp, c_vp]),
    "b200lev_ragged_to_padded": (ctypes.c_int, [c_vp, c_i32, c_vp, c_vp, c_i64, c_i64, c_i64, c_i64,
                                                c_vp, c_vp]),
    "b200lev_seqlp_forward": (ctypes.c_int, [c_vp, c_i32, c_i64, c_i64, c_i64, c_i64, c_vp, c_i32,
                                             c_i64, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "b200lev_seqlp_backward": (ctypes.c_int, [c_vp, c_i32, c_i64, c_i64, c_i64, c_i64, c_vp, c_vp,
                                              c_vp, c_vp, c_vp, c_vp]),
    "b200lev_ctc_greedy": (ctypes.c_int, [c_vp, c_i32, c_i64, c_i64, c_i64, c_i64, c_vp, c_i64, c_i32, c_vp,
                                          c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "b200lev_beam_topk": (ctypes.c_int, [c_vp, c_i32, c_i64, c_i64, c_i64, c_i64, c_i64, c_i64, c_vp, c_i64,
                                         c_i64, c_i64, c_vp, c_vp, c_vp, c_vp]),
    "b200lev_path_extend": (ctypes.c_int, [c_vp, c_i64, c_i64, c_i64, c_vp, c_vp, c_vp, c_i64, c_i64, c_i64,
                                           c_vp, c_vp, c_vp]),
    "b200lev_copy2d_async": (ctypes.c_int, [c_vp, c_sz, c_vp, c_sz, c_sz, c_sz, c_i32, c_vp]),
    "b200lev_profile": (ctypes.c_int, [ctypes.c_int]),
    "b200lev_profile_read": (ctypes.c_int, [ctypes.POINTER(ctypes.c_float), ctypes.c_int]),
    "b200lev_int32_peak_kernel": (ctypes.c_int, [c_i32, c_i64, c_i64, c_vp,
                                                 ctypes.POINTER(ctypes.c_double), c_vp]),
}

_lib: Optional[ctypes.CDLL] = None


class B200LevError(RuntimeError):
    pass


def _bind(lib: ctypes.CDLL) -> ctypes.CDLL:
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here == ABI mismatch; let it surface
        fn.restype = res
        fn.argtypes = args
    return lib


def lib() -> ctypes.CDLL:
    """The loaded ``libb200lev.so``; raises if it was never built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise B200LevError(
                f"{LIB_PATH} not found: build the CUDA library first "
                "(python pydrobert-pytorch_b200/build.py, or __graft_entry__.build()). "
                "b200lev has no CPU fallback."
            )
        _lib = _bind(ctypes.CDLL(LIB_PATH))
        if _lib.b200lev_abi_version() != 3:
            raise B200LevError("libb200lev.so ABI version mismatch")
    return _lib


def check(status: int) -> None:
    if status != OK:
        msg = lib().b200lev_last_error()
        raise B200LevError(f"b200lev error {status}: {msg.decode() if msg else '?'}")

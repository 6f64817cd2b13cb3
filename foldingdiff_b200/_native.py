"""
ctypes binding of the C ABI declared in include/foldingdiff_b200.h.

There is no Python / CPU fallback behind this module: if the shared library is
missing or a call fails, an exception is raised.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

from . import _build

FD_OK = 0
GEMM_FP32_SIMT = 0
GEMM_TC_3X = 1
GEMM_TC_1X = 2
GEMM_MODES = {"fp32": GEMM_FP32_SIMT, "tc3x": GEMM_TC_3X, "tc1x": GEMM_TC_1X}

W_HEAD, W_PER_LAYER, W_TAIL = 4, 17, 6


class FdDims(C.Structure):
    _fields_ = [
        ("hidden", C.c_int32), ("layers", C.c_int32), ("heads", C.c_int32),
        ("intermediate", C.c_int32), ("max_pos", C.c_int32), ("n_features", C.c_int32),
        ("timesteps", C.c_int32), ("ln_eps", C.c_float), ("head_ln_eps", C.c_float),
    ]


class NativeError(RuntimeError):
    pass


# name -> (restype, argtypes); this table is also what tests/test_abi.py checks against the header
SIGNATURES = {
    "fd_num_weights": (C.c_int32, [C.c_int32]),
    "fd_create": (C.c_int32, [C.POINTER(FdDims), C.POINTER(C.c_void_p), C.c_int32, C.c_void_p,
                              C.c_void_p, C.c_int32, C.c_int32, C.POINTER(C.c_void_p)]),
    "fd_destroy": (None, [C.c_void_p]),
    "fd_last_error": (C.c_char_p, []),
    "fd_abi_version": (C.c_int32, []),
    "fd_build_info": (C.c_char_p, []),
    "fd_set_schedule": (C.c_int32, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]),
    "fd_set_gemm_mode": (C.c_int32, [C.c_void_p, C.c_int32]),
    "fd_set_batch": (C.c_int32, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_int32,
                                 C.c_void_p, C.c_void_p]),
    "fd_forward": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "fd_p_sample_steps": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p,
                                      C.c_void_p, C.c_void_p, C.c_void_p]),
    "fd_p_sample_steps_philox": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_uint64, C.c_uint64,
                                             C.c_void_p, C.c_void_p, C.c_void_p]),
    "fd_status": (C.c_int32, [C.c_void_p]),
    "fd_sample_host": (C.c_int32, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                   C.c_int32, C.c_void_p, C.c_uint64, C.c_void_p, C.c_int32,
                                   C.c_void_p]),
    "fd_nerf_build": (C.c_int32, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32,
                                  C.c_void_p, C.c_void_p]),
    "fd_randn": (C.c_int32, [C.c_void_p, C.c_int64, C.c_uint64, C.c_uint64, C.c_void_p]),
    "fd_q_sample": (C.c_int32, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "fd_loss_terms": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p,
                                  C.c_int32, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p]),
    "fd_pdist_loss": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                  C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                  C.c_void_p]),
    "fd_launch_count": (C.c_int64, [C.c_void_p]),
    "fd_profile_begin": (C.c_int32, [C.c_void_p]),
    "fd_profile_end": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "fd_profile_num_categories": (C.c_int32, []),
    "fd_profile_category_name": (C.c_char_p, [C.c_int32]),
    "fd_debug_gemm": (C.c_int32, [C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                  C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "fd_debug_attention": (C.c_int32, [C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_int32,
                                       C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]),
    "fd_debug_tc_status": (C.c_int32, []),
    "fd_debug_graph_state": (C.c_int32, [C.c_void_p]),
    "fd_debug_attention_dump": (C.c_int32, [C.c_void_p]),
    "fd_write_angles_csv_gz": (C.c_int32, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_char_p), C.c_char_p,
                                           C.c_int32]),
    "fd_write_backbone_pdb": (C.c_int32, [C.c_void_p, C.c_int32, C.c_char_p]),
    "fd_write_batch": (C.c_int32, [C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.POINTER(C.c_char_p), C.c_void_p, C.c_int32,
                                   C.c_void_p, C.POINTER(C.c_char_p), C.POINTER(C.c_char_p), C.c_int32, C.c_int32]),
}

_lib: Optional[C.CDLL] = None


def lib() -> C.CDLL:
    """Load (once) the in-tree shared library and attach prototypes."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("FOLDINGDIFF_B200_LIB", _build.LIB_PATH)
    if not os.path.isfile(path):
        raise NativeError(
            f"CUDA library not found at {path}. Build it with "
            "`python -m foldingdiff_b200._build` (or __graft_entry__.build()). "
            "foldingdiff_b200 has no CPU fallback.")
    handle = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(handle, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = handle
    return handle


def check(status: int, what: str) -> None:
    if status != FD_OK:
        msg = lib().fd_last_error().decode("utf-8", "replace")
        raise NativeError(f"{what} failed with status {status}: {msg}")

"""ctypes binding of the C-ABI library (include/sow_b200.h).

The library is built in-tree by ``__graft_entry__.build()`` as ``sow_b200/csrc/libsow_b200.so``.  There is no
CPU fallback: if the library is missing, or a call fails, an exception is raised.
"""
from __future__ import annotations

import ctypes
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libsow_b200.so")

SOWB_BF16 = 0
SOWB_F32 = 1
SOWB_F16 = 2

OP_LINEAR_FWD = 0
OP_LINEAR_BWD = 1
OP_MERGE = 2
OP_THIN_QR = 3
OP_TT_PROJECT = 4


class SowB200Error(RuntimeError):
    pass


class MergeEntry(ctypes.Structure):
    _fields_ = [
        ("W", ctypes.c_void_p),
        ("W_prev", ctypes.c_void_p),
        ("A", ctypes.c_void_p),
        ("B", ctypes.c_void_p),
        ("in_features", ctypes.c_int),
        ("out_features", ctypes.c_int),
        ("r", ctypes.c_int),
        ("scale", ctypes.c_float),
    ]


class GroupMember(ctypes.Structure):
    """sowb_group_member (include/sow_b200.h)."""
    _fields_ = [
        ("W", ctypes.c_void_p),
        ("W_lo", ctypes.c_void_p),
        ("A", ctypes.c_void_p),
        ("B", ctypes.c_void_p),
        ("bias", ctypes.c_void_p),
        ("y", ctypes.c_void_p),
        ("dy", ctypes.c_void_p),
        ("dy_lo", ctypes.c_void_p),
        ("dA", ctypes.c_void_p),
        ("dB", ctypes.c_void_p),
        ("dbias", ctypes.c_void_p),
        ("out_features", ctypes.c_int),
        ("r", ctypes.c_int),
        ("scale", ctypes.c_float),
    ]


_vp, _i, _i64, _f, _sz = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_float, ctypes.c_size_t
_d = ctypes.c_double

# name -> (restype, argtypes).  Must list every symbol include/sow_b200.h declares (tests/test_abi.py checks).
SIGNATURES = {
    "sow_abi_version": (_i, []),
    "sow_last_error": (ctypes.c_char_p, []),
    "sow_profile_enable": (_i, [_i]),
    "sow_profile_read": (_i, [_i, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_int64)]),
    "sow_rank_pad": (_i, [_i]),
    "sow_group_workspace_bytes": (_sz, [_i, _i64, _i, ctypes.POINTER(GroupMember), _i]),
    "sow_group_fwd": (_i, [_vp, _vp, ctypes.POINTER(GroupMember), _i, _vp, _vp, _i64, _i, _i, _vp]),
    "sow_split_bf16x2": (_i, [_vp, _vp, _vp, _i64, _vp]),
    "sow_group_bwd": (_i, [_vp, _vp, _vp, ctypes.POINTER(GroupMember), _i, _vp, _vp, _i64, _i, _i, _vp, _sz, _vp]),
    "sow_merge_table_stride": (_sz, []),
    "sow_merge_grouped": (_i, [ctypes.POINTER(MergeEntry), _i, _i, _vp, _sz, _vp]),
    "sow_thin_qr": (_i, [_vp, _i64, _i, _vp, _i64, _i, _i, _i, _vp, _sz, _vp]),
    "sow_thin_qr_workspace_bytes": (_sz, [_i, _i, _i]),
    "tt_project": (_i, [_vp, _i64, _vp, _i64, _vp, _i64, _i, _i, _i, _i, _vp, _sz, _vp]),
    "tt_project_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "tt_interleave": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _i, _vp]),
    "tt_deinterleave": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _i, _vp]),
    "tt_gather2": (_i, [_vp, _i, _i, _i, _i, _vp, _i, _i, _vp]),
    "tt_project2": (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _i, _i, _vp, _sz, _vp]),
    "tt_project2_workspace_bytes": (_sz, [_i, _i, _i]),
    "tt_reconstruct2": (_i, [_vp, _vp, _i, _vp, _i, _i, _i, _i, _i, _vp]),
    "tt_matmul_rk": (_i, [_vp, _vp, _vp, _i, _i, _i, _vp]),
    "tt_adam_fused2": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _vp, _i, _i, _i, _i, _d, _d, _d, _d, _d, _i, _i, _vp]),
    "tt_adam2_head": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _vp, _vp, _i, _i, _i, _i, _d, _d, _i, _i, _vp]),
    "tt_adam2_fused": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _d, _d, _d, _d, _d, _i, _i,
                            _vp, _sz, _vp]),
    "tt_adam2_fused_workspace_bytes": (_sz, [_i, _i]),
    "tt_adam2_workspace_bytes": (_sz, [_i, _i]),
    "tt_adam_nd_workspace_bytes": (_sz, [_i, _i, _i, _vp]),
    "tt_nd_workspace_bytes": (_sz, [_i, _i, _i, _vp]),
    "tt_decompose_nd": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _sz, _vp]),
    "tt_reconstruct_nd": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _sz, _vp]),
    "tt_adam_nd_step": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _d, _d, _d, _d, _d, _i, _i, _vp, _sz, _vp]),
    "tt_adam2_step": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _d, _d, _d, _d, _d, _i, _i,
                           _vp, _sz, _vp]),
    "tt_adam_interleaved": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _d, _d, _d, _d, _d, _i, _vp]),
    "tt_adam_dense": (_i, [_vp, _vp, _vp, _vp, _i64, _d, _d, _d, _d, _d, _i, _vp]),
    "sow_adam_chunk_elems": (_i, []),
    "sow_adam_multi_ex": (_i, [_vp, _i, _i64, _d, _d, _d, _d, _d, _d, _d, _i, _i, _vp]),
    "sow_adam_multi": (_i, [_vp, _i, _d, _d, _d, _d, _d, _d, _d, _i, _i, _vp]),
    "sow_adam_multi_dev": (_i, [_vp, _i, _i64, _d, _d, _d, _d, _d, _vp, _i, _i, _vp]),
    "sow_adam_multi_amp": (_i, [_vp, _i, _i64, _d, _d, _d, _d, _d, _d, _d, _vp, _vp, _vp, _i, _i, _i, _vp]),
    "sow_adam_multi_clip": (_i, [_vp, _i, _i64, _d, _d, _d, _d, _d, _d, _d, _vp, _vp, _vp, _vp, _i, _i, _i, _vp]),
    "sow_grad_norm_partials": (_i, [_vp, _i, _i, _vp, _vp, _vp]),
    "sow_grad_norm_finalize": (_i, [_vp, _i, _d, _vp, _vp, _vp]),
    "sow_rope_fwd": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i64, _i64, _i64, _i64, _i64, _i64, _i64, _i, _vp]),
    "sow_rope_bwd": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i64, _i64, _i64, _i64, _i64, _i64, _i64, _i, _vp]),
    "sow_swiglu_fwd": (_i, [_vp, _vp, _vp, _i64, _i, _vp]),
    "sow_swiglu_bwd": (_i, [_vp, _vp, _vp, _vp, _vp, _i64, _i, _vp]),
    "sow_rmsnorm_fwd": (_i, [_vp, _vp, _vp, _vp, _i64, _i, _f, _i, _vp]),
    "sow_rmsnorm_bwd": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _i, _i, _vp]),
    "sow_ce_fwd": (_i, [_vp, _vp, _vp, _vp, _vp, _i64, _i, _i, _vp]),
    "sow_ce_bwd": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _i, _i, _vp]),
}

_lock = threading.Lock()
_lib = None


def load():
    """Load (once) and return the ctypes handle.  Raises SowB200Error when the extension has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise SowB200Error(
                f"{LIB_PATH} not found: build the CUDA extension first "
                "(python -c 'import __graft_entry__ as g; g.build()').  There is no CPU fallback."
            )
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if the symbol is missing -> loud failure
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = load().sow_last_error()
        raise SowB200Error(f"{what or 'sow_b200 call'} failed (code {rc}): {msg.decode() if msg else '?'}")

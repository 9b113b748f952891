"""ctypes binding of ``libstmgcn_b200.so`` (declared in ``include/stmgcn_b200.h``).

There is no CPU fallback: if the shared object is missing, importing this module raises, and every entry
point raises ``RuntimeError(stmgcn_last_error())`` on a non-zero return code.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_float, c_int32, c_int64, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("STMGCN_LIB_PATH") or os.path.join(os.path.dirname(_HERE), "lib", "libstmgcn_b200.so")

ACT_NONE, ACT_RELU = 0, 1
ABI_VERSION = 5

# (name, restype, argtypes) -- one row per symbol in include/stmgcn_b200.h
_P = c_void_p
SIGNATURES = [
    ("stmgcn_abi_version", c_int32, []),
    ("stmgcn_last_error", c_char_p, []),
    ("stmgcn_sm_count", c_int32, []),
    ("stmgcn_launch_count", c_int64, []),
    ("stmgcn_graph_from_dense", c_int32, [POINTER(c_void_p), _P, c_int64, c_int64, c_int32, _P]),
    ("stmgcn_graph_from_csr", c_int32, [POINTER(c_void_p), c_int64, c_int64, _P, _P, _P, c_int32, _P]),
    ("stmgcn_graph_destroy", c_int32, [_P]),
    ("stmgcn_graph_n", c_int64, [_P]),
    ("stmgcn_graph_nnz", c_int64, [_P]),
    ("stmgcn_graph_export", c_int32, [_P, c_int32, _P, _P, _P, _P]),
    ("stmgcn_cheb_spmm_step", c_int32, [_P, c_int32, c_float, _P, c_float, _P, c_float, _P, _P, c_int64, _P]),
    ("stmgcn_cheb_spmm_step16", c_int32, [_P, c_int32, c_float, _P, c_float, _P, c_float, _P, _P, _P, c_int64, _P]),
    ("stmgcn_to_bf16", c_int32, [_P, _P, c_int64, _P]),
    ("stmgcn_obs_to_node_major", c_int32, [_P, _P, _P, c_int64, c_int64, c_int64, c_int64, _P]),
    ("stmgcn_proj_fwd", c_int32, [_P, c_int64, c_int32, c_int64, c_int32, _P, _P, c_int32, c_int32, _P, _P,
                                  c_int64, _P]),
    ("stmgcn_proj_bwd", c_int32, [_P, c_int64, c_int32, c_int64, c_int32, _P, c_int32, c_int32, _P, _P, _P,
                                  c_float, c_int64, _P, _P, _P, _P, c_int64, _P]),
    ("stmgcn_proj_pack_tc", c_int32, [_P, c_int32, _P, _P, _P]),
    ("stmgcn_proj_fwd_tc", c_int32, [_P, c_int64, c_int32, c_int64, _P, _P, c_int32, _P, _P]),
    ("stmgcn_proj_bwd_tc", c_int32, [_P, c_int64, c_int32, c_int64, _P, c_int32, _P, _P, _P, _P, _P, _P, c_int64,
                                     _P]),
    ("stmgcn_gate_fwd", c_int32, [_P, c_int64, c_int32, c_int64, _P, _P, _P, _P, _P, _P]),
    ("stmgcn_gate_bwd", c_int32, [_P, _P, _P, _P, c_int64, c_int32, _P, _P, _P, _P, _P]),
    ("stmgcn_lstm_fwd", c_int32, [c_int32, c_int32, c_int64, c_int32, c_int32, c_int64, _P, _P, _P,
                                  POINTER(c_void_p), POINTER(c_void_p), _P, _P, _P, _P, _P, _P]),
    ("stmgcn_lstm_bwd", c_int32, [c_int32, c_int32, c_int64, c_int32, c_int32, c_int64, _P, _P, _P,
                                  POINTER(c_void_p), _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P,
                                  POINTER(c_void_p), POINTER(c_void_p), _P]),
    ("stmgcn_lstm16_pack", c_int32, [_P, _P, _P, _P, c_int32, c_int32, _P, _P, _P, _P]),
    ("stmgcn_lstm16_fwd", c_int32, [c_int32, c_int32, c_int64, c_int32, c_int64, c_int32, _P, _P,
                                    POINTER(c_void_p), POINTER(c_void_p), _P, _P, _P, _P, _P, _P, _P, _P]),
    ("stmgcn_lstm16_grid", c_int32, [c_int64]),
    ("stmgcn_lstm16_bwd", c_int32, [c_int32, c_int32, c_int64, c_int32, c_int64, c_int32, _P, _P,
                                    POINTER(c_void_p), POINTER(c_void_p), _P, _P, _P, _P, _P, _P, _P, _P, _P, _P,
                                    _P, _P, _P, POINTER(c_void_p), _P]),
    ("stmgcn_fuse_out_fwd", c_int32, [POINTER(c_void_p), c_int32, c_int64, c_int64, c_int32, c_int32, _P, _P,
                                      _P, _P, _P]),
    ("stmgcn_fuse_out_bwd", c_int32, [_P, _P, c_int64, c_int64, c_int32, c_int32, _P, _P, _P, _P, _P]),
]
EXPORTED_SYMBOLS = [s[0] for s in SIGNATURES]


def _load() -> ctypes.CDLL:
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: the ST-MGCN hot path has no CPU fallback. Build it with "
            f"`python -c 'import __graft_entry__ as g; g.build()'` (nvcc, sm_100a).")
    lib = ctypes.CDLL(LIB_PATH)
    for name, res, args in SIGNATURES:
        fn = getattr(lib, name)          # AttributeError here == header/library mismatch: fail loudly
        fn.restype = res
        fn.argtypes = args
    got = lib.stmgcn_abi_version()
    if got != ABI_VERSION:
        raise RuntimeError(f"libstmgcn_b200.so ABI {got} != binding ABI {ABI_VERSION}; rebuild")
    return lib


lib = _load()


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = lib.stmgcn_last_error()
        raise RuntimeError(f"libstmgcn_b200 {what} failed (rc={rc}): {msg.decode() if msg else '?'}")


def ptr_array(ptrs):
    """Host array of device pointers for ``const float* const*`` parameters."""
    arr = (c_void_p * len(ptrs))()
    for i, p in enumerate(ptrs):
        arr[i] = p
    return arr


def launch_count() -> int:
    return int(lib.stmgcn_launch_count())

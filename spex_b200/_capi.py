"""ctypes binding of libspex_b200.so (the C-ABI declared in include/spex_b200.h).

This module is the only place that touches the shared library.  It fails loudly: if the library
has not been built, importing it raises; if a call returns non-zero, a RuntimeError carries the
library's own error string.  There is no CPU or PyTorch fallback for any entry point.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SPEX_B200_LIB") or os.path.join(_HERE, "libspex_b200.so")  # env: tuning builds

_p = C.c_void_p
_i32 = C.c_int32
_i64 = C.c_int64
_f = C.c_float


class LongPlan(C.Structure):
    """spex_long_plan (include/spex_b200.h)."""

    _fields_ = [
        ("seg_len", _i32),
        ("n_long", _i32),
        ("n_seg", _i32),
        ("flags", _i32),
        ("long_rows", _p),
        ("long_segptr", _p),
        ("partial", _p),
        ("seg_start", _p),
        ("seg_count", _p),
        ("row_seg", _p),
        ("n_hub_seg", _i32),
    ]


_PLAN = C.POINTER(LongPlan)

# name -> (restype, argtypes); mirrors include/spex_b200.h declaration by declaration
SIGNATURES = {
    "spex_abi_version": (C.c_int, []),
    "spex_error_string": (C.c_char_p, [C.c_int]),
    "spex_device_check": (C.c_int, [C.POINTER(C.c_int)] * 3),
    "spex_launch_count": (_i64, []),
    "spex_spmm_csr_f32": (C.c_int, [_p, _p, _p, _p, _i64, _i32, _p, _p, _f, _p, _f, _PLAN, _p]),
    "spex_spmm_csr_rows_f32": (C.c_int, [_p, _p, _p, _p, _i64, _i32, _p, _i64, _p, _i32, _p, _i32, _p, _p, _p, _f, _p, _f,
                                         _PLAN, _p]),
    "spex_spmm_csr_rows_exchange_f32": (C.c_int, [_p, _p, _p, _p, _i64, _i32, _p, _i64, _p, _i32, _p, _i32, _p, _i64, _p,
                                                  _p, _i32, _p, _f, _p, _f, _PLAN, _p]),
    "spex_propagate_mean_f32": (C.c_int, [_p, _p, _p, _p, _i64, _i32, _i32, _p, _p, _p, _PLAN, _p]),
    "spex_propagate_mean_bwd_f32": (C.c_int, [_p, _p, _p, _p, _i64, _i32, _i32, _p, _p, _p, _PLAN, _p]),
    "spex_gather_f32": (C.c_int, [_p, _p, _p, _f, _p, _i64, _p]),
    "spex_edge_dropout_f32": (C.c_int, [_p, _p, _p, _p, _i64, _i64, C.c_uint64, _f, _p, _p, _p]),
    "spex_bce_fwd_f32": (C.c_int, [_p, _p, _i32, _p, _p, _p, _i64, _p, _p, _p, _p]),
    "spex_bce_bwd_f32": (C.c_int, [_p, _p, _i32, _p, _p, _p, _p, _i64, _p, _p, _p]),
    "spex_scatter_workspace_bytes": (_i64, [_i64]),
    "spex_bce_bwd_ws_f32": (C.c_int, [_p, _p, _i32, _p, _p, _p, _p, _i64, _p, _p, _p, _i64, _p]),
    "spex_clear_rows_f32": (C.c_int, [_p, _p, _i64, _i32, _p]),
    "spex_gather_owned_rows_f32": (C.c_int, [_p, _p, _i64, _i32, _i64, _i64, _p, _p]),
    "spex_scatter_rows_f32": (C.c_int, [_p, _p, _p, _p, _f, _i64, _p, _i32, _p, _i64, _i64, _p, _i64, _p]),
    "spex_bpr_bwd_ws_f32": (C.c_int, [_p, _p, _p, _p, _i32, _p, _p, _p, _p, _p, _i64, _p, _p, _p, _p, _p, _i64, _p]),
    "spex_bpr_fwd_f32": (C.c_int, [_p, _p, _p, _p, _i32, _p, _p, _p, _i64, _p, _p, _p, _p]),
    "spex_bpr_bwd_f32": (C.c_int, [_p, _p, _p, _p, _i32, _p, _p, _p, _p, _p, _i64, _p, _p, _p, _p, _p]),
    "spex_adam_f32": (C.c_int, [_p, _p, _p, _p, _i64, _f, _f, _f, _f, _i32, _p]),
    "spex_sample_negatives": (C.c_int, [_p, _p, _i32, _i32, _p, _i64, _i32, C.c_uint64, _p, _p]),
    "spex_sample_bpr": (C.c_int, [_p, _p, _i32, _i32, _i64, _i64, C.c_uint64, _p, _p, _p, _p]),
    "spex_expert_gate_f32": (C.c_int, [_p, _p, _p, _i64, _i32, _p, _p]),
    "spex_expert_gate_bwd_f32": (C.c_int, [_p, _p, _p, _p, _i64, _i32, _p, _p, _p, _p, _p]),
    "spex_score_topk_f32": (C.c_int, [_p, _p, _i32, _p, _i64, _i64, _p, _p, _i32, _p, _p, _p]),
    "spex_rating_f32": (C.c_int, [_p, _p, _i32, _p, _i64, _i64, _i32, _p, _p]),
    "spex_pack_bf16": (C.c_int, [_p, _p, _i64, _i64, _i32, _p, _p]),
    "spex_score_topk_bf16": (C.c_int, [_p, _p, _i64, _i64, _i64, _i64, _p, _p, _p, _i32, _p, _p, _p]),
    "spex_pack_f16": (C.c_int, [_p, _p, _i64, _i64, _i32, _p, _p, _p]),
    "spex_score_topk_f16": (C.c_int, [_p, _p, _i32, _i64, _i64, _i64, _i64, _p, _p, _p, _p, _p, _i32, _p, _p, _p]),
    "spex_score_candidates_f32": (C.c_int, [_p, _p, _i32, _p, _p, _i64, _i32, _p, _p]),
    "spex_ngcf_epilogue_f32": (C.c_int, [_p, _p, _p, _p, _p, _p, _i64, _i32, _f, _p, _p, _i64, _p]),
    "spex_ngcf_layer_fwd_f32": (C.c_int, [_p, _p, _p, _p, _p, _p, _p, _i64, _i32, _f, _p, _p, _i64, _p]),
    "spex_ngcf_layer_bwd_f32": (C.c_int, [_p, _p, _p, _p, _p, _p, _p, _p, _p, _i64, _i64, _i32, _f, _p, _p, _p, _p,
                                          _p, _p, _p, _p]),
    "spex_ipc_alloc": (C.c_int, [_i64, C.POINTER(_p), _p]),
    "spex_ipc_open": (C.c_int, [_p, C.POINTER(_p)]),
    "spex_ipc_close": (C.c_int, [_p]),
    "spex_ipc_free": (C.c_int, [_p]),
    "spex_spmm_csr_f32_mcast": (C.c_int, [_p, _p, _p, _p, _i64, _i32, _i64, _p, _p, _f, _p, _f, _PLAN, _p]),
    "spex_mcast_rows_f32": (C.c_int, [_p, _i64, _i32, _i64, _p, _p]),
    "spex_mcast_rows_f32_ex": (C.c_int, [_p, _i64, _i32, _i64, _p, _i32, _p]),
    "spex_push_rows_f32_ex": (C.c_int, [_p, _i64, _i32, _i64, C.POINTER(_p), _i32, _i32, _p]),
    "spex_spmm_csr_f32_publish": (C.c_int, [_p, _p, _p, _p, _i64, _i32, _i64, _p, _f, _p, _f, _p, _p,
                                            C.POINTER(_p), _i32, _PLAN, _p]),
    "spex_spmm_csr_f32_adam": (C.c_int, [_p, _p, _p, _p, _i64, _i32, _i64, _p, _f, _p, _f, _p, _p, _p, _f, _f, _f, _f,
                                         _i32, _p, C.POINTER(_p), _i32, _PLAN, _p]),
    "spex_memcpy_peer_async": (C.c_int, [_p, _p, _i64, _p]),
    "spex_push_rows_f32": (C.c_int, [_p, _i64, _i32, _i64, C.POINTER(_p), _i32, _p]),
    "spex_spmm_csr_f32_push": (
        C.c_int,
        [_p, _p, _p, _p, _i64, _i32, _i64, C.POINTER(_p), _i32, _p, _f, _p, _f, _PLAN, _p],
    ),
}

_NO_STATUS = {"spex_abi_version", "spex_error_string", "spex_launch_count", "spex_scatter_workspace_bytes"}


class SpexLibraryMissing(ImportError):
    pass


def _load():
    if not os.path.exists(LIB_PATH):
        raise SpexLibraryMissing(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C spex_b200/csrc`). spex_b200 has no CPU / PyTorch fallback."
        )
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the .so is stale: loud on purpose
        fn.restype = res
        fn.argtypes = args
    # SURVEY §8b: sm_100a only, import fails loudly on any other GPU.  A box with no CUDA device at
    # all (the CPU build/test container) may still import the binding to check the exported ABI;
    # every compute entry point fails there on its own.
    sm, ma, mi = C.c_int(0), C.c_int(0), C.c_int(0)
    rc = lib.spex_device_check(C.byref(sm), C.byref(ma), C.byref(mi))
    if rc == SPEX_E_ARCH:
        raise ImportError(
            f"spex_b200 is built for sm_100a (B200) only; the current device is sm_{ma.value}{mi.value}. "
            "There is no fallback path."
        )
    return lib


SPEX_E_ARCH = -4  # include/spex_b200.h
lib = _load()


def error_string(code: int) -> str:
    return lib.spex_error_string(int(code)).decode()


def call(name: str, *args):
    """Call a status-returning entry point; raise RuntimeError(name: reason) on failure."""
    rc = getattr(lib, name)(*args)
    if name in _NO_STATUS:
        return rc
    if rc != 0:
        raise RuntimeError(f"{name} failed ({rc}): {error_string(rc)}")
    return 0


def launch_count() -> int:
    return int(lib.spex_launch_count())


def abi_version() -> int:
    return int(lib.spex_abi_version())


def device_check():
    sm, ma, mi = C.c_int(0), C.c_int(0), C.c_int(0)
    call("spex_device_check", C.byref(sm), C.byref(ma), C.byref(mi))
    return sm.value, ma.value, mi.value


def ptr(t):
    """Device pointer of a torch tensor (None -> NULL)."""
    return None if t is None else C.c_void_p(t.data_ptr())


def stream_ptr():
    import torch

    return C.c_void_p(torch.cuda.current_stream().cuda_stream)

"""ctypes binding of libgcnb200.so (the C ABI declared in include/gcnb200.h).

This is the stub a pygcn maintainer would add next to pygcn/layers.py (see
INTEGRATION.md).  There is no CPU or eager-PyTorch fallback: if the CUDA library is
missing or fails to load, importing the hot path raises.
"""
from __future__ import annotations

import ctypes
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libgcnb200.so")

c_i64 = ctypes.c_int64
c_int = ctypes.c_int
c_vp = ctypes.c_void_p
c_sz = ctypes.c_size_t
c_double = ctypes.c_double

NUM_BINS = 5
BIN_EDGES = (0, 1, 9, 33, 1025)

# flags (mirror include/gcnb200.h)
BUILD_SYMMETRIZE, BUILD_SELF_LOOPS, BUILD_ROW_NORMALIZE, BUILD_KEEP_F64 = 1, 2, 4, 8
SPMM_TRANSPOSE, SPMM_RELU, SPMM_ACCUMULATE = 1, 2, 4
GEMM_FP32, GEMM_TF32X3, GEMM_AUTO = 0, 1, 2
LAYER_RELU, LAYER_NEED_DX, LAYER_NEED_DW, LAYER_NEED_DB, LAYER_AGG_FIRST = 1, 2, 4, 8, 16
TUNE_SPMM_KERNEL, TUNE_SPMM_GROUP_VARIANT, TUNE_PDL = 1, 2, 3
TUNE_SPMM_STREAM, TUNE_STREAM_HOT_MB, TUNE_STREAM_HINT, TUNE_STREAM_MIN_ROW_BYTES, TUNE_STREAM_BATCH = 4, 5, 6, 7, 8


class GraphInfo(ctypes.Structure):
    _fields_ = [
        ("n_rows", c_i64), ("n_cols", c_i64), ("nnz", c_i64),
        ("bin_rows", c_i64 * NUM_BINS), ("t_bin_rows", c_i64 * NUM_BINS),
        ("max_degree", c_i64), ("t_max_degree", c_i64),
        ("n_long_chunks", c_i64), ("t_n_long_chunks", c_i64),
        ("pattern_symmetric", ctypes.c_int32), ("dense_route", ctypes.c_int32),
        ("device_bytes", c_i64),
        ("d_rowptr", c_vp), ("d_col", c_vp), ("d_val", c_vp),
        ("d_t_rowptr", c_vp), ("d_t_col", c_vp), ("d_t_val", c_vp),
    ]


# name -> (restype, argtypes); every symbol include/gcnb200.h declares
SIGNATURES = {
    "gcnb_version": (c_int, []),
    "gcnb_last_error": (ctypes.c_char_p, []),
    "gcnb_check_device": (c_int, []),
    "gcnb_graph_from_edges": (c_int, [c_i64, c_i64, c_vp, c_vp, c_int, c_vp, ctypes.POINTER(c_vp)]),
    "gcnb_graph_from_coo": (c_int, [c_i64, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, ctypes.POINTER(c_vp)]),
    "gcnb_graph_from_csr": (c_int, [c_i64, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, ctypes.POINTER(c_vp)]),
    "gcnb_graph_from_dense": (c_int, [c_i64, c_i64, c_vp, c_i64, c_vp, ctypes.POINTER(c_vp)]),
    "gcnb_graph_free": (None, [c_vp]),
    "gcnb_graph_get_info": (c_int, [c_vp, ctypes.POINTER(GraphInfo)]),
    "gcnb_graph_block": (c_int, [c_vp, c_int, c_i64, c_i64, c_i64, c_i64, c_i64, c_i64, c_vp, ctypes.POINTER(c_vp)]),
    "gcnb_graph_block_gathered": (c_int, [c_vp, c_int, c_i64, c_i64, c_int, ctypes.POINTER(c_i64), c_i64, c_int, c_vp,
                                          ctypes.POINTER(c_vp)]),
    "gcnb_graph_export_coo": (c_int, [c_vp, c_vp, c_vp, c_vp]),
    "gcnb_graph_export_csr": (c_int, [c_vp, c_int, c_vp, c_vp, c_vp, c_vp]),
    "gcnb_spmm": (c_int, [c_vp, c_int, c_vp, c_i64, c_i64, c_vp, c_vp, c_i64, c_vp, c_sz, c_vp]),
    "gcnb_spmm_bf16": (c_int, [c_vp, c_int, c_vp, c_i64, c_i64, c_vp, c_vp, c_i64, c_vp, c_sz, c_vp]),
    "gcnb_to_bf16": (c_int, [c_i64, c_i64, c_vp, c_i64, c_vp, c_i64, c_vp]),
    "gcnb_spmm_workspace_bytes": (c_sz, [c_vp, c_int, c_i64]),
    "gcnb_gemm": (c_int, [c_i64, c_i64, c_i64, c_vp, c_i64, c_i64, c_vp, c_i64, c_i64, c_vp, c_i64, c_int,
                          c_vp, c_sz, c_vp]),
    "gcnb_gemm_ex": (c_int, [c_i64, c_i64, c_i64, c_vp, c_i64, c_i64, c_vp, c_i64, c_i64, c_vp, c_i64, c_vp, c_int, c_int,
                             c_vp, c_sz, c_vp]),
    "gcnb_gemm_workspace_bytes": (c_sz, [c_i64, c_i64, c_i64, c_int]),
    "gcnb_colsum": (c_int, [c_i64, c_i64, c_vp, c_i64, c_vp, c_i64, c_vp, c_i64, c_vp, c_vp, c_sz, c_vp]),
    "gcnb_colsum_workspace_bytes": (c_sz, [c_i64, c_i64]),
    "gcnb_layer_forward": (c_int, [c_vp, c_vp, c_i64, c_vp, c_vp, c_i64, c_i64, c_int, c_int, c_vp, ctypes.c_float,
                                   c_vp, c_vp, c_vp, c_sz, c_vp]),
    "gcnb_layer_backward": (c_int, [c_vp, c_vp, c_i64, c_vp, c_vp, c_i64, c_vp, c_i64, c_i64, c_int, c_int,
                                    c_vp, ctypes.c_float, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_sz, c_vp]),
    "gcnb_layer_workspace_bytes": (c_sz, [c_vp, c_i64, c_i64, c_int]),
    "gcnb_l2_flush": (c_int, [c_vp, c_sz, c_vp]),
    "gcnb_set_tuning": (c_int, [c_int, c_int]),
    "gcnb_symm_alloc": (c_int, [c_sz, c_vp, c_vp]),
    "gcnb_symm_open": (c_int, [c_vp, c_vp]),
    "gcnb_symm_close": (c_int, [c_vp]),
    "gcnb_symm_free": (c_int, [c_vp]),
    "gcnb_peer_epoch_bump": (c_int, [c_vp, c_vp, c_int, c_vp]),
    "gcnb_peer_push": (c_int, [c_vp, c_sz, c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_int, c_vp]),
    "gcnb_peer_wait": (c_int, [c_vp, c_vp, c_vp]),
    "gcnb_peer_wait_lag": (c_int, [c_vp, c_vp, ctypes.c_uint32, c_vp]),
    "gcnb_peer_copy": (c_int, [c_vp, c_vp, c_sz, c_vp]),
    "gcnb_fresh_bn_workspace_bytes": (c_sz, [c_i64, c_i64]),
    "gcnb_fresh_bn_forward": (c_int, [c_i64, c_i64, c_vp, c_i64, c_int, ctypes.c_float, c_vp, c_i64, c_vp, c_vp, c_vp, c_sz,
                                      c_vp]),
    "gcnb_fresh_bn_backward": (c_int, [c_i64, c_i64, c_vp, c_i64, c_int, c_vp, c_i64, c_vp, c_vp, c_vp, c_i64, c_vp, c_vp,
                                       c_sz, c_vp]),
    "gcnb_graph_block_sources": (c_int, [c_vp, c_int, c_i64, c_i64, c_int, ctypes.POINTER(c_i64), c_i64, ctypes.c_uint64,
                                         c_vp, ctypes.POINTER(c_vp)]),
    "gcnb_peer_ack": (c_int, [c_vp, c_vp, c_vp]),
    "gcnb_launch_count": (ctypes.c_longlong, []),
    "gcnb_halo_create": (c_int, [c_int, c_int, ctypes.POINTER(c_i64), c_vp, ctypes.POINTER(c_i64), ctypes.POINTER(c_i64), c_vp,
                                 ctypes.POINTER(c_vp)]),
    "gcnb_halo_free": (None, [c_vp]),
    "gcnb_halo_send_rows": (c_i64, [c_vp]),
    "gcnb_halo_recv_rows": (c_i64, [c_vp]),
    "gcnb_halo_nccl_available": (c_int, []),
    "gcnb_halo_pack": (c_int, [c_vp, c_vp, c_i64, c_i64, c_vp, c_vp]),
    "gcnb_halo_exchange": (c_int, [c_vp, c_vp, c_vp, c_i64, c_vp, c_vp]),
    # fp64 tier
    "gcnb_graph_from_coo_f64": (c_int, [c_i64, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, ctypes.POINTER(c_vp)]),
    "gcnb_graph_from_csr_f64": (c_int, [c_i64, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, ctypes.POINTER(c_vp)]),
    "gcnb_graph_from_dense_f64": (c_int, [c_i64, c_i64, c_vp, c_i64, c_vp, ctypes.POINTER(c_vp)]),
    "gcnb_graph_export_csr_f64": (c_int, [c_vp, c_int, c_vp, c_vp, c_vp, c_vp]),
    "gcnb_spmm_f64": (c_int, [c_vp, c_int, c_vp, c_i64, c_i64, c_vp, c_vp, c_i64, c_double, c_vp, c_i64, c_vp, c_sz, c_vp]),
    "gcnb_spmm_f64_workspace_bytes": (c_sz, [c_vp, c_int, c_i64]),
    "gcnb_gemm_f64": (c_int, [c_i64, c_i64, c_i64, c_vp, c_i64, c_i64, c_vp, c_i64, c_i64, c_vp, c_i64, c_vp, c_sz, c_vp]),
    "gcnb_gemm_f64_ex": (c_int, [c_i64, c_i64, c_i64, c_vp, c_i64, c_i64, c_vp, c_i64, c_i64, c_vp, c_i64, c_vp, c_int,
                                 c_vp, c_sz, c_vp]),
    "gcnb_gemm_f64_workspace_bytes": (c_sz, [c_i64, c_i64, c_i64]),
    "gcnb_colsum_f64": (c_int, [c_i64, c_i64, c_vp, c_i64, c_vp, c_i64, c_vp, c_i64, c_vp, c_vp, c_sz, c_vp]),
    "gcnb_colsum_f64_workspace_bytes": (c_sz, [c_i64, c_i64]),
    "gcnb_layer_forward_f64": (c_int, [c_vp, c_vp, c_i64, c_vp, c_vp, c_i64, c_i64, c_int, c_vp, c_double, c_vp, c_vp,
                                       c_vp, c_sz, c_vp]),
    "gcnb_layer_backward_f64": (c_int, [c_vp, c_vp, c_i64, c_vp, c_vp, c_i64, c_vp, c_i64, c_i64, c_int, c_vp, c_double,
                                        c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_sz, c_vp]),
    "gcnb_layer_f64_workspace_bytes": (c_sz, [c_vp, c_i64, c_i64]),
}

_lock = threading.Lock()
_lib = None


class GcnbError(RuntimeError):
    pass


def load(build_if_missing=True):
    """Load libgcnb200.so (building it with nvcc when it is absent and nvcc is here)."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        from . import build as _build

        # a library older than csrc/ or include/gcnb200.h would be called with the NEW signatures below: rebuild it
        # when nvcc is here, refuse to load it otherwise (GCNB_SKIP_STALE_CHECK=1 for a tree shipped without sources)
        stale = os.path.exists(LIB_PATH) and os.environ.get("GCNB_SKIP_STALE_CHECK") != "1" and _build.needs_build()
        if (stale or not os.path.exists(LIB_PATH)) and build_if_missing:
            try:
                _build.build()
                stale = False
            except RuntimeError:
                if not os.path.exists(LIB_PATH):
                    raise
        if stale:
            raise GcnbError(
                "libgcnb200.so at %s is older than its sources (pygcn_b200/csrc, include/gcnb200.h): rebuild it with "
                "`python -m pygcn_b200.build`" % LIB_PATH)
        if not os.path.exists(LIB_PATH):
            raise GcnbError(
                "libgcnb200.so not found at %s: build it with `python -m pygcn_b200.build` "
                "(there is no CPU/PyTorch fallback for the GCN hot path)" % LIB_PATH
            )
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if the library does not export it
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def last_error():
    msg = load().gcnb_last_error()
    return msg.decode("utf-8", "replace") if msg else ""


def check(status, what=""):
    if status != 0:
        raise GcnbError("%s failed (status %d): %s" % (what or "gcnb call", status, last_error()))

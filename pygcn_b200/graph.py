"""Device-resident adjacency: CSR + CSR^T + row-length-binned schedule, built on the GPU.

Replaces, for the GCN hot path, the reference's host-side graph helpers
  pygcn/utils.py:360-368  (edge list -> symmetric A + I; commented Cora loader)
  pygcn/utils.py:390-397  (normalize)
  pygcn/utils.py:407-414  (sparse_mx_to_torch_sparse_tensor)
and the per-call coalesce / COO->CSR conversion hidden inside `torch.spmm(adj, .)`
(pygcn/layers.py:34): the handle is built once per adjacency and reused by every call.
"""
from __future__ import annotations

import ctypes
import threading
import weakref

import torch

from . import _lib


def _stream_ptr(device):
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _require_cuda(t, what):
    if not isinstance(t, torch.Tensor):
        raise TypeError("%s must be a torch.Tensor, got %s" % (what, type(t).__name__))
    if not t.is_cuda:
        raise RuntimeError(
            "%s is on %s: pygcn_b200 runs the GCN layer on a CUDA device only "
            "(no CPU fallback); move the tensor with .cuda()" % (what, t.device)
        )


class Graph:
    """Opaque handle to a gcnb_graph living in HBM.  Accepted wherever `adj` is."""

    def __init__(self, handle, device, source="unknown", dtype=torch.float32):
        self._h = ctypes.c_void_p(handle)
        self.device = torch.device(device)
        self.source = source
        # torch.float64: the handle keeps fp64 values (and their fp32 rounding); layers on it compute in fp64
        self.dtype = dtype
        info = _lib.GraphInfo()
        _lib.check(_lib.load().gcnb_graph_get_info(self._h, ctypes.byref(info)), "gcnb_graph_get_info")
        self.n_rows, self.n_cols, self.nnz = int(info.n_rows), int(info.n_cols), int(info.nnz)
        self.bin_rows = [int(v) for v in info.bin_rows]
        self.t_bin_rows = [int(v) for v in info.t_bin_rows]
        self.max_degree, self.t_max_degree = int(info.max_degree), int(info.t_max_degree)
        self.n_long_chunks, self.t_n_long_chunks = int(info.n_long_chunks), int(info.t_n_long_chunks)
        self.pattern_symmetric = bool(info.pattern_symmetric)
        self.dense_route = bool(info.dense_route)
        self.device_bytes = int(info.device_bytes)
        self._finalizer = weakref.finalize(self, _lib.load().gcnb_graph_free, self._h)

    # ------------------------------------------------------------------ constructors
    @classmethod
    def from_edges(cls, src, dst, num_nodes, symmetrize=True, self_loops=True, row_normalize=True, dtype=torch.float32):
        """Edge list -> (optionally) max-symmetrised, + I, row-normalised adjacency.

        With all three flags set this is the reference's Cora pipeline
        (pygcn/utils.py:360-368, 390-397, 407-414) bit for bit.  dtype=torch.float64 keeps the fp64 values
        `normalize` computes before the cast of utils.py:409 (an fp64 handle).
        """
        if dtype not in (torch.float32, torch.float64):
            raise ValueError("dtype must be torch.float32 or torch.float64, got %s" % (dtype,))
        _require_cuda(src, "src")
        _require_cuda(dst, "dst")
        if src.dim() != 1 or src.shape != dst.shape:
            raise RuntimeError("src and dst must be 1-D tensors of equal length")
        src = src.to(torch.int32).contiguous()
        dst = dst.to(torch.int32).contiguous()
        flags = (_lib.BUILD_SYMMETRIZE if symmetrize else 0) | (_lib.BUILD_SELF_LOOPS if self_loops else 0) | (
            _lib.BUILD_ROW_NORMALIZE if row_normalize else 0) | (_lib.BUILD_KEEP_F64 if dtype == torch.float64 else 0)
        out = ctypes.c_void_p()
        with torch.cuda.device(src.device):
            st = _lib.load().gcnb_graph_from_edges(
                int(num_nodes), src.numel(), src.data_ptr(), dst.data_ptr(), flags, _stream_ptr(src.device),
                ctypes.byref(out),
            )
        _lib.check(st, "gcnb_graph_from_edges")
        return cls(out.value, src.device, "edges", dtype)

    @classmethod
    def from_torch(cls, adj):
        """torch adjacency (sparse COO, sparse CSR or dense strided; fp32, or fp64 for an fp64 handle) -> Graph."""
        _require_cuda(adj, "adj")
        if adj.dim() != 2:
            raise RuntimeError("adj must be a matrix, got %d-D" % adj.dim())
        if adj.dtype not in (torch.float32, torch.float64):
            raise RuntimeError("adj must be float32 (the reference builds FloatTensors) or float64, got %s" % adj.dtype)
        f64 = adj.dtype == torch.float64
        sfx = "_f64" if f64 else ""
        lib = _lib.load()
        out = ctypes.c_void_p()
        n_rows, n_cols = adj.shape
        with torch.cuda.device(adj.device):
            sp = _stream_ptr(adj.device)
            if adj.layout == torch.sparse_coo:
                if adj.dense_dim() != 0 or adj.sparse_dim() != 2:
                    raise RuntimeError("hybrid sparse tensors are not supported")
                idx = adj._indices()
                val = adj._values().contiguous()
                row = idx[0].contiguous()
                col = idx[1].contiguous()
                st = getattr(lib, "gcnb_graph_from_coo" + sfx)(n_rows, n_cols, val.numel(), row.data_ptr(), col.data_ptr(),
                                                               val.data_ptr(), sp, ctypes.byref(out))
                src = "coo"
            elif adj.layout == torch.sparse_csr:
                crow = adj.crow_indices().to(torch.int64).contiguous()
                col = adj.col_indices().to(torch.int64).contiguous()
                val = adj.values().contiguous()
                st = getattr(lib, "gcnb_graph_from_csr" + sfx)(n_rows, n_cols, val.numel(), crow.data_ptr(), col.data_ptr(),
                                                               val.data_ptr(), sp, ctypes.byref(out))
                src = "csr"
            elif adj.layout == torch.strided:
                a = adj if adj.stride(1) == 1 or n_cols <= 1 else adj.contiguous()
                lda = a.stride(0) if n_rows > 1 else max(n_cols, 1)
                if lda < n_cols:
                    a = a.contiguous()
                    lda = n_cols
                st = getattr(lib, "gcnb_graph_from_dense" + sfx)(n_rows, n_cols, a.data_ptr(), lda, sp, ctypes.byref(out))
                src = "dense"
            else:
                raise RuntimeError("unsupported adjacency layout %s" % adj.layout)
        _lib.check(st, "gcnb_graph_from_" + src + sfx)
        return cls(out.value, adj.device, src, adj.dtype)

    # ------------------------------------------------------------------ exports
    def to_sparse_coo(self):
        """torch sparse COO tensor in the exact layout utils.py:407-414 returns
        (int64 [2,nnz] indices, row-major / columns ascending, fp32 values -- fp64 on an fp64 handle -- uncoalesced flag)."""
        idx = torch.empty((2, self.nnz), dtype=torch.int64, device=self.device)
        val = torch.empty((self.nnz,), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(
                _lib.load().gcnb_graph_export_coo(self._h, idx.data_ptr(), val.data_ptr(), _stream_ptr(self.device)),
                "gcnb_graph_export_coo",
            )
        if self.dtype == torch.float64:  # the COO values are the CSR's, in the same order
            val = self.csr()[2]
        return torch.sparse_coo_tensor(idx, val, (self.n_rows, self.n_cols), check_invariants=False)

    def csr(self, transpose=False):
        """(rowptr int32, col int32, val) copies of the device CSR (or of the CSR of A^T); val is fp32, or fp64 on an
        fp64 handle."""
        rows = self.n_cols if transpose else self.n_rows
        f64 = self.dtype == torch.float64
        rowptr = torch.empty((rows + 1,), dtype=torch.int32, device=self.device)
        col = torch.empty((self.nnz,), dtype=torch.int32, device=self.device)
        val = torch.empty((self.nnz,), dtype=self.dtype, device=self.device)
        name = "gcnb_graph_export_csr_f64" if f64 else "gcnb_graph_export_csr"
        with torch.cuda.device(self.device):
            _lib.check(
                getattr(_lib.load(), name)(self._h, 1 if transpose else 0, rowptr.data_ptr(), col.data_ptr(),
                                           val.data_ptr(), _stream_ptr(self.device)),
                name,
            )
        return rowptr, col, val

    @property
    def shape(self):
        return (self.n_rows, self.n_cols)

    def __repr__(self):
        return "Graph(%d x %d, nnz=%d, bins=%s, long_chunks=%d, sym_pattern=%s, %s%s%s, %.1f MB)" % (
            self.n_rows, self.n_cols, self.nnz, self.bin_rows, self.n_long_chunks, self.pattern_symmetric,
            "dense route, " if self.dense_route else "", "fp64, " if self.dtype == torch.float64 else "", self.device,
            self.device_bytes / 1e6,
        )


# ---------------------------------------------------------------------- adjacency cache
# The reference passes the same `adj` tensor to every layer call of a run
# (SURVEY.md 8b); the handle is built on first sight and dropped with the tensor.
_cache = {}
_cache_lock = threading.Lock()


def _adj_fingerprint(adj):
    if adj.layout == torch.sparse_coo:
        return (adj._values().data_ptr(), adj._indices().data_ptr(), adj._values()._version, tuple(adj.shape),
                adj._nnz())
    if adj.layout == torch.sparse_csr:
        return (adj.values().data_ptr(), adj.col_indices().data_ptr(), adj.values()._version, tuple(adj.shape))
    return (adj.data_ptr(), adj._version, tuple(adj.shape), tuple(adj.stride()))


def as_graph(adj):
    """Graph for `adj` (Graph passes through; torch tensors are converted once and cached)."""
    if isinstance(adj, Graph):
        return adj
    _require_cuda(adj, "adj")
    key = id(adj)
    fp = _adj_fingerprint(adj)
    with _cache_lock:
        hit = _cache.get(key)
        if hit is not None and hit[0] == fp and hit[1]() is adj:
            return hit[2]
    g = Graph.from_torch(adj)
    with _cache_lock:
        try:
            ref = weakref.ref(adj, lambda _r, k=key: _cache.pop(k, None))
        except TypeError:  # pragma: no cover
            return g
        _cache[key] = (fp, ref, g)
    return g


def clear_cache():
    with _cache_lock:
        _cache.clear()

"""Multi-GPU GCN layer: 1-D row partition of A-hat over the GPUs of one node (SURVEY.md 8e).

The reference is single-process / single-GPU (no torch.distributed anywhere); this is the
B200-native scaling of its hot path (pygcn/layers.py:32-38 + autograd):

  * rank p owns the contiguous row block p of A-hat (and the matching rows of X, out, G), block
    boundaries balance stored entries (nnz), W and b are replicated;
  * the row block is cut into the diagonal block A[p,p] (columns this rank owns) and the remote
    block A[p,~p] whose column ids address the all-gathered panel directly:
        out_p = A[p,p] . S_p + A[p,~p] . allgather(S) ,      S_q = X_q W  computed on rank q
    the diagonal block runs first while the NCCL all-gather of the panels is in flight over NVLink
    (communicator stream); the remote block accumulates once it has landed and applies bias/ReLU.
    (A finer per-source-rank column blocking was measured first and rejected: every extra pass over
    the rows costs a read-modify-write of the output rows and shorter gather loops; profiles/.)
  * backward uses the same scheme on the row block of A-hat^T with G as the exchanged panel
    (atomic-free, deterministic), then dW/db are summed with one all-reduce.

  * exchange "peer" (default on GPUs with peer access): the all-gather is replaced by our own push
    kernel over NVLink peer memory (csrc/peer.cu) and the row block is cut into one column block per
    source rank, consumed in the order p, p+1, ... as the slots land (flag per source), so the
    transfer of slot q+1 overlaps the SpMM over block q.  `PeerExchange` below; the NCCL path stays as
    exchange "nccl".

One process per GPU (`torchrun`), `torch.distributed` for the plumbing.  The arithmetic is behind
an `ops` object: `CudaOps` (libgcnb200.so) in production; the CPU tests of the host logic
(tests/test_dist_gloo.py, gloo, world size 2) inject a numpy implementation.
"""
from __future__ import annotations

import ctypes
import json
import os
import sys
import time

import torch
import torch.distributed as dist
from torch.autograd.function import once_differentiable


# ---------------------------------------------------------------------------- host logic
def partition_rows_by_nnz(rowptr, world, row_weight=0.0):
    """Row-block boundaries [b_0=0, ..., b_world=N] with ~equal cost per block, cost = stored entries +
    row_weight * rows.

    rowptr: 1-D integer tensor/array of length N+1 (host).  Boundaries are non-decreasing; a block
    may be empty when there are fewer rows than ranks.
    row_weight = 0 (default) balances stored entries alone: right for the SpMM, and on graphs with even
    degrees the blocks then hold equal row counts too.  On power-law graphs they do not (products-shaped R-MAT,
    8 ranks: 21 K ... 909 K rows, tools/halo_fraction.py), and the all-gather ships world * max(rows) padded
    panel rows; row_weight = the average degree weighs both equally and bounds that padding.
    """
    rp = torch.as_tensor(rowptr, dtype=torch.int64).cpu()
    n = rp.numel() - 1
    if row_weight:
        rp = rp.to(torch.float64) + float(row_weight) * torch.arange(n + 1, dtype=torch.float64)
    total = rp[-1].item()
    bounds = [0]
    for k in range(1, world):
        target = (total * k) // world if not row_weight else total * k / world
        r = int(torch.searchsorted(rp, torch.tensor([target], dtype=rp.dtype), right=False)[0])
        r = min(max(r, bounds[-1]), n)
        bounds.append(r)
    bounds.append(n)
    return bounds


def balanced_node_partition(row_len, world):
    """A 1-D partition of the NODES in which every block holds the same number of rows AND (nearly) the same number of
    stored entries: nodes sorted by row length, dealt to the ranks in snake order (0 .. P-1, P-1 .. 0, ...), each
    rank's nodes kept in ascending id order.

    Contiguous row blocks cannot give both on a power-law graph (products-shaped R-MAT, 2 ranks: the block with half
    the entries holds 30 % of the rows), and the layer step alternates phases that scale with rows (dense products,
    element-wise passes) and with entries (SpMMs), separated by exchanges that synchronise the ranks -- so the step
    costs the sum over phases of the slowest rank, and a partition that balances only the total helps nobody
    (profiles/r02_dist_tune_n2.txt: 33 ms at 2 GPUs against 35 ms at one).

    row_len: 1-D integer tensor [N] (any device).  Returns (new_id int64 [N]: node i becomes row new_id[i] of the
    relabelled graph; bounds [world + 1]: rank p owns relabelled rows bounds[p] .. bounds[p + 1])."""
    rl = torch.as_tensor(row_len).to(torch.int64)
    n = rl.numel()
    order = torch.argsort(rl, descending=True, stable=True)
    k = torch.arange(n, device=rl.device)
    lap, pos = torch.div(k, world, rounding_mode="floor"), k % world
    owner_sorted = torch.where(lap % 2 == 0, pos, world - 1 - pos)
    owner = torch.empty(n, dtype=torch.int64, device=rl.device)
    owner[order] = owner_sorted
    counts = torch.bincount(owner, minlength=world)
    bounds = [0] + [int(v) for v in torch.cumsum(counts, 0).cpu()]
    # within a rank: ascending original id (a stable sort of the owners keeps it)
    by_owner = torch.argsort(owner, stable=True)
    new_id = torch.empty(n, dtype=torch.int64, device=rl.device)
    new_id[by_owner] = k
    return new_id, bounds


def exchange_phases(rank, world):
    """Consumption order of the source ranks for the pipelined exchange, grouped into phases:
    [[p], [p+1, p+2], [p+3, p+4], ..., [last]] (mod world).  One SpMM per phase: this rank's own slot
    first (nothing to wait for), pairs in the middle (a row restricted to ONE of 8 sources is ~12
    stored entries -- too short to gather efficiently), and a single source at the end so that little
    work is left once the last slot has landed."""
    order = [(rank + k) % world for k in range(world)]
    phases = [[order[0]]]
    rest = order[1:]
    while len(rest) > 1:
        phases.append(rest[:2])
        rest = rest[2:]
    if rest:
        phases.append(rest)
    return phases


class DistGraph:
    """Row block `rank` of A-hat and of A-hat^T, each split into the diagonal block (columns owned
    by this rank, local ids) and the remote block (all other columns, ids remapped to the layout of
    the all-gathered panel: source q occupies rows [q*pad_rows, q*pad_rows + n_q))."""

    # Splitting the row block costs a second pass over the rows (read-modify-write of the output,
    # shorter gather loops: measured +35 % SpMM time on the uniform CBG graph), and can hide at most
    # the diagonal block's share of the work behind the all-gather.  It pays only when the partition
    # has locality, i.e. most stored entries sit in the diagonal block.
    SPLIT_MIN_DIAG_FRACTION = 0.6

    def __init__(self, rank, world, bounds, pad_rows, fwd_diag, fwd_remote, bwd_diag, bwd_remote, nnz_local,
                 nnz_global, split=True):
        self.rank, self.world = rank, world
        self.bounds = list(bounds)
        self.pad_rows = pad_rows
        # split=True : (diag, remote) pairs.  split=False: *_diag is None and *_remote holds the whole
        # row block in the all-gather column layout (own slot included).
        self.split = split
        self.fwd_diag, self.fwd_remote = fwd_diag, fwd_remote
        self.bwd_diag, self.bwd_remote = bwd_diag, bwd_remote
        self.nnz_local, self.nnz_global = nnz_local, nnz_global
        # exchange "peer": one column block per phase (group of source ranks, exchange_phases), columns in
        # the gathered layout, for A and A^T
        self.phases = None
        self.fwd_blocks = None
        self.bwd_blocks = None

    def n_rows(self, q=None):
        q = self.rank if q is None else q
        return self.bounds[q + 1] - self.bounds[q]

    @staticmethod
    def padded_rows(bounds):
        """Rows per source slot of the all-gathered panel: the largest block, rounded up to 8."""
        m = max(bounds[q + 1] - bounds[q] for q in range(len(bounds) - 1))
        return max(8, (m + 7) // 8 * 8)

    @classmethod
    def from_graph(cls, graph, rank, world, bounds=None, split=None, per_source=False, row_weight=0.0):
        """Cut the row block of `rank` out of a full device `Graph` (CUDA).  split=None decides from
        the share of stored entries in the diagonal block (SPLIT_MIN_DIAG_FRACTION).
        per_source=True additionally cuts one column block per source rank (exchange "peer")."""
        from . import _lib
        from .graph import Graph, _stream_ptr

        lib = _lib.load()
        if bounds is None:
            bounds = partition_rows_by_nnz(graph.csr()[0].cpu(), world, row_weight)
        r0, r1 = bounds[rank], bounds[rank + 1]
        pad = cls.padded_rows(bounds)
        hb = (ctypes.c_int64 * (world + 1))(*bounds)

        def cut_diag(transpose):
            with torch.cuda.device(graph.device):
                out = ctypes.c_void_p()
                st = lib.gcnb_graph_block(graph._h, 1 if transpose else 0, r0, r1, r0, r1, 0, max(pad, 1),
                                          _stream_ptr(graph.device), ctypes.byref(out))
                _lib.check(st, "gcnb_graph_block")
                return Graph(out.value, graph.device, "diag[%d]%s" % (rank, "^T" if transpose else ""))

        def cut_gathered(transpose, exclude):
            with torch.cuda.device(graph.device):
                out = ctypes.c_void_p()
                st = lib.gcnb_graph_block_gathered(graph._h, 1 if transpose else 0, r0, r1, world, hb, pad, exclude,
                                                   _stream_ptr(graph.device), ctypes.byref(out))
                _lib.check(st, "gcnb_graph_block_gathered")
                return Graph(out.value, graph.device, "%s[%d]%s" % ("remote" if exclude >= 0 else "rows", rank,
                                                                    "^T" if transpose else ""))

        def cut_sources(transpose, qs):
            mask = 0
            for q in qs:
                mask |= 1 << q
            with torch.cuda.device(graph.device):
                out = ctypes.c_void_p()
                st = lib.gcnb_graph_block_sources(graph._h, 1 if transpose else 0, r0, r1, world, hb, pad, mask,
                                                  _stream_ptr(graph.device), ctypes.byref(out))
                _lib.check(st, "gcnb_graph_block_sources")
                return Graph(out.value, graph.device, "A[%d,%s]%s" % (rank, qs, "^T" if transpose else ""))

        fd = cut_diag(False)
        if world == 1:
            return cls(rank, world, bounds, pad, fd, None, cut_diag(True), None, fd.nnz, graph.nnz, True)
        full = cut_gathered(False, -1)
        if split is None:
            split = fd.nnz >= cls.SPLIT_MIN_DIAG_FRACTION * max(full.nnz, 1)
        if split:
            dg = cls(rank, world, bounds, pad, fd, cut_gathered(False, rank), cut_diag(True),
                     cut_gathered(True, rank), full.nnz, graph.nnz, True)
        else:
            dg = cls(rank, world, bounds, pad, None, full, None, cut_gathered(True, -1), full.nnz, graph.nnz, False)
        if per_source:
            dg.phases = exchange_phases(rank, world)
            dg.fwd_blocks = [cut_sources(False, qs) for qs in dg.phases]
            dg.bwd_blocks = [cut_sources(True, qs) for qs in dg.phases]
        return dg


# ---------------------------------------------------------------------------- partitioned graph build
def _partition_counts(src, dst, n, r0, r1):
    """Stage 1 of the partitioned build on one rank: the rows [r0, r1) of the UN-normalised adjacency
    max(C, C^T) + I (C = edge counts; pygcn/utils.py:360-368) from the edges that touch those rows.
    A row of the symmetrised matrix depends only on the edges incident to its node, so the block is exact
    although the rank never sees the rest of the graph.  Returns (local rowptr int64, global col int64,
    counts fp64, row sums fp64)."""
    from .graph import Graph

    touch = ((src >= r0) & (src < r1)) | ((dst >= r0) & (dst < r1))
    u = Graph.from_edges(src[touch], dst[touch], n, symmetrize=True, self_loops=True, row_normalize=False)
    rowptr, col, val = u.csr()
    e0, e1 = int(rowptr[r0]), int(rowptr[r1])
    lrp = (rowptr[r0:r1 + 1] - e0).to(torch.int64)
    lcol = col[e0:e1].to(torch.int64)
    a = val[e0:e1].to(torch.float64)
    rows = torch.repeat_interleave(torch.arange(r1 - r0, device=src.device), lrp[1:] - lrp[:-1])
    rowsum = torch.zeros(r1 - r0, dtype=torch.float64, device=src.device).index_add_(0, rows, a)  # small integers: exact
    del u
    return lrp, lcol, a, rows, rowsum


def _partition_blocks(rank, world, bounds, pad, lrp, lcol, a, rows, rowsum_global, n_global_nnz=0):
    """Stage 2: with every node's row sum known (all-gathered), normalise like utils.normalize
    (pygcn/utils.py:390-397: r_inv = rowsum^-1 in fp64, inf -> 0, fp32 cast of the product) and build the
    rank's row block of A (values r_inv[row] * a) and of A^T (values r_inv[col] * a: the counts are
    symmetric, so row j of A^T has the pattern of row j of A), columns remapped to the gathered layout."""
    from . import _lib
    from .graph import Graph, _stream_ptr

    dev = lcol.device
    r0, r1 = bounds[rank], bounds[rank + 1]
    r_inv = 1.0 / rowsum_global
    r_inv[torch.isinf(r_inv)] = 0.0
    val_f = (r_inv[r0:r1][rows] * a).to(torch.float32)
    val_b = (r_inv[lcol] * a).to(torch.float32)
    bt = torch.tensor(bounds, dtype=torch.int64, device=dev)
    part = torch.searchsorted(bt, lcol, right=True) - 1
    gcol = (part * pad + (lcol - bt[part])).contiguous()
    lib = _lib.load()

    def make(vals, name):
        out = ctypes.c_void_p()
        v = vals.contiguous()
        crow = lrp.contiguous()
        with torch.cuda.device(dev):
            st = lib.gcnb_graph_from_csr(r1 - r0, world * pad, v.numel(), crow.data_ptr(), gcol.data_ptr(), v.data_ptr(),
                                         _stream_ptr(dev), ctypes.byref(out))
        _lib.check(st, "gcnb_graph_from_csr")
        return Graph(out.value, dev, name)

    fwd = make(val_f, "rows[%d] (partitioned build)" % rank)
    bwd = make(val_b, "rows[%d]^T (partitioned build)" % rank)
    return DistGraph(rank, world, bounds, pad, None, fwd, None, bwd, fwd.nnz, n_global_nnz, False)


def build_partitioned(src, dst, n, rank, world, bounds=None, group=None, row_weight=0.0):
    """This rank's DistGraph from a (replicated) edge list WITHOUT building the whole adjacency on any GPU:
    what a papers100M-sized graph needs (3.2 G stored entries exceed one int32 handle, SURVEY.md 7).
    Bit-identical to cutting the block out of the single-GPU `Graph.from_edges` result.  Collective:
    one all-gather of the fp64 row sums (8 B per node) and one all-reduce of the entry counts."""
    dev = src.device
    if bounds is None:  # balance stored entries with the incident-edge count as the estimate
        deg = torch.bincount(src.long(), minlength=n) + torch.bincount(dst.long(), minlength=n) + 1
        rp = torch.cat([torch.zeros(1, dtype=torch.int64, device=dev), deg.cumsum(0)])
        bounds = partition_rows_by_nnz(rp, world, row_weight)
    pad = DistGraph.padded_rows(bounds)
    lrp, lcol, a, rows, rowsum = _partition_counts(src, dst, n, bounds[rank], bounds[rank + 1])
    slot = torch.ones(pad, dtype=torch.float64, device=dev)
    slot[: rowsum.numel()] = rowsum
    gathered = torch.empty(world * pad, dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_gather_into_tensor(gathered, slot, group=group)
    else:
        gathered.copy_(slot)
    rowsum_global = torch.cat([gathered[q * pad: q * pad + bounds[q + 1] - bounds[q]] for q in range(world)])
    nnz = torch.tensor([a.numel()], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(nnz, group=group)
    return _partition_blocks(rank, world, bounds, pad, lrp, lcol, a, rows, rowsum_global, int(nnz.item()))


# ---------------------------------------------------------------------------- arithmetic backends
class CudaOps:
    """The product backend: every call is a kernel of libgcnb200.so on the current stream."""

    def __init__(self, precision="auto"):
        from . import _lib
        from . import functional as F_

        self._lib = _lib
        self.lib = _lib.load()
        self.F = F_
        self.precision = F_._PRECISIONS[precision]

    def _sp(self, dev):
        return ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)

    def gemm(self, a, b, out=None):
        """a [m,k] @ b [k,n] (any strides); written to the first m rows of `out` when given."""
        m, k = a.shape
        n = b.shape[1]
        if out is None:
            out = torch.empty((m, n), dtype=torch.float32, device=a.device)
        with torch.cuda.device(a.device):
            ws = self.F._ws(self.lib.gcnb_gemm_workspace_bytes(m, n, k, self.precision), a.device)
            st = self.lib.gcnb_gemm(m, n, k, a.data_ptr(), a.stride(0), a.stride(1), b.data_ptr(), b.stride(0),
                                    b.stride(1), out.data_ptr(), max(n, 1), self.precision, ws.data_ptr(), ws.numel(),
                                    self._sp(a.device))
        self._lib.check(st, "gcnb_gemm")
        return out

    def gemm_bias_act(self, a, b, bias=None, relu=False):
        """relu?(a @ b + bias): gcnb_gemm_ex (the epilogue rides in the TMA-fed tcgen05 kernel when that runs)."""
        m, k = a.shape
        n = b.shape[1]
        out = torch.empty((m, n), dtype=torch.float32, device=a.device)
        with torch.cuda.device(a.device):
            ws = self.F._ws(self.lib.gcnb_gemm_workspace_bytes(m, n, k, self.precision), a.device)
            st = self.lib.gcnb_gemm_ex(m, n, k, a.data_ptr(), a.stride(0), a.stride(1), b.data_ptr(), b.stride(0),
                                       b.stride(1), out.data_ptr(), max(n, 1), bias.data_ptr() if bias is not None else None,
                                       1 if relu else 0, self.precision, ws.data_ptr(), ws.numel(), self._sp(a.device))
        self._lib.check(st, "gcnb_gemm_ex")
        return out

    def spmm_block(self, block, dense, out, accumulate, bias=None, relu=False):
        """out (+)= block @ dense (+ bias) (relu)."""
        f = dense.shape[1]
        flags = (self._lib.SPMM_ACCUMULATE if accumulate else 0) | (self._lib.SPMM_RELU if relu else 0)
        with torch.cuda.device(dense.device):
            ws = self.F._ws(self.lib.gcnb_spmm_workspace_bytes(block._h, 0, f), dense.device)
            st = self.lib.gcnb_spmm(block._h, flags, dense.data_ptr(), dense.stride(0) if dense.shape[0] > 1 else f, f,
                                    bias.data_ptr() if bias is not None else None, out.data_ptr(), out.stride(0)
                                    if out.shape[0] > 1 else f, ws.data_ptr(), ws.numel(), self._sp(dense.device))
        self._lib.check(st, "gcnb_spmm")
        return out

    def colsum(self, g, y=None, gm=None):
        """(column sums of g [masked by y > 0], the masked g).  When `gm` (>= n rows) is given the
        masked gradient -- or a plain copy of g -- is staged into its first n rows."""
        n, f = g.shape
        out = torch.empty((f,), dtype=torch.float32, device=g.device)
        if gm is None and y is not None:
            gm = torch.empty_like(g)
        with torch.cuda.device(g.device):
            ws = self.F._ws(self.lib.gcnb_colsum_workspace_bytes(n, f), g.device)
            st = self.lib.gcnb_colsum(n, f, g.data_ptr(), g.stride(0) if n > 1 else f,
                                      y.data_ptr() if y is not None else None, (y.stride(0) if n > 1 else f) if y is not None else f,
                                      gm.data_ptr() if gm is not None else None, f, out.data_ptr(), ws.data_ptr(),
                                      ws.numel(), self._sp(g.device))
        self._lib.check(st, "gcnb_colsum")
        return out, (gm if gm is not None else g)

    def empty(self, shape, like):
        return torch.empty(shape, dtype=torch.float32, device=like.device)

    # -- the halo exchange through the library's own C ABI (csrc/dist.cu): one pack kernel + one grouped ncclSend /
    # ncclRecv round on an NCCL communicator of ours, on a side stream so that the diagonal block's SpMM overlaps it
    _halo_group = None  # (process group kept alive, ncclComm_t as int): one per process, made on first use (collective)

    @classmethod
    def halo_comm(cls, device):
        if cls._halo_group is None:
            pg = dist.new_group(backend="nccl")          # its own communicator: never interleaves with torch's collectives
            t = torch.zeros(1, device=device)
            dist.all_reduce(t, group=pg)                  # NCCL communicators are created lazily: force it now
            torch.cuda.synchronize(device)
            cls._halo_group = (pg, int(pg._get_backend(torch.device(device))._comm_ptr()))
        return cls._halo_group[1]

    def halo_create(self, plan, dgraph, device):
        """gcnb_halo handle of a HaloPlan (rows to send grouped by destination rank, receive offsets into the compact
        panel) + the side stream the exchange runs on.  None when NCCL could not be bound."""
        if not self.lib.gcnb_halo_nccl_available():
            return None
        world, p = dgraph.world, dgraph.rank
        i64 = ctypes.c_int64 * world
        send = [int(plan.give[r].numel()) if r != p else 0 for r in range(world)]
        recv = [int(plan.need[q].numel()) if q != p else 0 for q in range(world)]
        offs = [int(plan.offset[q]) if q != p else 0 for q in range(world)]
        rows = [plan.give[r].to(torch.int32) for r in range(world) if r != p and plan.give[r].numel()]
        send_rows = torch.cat(rows).contiguous() if rows else torch.zeros(1, dtype=torch.int32, device=device)
        h = ctypes.c_void_p()
        with torch.cuda.device(device):
            st = self.lib.gcnb_halo_create(p, world, i64(*send), send_rows.data_ptr(), i64(*recv), i64(*offs),
                                           self._sp(device), ctypes.byref(h))
        self._lib.check(st, "gcnb_halo_create")
        import weakref

        weakref.finalize(plan, self.lib.gcnb_halo_free, h)
        # the side stream has HIGH priority: its pack-free exchange kernels (NCCL's send / recv CTAs) must get SM slots while
        # a SpMM grid of the main stream is resident, not after that grid has been dispatched to the end
        prio = -1 if os.environ.get("GCNB_DIST_SIDE_PRIORITY", "1") == "1" else 0
        return {"h": h, "comm": self.halo_comm(device), "stream": torch.cuda.Stream(device=device, priority=prio),
                "send_rows": sum(send)}

    def halo_exchange_async(self, c, panel, compact):
        """Pack on the current stream, exchange on the side stream; returns the event the consumer waits for."""
        dev = panel.device
        f = panel.shape[1]
        main = torch.cuda.current_stream(dev)
        sendbuf = torch.empty((max(c["send_rows"], 1), f), dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            st = self.lib.gcnb_halo_pack(c["h"], panel.data_ptr(), panel.stride(0) if panel.shape[0] > 1 else f, f,
                                         sendbuf.data_ptr(), self._sp(dev))
            self._lib.check(st, "gcnb_halo_pack")
            side = c["stream"]
            side.wait_stream(main)                        # the packed rows (and the compact panel's allocation) are ready
            sendbuf.record_stream(side)
            compact.record_stream(side)
            with torch.cuda.stream(side):
                st = self.lib.gcnb_halo_exchange(c["h"], ctypes.c_void_p(c["comm"]), sendbuf.data_ptr(), f, compact.data_ptr(),
                                                 ctypes.c_void_p(side.cuda_stream))
                self._lib.check(st, "gcnb_halo_exchange")
                done = torch.cuda.Event()
                done.record(side)
        return done

    # -- build-time helpers of the halo exchange (HaloPlan): blocks as CSR tensors and back
    def block_csr(self, block):
        rowptr, col, val = block.csr()
        return rowptr.long(), col.long(), val

    def block_from_csr(self, rowptr, col, val, n_rows, n_cols):
        from .graph import Graph

        adj = torch.sparse_csr_tensor(rowptr, col, val, size=(n_rows, n_cols), check_invariants=False)
        return Graph.from_torch(adj)

    def selection_block(self, ids, n_cols):
        """[len(ids), n_cols] with a single 1.0 per row: block @ dense packs the rows `ids` of dense (exact copies)."""
        k = ids.numel()
        rowptr = torch.arange(k + 1, dtype=torch.int64, device=ids.device)
        return self.block_from_csr(rowptr, ids.long(), torch.ones(k, dtype=torch.float32, device=ids.device), k, n_cols)


# ---------------------------------------------------------------------------- peer-memory exchange
class _DevMem:
    """A raw device allocation seen as a tensor through __cuda_array_interface__."""

    def __init__(self, ptr, shape, typestr="<f4"):
        self.__cuda_array_interface__ = {"data": (ptr, False), "shape": tuple(shape), "typestr": typestr, "version": 3,
                                         "strides": None}


class PeerExchangeUnavailable(RuntimeError):
    """CUDA IPC / peer access is not available between the ranks (raised on EVERY rank, after a collective
    agreement, so that all of them fall back to the NCCL exchange together)."""


class PeerExchange:
    """One panel exchange buffer: gathered [world * pad_rows, f] fp32 on every rank, written by the
    peers' push kernels over NVLink peer memory, plus flag / ack words per source rank (csrc/peer.cu).

    Protocol per exchange (all on device, CUDA-graph replayable):
      start(): epoch += 1 on the compute stream, then on the communication stream the push kernel
               copies this rank's slot to ranks p-1, p-2, ... and publishes flag[p] = epoch there;
      wait(q): the compute stream spins until slot q has landed;  done(q): acks it to rank q so q's next
               push may overwrite it;  finish(): joins the communication stream."""

    CTRL_BYTES = 1024
    PUSH_CTAS = 32
    # "ce": the slot is moved by the copy engines (cudaMemcpyAsync to the mapped peer pointer, 635 GB/s
    # per peer pair measured, no SMs taken from the SpMM) between our wait-for-ack and publish-flag
    # kernels; "sm": our push kernel stores it over NVLink itself (P2P stores, ~380-460 GB/s with 32-296
    # CTAs, tools/peer_bw.py).  GCNB_PEER_PUSH overrides.
    PUSH_MODE = os.environ.get("GCNB_PEER_PUSH", "ce")

    def __init__(self, rank, world, pad_rows, f, device, group=None):
        from . import _lib

        self._lib = _lib
        self.lib = _lib.load()
        self.rank, self.world, self.pad_rows, self.f = rank, world, pad_rows, f
        self.device = device
        if world - 1 > 15:
            raise RuntimeError("peer exchange supports at most 16 ranks")
        self.slot_bytes = pad_rows * f * 4
        data = (world * self.slot_bytes + 255) // 256 * 256
        self.off_flags, self.off_acks = data, data + 256
        self.off_epoch, self.off_counters = data + 512, data + 768
        self.bytes = data + self.CTRL_BYTES
        ok, why = 1, ""
        self.ptr, self.peer_ptr = None, {}
        with torch.cuda.device(device):
            ptr = ctypes.c_void_p()
            handle = ctypes.create_string_buffer(64)
            try:
                _lib.check(self.lib.gcnb_symm_alloc(self.bytes, ctypes.byref(ptr), handle), "gcnb_symm_alloc")
                self.ptr = ptr.value
            except Exception as e:  # no IPC in this environment: every rank must learn it (collectives below)
                ok, why = 0, repr(e)
            handles = [None] * world
            dist.all_gather_object(handles, handle.raw if ok else None, group=group)
            if ok and all(h is not None for h in handles):
                try:
                    for q in range(world):
                        if q == rank:
                            continue
                        pp = ctypes.c_void_p()
                        _lib.check(self.lib.gcnb_symm_open(ctypes.create_string_buffer(handles[q], 64), ctypes.byref(pp)),
                                   "gcnb_symm_open")
                        self.peer_ptr[q] = pp.value
                except Exception as e:
                    ok, why = 0, repr(e)
            else:
                ok = 0
            flag = torch.tensor([float(ok)], device=device)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=group)  # also: every rank has mapped every buffer
            if flag.item() < 1:
                self.close()
                raise PeerExchangeUnavailable("peer-memory exchange unavailable on at least one rank (%s)" % (why or "peer"))
        # push order: the rank that consumes our slot first (p-1) is served first
        order = [(rank - k) % world for k in range(1, world)]
        n = len(order)
        self._n_peers = n
        self._dst = (ctypes.c_void_p * max(n, 1))(*[self.peer_ptr[r] + rank * self.slot_bytes for r in order])
        self._flag = (ctypes.c_void_p * max(n, 1))(*[self.peer_ptr[r] + self.off_flags + 4 * rank for r in order])
        self._ack = (ctypes.c_void_p * max(n, 1))(*[self.ptr + self.off_acks + 4 * r for r in order])
        self.gathered = torch.as_tensor(_DevMem(self.ptr, (world * pad_rows, f)), device=device)
        self.my_slot = self.gathered[rank * pad_rows:(rank + 1) * pad_rows]
        self.comm = torch.cuda.Stream(device=device, priority=-1)
        self._ev = torch.cuda.Event()

    def _sp(self, stream=None):
        return ctypes.c_void_p((stream or torch.cuda.current_stream(self.device)).cuda_stream)

    def start(self):
        lib, ck = self.lib, self._lib.check
        with torch.cuda.device(self.device):
            ck(lib.gcnb_peer_epoch_bump(self.ptr + self.off_epoch, self.ptr + self.off_counters, self._n_peers, self._sp()),
               "gcnb_peer_epoch_bump")
            self._ev.record(torch.cuda.current_stream(self.device))
            self.comm.wait_event(self._ev)
            cs = self._sp(self.comm)
            if self.PUSH_MODE == "sm":
                ck(lib.gcnb_peer_push(self.ptr + self.rank * self.slot_bytes, self.slot_bytes, self._n_peers, self._dst,
                                      self._flag, self._ack, self.ptr + self.off_epoch, self.ptr + self.off_counters,
                                      self.PUSH_CTAS, cs), "gcnb_peer_push")
            else:
                ep = self.ptr + self.off_epoch
                for k in range(self._n_peers):
                    ck(lib.gcnb_peer_wait_lag(self._ack[k], ep, 1, cs), "gcnb_peer_wait_lag")  # peer done with the old slot
                    ck(lib.gcnb_peer_copy(self._dst[k], self.ptr + self.rank * self.slot_bytes, self.slot_bytes, cs),
                       "gcnb_peer_copy")
                    ck(lib.gcnb_peer_ack(self._flag[k], ep, cs), "gcnb_peer_ack")               # publish flag = epoch

    def wait(self, q):
        if q != self.rank:
            with torch.cuda.device(self.device):
                self._lib.check(self.lib.gcnb_peer_wait(self.ptr + self.off_flags + 4 * q, self.ptr + self.off_epoch,
                                                        self._sp()), "gcnb_peer_wait")

    def done(self, q):
        if q != self.rank:
            with torch.cuda.device(self.device):
                self._lib.check(self.lib.gcnb_peer_ack(self.peer_ptr[q] + self.off_acks + 4 * self.rank,
                                                       self.ptr + self.off_epoch, self._sp()), "gcnb_peer_ack")

    def finish(self):
        torch.cuda.current_stream(self.device).wait_stream(self.comm)

    def close(self):
        with torch.cuda.device(self.device):
            torch.cuda.synchronize(self.device)
            for p in getattr(self, "peer_ptr", {}).values():
                self.lib.gcnb_symm_close(p)
            self.peer_ptr = {}
            if getattr(self, "ptr", None):
                self.lib.gcnb_symm_free(self.ptr)
            self.ptr = None


class CollectiveExchange:
    """The same interface on top of one all-gather (gloo in the CPU tests of the host logic, or NCCL):
    start() gathers every slot at once, wait / done are no-ops."""

    def __init__(self, rank, world, pad_rows, f, like, group=None):
        self.rank, self.world, self.pad_rows, self.f, self.group = rank, world, pad_rows, f, group
        self.gathered = torch.zeros((world * pad_rows, f), dtype=torch.float32, device=like.device)
        self.my_slot = self.gathered[rank * pad_rows:(rank + 1) * pad_rows]

    def start(self):
        dist.all_gather_into_tensor(self.gathered, self.my_slot.clone(), group=self.group)

    def wait(self, q):
        pass

    def done(self, q):
        pass

    def finish(self):
        pass

    def close(self):
        pass


def dist_spmm_pipelined(ops, dgraph, blocks, exch, bias=None, relu=False):
    """out_p = sum_i blocks[i] @ gathered (+ bias) (relu) over the phases of dgraph.phases (groups of
    source ranks p, p+1, ...): this rank's slot is already in exch.my_slot; every other slot is consumed
    as soon as it has landed (exch.wait) and released to its owner right after (exch.done).  The bias /
    ReLU epilogue rides on the last block."""
    out = ops.empty((dgraph.n_rows(), exch.f), exch.gathered)
    exch.start()
    n = len(dgraph.phases)
    for i, qs in enumerate(dgraph.phases):
        last = i == n - 1
        for q in qs:
            exch.wait(q)
        ops.spmm_block(blocks[i], exch.gathered, out, i > 0, bias if last else None, relu and last)
        for q in qs:
            exch.done(q)
    exch.finish()
    return out


# ---------------------------------------------------------------------------- the exchange + layer
class HaloPlan:
    """Needed-rows-only ("halo") exchange for one direction of one DistGraph (opt-in, exchange "halo"; host logic
    covered by the gloo tests, composed of kernels that are measured -- the packing is an SpMM with a selection
    block -- but NOT yet run on GPUs as a whole).

    The all-gather ships every row of every slot; a rank only reads the rows that appear as a column in its block:
    95.6 % of them on a uniform graph, 35 % on a products-shaped R-MAT graph (tools/halo_fraction.py).  Built once
    (collective: the lists of needed rows are exchanged): need[q] = sorted local ids of source q's rows this rank
    reads; give[r] = ids of this rank's rows that rank r reads; pack[r] = selection block so that pack[r] @ panel is
    the send buffer for r; block = the rank's (remote or whole) row block with its columns renumbered to the compact
    panel [own slot (unsplit blocks only) | halo of source 0 | halo of source 1 | ...]."""

    def __init__(self, ops, dgraph, block, group=None):
        p, world, pad = dgraph.rank, dgraph.world, dgraph.pad_rows
        rowptr, col, val = ops.block_csr(block)
        src = torch.div(col, pad, rounding_mode="floor")
        loc = col - src * pad
        self.own = 0 if dgraph.split else pad  # a split row block keeps its own columns in the diagonal block
        self.need, self.offset = {}, {}
        new_col = torch.empty_like(col)
        mine = src == p
        new_col[mine] = loc[mine]
        off = self.own
        for q in range(world):
            if q == p:
                continue
            m = src == q
            ids = torch.unique(loc[m])  # sorted
            self.need[q], self.offset[q] = ids, off
            if ids.numel():
                new_col[m] = off + torch.searchsorted(ids, loc[m])
            off += ids.numel()
        self.n_compact = max(off, 1)
        lists = [None] * world
        dist.all_gather_object(lists, {q: v.cpu() for q, v in self.need.items()}, group=group)
        self.give = {r: lists[r][p].to(col.device) for r in range(world) if r != p}
        n_p = dgraph.n_rows()
        self.pack = {r: ops.selection_block(ids, max(pad, 1)) for r, ids in self.give.items() if ids.numel()}
        self.block = ops.block_from_csr(rowptr, new_col, val, n_p, self.n_compact)
        self.rows_received = off - self.own
        self.rows_all_gather = (world - 1) * pad
        # the product path: the library's own exchange (gcnb_halo_*, csrc/dist.cu) over an NCCL communicator of its own;
        # backends without it (the numpy backend of the CPU tests) use torch.distributed's grouped send / recv below
        self.c = ops.halo_create(self, dgraph, col.device) if hasattr(ops, "halo_create") and world > 1 else None


def halo_compact(ops, dgraph, transpose, f, like, exch, group=None):
    """The compact panel [own slot | halo rows] of an unsplit row block, allocated BEFORE the panel is produced: the
    producer (X W, the staged masked G, G W^T) writes its rows straight into the own slot `compact[:n_p]` and the
    exchange skips the copy (1.25 GB read + written per exchange at 2 GPUs and F = 256).  None when the exchange is
    not "halo", the row block is split (its compact panel has no own slot) or the width needs padding."""
    if exch != "halo" or dgraph.world == 1 or dgraph.split or f % 4 != 0:
        return None
    plan = halo_plans(ops, dgraph, group)[1 if transpose else 0]
    return ops.empty((plan.n_compact, f), like)


def _halo_start(ops, dgraph, plan, panel, compact, group=None):
    """Starts the exchange of one panel (this rank's rows `panel`, halo rows into `compact`) and returns the callable
    that makes the caller wait for the halo rows: a stream wait on the exchange's event (library path: pack kernel on
    the current stream, grouped ncclSend / ncclRecv on the side stream), or the completion of the grouped
    torch.distributed send / recv (backends without the library: the CPU tests)."""
    f = panel.shape[1]
    p, world = dgraph.rank, dgraph.world
    if getattr(plan, "c", None) is not None:
        done = ops.halo_exchange_async(plan.c, panel, compact)
        return lambda: torch.cuda.current_stream(panel.device).wait_event(done)
    sends, p2p = [], []
    for k in range(1, world):
        r = (p + k) % world
        if r in plan.pack:
            buf = ops.empty((plan.give[r].numel(), f), panel)
            ops.spmm_block(plan.pack[r], panel, buf, False)
            sends.append(buf)
            p2p.append(dist.P2POp(dist.isend, buf, r if group is None else dist.get_global_rank(group, r), group))
        q = (p - k) % world
        n_q = plan.need[q].numel()
        if n_q:
            p2p.append(dist.P2POp(dist.irecv, compact[plan.offset[q]: plan.offset[q] + n_q],
                                  q if group is None else dist.get_global_rank(group, q), group))
    reqs = dist.batch_isend_irecv(p2p) if p2p else []

    def finish(sends=sends):  # (the send buffers live until the requests are done)
        for rq in reqs:
            rq.wait()
    return finish


def dist_spmm_halo(ops, dgraph, plan, diag, panel, bias=None, relu=False, group=None, compact=None):
    """out_p with the needed-rows-only exchange: every peer r gets pack[r] @ panel (the rows of this rank it reads),
    this rank receives need[q] rows from every source q into the compact panel, then one SpMM over the renumbered
    block (after the diagonal block when the row block is split).  compact: the panel already IS compact[:n_p]
    (halo_compact)."""
    f = panel.shape[1]
    out = ops.empty((dgraph.n_rows(), f), panel)
    in_place = compact is not None
    if not in_place:
        compact = ops.empty((plan.n_compact, f), panel)
    finish = _halo_start(ops, dgraph, plan, panel, compact, group)
    if dgraph.split:
        ops.spmm_block(diag, panel, out, False)           # runs while the halo rows are on the wire
    elif not in_place:
        compact[: panel.shape[0]].copy_(panel)            # own slot at the front of the compact panel
    finish()
    return ops.spmm_block(plan.block, compact, out, dgraph.split, bias, relu)


# Column chunks of the exchanged panel (unsplit row blocks, halo exchange): chunk k + 1 is produced and packed while
# chunk k is on the wire, and chunk k is aggregated while chunk k + 1 is on the wire.  Only where a chunk is still a
# wide gather (>= 128 columns: the streaming SpMM at 512-byte rows costs what half a 1 KB-row launch costs; narrower
# chunks lose more in the SpMM than the overlap returns -- profiles/r02_rmat_probe_column_slices_old_kernels.txt).
CHUNK_MIN_COLS = int(os.environ.get("GCNB_DIST_CHUNK_MIN_COLS", "128"))
CHUNKS_MAX = int(os.environ.get("GCNB_DIST_CHUNKS", "2"))


def column_chunks(f):
    """[(c0, c1)] column ranges of the pipelined exchange: at most CHUNKS_MAX, each a multiple of 4 columns and at least
    CHUNK_MIN_COLS wide; one range = not pipelined."""
    k = max(1, min(CHUNKS_MAX, f // max(CHUNK_MIN_COLS, 4)))
    if k == 1 or f % 4 != 0:
        return [(0, f)]
    w = -(-(f // 4) // k) * 4
    return [(c, min(c + w, f)) for c in range(0, f, w)]


def chunked_halo_applies(ops, dgraph, f, exch):
    return exch == "halo" and dgraph.world > 1 and not dgraph.split and len(column_chunks(f)) > 1


def dist_spmm_halo_chunked(ops, dgraph, transpose, f, like, produce, bias=None, relu=False, group=None):
    """Rows p of A @ P (transpose: A^T @ P) where the rank's rows of P are PRODUCED chunk by chunk: produce(c0, c1, dst)
    writes columns [c0, c1) of this rank's rows into dst [n_p, c1 - c0] -- the own slot of that chunk's compact panel.
    Order on the current stream: produce 0, pack 0, produce 1, pack 1, ..., wait 0, SpMM 0, wait 1, SpMM 1, ...; the
    exchanges follow one another on the side stream."""
    plan = halo_plans(ops, dgraph, group)[1 if transpose else 0]
    n_p = dgraph.n_rows()
    out = ops.empty((n_p, f), like)
    pending = []
    for c0, c1 in column_chunks(f):
        compact = ops.empty((plan.n_compact, c1 - c0), like)
        own = compact[:n_p]
        produce(c0, c1, own)
        pending.append((c0, c1, compact, _halo_start(ops, dgraph, plan, own, compact, group)))
    for c0, c1, compact, finish in pending:
        finish()
        ops.spmm_block(plan.block, compact, out[:, c0:c1], False, bias[c0:c1] if bias is not None else None, relu)
    return out


def dist_spmm(ops, dgraph, diag, remote, panel, bias=None, relu=False, group=None):
    """out_p = diag @ panel[:n_p] + remote @ allgather(panel) (+ bias) (relu).

    `panel` is this rank's [pad_rows, F] slot (rows past n_p are padding nobody references).  The
    all-gather of the slots (NCCL over NVLink, on the communicator's stream) runs while the
    diagonal block is multiplied; the remote block is accumulated once the panel has landed."""
    world = dgraph.world
    out = ops.empty((dgraph.n_rows(), panel.shape[1]), panel)
    if world == 1:
        return ops.spmm_block(diag, panel, out, False, bias, relu)
    gathered = ops.empty((world * dgraph.pad_rows, panel.shape[1]), panel)
    if not dgraph.split:  # no locality to exploit: one pass over the whole row block
        dist.all_gather_into_tensor(gathered, panel, group=group)
        return ops.spmm_block(remote, gathered, out, False, bias, relu)
    work = dist.all_gather_into_tensor(gathered, panel, group=group, async_op=True)
    ops.spmm_block(diag, panel, out, False)
    work.wait()
    return ops.spmm_block(remote, gathered, out, True, bias, relu)


def halo_plans(ops, dgraph, group=None):
    """(forward, backward) HaloPlan of a DistGraph, built on first use (collective) and kept on the graph."""
    plans = getattr(dgraph, "_halo_plans", None)
    if plans is None:
        plans = (HaloPlan(ops, dgraph, dgraph.fwd_remote, group), HaloPlan(ops, dgraph, dgraph.bwd_remote, group))
        dgraph._halo_plans = plans
    return plans


def halo_fraction(ops, dgraph, group=None):
    """Largest share, over ranks and directions, of the all-gathered remote rows a rank actually reads (collective)."""
    frac = getattr(dgraph, "_halo_fraction", None)
    if frac is None:
        plans = halo_plans(ops, dgraph, group)
        mine = max(p.rows_received / max(p.rows_all_gather, 1) for p in plans)
        t = torch.tensor([mine], dtype=torch.float64, device=plans[0].block.device if hasattr(plans[0].block, "device") else "cpu")
        if dgraph.world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
        frac = dgraph._halo_fraction = float(t.item())
    return frac


def exchanged_spmm(ops, dgraph, transpose, panel, exch, bias=None, relu=False, group=None, compact=None):
    """Rows p of  A @ P  (transpose: A^T @ P) for the row-partitioned panel P whose rows of this rank are `panel`
    [n_p, F]: the exchange step of the layer.  exch: None / "nccl" = all-gather of the padded slots, "halo" = needed
    rows only, or a PeerExchange (pipelined per-source blocks over NVLink peer memory)."""
    diag, remote = (dgraph.bwd_diag, dgraph.bwd_remote) if transpose else (dgraph.fwd_diag, dgraph.fwd_remote)
    n_p, f = dgraph.n_rows(), panel.shape[1]
    if f % 4 != 0 and (exch is None or isinstance(exch, str)):
        # panel rows must be 16-byte aligned for the vector gathers (47 classes): exchange a zero-padded panel (the peer
        # exchange's slots are laid out by the exchange object itself)
        f4 = (f + 3) // 4 * 4
        wide = ops.empty((panel.shape[0], f4), panel)
        wide.zero_()
        wide[:, :f].copy_(panel)
        b4 = None
        if bias is not None:
            b4 = ops.empty((f4,), panel)
            b4.zero_()
            b4[:f].copy_(bias)
        return exchanged_spmm(ops, dgraph, transpose, wide, exch, b4, relu, group)[:, :f].contiguous()
    if dgraph.world == 1:
        out = ops.empty((n_p, f), panel)
        return ops.spmm_block(diag, panel, out, False, bias, relu)
    if exch == "halo":
        return dist_spmm_halo(ops, dgraph, halo_plans(ops, dgraph, group)[1 if transpose else 0], diag, panel, bias, relu, group,
                              compact)
    if exch is not None and exch != "nccl":  # PeerExchange: the panel goes into this rank's slot, blocks follow the phases
        exch.my_slot[:n_p].copy_(panel[:n_p])
        return dist_spmm_pipelined(ops, dgraph, dgraph.bwd_blocks if transpose else dgraph.fwd_blocks, exch, bias, relu)
    if panel.shape[0] != dgraph.pad_rows:  # the all-gather moves equal slots
        slot = ops.empty((dgraph.pad_rows, f), panel)
        slot[:n_p].copy_(panel[:n_p])
        panel = slot
    return dist_spmm(ops, dgraph, diag, remote, panel, bias, relu, group)


def aggregate_first(fin, fout, need_dx, need_dw=True):
    """The association order of functional._aggregate_first for the row-partitioned layer: (A X) W when its SpMMs --
    and here its EXCHANGES, one per SpMM -- move fewer panel columns than A (X W)'s."""
    cost_ref = fout * (2 if (need_dx or need_dw) else 1)
    cost_agg = fin * (2 if need_dx else 1)
    return fin % 4 == 0 and cost_agg < cost_ref


def dist_layer_forward(ops, dgraph, x, w, b, relu=False, group=None, exch=None, agg=False):
    """Row block of  A (X W) + b  (pygcn/layers.py:33-36) for this rank; agg: (A X) W + b, the exchanged panel is X.
    Returns (out, what backward needs beside it: A X for the aggregate-first order, else None)."""
    if agg:
        if chunked_halo_applies(ops, dgraph, x.shape[1], exch):
            ax = dist_spmm_halo_chunked(ops, dgraph, False, x.shape[1], x, lambda c0, c1, dst: dst.copy_(x[:, c0:c1]),
                                        None, False, group)
        else:
            ax = exchanged_spmm(ops, dgraph, False, x, exch, None, False, group)
        return ops.gemm_bias_act(ax, w, b, relu), ax
    if exch is not None and not isinstance(exch, str) and dgraph.world > 1:
        ops.gemm(x, w, out=exch.my_slot)             # X_p W straight into this rank's slot of the peer exchange
        return dist_spmm_pipelined(ops, dgraph, dgraph.fwd_blocks, exch, b, relu), None
    if chunked_halo_applies(ops, dgraph, w.shape[1], exch):   # X_p W[:, chunk] while the previous chunk is on the wire
        return dist_spmm_halo_chunked(ops, dgraph, False, w.shape[1], x, lambda c0, c1, dst: ops.gemm(x, w[:, c0:c1], out=dst),
                                      b, relu, group), None
    compact = halo_compact(ops, dgraph, False, w.shape[1], x, exch, group)
    if compact is not None:
        support = compact[: x.shape[0]]              # X_p W lands in the own slot of the compact panel
    else:
        support = ops.empty((dgraph.pad_rows if exch != "halo" else x.shape[0], w.shape[1]), x)
    ops.gemm(x, w, out=support)
    return exchanged_spmm(ops, dgraph, False, support, exch, b, relu, group, compact), None


def dist_layer_backward(ops, dgraph, x, w, g, y=None, need_dx=True, has_bias=True, group=None, exch=None, agg=False, ax=None,
                        reduce=True):
    """(dX rows of this rank or None, dW, db): dW/db are summed over ranks when `reduce` (one all-reduce)."""
    fin, fout = w.shape
    if not agg and chunked_halo_applies(ops, dgraph, fout, exch):
        # the masked gradient staged chunk by chunk into the compact panels (its column sums = that chunk of db)
        dbs = []
        ds = dist_spmm_halo_chunked(
            ops, dgraph, True, fout, g,
            lambda c0, c1, dst: dbs.append(ops.colsum(g[:, c0:c1], y[:, c0:c1] if y is not None else None, dst)[0]),
            None, False, group)
        return _finish_backward(ops, dgraph, x, w, torch.cat(dbs), None, ds, need_dx, has_bias, group, exch, False, None, reduce)
    compact = None if agg else halo_compact(ops, dgraph, True, fout, g, exch, group)
    # local part of db; G masked by [y > 0] when the ReLU is fused (staged into the compact panel's own slot when the
    # exchange takes it from there)
    db, gm = ops.colsum(g, y, compact[: g.shape[0]] if compact is not None else None)
    if agg:
        dw = ops.gemm(ax.t(), gm)                    # (A X)_p^T G_p: no exchange at all for dW
        ds = None
    else:
        ds = exchanged_spmm(ops, dgraph, True, gm, exch, None, False, group, compact)   # rows p of A^T G
    return _finish_backward(ops, dgraph, x, w, db, gm, ds, need_dx, has_bias, group, exch, agg, dw if agg else None, reduce)


def _finish_backward(ops, dgraph, x, w, db, gm, ds, need_dx, has_bias, group, exch, agg, dw, reduce):
    """dW (reference order: X_p^T dS_p), the all-reduce of dW / db, dX."""
    fin, fout = w.shape
    if not agg:
        dw = ops.gemm(x.t(), ds)                     # local part of X^T dS
    if dgraph.world > 1 and reduce:
        flat = torch.cat([dw.reshape(-1), db.reshape(-1)])
        dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
        dw = flat[: fin * fout].reshape(fin, fout)
        db = flat[fin * fout:]
    dx = None
    if need_dx and agg and chunked_halo_applies(ops, dgraph, fin, exch):
        dx = dist_spmm_halo_chunked(ops, dgraph, True, fin, gm, lambda c0, c1, dst: ops.gemm(gm, w[c0:c1].t(), out=dst),
                                    None, False, group)
    elif need_dx and agg:
        compact = halo_compact(ops, dgraph, True, fin, gm, exch, group)
        gw = ops.gemm(gm, w.t(), out=compact[: gm.shape[0]] if compact is not None else None)
        dx = exchanged_spmm(ops, dgraph, True, gw, exch, None, False, group, compact)
    elif need_dx:
        dx = ops.gemm(ds, w.t())
    return dx, dw, (db if has_bias else None)


class _DistGCNLayerFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight, bias, dgraph, relu, ops, group, exch_f=None, exch_b=None, association="auto"):
        fin, fout = weight.shape
        agg = association == "aggregate_first" or (
            association == "auto" and aggregate_first(fin, fout, ctx.needs_input_grad[0], ctx.needs_input_grad[1]))
        out, ax = dist_layer_forward(ops, dgraph, x, weight, bias, relu, group, exch_f, agg)
        ctx.dgraph, ctx.relu, ctx.ops, ctx.group, ctx.exch_b, ctx.agg = dgraph, relu, ops, group, exch_b, agg
        ctx.has_bias = bias is not None
        ctx.save_for_backward(ax if agg else x, weight, out if relu else None)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        x, w, y = ctx.saved_tensors
        dx, dw, db = dist_layer_backward(ctx.ops, ctx.dgraph, None if ctx.agg else x, w, g.contiguous(), y,
                                         ctx.needs_input_grad[0], ctx.has_bias, ctx.group, ctx.exch_b, ctx.agg,
                                         x if ctx.agg else None)
        return dx, dw, db, None, None, None, None, None, None, None


class DistGraphConvolution(torch.nn.Module):
    """`GraphConvolution` over a row-partitioned graph: forward(x_local, dist_graph) -> out_local.
    Parameters are replicated (same seed on every rank = same init as the reference layer);
    `.grad` of weight/bias comes out already all-reduced.

    exchange: "nccl"  all-gather of the padded panel slots, overlapped with the diagonal block when the row block is split;
              "halo"  only the rows a rank reads travel (HaloPlan): on a power-law graph a third of them;
              "peer"  own push kernel over NVLink peer memory, per-source blocks consumed as they land (2 GPUs);
              "auto"  halo when a rank reads less than HALO_MAX_FRACTION of the remote rows, else nccl."""

    HALO_MAX_FRACTION = 0.7

    def __init__(self, in_features, out_features, bias=True, *, fuse_relu=False, precision="auto", group=None,
                 exchange="auto", association="auto"):
        super().__init__()
        from .layers import GraphConvolution

        if exchange not in ("auto", "peer", "nccl", "halo"):
            raise ValueError("exchange must be 'auto', 'peer', 'nccl' or 'halo'")
        if precision == "bf16":
            raise ValueError("the row-partitioned layer has no bf16 panel tier (single-GPU GraphConvolution only)")
        self.inner = GraphConvolution(in_features, out_features, bias, fuse_relu=fuse_relu, precision=precision)
        self.group = group
        self.exchange = exchange
        self.association = association
        self._ops = None
        self._exch = None  # (dgraph id, forward exchange, backward exchange): per layer, so that a slot is
        #                    never overwritten by another layer's panel while a peer still reads it

    def resolve_exchange(self, dgraph):
        if self.exchange != "auto" or dgraph.world == 1:
            return self.exchange if self.exchange != "auto" else "nccl"
        return "halo" if halo_fraction(self._ops, dgraph, self.group) < self.HALO_MAX_FRACTION else "nccl"

    def _exchanges(self, dgraph, dev):
        kind = self.resolve_exchange(dgraph)
        if dgraph.world == 1 or kind in ("nccl", "halo"):
            return kind, kind
        if dgraph.fwd_blocks is None:
            raise RuntimeError("exchange='peer' needs a DistGraph cut per source rank (DistGraph.from_graph(per_source=True))")
        if self._exch is None or self._exch[0] is not dgraph:
            if self._exch is not None:
                self._exch[1].close()
                self._exch[2].close()
                self._exch = None
            f = self.inner.out_features
            try:
                ef = PeerExchange(dgraph.rank, dgraph.world, dgraph.pad_rows, f, dev, self.group)
                try:
                    eb = PeerExchange(dgraph.rank, dgraph.world, dgraph.pad_rows, f, dev, self.group)
                except PeerExchangeUnavailable:
                    ef.close()
                    raise
            except PeerExchangeUnavailable as e:  # agreed on by all ranks: use the NCCL exchange from now on
                sys.stderr.write("pygcn_b200.dist: %s; falling back to exchange='nccl'\n" % e)
                self.exchange = "nccl"
                return "nccl", "nccl"
            self._exch = (dgraph, ef, eb)
        return self._exch[1], self._exch[2]

    @property
    def weight(self):
        return self.inner.weight

    @property
    def bias(self):
        return self.inner.bias

    def forward(self, input, dgraph):
        if self._ops is None:
            self._ops = CudaOps(self.inner.precision)
        if not input.is_cuda:
            raise RuntimeError("DistGraphConvolution runs on CUDA devices only (no CPU fallback)")
        if input.dtype != torch.float32 or self.inner.weight.dtype != torch.float32:
            raise RuntimeError("DistGraphConvolution computes in float32 only (got input %s, weight %s); the fp64 layer is "
                               "the single-GPU GraphConvolution" % (input.dtype, self.inner.weight.dtype))
        ef, eb = self._exchanges(dgraph, input.device)
        assoc = self.association if isinstance(ef, str) else "reference"  # the peer exchange's slots are Fout wide
        return _DistGCNLayerFn.apply(input.contiguous(), self.inner.weight, self.inner.bias, dgraph,
                                     self.inner.fuse_relu, self._ops, self.group, ef, eb, assoc)


# ---------------------------------------------------------------------------- bench entry (N > 1)
def bench_main(args, wl):
    """`bench.py --gpus N` under torchrun: the workload's graph row-partitioned over N GPUs (fixed total size: strong
    scaling), the workload's whole model per step.  One JSON line on rank 0, with a parity gate against the
    single-GPU layer and an fp64 run of the reference's lines (graphs that fit one GPU)."""
    import bench as B
    import pygcn_b200 as P
    from . import _lib

    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local_rank = int(os.environ.get("LOCAL_RANK", rank))
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()
    _lib.check(lib.gcnb_check_device(), "gcnb_check_device")
    sampler = B.ClockSampler(local_rank) if rank == 0 else None
    timer = B.Timer(torch, lib, _lib, dev)
    dims, relu = wl["dims"], wl["relu"]
    layers_n = len(dims) - 1
    partitioned = bool(wl.get("partitioned"))
    exchange = os.environ.get("GCNB_DIST_EXCHANGE", "auto")
    # cost of a row against a stored entry when cutting the row blocks: the dense products and element-wise passes
    # scale with rows, the SpMMs with entries (products-shaped 3-layer step on one GPU: ~0.33 ns per entry, ~4 ns per row)
    row_weight = float(os.environ.get("GCNB_DIST_ROW_WEIGHT", "12" if layers_n > 1 else "0"))
    balance = os.environ.get("GCNB_DIST_BALANCE", "1") == "1"  # balanced_node_partition instead of contiguous row blocks
    split_env = os.environ.get("GCNB_DIST_SPLIT", "auto")
    split = None if split_env == "auto" else split_env == "1"

    t0 = time.perf_counter()
    full = None
    if partitioned:
        # the whole adjacency never exists on one GPU: every rank builds its row block of A and A^T from the
        # replicated edge list (drawn on the device: 752 M edges)
        n_global = wl["n"]
        gen = torch.Generator(device=dev).manual_seed(0)
        src = torch.randint(0, n_global, (wl["n_raw"],), generator=gen, device=dev, dtype=torch.int32)
        dst = torch.randint(0, n_global, (wl["n_raw"],), generator=gen, device=dev, dtype=torch.int32)
        dgraph = build_partitioned(src, dst, n_global, rank, world, row_weight=row_weight)
        nnz_global = dgraph.nnz_global
        del src, dst
        torch.cuda.empty_cache()
        if exchange == "auto":
            exchange = "nccl"  # uniform graph: a rank reads ~96 % of every slot (tools/halo_fraction.py)
    else:
        src, dst, n_global = B.make_edges(torch, wl, 0)      # CPU generator, same seed on every rank: the single-GPU arm's graph
        src, dst = src.to(dev), dst.to(dev)
        full = P.Graph.from_edges(src, dst, n_global)        # kept for the parity gate (the single-GPU layer on this GPU)
        nnz_global = full.nnz
        if split is None and exchange in ("auto", "halo"):
            split = False  # one pass over [own rows | halo rows] (profiles/r02_dist_tune_n2.txt: 33.2 vs 33.4 ms split)
        if balance:
            # nodes dealt to the ranks by row length: every rank owns N / P rows and ~nnz / P stored entries; the graph
            # is rebuilt with the nodes renumbered rank by rank (same entries, same values), rank p owns new rows
            # bounds[p] .. bounds[p + 1] = the original nodes `mine`
            rp = full.csr()[0].long()
            new_id, bounds = balanced_node_partition(rp[1:] - rp[:-1], world)
            relabelled = P.Graph.from_edges(new_id[src.long()].int(), new_id[dst.long()].int(), n_global)
            dgraph = DistGraph.from_graph(relabelled, rank, world, bounds=bounds, split=split)
            mine = torch.argsort(new_id)[bounds[rank]:bounds[rank + 1]].cpu()  # original ids of this rank's rows, in row order
            del relabelled, rp
        else:
            dgraph = DistGraph.from_graph(full, rank, world, split=split, row_weight=row_weight)
            mine = torch.arange(dgraph.bounds[rank], dgraph.bounds[rank + 1])
        del src, dst
    torch.cuda.synchronize()
    build_s = time.perf_counter() - t0
    r0, r1 = dgraph.bounds[rank], dgraph.bounds[rank + 1]
    n_local = r1 - r0

    params = B.init_params(torch, dims)
    layers = torch.nn.ModuleList([DistGraphConvolution(a, b, fuse_relu=relu, exchange=exchange) for a, b in zip(dims[:-1], dims[1:])])
    with torch.no_grad():
        for l, (w, b) in zip(layers, params):
            l.inner.weight.copy_(w)
            l.inner.bias.copy_(b)
    layers = layers.to(dev)
    gen = torch.Generator(device="cpu")
    if partitioned:  # 57 GB of features: every rank draws its own rows
        x_host = torch.randn(n_local, dims[0], generator=gen.manual_seed(1 + rank)).pin_memory()
        g_host = torch.randn(n_local, dims[-1], generator=gen.manual_seed(100 + rank)).pin_memory()
        x_full = g_full = None
    else:            # the single-GPU arm's X and G, this rank's rows
        x_full = torch.randn(n_global, dims[0], generator=gen.manual_seed(1))
        g_full = torch.randn(n_global, dims[-1], generator=gen.manual_seed(2))
        x_host, g_host = x_full[mine].clone().pin_memory(), g_full[mine].clone().pin_memory()
    x, g = x_host.to(dev), g_host.to(dev)

    def run(xx, gg):
        for l in layers:
            l.inner.weight.grad = None
            l.inner.bias.grad = None
        h = xx
        for l in layers:
            h = l(h, dgraph)
        h.backward(gg)
        return h

    def step_eager():
        return run(x, g)

    if sampler:
        sampler.start()
    warm = max(args.warmup, 3)
    for _ in range(warm):
        step_eager()
    torch.cuda.synchronize()
    dist.barrier()
    c0 = lib.gcnb_launch_count()
    step_eager()
    launches_per_step = int(lib.gcnb_launch_count() - c0)
    resolved = [l.resolve_exchange(dgraph) for l in layers]

    # capture the step (kernels + NCCL sends / receives / all-reduces) in a CUDA graph: removes the Python and launch
    # gaps from the device time, like the single-GPU arm.  All ranks must agree.
    cg = None
    if not args.no_cuda_graph and not partitioned and os.environ.get("GCNB_DIST_CUDA_GRAPH", "1") == "1":
        ok = torch.ones(1, device=dev)
        try:
            s_ = torch.cuda.Stream()
            s_.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s_):
                for _ in range(2):
                    step_eager()
            torch.cuda.current_stream().wait_stream(s_)
            torch.cuda.synchronize()
            cg = torch.cuda.CUDAGraph()
            with torch.cuda.graph(cg):
                step_eager()
            torch.cuda.synchronize()
        except Exception as e:  # pragma: no cover
            sys.stderr.write("rank %d: CUDA graph capture failed (%r); timing eager launches\n" % (rank, e))
            cg = None
            ok.zero_()
            torch.cuda.synchronize()
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if ok.item() == 0:
            cg = None
    step = cg.replay if cg is not None else step_eager
    for _ in range(warm):
        timer.flush()
        step()
    torch.cuda.synchronize()
    dist.barrier()
    torch.cuda.synchronize()

    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    if sampler:
        sampler.in_region = True
    for i in range(args.steps):
        timer.flush()
        ev[i][0].record()
        step()
        ev[i][1].record()
    torch.cuda.synchronize()
    dist.barrier()
    torch.cuda.synchronize()
    if sampler:
        sampler.in_region = False
    total_ms = torch.tensor([sum(a.elapsed_time(b) for a, b in ev)], device=dev, dtype=torch.float64)
    mine_ms = total_ms.clone()
    dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
    ms_per_step = total_ms.item() / args.steps
    value = layers_n * nnz_global / (ms_per_step * 1e-3)
    per_rank = [torch.zeros_like(mine_ms) for _ in range(world)]
    dist.all_gather(per_rank, mine_ms)

    # ---- end to end from pinned host buffers, the single-GPU arm's method at every N: step i+1's H2D copies run on a
    # copy stream while step i computes; every step copies its own X and G rows in and reads every dW / db back
    copy_stream = torch.cuda.Stream()
    bufs = [(torch.empty_like(x), torch.empty_like(g)) for _ in range(2)]
    ready = [torch.cuda.Event() for _ in range(2)]
    done = [torch.cuda.Event() for _ in range(2)]

    def prefetch(i):
        b = i % 2
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(done[b])
            bufs[b][0].copy_(x_host, non_blocking=True)
            bufs[b][1].copy_(g_host, non_blocking=True)
            ready[b].record(copy_stream)

    def e2e_loop(k):
        for b in range(2):
            done[b].record()
        torch.cuda.synchronize()
        dist.barrier()
        t0 = time.perf_counter()
        prefetch(0)
        for i in range(k):
            if i + 1 < k:
                prefetch(i + 1)
            b = i % 2
            torch.cuda.current_stream().wait_event(ready[b])
            run(bufs[b][0], bufs[b][1])
            done[b].record()
            [(l.inner.weight.grad.cpu(), l.inner.bias.grad.cpu()) for l in layers]
        torch.cuda.synchronize()
        return time.perf_counter() - t0

    quick = bool(getattr(args, "quick", False))
    if not quick:
        e2e_loop(2)
    e2e_t = torch.tensor([e2e_loop(args.steps) if not quick else float("nan")], device=dev, dtype=torch.float64)
    dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
    e2e_value = layers_n * nnz_global / (e2e_t.item() / args.steps)
    del bufs
    if sampler:
        sampler.stop()

    # ---- parity gate: this rank's rows of the output and the all-reduced gradients against (a) the single-GPU layer
    # of this package on the whole graph and (b) an fp64 run of the reference's lines, both on this GPU.  Rule as in
    # the single-GPU arm (SURVEY.md 8d): error against fp64 <= max(1e-5, 2 x the single-GPU step's error against fp64).
    parity = None
    if not partitioned and not quick:
        try:
            o_d = step_eager().detach().clone()
            g_d = [(l.inner.weight.grad.clone(), l.inner.bias.grad.clone()) for l in layers]
            single = B.build_stack(P, torch, dims, relu, params, dev)
            xf, gf = x_full.to(dev), g_full.to(dev)
            o_s = B.stack_step(single, xf, full, gf).detach()
            g_s = [(l.weight.grad.clone(), l.bias.grad.clone()) for l in single]
            o64, g64, _ = B.torch_reference_lines(torch, full, params, relu, xf, gf, "csr", 1, dtype=torch.float64)

            def nerr(a, b):
                return ((a - b).abs().max() / b.abs().max().clamp_min(1e-30)).item()
            rows_ = mine.to(dev)
            errs = {"dist_vs_fp64": {"out": nerr(o_d.double(), o64[rows_])}, "single_gpu_vs_fp64": {"out": nerr(o_s[rows_].double(), o64[rows_])},
                    "dist_vs_single_gpu": {"out": nerr(o_d, o_s[rows_])}}
            for i, ((dw, db), (sw, sb), (w64, b64)) in enumerate(zip(g_d, g_s, g64), 1):
                for nm, a_, s__, d_ in (("dW%d" % i, dw, sw, w64), ("db%d" % i, db, sb, b64)):
                    errs["dist_vs_fp64"][nm] = nerr(a_.double(), d_)
                    errs["single_gpu_vs_fp64"][nm] = nerr(s__.double(), d_)
                    errs["dist_vs_single_gpu"][nm] = nerr(a_, s__)
            okv = torch.tensor([1.0 if errs["dist_vs_fp64"]["out"] <= 1e-5 and all(
                v <= max(1e-5, 2 * errs["single_gpu_vs_fp64"][k]) for k, v in errs["dist_vs_fp64"].items()) else 0.0], device=dev)
            worst = torch.tensor([max(errs["dist_vs_fp64"].values())], device=dev, dtype=torch.float64)
            dist.all_reduce(okv, op=dist.ReduceOp.MIN)
            dist.all_reduce(worst, op=dist.ReduceOp.MAX)
            parity = {"ok": bool(okv.item() == 1.0), "tolerance": 1e-5, "worst_dist_vs_fp64_over_ranks": worst.item(),
                      "rule": "dist_vs_fp64 <= max(1e-5, 2 * single_gpu_vs_fp64) on every rank, norm-wise max|a-b| / max|b|",
                      "rank0": errs}
            del single, xf, gf, o_s, g_s, o64, g64, o_d, g_d
        except Exception as e:  # pragma: no cover
            parity = {"ok": False, "error": repr(e)}
        torch.cuda.empty_cache()

    if partitioned and not quick:
        # no GPU holds the whole graph: the gate is what a row-normalised adjacency must satisfy at any size -- every row
        # of A sums to one, through the real exchange (a panel of ones) and the real row block
        try:
            ones = torch.ones(n_local, 4, device=dev)
            rs = exchanged_spmm(CudaOps(), dgraph, False, ones, "nccl")
            dev_max = torch.tensor([(rs - 1).abs().max().item()], device=dev, dtype=torch.float64)
            dist.all_reduce(dev_max, op=dist.ReduceOp.MAX)
            parity = {"ok": bool(dev_max.item() < 1e-5), "what": "max |rowsum(A) - 1| over all ranks through the exchanged SpMM",
                      "row_sums_max_deviation": dev_max.item(), "tolerance": 1e-5}
            del ones, rs
        except Exception as e:  # pragma: no cover
            parity = {"ok": False, "error": repr(e)}
        torch.cuda.empty_cache()

    # ---- the exchange alone and the dominant SpMM alone on this rank, at the widest panel of the model
    fw = max(f for (_, f, _, _) in B.spmm_plan(dims))
    ops = CudaOps()
    panel = torch.randn(n_local if resolved[0] == "halo" else dgraph.pad_rows, fw, device=dev)
    kind = "halo" if "halo" in resolved else "nccl"

    chunked = chunked_halo_applies(ops, dgraph, fw, kind)

    def exchange_and_spmm():  # as the layer runs it: in column chunks where that applies (the producer here is a copy)
        if chunked:
            dist_spmm_halo_chunked(ops, dgraph, False, fw, panel, lambda c0, c1, dst: dst.copy_(panel[:, c0:c1]))
        else:
            exchanged_spmm(ops, dgraph, False, panel, kind)
    ex_ms = timer.time(exchange_and_spmm, max(3, min(args.steps, 10)))[0]
    blk = dgraph.fwd_remote if kind == "nccl" else halo_plans(ops, dgraph)[0].block
    dense = torch.randn(blk.n_cols, fw, device=dev)
    outb = torch.empty(n_local, fw, device=dev)
    sp_ms = timer.time(lambda: ops.spmm_block(blk, dense, outb, False), max(3, min(args.steps, 10)))[0]
    t2 = torch.tensor([ex_ms, sp_ms], device=dev, dtype=torch.float64)
    dist.all_reduce(t2, op=dist.ReduceOp.MAX)
    halo = None
    if kind == "halo":
        pl = halo_plans(ops, dgraph)
        rows = torch.tensor([pl[0].rows_received, pl[0].rows_all_gather, n_local, dgraph.fwd_diag.nnz if dgraph.split else 0,
                             pl[0].block.nnz], device=dev, dtype=torch.float64)
        allrows = [torch.zeros_like(rows) for _ in range(world)]
        dist.all_gather(allrows, rows)
        halo = {"rows_received_per_rank": [int(r[0].item()) for r in allrows], "rows_an_all_gather_would_move": int(allrows[0][1].item()),
                "rows_owned_per_rank": [int(r[2].item()) for r in allrows],
                "stored_entries_diag_block": [int(r[3].item()) for r in allrows], "stored_entries_halo_block": [int(r[4].item()) for r in allrows]}
    peak, peak_src = B.peaks()
    alg = B.algorithmic_bytes_spmm(blk.nnz, n_local, fw)
    if rank == 0:
        cfg = B.config_of(wl, nnz_global, n_global)  # the same object as the reference arm's, key for key
        run = {}
        run.update({"partition": ("1-D partition of the nodes, dealt by row length: equal rows and ~equal stored entries per rank "
                                  "(dist.balanced_node_partition)" if (balance and not partitioned) else
                                  "1-D contiguous row blocks, cost = stored entries + %g x rows" % row_weight),
                    "bounds": dgraph.bounds,
                    "row_block_split": dgraph.split, "exchange": resolved, "cuda_graph": cg is not None,
                    "graph_build_s": build_s,
                    "association": [o for (_, _, _, o) in B.spmm_plan(dims)], "halo": halo,
                    "exchange_note": "halo: every rank sends each peer only the panel rows that peer's block reads (selection SpMM "
                                     "packs them, grouped NCCL send / recv into a compact panel) while the diagonal block's SpMM "
                                     "runs; nccl: all-gather of the padded slots; dW / db: one NCCL all-reduce per layer"})
        line = {
            "metric": B.METRIC, "value": value, "unit": "edges/s", "n_gpus": world,
            "steps": args.steps, "warmup": warm, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": cfg,
            "run": run,
            "clocks": sampler.summary(),
            "e2e": {"value": e2e_value, "unit": "edges/s", "h2d_bytes_per_step": (x_host.numel() + g_host.numel()) * 4,
                    "d2h_bytes_per_step": sum(w.numel() + b.numel() for w, b in params) * 4,
                    "ms_per_step": e2e_t.item() / args.steps * 1e3,
                    "how": "wall clock over K steps through DistGraphConvolution (max over ranks); every step's X and G rows "
                           "copied from pinned host memory (double-buffered on a copy stream), every dW / db read back; bytes are rank 0's"},
            "parity": parity,
            "per_rank_ms_per_step": [t.item() / args.steps for t in per_rank],
            "gpu_launches": launches_per_step * args.steps, "gpu_launches_per_step": launches_per_step,
            "roofline": {"bound": "hbm", "achieved": alg / (t2[1].item() * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": alg / (t2[1].item() * 1e-3) / 1e9 / peak, "traffic": None,
                         "kernel": "CSR SpMM over rank 0's row block (width %d), slowest rank's time" % fw,
                         "algorithmic_bytes_per_launch": alg, "kernel_ms": t2[1].item(), "peak_source": peak_src,
                         "exchange_plus_spmm_ms": t2[0].item(), "exchange_column_chunks": column_chunks(fw) if chunked else None, "exchange_share": max(0.0, 1.0 - t2[1].item() / max(t2[0].item(), 1e-9))},
        }
        print(json.dumps(line), flush=True)
    # a captured graph that holds NCCL kernels must go before the communicator does
    del step, cg
    torch.cuda.synchronize()
    dist.barrier()
    torch.cuda.synchronize()
    dist.destroy_process_group()
    return 0

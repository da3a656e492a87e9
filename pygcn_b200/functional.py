"""autograd wrappers around the C ABI: the GCN layer and the `torch.spmm` drop-in.

Forward  : pygcn/layers.py:32-38   support = mm(input, W); out = spmm(adj, support) (+ bias)
Backward : the autograd graph of those lines (SURVEY.md 3.2), hand-written here:
           db = colsum(G); dS = adj^T G; dW = X^T dS; dX = dS W^T  (only what
           ctx.needs_input_grad asks for).
All arithmetic happens in libgcnb200.so on the current CUDA stream; nothing here falls back
to PyTorch ops.  fp64 operands on an fp64 adjacency (`model.double()`) run the library's fp64 tier
(the *_f64 entry points): same products, same epilogue, fp64 throughout.
"""
from __future__ import annotations

import ctypes

import torch
from torch.autograd.function import once_differentiable

from . import _lib
from .graph import Graph, _require_cuda, _stream_ptr, as_graph

# "bf16": bf16 panels for the SpMM (the 2e-2 tier); its dense products, and the layer on a dense-route or
# batched input, use the "auto" kernels
_PRECISIONS = {"fp32": _lib.GEMM_FP32, "tf32x3": _lib.GEMM_TF32X3, "auto": _lib.GEMM_AUTO, "bf16": _lib.GEMM_AUTO}


def _ld4(f):
    return (f + 3) // 4 * 4


def _ld2(f):
    return (f + 1) // 2 * 2


def _rowmajor(t, dtype=torch.float32):
    """2-D tensor of `dtype` with unit column stride (row stride may exceed the width:
    the fork passes column-slice views, pygcn/models.py:345)."""
    if t.dim() != 2:
        raise RuntimeError("expected a 2-D tensor, got %d-D" % t.dim())
    if t.dtype != dtype:
        raise RuntimeError("expected %s, got %s" % (str(dtype).replace("torch.", ""), t.dtype))
    if t.shape[1] > 1 and t.stride(1) != 1:
        t = t.contiguous()
    if t.shape[0] > 1 and t.stride(0) < t.shape[1]:
        t = t.contiguous()
    return t


def _ld(t):
    return t.stride(0) if t.shape[0] > 1 else max(t.shape[1], 1)


def _ws(nbytes, device):
    return torch.empty((max(int(nbytes), 256),), dtype=torch.uint8, device=device)


def _ptr(t):
    # ctypes converts a plain int for c_void_p parameters; None is NULL
    return t.data_ptr() if t is not None else None


class _on_device:
    """`with torch.cuda.device(dev)` only when dev is not already current (the common case costs nothing)."""

    __slots__ = ("ctx",)

    def __init__(self, dev):
        self.ctx = None if torch.cuda.current_device() == dev.index else torch.cuda.device(dev)

    def __enter__(self):
        if self.ctx is not None:
            self.ctx.__enter__()

    def __exit__(self, *exc):
        if self.ctx is not None:
            return self.ctx.__exit__(*exc)
        return False


def _layer_ws_bytes(lib, graph, fin, fout, precision):
    """gcnb_layer_workspace_bytes, cached on the graph handle (constant per shape)."""
    cache = graph.__dict__.setdefault("_ws_cache", {})
    key = (fin, fout, precision)
    v = cache.get(key)
    if v is None:
        v = cache[key] = int(lib.gcnb_layer_workspace_bytes(graph._h, fin, fout, precision))
    return v


_ASSOCIATIONS = ("auto", "reference", "aggregate_first")


def _aggregate_first(association, graph, xr, fin, fout, need_dx, need_dw, lane=4):
    """Which product comes first.  The reference computes adj @ (X @ W) (pygcn/layers.py:33-34); (adj @ X) @ W is the
    same function and the same gradients to fp32 rounding, and its SpMMs gather rows of width fin instead of fout:
    forward one SpMM either way; backward one SpMM of width fout in the reference order (dS = adj^T G, for dW and
    dX), in the aggregate-first order none for dW = (adj X)^T G and one of width fin for dX = adj^T (G W^T).
    "auto" picks the order whose SpMMs move fewer panel columns; ties keep the reference order."""
    if association == "reference" or graph.dense_route:
        return False
    # 16-byte gathers of X's rows: lane = elements per 16 bytes (4 fp32, 2 fp64)
    ok = xr.data_ptr() % 16 == 0 and _ld(xr) % lane == 0 and _ld(xr) >= (fin + lane - 1) // lane * lane
    if association == "aggregate_first":
        if not ok:
            raise RuntimeError("association='aggregate_first' needs 16-byte aligned input rows (stride a multiple of %d)"
                               % lane)
        return True
    cost_ref = fout * (2 if (need_dx or need_dw) else 1)
    cost_agg = fin * (2 if need_dx else 1)
    return ok and cost_agg < cost_ref


class _GCNLayerFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight, bias, graph, relu, precision, mask=None, mask_scale=1.0, association="auto"):
        lib = _lib.load()
        dev = x.device
        fin, fout = weight.shape
        xr = _rowmajor(x)
        w = weight.contiguous()
        b = bias.contiguous() if bias is not None else None
        agg = _aggregate_first(association, graph, xr, fin, fout, ctx.needs_input_grad[0], ctx.needs_input_grad[1])
        if agg:  # A X, kept for dW = (A X)^T G
            support = torch.empty((graph.n_rows, _ld4(fin)), dtype=torch.float32, device=dev)
        else:
            support = torch.empty((graph.n_cols, _ld4(fout)), dtype=torch.float32, device=dev)
        out = torch.empty((graph.n_rows, fout), dtype=torch.float32, device=dev)
        flags = (_lib.LAYER_RELU if relu else 0) | (_lib.LAYER_AGG_FIRST if agg else 0)
        with _on_device(dev):
            ws = _ws(_layer_ws_bytes(lib, graph, fin, fout, precision), dev)
            st = lib.gcnb_layer_forward(
                graph._h, _ptr(xr), _ld(xr), _ptr(w), _ptr(b), fin, fout, flags, precision,
                _ptr(mask), mask_scale, _ptr(support), _ptr(out), _ptr(ws), ws.numel(),
                torch.cuda.current_stream(dev).cuda_stream,
            )
        if st:
            _lib.check(st, "gcnb_layer_forward")
        ctx.graph = graph
        ctx.relu = relu
        ctx.precision = precision
        ctx.has_bias = bias is not None
        ctx.x_shape = tuple(x.shape)
        ctx.mask = mask
        ctx.mask_scale = mask_scale
        ctx.agg = agg
        ctx.save_for_backward(support if agg else xr, w, out if relu else None)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        lib = _lib.load()
        xr, w, y = ctx.saved_tensors
        graph = ctx.graph
        dev = g.device
        fin, fout = w.shape
        need_dx, need_dw = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        need_db = ctx.has_bias and ctx.needs_input_grad[2]
        gr = _rowmajor(g)
        flags = (_lib.LAYER_RELU if ctx.relu else 0) | (_lib.LAYER_NEED_DX if need_dx else 0) | (
            _lib.LAYER_NEED_DW if need_dw else 0) | (_lib.LAYER_NEED_DB if need_db else 0) | (
            _lib.LAYER_AGG_FIRST if ctx.agg else 0)
        if ctx.agg:  # scratch for G W^T, only on the way to dX
            ds = torch.empty((graph.n_rows, _ld4(fin)), dtype=torch.float32, device=dev) if need_dx else None
        else:
            ds = torch.empty((graph.n_cols, _ld4(fout)), dtype=torch.float32, device=dev)
        # the copy of G the SpMM / dW product read: the masked gradient, or G itself re-laid with 16-byte aligned rows
        # when the caller's are not (fout = 47)
        staged = ctx.relu or ctx.mask is not None or _ld(gr) % 4 != 0 or gr.data_ptr() % 16 != 0
        gm = torch.empty((graph.n_rows, _ld4(fout)), dtype=torch.float32, device=dev) if staged else None
        dw = torch.empty((fin, fout), dtype=torch.float32, device=dev) if need_dw else None
        db = torch.empty((fout,), dtype=torch.float32, device=dev) if need_db else None
        dx = torch.empty((graph.n_cols, fin), dtype=torch.float32, device=dev) if need_dx else None
        with _on_device(dev):
            ws = _ws(_layer_ws_bytes(lib, graph, fin, fout, ctx.precision), dev)
            st = lib.gcnb_layer_backward(
                graph._h, _ptr(xr), _ld(xr), _ptr(w), _ptr(gr), _ld(gr), _ptr(y), fin, fout, flags, ctx.precision,
                _ptr(ctx.mask), ctx.mask_scale, _ptr(gm), _ptr(ds), _ptr(dw), _ptr(db), _ptr(dx), fin, _ptr(ws),
                ws.numel(),
                torch.cuda.current_stream(dev).cuda_stream,
            )
        if st:
            _lib.check(st, "gcnb_layer_backward")
        return dx, dw, db, None, None, None, None, None, None


def _ld8(f):
    return (f + 7) // 8 * 8


def _gemm(lib, m, n, k, a, a_rs, a_cs, b, b_rs, b_cs, out, ldc, dev, sp, bias=None, relu=False):
    """out[m, n] (ld ldc) = a b (+ bias) (relu) through gcnb_gemm / gcnb_gemm_ex, precision "auto"."""
    auto = _lib.GEMM_AUTO
    ws = _ws(lib.gcnb_gemm_workspace_bytes(m, n, k, auto), dev)
    if bias is None and not relu:
        _lib.check(lib.gcnb_gemm(m, n, k, _ptr(a), a_rs, a_cs, _ptr(b), b_rs, b_cs, _ptr(out), ldc, auto, _ptr(ws), ws.numel(), sp),
                   "gcnb_gemm")
    else:
        _lib.check(lib.gcnb_gemm_ex(m, n, k, _ptr(a), a_rs, a_cs, _ptr(b), b_rs, b_cs, _ptr(out), ldc, _ptr(bias), 1 if relu else 0,
                                    auto, _ptr(ws), ws.numel(), sp), "gcnb_gemm_ex")
    return out


def _spmm_bf16_panel(lib, graph, flags, src, f, bias, out, ldo, dev, sp):
    """out = A (or A^T) @ bf16(src[:, :f]) (+ bias) (relu): the panel is rounded once (gcnb_to_bf16) and gathered at half
    the bytes per row (gcnb_spmm_bf16); accumulation and output fp32."""
    rows = src.shape[0]
    panel = torch.empty((rows, _ld8(f)), dtype=torch.bfloat16, device=dev)
    _lib.check(lib.gcnb_to_bf16(rows, f, _ptr(src), _ld(src), _ptr(panel), _ld8(f), sp), "gcnb_to_bf16")
    ws = _ws(lib.gcnb_spmm_workspace_bytes(graph._h, flags & _lib.SPMM_TRANSPOSE, f), dev)
    _lib.check(lib.gcnb_spmm_bf16(graph._h, flags, _ptr(panel), _ld8(f), f, _ptr(bias), _ptr(out), ldo, _ptr(ws), ws.numel(), sp),
               "gcnb_spmm_bf16")
    return out


class _GCNLayerBf16Fn(torch.autograd.Function):
    """The layer with bf16 PANELS (precision="bf16", the <= 2e-2 tier of BASELINE's north_star): the operand the
    SpMM gathers -- support = X W (or X itself in the aggregate-first order) forward, the (masked) upstream gradient (or
    G W^T) backward -- is rounded to bf16 once and gathered at half the bytes per row; X, W, the dense products, the
    accumulation of the SpMM, bias, ReLU and every output stay fp32.  Same association rule as the fp32 tier."""

    @staticmethod
    def forward(ctx, x, weight, bias, graph, relu, association="auto"):
        lib = _lib.load()
        dev = x.device
        fin, fout = weight.shape
        xr = _rowmajor(x)
        w = weight.contiguous()
        b = bias.contiguous() if bias is not None else None
        n = graph.n_cols
        agg = association == "aggregate_first" or (association == "auto" and fin * (2 if ctx.needs_input_grad[0] else 1) < fout * (
            2 if (ctx.needs_input_grad[0] or ctx.needs_input_grad[1]) else 1))
        out = torch.empty((graph.n_rows, fout), dtype=torch.float32, device=dev)
        with _on_device(dev):
            sp = _stream_ptr(dev)
            if agg:  # out = (A bf16(X)) W + b
                ax = torch.empty((graph.n_rows, _ld4(fin)), dtype=torch.float32, device=dev)
                if _ld4(fin) != fin:
                    ax.zero_()
                _spmm_bf16_panel(lib, graph, 0, xr, fin, None, ax, _ld4(fin), dev, sp)
                _gemm(lib, graph.n_rows, fout, fin, ax, _ld4(fin), 1, w, fout, 1, out, fout, dev, sp, b, relu)
                keep = ax
            else:    # out = A bf16(X W) + b
                support = torch.empty((n, _ld4(fout)), dtype=torch.float32, device=dev)
                _gemm(lib, n, fout, fin, xr, _ld(xr), 1, w, fout, 1, support, _ld4(fout), dev, sp)
                _spmm_bf16_panel(lib, graph, _lib.SPMM_RELU if relu else 0, support[:, :fout], fout, b, out, fout, dev, sp)
                keep = xr
        ctx.graph, ctx.relu, ctx.has_bias, ctx.agg = graph, relu, bias is not None, agg
        ctx.save_for_backward(keep, w, out if relu else None)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        lib = _lib.load()
        xk, w, y = ctx.saved_tensors  # xk = X, or A X in the aggregate-first order
        graph = ctx.graph
        dev = g.device
        fin, fout = w.shape
        need_dx, need_dw = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        need_db = ctx.has_bias and ctx.needs_input_grad[2]
        gr = _rowmajor(g)
        dx = dw = db = None
        with _on_device(dev):
            sp = _stream_ptr(dev)
            gsrc = gr
            staged = ctx.relu or _ld(gr) % 4 != 0 or gr.data_ptr() % 16 != 0  # (aligned rows for the dense products)
            if staged or need_db:
                gm = torch.empty((graph.n_rows, _ld4(fout)), dtype=torch.float32, device=dev) if staged else None
                db = torch.empty((fout,), dtype=torch.float32, device=dev)
                ws = _ws(lib.gcnb_colsum_workspace_bytes(graph.n_rows, fout), dev)
                _lib.check(lib.gcnb_colsum(graph.n_rows, fout, _ptr(gr), _ld(gr), _ptr(y) if ctx.relu else None, fout,
                                           _ptr(gm), _ld4(fout), _ptr(db), _ptr(ws), ws.numel(), sp), "gcnb_colsum")
                if gm is not None:
                    gsrc = gm[:, :fout]
                if not need_db:
                    db = None
            n = graph.n_cols
            if ctx.agg:
                if need_dw:  # dW = (A X)^T G: no SpMM
                    dw = torch.empty((fin, fout), dtype=torch.float32, device=dev)
                    _gemm(lib, fin, fout, graph.n_rows, xk, 1, _ld(xk), gsrc, _ld(gsrc), 1, dw, fout, dev, sp)
                if need_dx:  # dX = A^T bf16(G W^T)
                    t = torch.empty((graph.n_rows, _ld4(fin)), dtype=torch.float32, device=dev)
                    _gemm(lib, graph.n_rows, fin, fout, gsrc, _ld(gsrc), 1, w, 1, fout, t, _ld4(fin), dev, sp)
                    dx = torch.empty((n, fin), dtype=torch.float32, device=dev)
                    _spmm_bf16_panel(lib, graph, _lib.SPMM_TRANSPOSE, t[:, :fin], fin, None, dx, fin, dev, sp)
            elif need_dw or need_dx:
                ds = torch.empty((n, _ld4(fout)), dtype=torch.float32, device=dev)
                _spmm_bf16_panel(lib, graph, _lib.SPMM_TRANSPOSE, gsrc, fout, None, ds, _ld4(fout), dev, sp)
                if need_dw:
                    dw = torch.empty((fin, fout), dtype=torch.float32, device=dev)
                    _gemm(lib, fin, fout, n, xk, 1, _ld(xk), ds, _ld4(fout), 1, dw, fout, dev, sp)
                if need_dx:
                    dx = torch.empty((n, fin), dtype=torch.float32, device=dev)
                    _gemm(lib, n, fin, fout, ds, _ld4(fout), 1, w, 1, fout, dx, fin, dev, sp)
        return dx, dw, db, None, None, None


class _GCNLayerBatchedFn(torch.autograd.Function):
    """The layer over a batch of feature matrices that share one adjacency: x [B, N, Fin] -> [B, N, Fout].

    The fork's real training step calls the 3-layer GCN once per sample with the same `adj`
    (GCN_OVER_MLP.forward, pygcn/models.py:343-349: 20 samples -> 60 layer calls per step).  Here the
    batch is laid out node-major, Xn [(N*B), Fin], so that X.W is ONE GEMM whose result, seen as
    [N, B*Fout], is the dense operand of ONE SpMM: the index/value stream of the adjacency is read
    once per layer instead of B times, and B*Fout-wide rows gather at the wide-row rate."""

    @staticmethod
    def forward(ctx, x, weight, bias, graph, relu, precision):
        lib = _lib.load()
        dev = x.device
        bsz, n, fin = x.shape
        fout = weight.shape[1]
        wide = bsz * fout
        xn = x.permute(1, 0, 2).contiguous().view(n * bsz, fin)   # node-major rows (n, b); free if already so
        w = weight.contiguous()
        s2 = torch.empty((n * bsz, fout), dtype=torch.float32, device=dev)
        out2 = torch.empty((graph.n_rows, wide), dtype=torch.float32, device=dev)
        brep = bias.detach().repeat(bsz).contiguous() if bias is not None else None
        with _on_device(dev):
            sp = _stream_ptr(dev)
            ws = _ws(lib.gcnb_gemm_workspace_bytes(n * bsz, fout, fin, precision), dev)
            st = lib.gcnb_gemm(n * bsz, fout, fin, _ptr(xn), fin, 1, _ptr(w), fout, 1, _ptr(s2), fout, precision,
                               _ptr(ws), ws.numel(), sp)
            _lib.check(st, "gcnb_gemm")
            ws2 = _ws(lib.gcnb_spmm_workspace_bytes(graph._h, 0, wide), dev)
            st = lib.gcnb_spmm(graph._h, _lib.SPMM_RELU if relu else 0, _ptr(s2), wide, wide, _ptr(brep), _ptr(out2),
                               wide, _ptr(ws2), ws2.numel(), sp)
            _lib.check(st, "gcnb_spmm")
        ctx.graph, ctx.relu, ctx.precision = graph, relu, precision
        ctx.has_bias = bias is not None
        ctx.dims = (bsz, n, fin, fout)
        ctx.save_for_backward(xn, w, out2 if relu else None)
        return out2.view(graph.n_rows, bsz, fout).permute(1, 0, 2)

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        lib = _lib.load()
        xn, w, y2 = ctx.saved_tensors
        graph, precision = ctx.graph, ctx.precision
        bsz, n, fin, fout = ctx.dims
        wide = bsz * fout
        dev = g.device
        need_dx, need_dw, need_db = ctx.needs_input_grad[0], ctx.needs_input_grad[1], ctx.has_bias and ctx.needs_input_grad[2]
        g2 = g.permute(1, 0, 2).contiguous().view(graph.n_rows, wide)
        dx = dw = db = None
        with _on_device(dev):
            sp = _stream_ptr(dev)
            gm2 = g2
            if ctx.relu or need_db:
                gm2 = torch.empty_like(g2) if ctx.relu else None
                dbrep = torch.empty((wide,), dtype=torch.float32, device=dev)
                ws = _ws(lib.gcnb_colsum_workspace_bytes(graph.n_rows, wide), dev)
                st = lib.gcnb_colsum(graph.n_rows, wide, _ptr(g2), wide, _ptr(y2) if ctx.relu else None, wide,
                                     _ptr(gm2), wide, _ptr(dbrep), _ptr(ws), ws.numel(), sp)
                _lib.check(st, "gcnb_colsum")
                if gm2 is None:
                    gm2 = g2
                if need_db:  # db = sum over the batch of the per-sample column sums
                    db = torch.empty((fout,), dtype=torch.float32, device=dev)
                    ws = _ws(lib.gcnb_colsum_workspace_bytes(bsz, fout), dev)
                    st = lib.gcnb_colsum(bsz, fout, _ptr(dbrep), fout, None, fout, None, fout, _ptr(db), _ptr(ws),
                                         ws.numel(), sp)
                    _lib.check(st, "gcnb_colsum")
            if need_dw or need_dx:
                ds2 = torch.empty((graph.n_cols, wide), dtype=torch.float32, device=dev)
                ws = _ws(lib.gcnb_spmm_workspace_bytes(graph._h, _lib.SPMM_TRANSPOSE, wide), dev)
                st = lib.gcnb_spmm(graph._h, _lib.SPMM_TRANSPOSE, _ptr(gm2), wide, wide, None, _ptr(ds2), wide, _ptr(ws),
                                   ws.numel(), sp)
                _lib.check(st, "gcnb_spmm(transpose)")
                rows = n * bsz
                if need_dw:  # dW = Xn^T dS over the (n, b) rows: one split-K product
                    dw = torch.empty((fin, fout), dtype=torch.float32, device=dev)
                    ws = _ws(lib.gcnb_gemm_workspace_bytes(fin, fout, rows, precision), dev)
                    st = lib.gcnb_gemm(fin, fout, rows, _ptr(xn), 1, fin, _ptr(ds2), fout, 1, _ptr(dw), fout, precision,
                                       _ptr(ws), ws.numel(), sp)
                    _lib.check(st, "gcnb_gemm(dW)")
                if need_dx:
                    dxn = torch.empty((rows, fin), dtype=torch.float32, device=dev)
                    ws = _ws(lib.gcnb_gemm_workspace_bytes(rows, fin, fout, precision), dev)
                    st = lib.gcnb_gemm(rows, fin, fout, _ptr(ds2), fout, 1, _ptr(w), 1, fout, _ptr(dxn), fin, precision,
                                       _ptr(ws), ws.numel(), sp)
                    _lib.check(st, "gcnb_gemm(dX)")
                    dx = dxn.view(n, bsz, fin).permute(1, 0, 2)
        return dx, dw, db, None, None, None


class _GCNLayerF64Fn(torch.autograd.Function):
    """The layer in fp64 (gcnb_layer_forward_f64 / _backward_f64): what `model.double()` computes in the reference, on
    the handle's fp64 values.  Same association rule as the fp32 layer, with ld2 panels."""

    @staticmethod
    def forward(ctx, x, weight, bias, graph, relu, mask=None, mask_scale=1.0, association="auto"):
        lib = _lib.load()
        dev = x.device
        f64 = torch.float64
        fin, fout = weight.shape
        xr = _rowmajor(x, f64)
        w = weight.contiguous()
        b = bias.contiguous() if bias is not None else None
        agg = _aggregate_first(association, graph, xr, fin, fout, ctx.needs_input_grad[0], ctx.needs_input_grad[1], lane=2)
        if agg:  # A X, kept for dW = (A X)^T G
            support = torch.empty((graph.n_rows, _ld2(fin)), dtype=f64, device=dev)
        else:
            support = torch.empty((graph.n_cols, _ld2(fout)), dtype=f64, device=dev)
        out = torch.empty((graph.n_rows, fout), dtype=f64, device=dev)
        flags = (_lib.LAYER_RELU if relu else 0) | (_lib.LAYER_AGG_FIRST if agg else 0)
        with _on_device(dev):
            ws = _ws(lib.gcnb_layer_f64_workspace_bytes(graph._h, fin, fout), dev)
            _lib.check(lib.gcnb_layer_forward_f64(graph._h, _ptr(xr), _ld(xr), _ptr(w), _ptr(b), fin, fout, flags, _ptr(mask),
                                                  mask_scale, _ptr(support), _ptr(out), _ptr(ws), ws.numel(),
                                                  torch.cuda.current_stream(dev).cuda_stream), "gcnb_layer_forward_f64")
        ctx.graph, ctx.relu, ctx.has_bias, ctx.agg = graph, relu, bias is not None, agg
        ctx.mask, ctx.mask_scale = mask, mask_scale
        ctx.save_for_backward(support if agg else xr, w, out if relu else None)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        lib = _lib.load()
        xr, w, y = ctx.saved_tensors
        graph = ctx.graph
        dev = g.device
        f64 = torch.float64
        fin, fout = w.shape
        need_dx, need_dw = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        need_db = ctx.has_bias and ctx.needs_input_grad[2]
        gr = _rowmajor(g, f64)
        flags = (_lib.LAYER_RELU if ctx.relu else 0) | (_lib.LAYER_NEED_DX if need_dx else 0) | (
            _lib.LAYER_NEED_DW if need_dw else 0) | (_lib.LAYER_NEED_DB if need_db else 0) | (
            _lib.LAYER_AGG_FIRST if ctx.agg else 0)
        if ctx.agg:  # scratch for G W^T, only on the way to dX
            ds = torch.empty((graph.n_rows, _ld2(fin)), dtype=f64, device=dev) if need_dx else None
        else:
            ds = torch.empty((graph.n_cols, _ld2(fout)), dtype=f64, device=dev) if (need_dx or need_dw) else None
        masked = ctx.relu or ctx.mask is not None  # the masked gradient is staged with ld2 rows
        gm = torch.empty((graph.n_rows, _ld2(fout)), dtype=f64, device=dev) if masked else None
        dw = torch.empty((fin, fout), dtype=f64, device=dev) if need_dw else None
        db = torch.empty((fout,), dtype=f64, device=dev) if need_db else None
        dx = torch.empty((graph.n_cols, fin), dtype=f64, device=dev) if need_dx else None
        with _on_device(dev):
            ws = _ws(lib.gcnb_layer_f64_workspace_bytes(graph._h, fin, fout), dev)
            _lib.check(lib.gcnb_layer_backward_f64(
                graph._h, _ptr(xr), _ld(xr), _ptr(w), _ptr(gr), _ld(gr), _ptr(y), fin, fout, flags, _ptr(ctx.mask),
                ctx.mask_scale, _ptr(gm), _ptr(ds), _ptr(dw), _ptr(db), _ptr(dx), fin, _ptr(ws), ws.numel(),
                torch.cuda.current_stream(dev).cuda_stream), "gcnb_layer_backward_f64")
        return dx, dw, db, None, None, None, None, None


class _GCNLayerBatchedF64Fn(torch.autograd.Function):
    """_GCNLayerBatchedFn in fp64: one fp64 product over the node-major rows, one fp64 SpMM over the [N, B*Fout] panel."""

    @staticmethod
    def forward(ctx, x, weight, bias, graph, relu):
        lib = _lib.load()
        dev = x.device
        f64 = torch.float64
        bsz, n, fin = x.shape
        fout = weight.shape[1]
        wide = bsz * fout
        xn = x.permute(1, 0, 2).contiguous().view(n * bsz, fin)
        w = weight.contiguous()
        s2 = torch.empty((n * bsz, fout), dtype=f64, device=dev)
        out2 = torch.empty((graph.n_rows, wide), dtype=f64, device=dev)
        brep = bias.detach().repeat(bsz).contiguous() if bias is not None else None
        with _on_device(dev):
            sp = _stream_ptr(dev)
            _gemm_f64(lib, n * bsz, fout, fin, xn, fin, 1, w, fout, 1, s2, fout, dev, sp)
            _spmm_f64(lib, graph, _lib.SPMM_RELU if relu else 0, s2, wide, wide, brep, out2, wide, dev, sp)
        ctx.graph, ctx.relu, ctx.has_bias = graph, relu, bias is not None
        ctx.dims = (bsz, n, fin, fout)
        ctx.save_for_backward(xn, w, out2 if relu else None)
        return out2.view(graph.n_rows, bsz, fout).permute(1, 0, 2)

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        lib = _lib.load()
        xn, w, y2 = ctx.saved_tensors
        graph = ctx.graph
        bsz, n, fin, fout = ctx.dims
        wide = bsz * fout
        dev = g.device
        f64 = torch.float64
        need_dx, need_dw, need_db = ctx.needs_input_grad[0], ctx.needs_input_grad[1], ctx.has_bias and ctx.needs_input_grad[2]
        g2 = g.permute(1, 0, 2).contiguous().view(graph.n_rows, wide)
        dx = dw = db = None
        with _on_device(dev):
            sp = _stream_ptr(dev)
            gm2 = g2
            if ctx.relu or need_db:
                gm2 = torch.empty_like(g2) if ctx.relu else g2
                dbrep = torch.empty((wide,), dtype=f64, device=dev)
                _colsum_f64(lib, graph.n_rows, wide, g2, wide, y2 if ctx.relu else None, wide,
                            gm2 if ctx.relu else None, wide, dbrep, dev, sp)
                if need_db:  # db = sum over the batch of the per-sample column sums
                    db = torch.empty((fout,), dtype=f64, device=dev)
                    _colsum_f64(lib, bsz, fout, dbrep, fout, None, fout, None, fout, db, dev, sp)
            if need_dw or need_dx:
                ds2 = torch.empty((graph.n_cols, wide), dtype=f64, device=dev)
                _spmm_f64(lib, graph, _lib.SPMM_TRANSPOSE, gm2, wide, wide, None, ds2, wide, dev, sp)
                rows = n * bsz
                if need_dw:
                    dw = torch.empty((fin, fout), dtype=f64, device=dev)
                    _gemm_f64(lib, fin, fout, rows, xn, 1, fin, ds2, fout, 1, dw, fout, dev, sp)
                if need_dx:
                    dxn = torch.empty((rows, fin), dtype=f64, device=dev)
                    _gemm_f64(lib, rows, fin, fout, ds2, fout, 1, w, 1, fout, dxn, fin, dev, sp)
                    dx = dxn.view(n, bsz, fin).permute(1, 0, 2)
        return dx, dw, db, None, None


def _gemm_f64(lib, m, n, k, a, a_rs, a_cs, b, b_rs, b_cs, out, ldc, dev, sp, bias=None, relu=False):
    ws = _ws(lib.gcnb_gemm_f64_workspace_bytes(m, n, k), dev)
    if bias is None and not relu:
        _lib.check(lib.gcnb_gemm_f64(m, n, k, _ptr(a), a_rs, a_cs, _ptr(b), b_rs, b_cs, _ptr(out), ldc, _ptr(ws), ws.numel(), sp),
                   "gcnb_gemm_f64")
    else:
        _lib.check(lib.gcnb_gemm_f64_ex(m, n, k, _ptr(a), a_rs, a_cs, _ptr(b), b_rs, b_cs, _ptr(out), ldc, _ptr(bias),
                                        1 if relu else 0, _ptr(ws), ws.numel(), sp), "gcnb_gemm_f64_ex")
    return out


def _spmm_f64(lib, graph, flags, src, ldb, f, bias, out, ldo, dev, sp):
    ws = _ws(lib.gcnb_spmm_f64_workspace_bytes(graph._h, flags & _lib.SPMM_TRANSPOSE, f), dev)
    _lib.check(lib.gcnb_spmm_f64(graph._h, flags, _ptr(src), ldb, f, _ptr(bias), None, 0, 1.0, _ptr(out), ldo, _ptr(ws),
                                 ws.numel(), sp), "gcnb_spmm_f64")
    return out


def _colsum_f64(lib, n_rows, f, g, ldg, y, ldy, gm, ldgm, out, dev, sp):
    ws = _ws(lib.gcnb_colsum_f64_workspace_bytes(n_rows, f), dev)
    _lib.check(lib.gcnb_colsum_f64(n_rows, f, _ptr(g), ldg, _ptr(y), ldy, _ptr(gm), ldgm, _ptr(out), _ptr(ws), ws.numel(), sp),
               "gcnb_colsum_f64")
    return out


def _check_layer_args(x, graph, weight, bias):
    _require_cuda(x, "input")
    _require_cuda(weight, "weight")
    if x.dim() != 2 or weight.dim() != 2:
        raise RuntimeError("input and weight must be matrices")
    if x.shape[1] != weight.shape[0]:
        raise RuntimeError(
            "mat1 and mat2 shapes cannot be multiplied (%dx%d and %dx%d)" % (*x.shape, *weight.shape)
        )
    if x.shape[0] != graph.n_cols:
        raise RuntimeError(
            "size mismatch: adj is %dx%d but input has %d rows" % (graph.n_rows, graph.n_cols, x.shape[0])
        )
    if x.dtype not in (torch.float32, torch.float64):
        raise RuntimeError("expected float32 or float64 input, got %s" % x.dtype)
    if weight.dtype != x.dtype or graph.dtype != x.dtype or (bias is not None and bias.dtype != x.dtype):
        raise RuntimeError("input (%s), weight (%s), bias (%s) and adj (%s) must have one dtype" % (
            x.dtype, weight.dtype, None if bias is None else bias.dtype, graph.dtype))
    if x.device != graph.device or weight.device != graph.device:
        raise RuntimeError("input (%s), weight (%s) and adj (%s) must be on the same device" %
                           (x.device, weight.device, graph.device))
    if bias is not None:
        if bias.shape != (weight.shape[1],) or bias.device != graph.device:
            raise RuntimeError("bias must be a %s [%d] tensor on %s" % (x.dtype, weight.shape[1], graph.device))


def gcn_layer(input, adj, weight, bias=None, relu=False, precision="auto", dropout_mask=None, dropout_p=0.0,
              association="auto"):
    """`adj @ (input @ weight) + bias` (optionally followed by ReLU, then dropout) -- pygcn/layers.py:32-38.

    adj: torch sparse COO / sparse CSR / dense tensor, or a `Graph`.
    relu=True fuses the `F.relu` the reference's models apply to every layer output
    (pygcn/models.py:49,53,56); applying F.relu again on the result is a no-op, so unchanged
    callers stay correct.
    dropout_mask: optional keep-mask (bool/uint8 [n_rows, out_features]) fused into the same epilogue
    with scale 1/(1-dropout_p) -- upstream pygcn's `F.dropout` on the layer output (commented out in
    the fork, pygcn/models.py:50,54); the backward masks the incoming gradient the same way.
    association: "auto" (default) computes (adj @ input) @ weight instead of the reference's adj @ (input @ weight)
    when that moves fewer bytes through the SpMMs (in_features < out_features; see _aggregate_first) -- same result
    to fp32 rounding; "reference" / "aggregate_first" force one order.
    fp64 input, weight, bias and adj (all one dtype, as torch requires) compute the layer in fp64; precision must then be
    "auto".
    """
    if association not in _ASSOCIATIONS:
        raise ValueError("association must be one of %s, got %r" % (_ASSOCIATIONS, association))
    graph = as_graph(adj)
    f64 = isinstance(input, torch.Tensor) and input.dtype == torch.float64
    if f64 and precision != "auto":
        raise ValueError("precision=%r selects an fp32 kernel tier; with float64 operands precision must be 'auto'" % (precision,))
    if input.dim() == 3:  # [B, N, Fin]: the batch shares the adjacency (pygcn/models.py:343-349)
        if dropout_mask is not None:
            raise NotImplementedError("the fused dropout mask is not available for batched input")
        if input.shape[0] == 0:
            return input.new_empty((0, graph.n_rows, weight.shape[1]))
        _check_layer_args(input[0], graph, weight, bias)
        if f64:
            return _GCNLayerBatchedF64Fn.apply(input, weight, bias, graph, bool(relu))
        return _GCNLayerBatchedFn.apply(input, weight, bias, graph, bool(relu), _PRECISIONS[precision])
    _check_layer_args(input, graph, weight, bias)
    if precision == "bf16" and not graph.dense_route:
        if dropout_mask is not None:
            raise NotImplementedError("the fused dropout mask is not available in the bf16 panel tier")
        return _GCNLayerBf16Fn.apply(input, weight, bias, graph, bool(relu), association)
    mask, scale = None, 1.0
    if dropout_mask is not None:
        if not 0.0 <= dropout_p < 1.0:
            raise ValueError("dropout probability has to be in [0, 1), got %r" % (dropout_p,))
        if tuple(dropout_mask.shape) != (graph.n_rows, weight.shape[1]) or dropout_mask.device != graph.device:
            raise RuntimeError("dropout_mask must be a [%d, %d] tensor on %s" % (graph.n_rows, weight.shape[1], graph.device))
        mask = dropout_mask.to(torch.uint8).contiguous()
        scale = 1.0 / (1.0 - dropout_p)
    if f64:
        return _GCNLayerF64Fn.apply(input, weight, bias, graph, bool(relu), mask, scale, association)
    return _GCNLayerFn.apply(input, weight, bias, graph, bool(relu), _PRECISIONS[precision], mask, scale, association)


class _SpmmFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, dense, graph):
        lib = _lib.load()
        dev = dense.device
        d = _rowmajor(dense)
        f = d.shape[1]
        out = torch.empty((graph.n_rows, f), dtype=torch.float32, device=dev)
        if f == 0 or graph.n_rows == 0:
            ctx.graph = graph
            return out
        with torch.cuda.device(dev):
            ws = _ws(lib.gcnb_spmm_workspace_bytes(graph._h, 0, f), dev)
            st = lib.gcnb_spmm(graph._h, 0, _ptr(d), _ld(d), f, None, _ptr(out), f, _ptr(ws), ws.numel(),
                               _stream_ptr(dev))
        _lib.check(st, "gcnb_spmm")
        ctx.graph = graph
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        lib = _lib.load()
        graph = ctx.graph
        dev = g.device
        gr = _rowmajor(g)
        f = gr.shape[1]
        out = torch.empty((graph.n_cols, f), dtype=torch.float32, device=dev)
        if f == 0 or graph.n_cols == 0:
            return out, None
        with torch.cuda.device(dev):
            ws = _ws(lib.gcnb_spmm_workspace_bytes(graph._h, _lib.SPMM_TRANSPOSE, f), dev)
            st = lib.gcnb_spmm(graph._h, _lib.SPMM_TRANSPOSE, _ptr(gr), _ld(gr), f, None, _ptr(out), f, _ptr(ws),
                               ws.numel(), _stream_ptr(dev))
        _lib.check(st, "gcnb_spmm(transpose)")
        return out, None


class _SpmmF64Fn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, dense, graph):
        lib = _lib.load()
        dev = dense.device
        d = _rowmajor(dense, torch.float64)
        f = d.shape[1]
        out = torch.empty((graph.n_rows, f), dtype=torch.float64, device=dev)
        ctx.graph = graph
        if f > 0 and graph.n_rows > 0:
            with torch.cuda.device(dev):
                _spmm_f64(lib, graph, 0, d, _ld(d), f, None, out, f, dev, _stream_ptr(dev))
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        lib = _lib.load()
        graph = ctx.graph
        dev = g.device
        gr = _rowmajor(g, torch.float64)
        f = gr.shape[1]
        out = torch.empty((graph.n_cols, f), dtype=torch.float64, device=dev)
        if f > 0 and graph.n_cols > 0:
            with torch.cuda.device(dev):
                _spmm_f64(lib, graph, _lib.SPMM_TRANSPOSE, gr, _ld(gr), f, None, out, f, dev, _stream_ptr(dev))
        return out, None


def spmm(adj, dense):
    """Drop-in for `torch.spmm(adj, dense)` as the layer uses it (pygcn/layers.py:34).

    Differentiable w.r.t. `dense`; `adj` never requires grad in the reference.
    """
    graph = as_graph(adj)
    _require_cuda(dense, "dense")
    if isinstance(adj, torch.Tensor) and adj.requires_grad:
        raise NotImplementedError("gradients w.r.t. the adjacency are not part of the GCN hot path")
    if dense.dim() != 2 or dense.shape[0] != graph.n_cols:
        raise RuntimeError("mat1 and mat2 shapes cannot be multiplied (%dx%d and %s)" %
                           (graph.n_rows, graph.n_cols, "x".join(str(s) for s in dense.shape)))
    if dense.dtype not in (torch.float32, torch.float64):
        raise RuntimeError("expected float32 or float64 dense operand, got %s" % dense.dtype)
    if dense.dtype != graph.dtype:
        raise RuntimeError("adj (%s) and dense (%s) must have one dtype" % (graph.dtype, dense.dtype))
    if dense.device != graph.device:
        raise RuntimeError("adj (%s) and dense (%s) must be on the same device" % (graph.device, dense.device))
    if dense.dtype == torch.float64:
        return _SpmmF64Fn.apply(dense, graph)
    return _SpmmFn.apply(dense, graph)


def load_adj(avg_visits, precision="auto"):
    """The CBG adjacency of `utils.load_adj` (pygcn/utils.py:122-131) on the device:
    adj[i][j] = sum_p avg[p, i] * avg[p, j]  for the averaged POI x CBG visit matrix `avg` [n_poi, n_cbg]
    (the reference's O(N^2 M) Python double loop, cached as adj_<msa>.npy), returned as the dense fp32
    [n_cbg, n_cbg] tensor the scripts pass as `adj`.  One split-K tensor-core product per 256-column panel
    (gcnb_gemm, tcgen05 3xTF32 "tn" kernel) on a copy of `avg` whose rows are zero-padded to a multiple of 4."""
    lib = _lib.load()
    _require_cuda(avg_visits, "avg_visits")
    if avg_visits.dim() != 2:
        raise RuntimeError("avg_visits must be a [n_poi, n_cbg] matrix")
    a = avg_visits.to(torch.float32)
    p_, n = a.shape
    n4 = _ld4(n)
    a4 = torch.zeros((p_, n4), dtype=torch.float32, device=a.device)
    a4[:, :n] = a
    out = torch.empty((n4, n4), dtype=torch.float32, device=a.device)
    prec = _PRECISIONS[precision]
    with torch.cuda.device(a.device):
        for f0 in range(0, n4, 256):
            fw = min(256, n4 - f0)
            ws = _ws(lib.gcnb_gemm_workspace_bytes(n4, fw, p_, prec), a.device)
            st = lib.gcnb_gemm(n4, fw, p_, _ptr(a4), 1, n4, a4.data_ptr() + 4 * f0, n4, 1, out.data_ptr() + 4 * f0, n4,
                               prec, _ptr(ws), ws.numel(), _stream_ptr(a.device))
            _lib.check(st, "gcnb_gemm")
    return out[:n, :n].contiguous()


def mm(a, b, precision="auto"):
    """`torch.mm(a, b)` through gcnb_gemm (no autograd); used by tests and the benchmark.  fp64 a and b run the fp64
    product (gcnb_gemm_f64, precision "auto" only)."""
    lib = _lib.load()
    _require_cuda(a, "a")
    _require_cuda(b, "b")
    if a.dim() != 2 or b.dim() != 2 or a.shape[1] != b.shape[0]:
        raise RuntimeError("mat1 and mat2 shapes cannot be multiplied")
    m, k = a.shape
    n = b.shape[1]
    if a.dtype == torch.float64 or b.dtype == torch.float64:
        if a.dtype != b.dtype:
            raise RuntimeError("expected both operands of one dtype, got %s and %s" % (a.dtype, b.dtype))
        if precision != "auto":
            raise ValueError("with float64 operands precision must be 'auto', got %r" % (precision,))
        out = torch.empty((m, n), dtype=torch.float64, device=a.device)
        with torch.cuda.device(a.device):
            _gemm_f64(lib, m, n, k, a, a.stride(0), a.stride(1), b, b.stride(0), b.stride(1), out, max(n, 1), a.device,
                      _stream_ptr(a.device))
        return out
    out = torch.empty((m, n), dtype=torch.float32, device=a.device)
    prec = _PRECISIONS[precision]
    with torch.cuda.device(a.device):
        ws = _ws(lib.gcnb_gemm_workspace_bytes(m, n, k, prec), a.device)
        st = lib.gcnb_gemm(m, n, k, _ptr(a), a.stride(0), a.stride(1), _ptr(b), b.stride(0), b.stride(1), _ptr(out),
                           max(n, 1), prec, _ptr(ws), ws.numel(), _stream_ptr(a.device))
    _lib.check(st, "gcnb_gemm")
    return out


# ---------------------------------------------------------------------------- (ReLU ->) fresh BatchNorm (SURVEY.md 8f rank 2)
class _FreshBatchNormFn(torch.autograd.Function):
    """gcnb_fresh_bn_forward / _backward: `GCN.apply_bn(F.relu(y))` (pygcn/models.py:41-45, 49, 53) in one statistics
    pass and one apply pass each way."""

    @staticmethod
    def forward(ctx, y, relu, eps):
        lib = _lib.load()
        dev = y.device
        yr = _rowmajor(y)
        n, f = yr.shape
        out = torch.empty((n, f), dtype=torch.float32, device=dev)
        stat = torch.empty((2, _ld4(f)), dtype=torch.float32, device=dev)  # mean | rstd, rows 16-byte aligned
        with torch.cuda.device(dev):
            ws = _ws(lib.gcnb_fresh_bn_workspace_bytes(n, f), dev)
            st = lib.gcnb_fresh_bn_forward(n, f, _ptr(yr), _ld(yr), 1 if relu else 0, float(eps), _ptr(out), max(f, 1),
                                           stat[0].data_ptr(), stat[1].data_ptr(), _ptr(ws), ws.numel(), _stream_ptr(dev))
        _lib.check(st, "gcnb_fresh_bn_forward")
        ctx.relu = bool(relu)
        ctx.save_for_backward(yr, stat)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        lib = _lib.load()
        yr, stat = ctx.saved_tensors
        dev = yr.device
        gr = _rowmajor(g)
        n, f = yr.shape
        dy = torch.empty((n, f), dtype=torch.float32, device=dev)
        gstat = torch.empty((2 * f,), dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            ws = _ws(lib.gcnb_fresh_bn_workspace_bytes(n, f), dev)
            st = lib.gcnb_fresh_bn_backward(n, f, _ptr(yr), _ld(yr), 1 if ctx.relu else 0, _ptr(gr), _ld(gr),
                                            stat[0].data_ptr(), stat[1].data_ptr(), _ptr(dy), max(f, 1), _ptr(gstat),
                                            _ptr(ws), ws.numel(), _stream_ptr(dev))
        _lib.check(st, "gcnb_fresh_bn_backward")
        return dy, None, None


def apply_bn(x, relu=False, eps=1e-5):
    """Drop-in for `GCN.apply_bn` (pygcn/models.py:41-45): batch-normalise the [N, F] layer output with a FRESH
    BatchNorm1d -- affine weight 1 / bias 0, batch statistics (biased variance, eps 1e-5) whatever the model's
    train / eval mode.  relu=True folds the `F.relu` the models apply first (`apply_bn(F.relu(gc(x, adj)))`,
    models.py:49,53) and its backward mask into the same two passes:  apply_bn(y, relu=True) == apply_bn(F.relu(y)).
    x may also be this package's batched samples [B, N, F]: normalised per sample, as the per-sample loop does.
    Differentiable w.r.t. x.  Errors mirror torch's: fewer than 2 rows raise ValueError, CPU tensors raise (no
    fallback).  Opt-in: written at the end of round 1, not yet run on hardware (tests/test_gpu_optin.py)."""
    _require_cuda(x, "x")
    if x.dim() == 3:
        # this package's batched-samples layout x[B, N, F] (GraphConvolution.forward(x[B, N, Fin], adj), DESIGN 3.5): the
        # per-sample loop of GCN_OVER_MLP (pygcn/models.py:343-349) applies a fresh BatchNorm to every sample's [N, F]
        # output, i.e. statistics per (sample, feature) over the N nodes -- one pass over the node-major [N, B*F] panel,
        # which is how the batched layer stores its output (a free view).  NOT torch's [B, C, L] convention.
        if x.dtype != torch.float32:
            raise RuntimeError("expected float32, got %s" % x.dtype)
        b, n, f = x.shape
        if n < 2:
            raise ValueError("Expected more than 1 value per channel when training, got input size %s" % (tuple(x.shape),))
        if b == 0 or f == 0:
            return torch.empty_like(x)
        xn = x.permute(1, 0, 2)
        if not xn.is_contiguous():
            xn = xn.contiguous()
        out = _FreshBatchNormFn.apply(xn.reshape(n, b * f), bool(relu), float(eps))
        return out.view(n, b, f).permute(1, 0, 2)
    if x.dim() != 2:
        raise ValueError("expected 2D input [N, F] or batched samples [B, N, F] (got %dD input)" % x.dim())  # models.py:44
    if x.dtype != torch.float32:
        raise RuntimeError("expected float32, got %s" % x.dtype)
    if x.shape[0] < 2:
        raise ValueError("Expected more than 1 value per channel when training, got input size %s" % (tuple(x.shape),))
    if x.shape[1] == 0:
        return torch.empty_like(x)
    return _FreshBatchNormFn.apply(x, bool(relu), float(eps))

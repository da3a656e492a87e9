"""Every SpMM kernel on adversarial CSR structures, against exact-arithmetic references.

The inputs make every partial sum exact in fp32 -- in bf16 panels and in 3xTF32 too -- in any summation order:
stored values in {+-1/4, +-1/2, +-1, +-2}, panel entries integers in [-8, 8], integer bias, dropout scale 2, and all
sums far below 2^22.  The fp64 scipy product cast to fp32 is then the only correct answer, and every kernel must
produce it on every entry (torch.equal), whatever order it adds in.  On top of that, each case:
  * fills the panel's padding columns (ld > f) with NaN,
  * surrounds the output with a sentinel that must come back bit for bit outside [rows, 0:f),
  * runs twice and requires bit-identical results.
The structures put row lengths on the bin, chunk, stage and item edges (0, 1-9, 15-17, 31-33, 63-65, 1023-1025,
2047-2049, 3073), runs of empty rows, odd and even row starts, odd nnz, rectangular shapes (the transposed view gets
empty rows and hub-column long rows), a single-row and an empty handle, and the row blocks of the multi-GPU layer.
Non-finite panel values must propagate exactly as in the fp64 product, which touches stored entries only.
"""
import ctypes

import numpy as np
import pytest
import scipy.sparse as sp
import torch

pytestmark = pytest.mark.gpu

VALUES = np.array([-2, -1, -0.5, -0.25, 0.25, 0.5, 1, 2], np.float32)
SENTINEL = -12345.0
FP32_WIDTHS = [1, 2, 3, 4, 5, 8, 9, 16, 17, 31, 32, 33, 63, 64, 65, 127, 128, 129, 255, 256, 257, 511, 512, 513, 1025]
BF16_WIDTHS = [7, 8, 9, 63, 64, 65, 127, 128, 129, 1023, 1024, 1025]
FMAX = 1025
EDGE_LENGTHS = [1, 2, 3, 4, 5, 6, 7, 8, 9, 15, 16, 17, 31, 32, 33, 63, 64, 65, 1023, 1024, 1025, 2047, 2048, 2049, 3073]
# every short-row kernel: auto, warp-per-row, TMA-staged, the 16 group-per-row variants, and the streaming kernel with
# 0 (auto) / 2 / 4 / 8 gathered rows in flight
KERNELS = ["auto", "rows", "tma"] + [("group", v) for v in range(16)] + [("stream", u) for u in (0, 2, 4, 8)]


def _kid(k):
    return k if isinstance(k, str) else "%s%d" % k


def dev():
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def P():
    import pygcn_b200

    assert pygcn_b200._lib.load().gcnb_check_device() == 0, pygcn_b200._lib.last_error()
    return pygcn_b200


_KERNELS = {"auto": 0, "rows": 1, "group": 2, "tma": 3}


@pytest.fixture
def spmm_kernel(P, request):
    """Forces one of the SpMM kernels for the short-row bins (gcnb_set_tuning), restores auto after."""
    from pygcn_b200 import _lib

    lib = _lib.load()
    name, variant = request.param if isinstance(request.param, tuple) else (request.param, -1)
    if name == "stream":  # the streaming kernel wherever the view is eligible (auto keeps it for big graphs);
        # variant = gathered rows in flight per lane, paired with one of the L2 hint modes (2 -> 2, 4 -> 1, 8 -> 0)
        _lib.check(lib.gcnb_set_tuning(_lib.TUNE_SPMM_KERNEL, 0), "set_tuning")
        _lib.check(lib.gcnb_set_tuning(_lib.TUNE_SPMM_STREAM, 2), "set_tuning")
        _lib.check(lib.gcnb_set_tuning(_lib.TUNE_STREAM_BATCH, max(variant, 0)), "set_tuning")
        _lib.check(lib.gcnb_set_tuning(_lib.TUNE_STREAM_HINT, {2: 2, 4: 1, 8: 0}.get(variant, 0)), "set_tuning")
        _lib.check(lib.gcnb_set_tuning(_lib.TUNE_STREAM_HOT_MB, 1), "set_tuning")  # small graphs: some hot, some cold columns
    else:
        _lib.check(lib.gcnb_set_tuning(_lib.TUNE_SPMM_STREAM, 0 if name != "auto" else 1), "set_tuning")
        _lib.check(lib.gcnb_set_tuning(_lib.TUNE_SPMM_KERNEL, _KERNELS[name]), "set_tuning")
        _lib.check(lib.gcnb_set_tuning(_lib.TUNE_SPMM_GROUP_VARIANT, variant), "set_tuning")
    yield name
    lib.gcnb_set_tuning(_lib.TUNE_SPMM_KERNEL, 0)
    lib.gcnb_set_tuning(_lib.TUNE_SPMM_GROUP_VARIANT, -1)
    lib.gcnb_set_tuning(_lib.TUNE_SPMM_STREAM, 1)
    lib.gcnb_set_tuning(_lib.TUNE_STREAM_BATCH, 0)
    lib.gcnb_set_tuning(_lib.TUNE_STREAM_HINT, 0)
    lib.gcnb_set_tuning(_lib.TUNE_STREAM_HOT_MB, 48)


# ------------------------------------------------------------------ structures (host-side CSR)
def _csr(lengths, n_cols, cols, vals):
    indptr = np.concatenate([[0], np.cumsum(lengths)]).astype(np.int64)
    assert indptr[-1] == len(cols) == len(vals)
    return sp.csr_matrix((vals.astype(np.float64), cols.astype(np.int64), indptr), shape=(len(lengths), n_cols))


def _edge_lengths_both_parities():
    """Every edge length once at an even and once at an odd row start, empty rows around the long ones."""
    out, nnz = [], 0
    for n in EDGE_LENGTHS:
        for parity in (0, 1):
            if nnz % 2 != parity:
                out.append(1)
                nnz += 1
            if n >= 1023:
                out += [0, 0, 0]
            out.append(n)
            nnz += n
            if n >= 1023:
                out += [0, 0]
    return out


def _rectangular(rs):
    """R x C, R < C: leading / trailing / interior empty-row runs, edge lengths at both parities, odd nnz; columns
    skewed (low ids are hubs, so the transposed view has long rows), two column runs never referenced (empty rows of
    the transposed view) and one column referenced exactly once."""
    n_cols = 2500
    lengths = [0] * 5 + _edge_lengths_both_parities() + list(rs.integers(0, 41, 1500)) + [0] * 4
    if sum(lengths) % 2 == 0:
        lengths.append(1)
    lengths += [0] * 6
    nnz = sum(lengths)
    cols = (n_cols * rs.random(nnz) ** 3).astype(np.int64)
    unused = ((cols >= 700) & (cols < 720)) | (cols >= n_cols - 41)
    cols[unused] = cols[unused] % 600 + 1
    cols[nnz // 2] = n_cols - 41  # referenced once
    return _csr(lengths, n_cols, cols, rs.choice(VALUES, nnz))


def _square_without_empty_rows(rs):
    """n x n with a diagonal entry in every row: no empty row in either direction (the streaming kernel's views)."""
    lengths = _edge_lengths_both_parities()
    lengths = [max(n, 1) for n in lengths] + list(rs.integers(1, 41, 2500))
    n = len(lengths)
    nnz = sum(lengths)
    cols = rs.integers(0, n, nnz)
    starts = np.concatenate([[0], np.cumsum(lengths)[:-1]])
    cols[starts] = np.arange(n)
    return _csr(lengths, n, cols, rs.choice(VALUES, nnz))


class View:
    """One operand of a product: a graph handle + direction, its fp64 CSR, the panel rows NaN-filled (padding slots
    of an all-gathered panel), and the exact reference on the module's integer panel."""

    def __init__(self, name, gr, transpose, a64, nan_rows=None, layer=False):
        self.name, self.gr, self.transpose, self.a64 = name, gr, transpose, a64
        self.flags = 1 if transpose else 0  # GCNB_SPMM_TRANSPOSE
        self.rows, self.k = a64.shape
        self.layer = layer  # a full handle: also run the dropout-mask epilogue through the layer
        rs = np.random.default_rng(self.rows * 7 + self.k)
        b = rs.integers(-8, 9, (self.k, FMAX)).astype(np.float64)
        if nan_rows is not None:
            b[nan_rows] = np.nan
        self.b64 = b
        self.panel = torch.from_numpy(b.astype(np.float32)).to(dev())
        self.ref = torch.from_numpy((a64 @ b).astype(np.float32)).to(dev())
        self.bias = torch.from_numpy(rs.integers(-8, 9, FMAX).astype(np.float32)).to(dev())
        self.prev = torch.from_numpy(rs.integers(-8, 9, (self.rows, FMAX)).astype(np.float32)).to(dev())


def _graph(P, a):
    a = a.tocsr()
    t = torch.sparse_csr_tensor(torch.from_numpy(a.indptr.astype(np.int64)), torch.from_numpy(a.indices.astype(np.int64)),
                                torch.from_numpy(a.data.astype(np.float32)), a.shape)
    return P.Graph.from_torch(t.to(dev()))


def _block_csr(blk):
    rp, col, val = (t.cpu().numpy() for t in blk.csr())
    return sp.csr_matrix((val.astype(np.float64), col.astype(np.int64), rp.astype(np.int64)), shape=(blk.n_rows, blk.n_cols))


@pytest.fixture(scope="module")
def views(P):
    from pygcn_b200 import dist as D

    rs = np.random.default_rng(2024)
    out = []
    rect = _rectangular(rs)
    square = _square_without_empty_rows(rs)
    single = _csr([1025], 300, rs.integers(0, 300, 1025), rs.choice(VALUES, 1025))
    empty = _csr([0] * 20, 30, np.zeros(0, np.int64), np.zeros(0, np.float32))
    for name, a in (("rect", rect), ("square", square), ("single", single), ("empty", empty)):
        gr = _graph(P, a)
        assert gr.nnz == a.nnz and not gr.dense_route
        out.append(View(name, gr, False, a, layer=True))
        out.append(View(name + "^T", gr, True, a.T.tocsr()))
    rs_rect = rect.indptr[1:] - rect.indptr[:-1]
    assert (rs_rect == 0).sum() > 10 and rs_rect.max() == 3073 and rect.nnz % 2 == 1
    assert (np.bincount(rect.indices, minlength=rect.shape[1]) == 0).sum() >= 60
    assert np.bincount(rect.indices).max() > 1025  # a long row in the transposed view
    # the row blocks of the 3-rank layer, cut from the square graph (own and padding slots as the layer lays them out)
    gsq = out[2].gr
    world = 3
    bounds = D.partition_rows_by_nnz(gsq.csr()[0].cpu(), world)
    pad = D.DistGraph.padded_rows(bounds)
    padding = np.concatenate([np.arange(q * pad + bounds[q + 1] - bounds[q], (q + 1) * pad) for q in range(world)])
    dg = D.DistGraph.from_graph(gsq, 1, world, bounds, split=True)
    n1 = bounds[2] - bounds[1]
    for name, blk in (("fwd_diag", dg.fwd_diag), ("fwd_remote", dg.fwd_remote), ("bwd_diag", dg.bwd_diag),
                      ("bwd_remote", dg.bwd_remote)):
        a = _block_csr(blk)
        nan_rows = np.arange(n1, blk.n_cols) if "diag" in name else padding
        out.append(View(name, blk, False, a, nan_rows=nan_rows))
    assert any(v.a64.getnnz(axis=1).min() == 0 for v in out[-4:])  # the blocks have empty rows
    return out


# ------------------------------------------------------------------ calls
def _spmm(P, v, panel, f, out, flags=0, bias=None):
    from pygcn_b200 import _lib

    lib = _lib.load()
    flags |= v.flags
    ws = torch.empty(max(int(lib.gcnb_spmm_workspace_bytes(v.gr._h, flags, f)), 256), dtype=torch.uint8, device=dev())
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    fn = lib.gcnb_spmm_bf16 if panel.dtype == torch.bfloat16 else lib.gcnb_spmm
    _lib.check(fn(v.gr._h, flags, panel.data_ptr(), panel.stride(0), f, bias.data_ptr() if bias is not None else None,
                  out.data_ptr(), out.stride(0), ws.data_ptr(), ws.numel(), st), "spmm")


def _panel(src, f, dtype, ld=None):
    """src[:, :f] in a buffer of leading dimension ld > f (16-byte aligned rows by default), NaN past f."""
    step = 8 if dtype == torch.bfloat16 else 4
    ld = ld or (f + step - 1) // step * step + step
    buf = torch.full((src.shape[0], ld), float("nan"), dtype=dtype, device=dev())
    buf[:, :f] = src[:, :f].to(dtype)
    return buf


class Sentinel:
    """An output view out = big[1:1+rows, c0:c0+f] inside a sentinel-filled buffer."""

    def __init__(self, rows, f, c0=4, fill=None):
        ld = (f + 3) // 4 * 4 + 8
        self.big = torch.full((rows + 2, ld), SENTINEL, device=dev())
        self.rows, self.f, self.c0 = rows, f, c0
        self.out = self.big[1:1 + rows, c0:c0 + f]
        if fill is not None:
            self.out.copy_(fill)

    def check(self, want, what):
        assert torch.equal(self.out, want), (what, (self.out != want).sum().item())
        rest = self.big.clone()
        rest[1:1 + self.rows, self.c0:self.c0 + self.f] = SENTINEL
        assert bool((rest == SENTINEL).all()), ("wrote outside its output", what)


def _run_exact(P, v, f, dtype, what):
    from pygcn_b200 import _lib

    panel = _panel(v.panel, f, dtype)
    ref = v.ref[:, :f]
    o = Sentinel(v.rows, f)
    _spmm(P, v, panel, f, o.out)
    o.check(ref, what)
    first = o.big.clone()
    _spmm(P, v, panel, f, o.out)
    assert torch.equal(o.big, first), ("rerun differs", what)
    bias = v.bias[:f]
    o = Sentinel(v.rows, f)
    _spmm(P, v, panel, f, o.out, _lib.SPMM_RELU, bias)
    o.check(torch.relu(ref + bias), what + " bias+relu")
    c0 = 4 if f % 8 == 0 else 3  # aligned and unaligned strided outputs
    prev = v.prev[:, :f]
    o = Sentinel(v.rows, f, c0=c0, fill=prev)
    _spmm(P, v, panel, f, o.out, _lib.SPMM_ACCUMULATE)
    o.check(prev + ref, what + " accumulate")
    return ref


@pytest.mark.parametrize("spmm_kernel", KERNELS, indirect=True, ids=_kid)
@pytest.mark.parametrize("dtype,f", [("fp32", f) for f in FP32_WIDTHS] + [("bf16", f) for f in BF16_WIDTHS])
def test_exact_product_on_adversarial_structures(P, views, spmm_kernel, dtype, f):
    """Plain, bias + ReLU, accumulate into a strided output, and (fp32, full handles) the dropout-mask epilogue
    through the layer: equal to the exact product on every entry, nothing written outside the output, rerun
    bit-identical -- on every structure, forward and transposed."""
    tdt = torch.bfloat16 if dtype == "bf16" else torch.float32
    for v in views:
        what = "%s f=%d %s %s" % (v.name, f, dtype, spmm_kernel)
        ref = _run_exact(P, v, f, tdt, what)
        if dtype == "fp32" and spmm_kernel == "auto" and v.rows > 0:
            # rows that are not 16-byte aligned: the generic scalar kernel
            ld = f + 1 if (f + 1) % 4 else f + 2
            o = Sentinel(v.rows, f)
            _spmm(P, v, _panel(v.panel, f, tdt, ld=ld), f, o.out)
            o.check(ref, what + " unaligned panel")
        if v.layer and dtype == "fp32":
            keep = torch.from_numpy(np.random.default_rng(f).random((v.rows, f)) > 0.5).to(dev())
            x = v.panel[:, :f].contiguous()
            got = P.gcn_layer(x, v.gr, torch.eye(f, device=dev()), v.bias[:f], relu=True, precision="fp32",
                              dropout_mask=keep, dropout_p=0.5, association="reference")
            assert torch.equal(got, torch.relu(ref + v.bias[:f]) * keep * 2.0), what + " mask"


# ------------------------------------------------------------------ non-finite panel values
def _poison(a64):
    """Panel rows to poison for the product a64 @ B: +Inf in row 0 and in a row p that shares an output row with
    another row k, -Inf in k, NaN in a row that exactly one output row references."""
    a = a64.tocsr()
    pattern = sp.csr_matrix((np.ones(a.nnz), a.indices.copy(), a.indptr.copy()), shape=a.shape)
    pattern.sum_duplicates()  # (in place: not on a64's own index arrays)
    users = np.asarray((pattern > 0).sum(axis=0)).ravel()  # output rows referencing each panel row
    p = k = None
    for i in range(a.shape[0]):
        cols = np.unique(a.indices[a.indptr[i]:a.indptr[i + 1]])
        if len(cols) >= 2:
            p, k = (0, cols[cols != 0][0]) if 0 in cols else (cols[0], cols[1])
            break
    once = [c for c in np.nonzero(users == 1)[0] if c not in (0, p, k)]
    return p, k, (once[0] if once else None)


_CACHE = {}


def _poisoned(v, f):
    """(panel fp64 with +-Inf / NaN rows, the fp32 product) of view v at width f, computed once."""
    key = ("poison", v.name, f)
    if key not in _CACHE:
        p, k, once = _poison(v.a64)
        b = v.b64[:, :f].copy()
        b[0] = np.inf
        if p is not None:
            b[p] = np.inf
            b[k] = -np.inf
        if once is not None:
            b[once] = np.nan
        with np.errstate(invalid="ignore"):
            want = torch.from_numpy((v.a64 @ b).astype(np.float32)).to(dev())
        assert bool(torch.isnan(want).any()) or once is None
        _CACHE[key] = (torch.from_numpy(b.astype(np.float32)).to(dev()), want)
    return _CACHE[key]


@pytest.mark.parametrize("spmm_kernel", KERNELS, indirect=True, ids=_kid)
@pytest.mark.parametrize("dtype,f", [("fp32", 3), ("fp32", 8), ("fp32", 33), ("fp32", 64), ("fp32", 129), ("fp32", 513),
                                     ("bf16", 64), ("bf16", 129)])
def test_non_finite_panel_values_propagate_as_in_the_product(P, views, spmm_kernel, dtype, f):
    """+Inf in panel row 0, -Inf in a row sharing an output row with a +Inf row, NaN in a row one output row reads:
    the output has exactly the fp64 product's Inf / NaN pattern and its finite values.  A kernel that multiplies a
    padding entry (value 0) by a gathered row puts NaN where the product has none."""
    tdt = torch.bfloat16 if dtype == "bf16" else torch.float32
    for v in views:
        if v.a64.nnz == 0:
            continue
        b, want = _poisoned(v, f)
        panel = _panel(b, f, tdt)
        o = Sentinel(v.rows, f)
        _spmm(P, v, panel, f, o.out)
        torch.testing.assert_close(o.out, want, rtol=0, atol=0, equal_nan=True,
                                   msg=lambda m: "%s f=%d %s %s: %s" % (v.name, f, dtype, spmm_kernel, m))


# ------------------------------------------------------------------ real values: per-entry worst-case bound
@pytest.mark.parametrize("spmm_kernel", KERNELS, indirect=True, ids=_kid)
@pytest.mark.parametrize("dtype,f", [("fp32", 17), ("fp32", 257), ("bf16", 65)])
def test_real_values_within_the_per_entry_summation_bound(P, views, spmm_kernel, dtype, f):
    """Normal values and panel: |got - ref64| <= (len_i + 2) * 2^-24 * (|A| |B|)_ij on every entry, ref64 the fp64
    product (of the bf16-rounded panel for bf16).  The full handles' structures, each direction as a forward view."""
    tdt = torch.bfloat16 if dtype == "bf16" else torch.float32
    for v in views:
        if not v.name.startswith(("rect", "square", "single")):
            continue
        key = ("real", v.name, f, dtype)
        if key not in _CACHE:
            rs = np.random.default_rng(f + v.rows)
            a = v.a64.copy()
            a.data = rs.standard_normal(a.nnz).astype(np.float32).astype(np.float64)
            fv = View.__new__(View)
            fv.gr, fv.flags = _graph(P, a), 0
            b32 = torch.from_numpy(rs.standard_normal((v.k, f)).astype(np.float32)).to(dev())
            b64 = b32.to(tdt).double().cpu().numpy()
            # (|A| by hand: scipy's abs() first merges duplicate entries in place, which would give |a + a'|)
            abs_a = sp.csr_matrix((np.abs(a.data), a.indices.copy(), a.indptr.copy()), shape=a.shape)
            bound = (np.diff(a.indptr)[:, None] + 2) * 2.0 ** -24 * (abs_a @ np.abs(b64))
            _CACHE[key] = (fv, _panel(b32, f, tdt), a @ b64, bound)
        fv, panel, ref, bound = _CACHE[key]
        out = torch.empty(v.rows, f, device=dev())
        _spmm(P, fv, panel, f, out)
        err = np.abs(out.cpu().numpy().astype(np.float64) - ref)
        assert (err <= bound).all(), (v.name, f, dtype, spmm_kernel, float((err - bound).max()))


# ------------------------------------------------------------------ dense route
def test_dense_route_tensor_core_and_simt_panels_exact(P):
    """A 16384^2 dense handle (12.5 % dense, exact values), f = 300: column panels of 256 and 44 on the tcgen05 tn
    kernel; f = 260: the 4-column tail on the SIMT kernel.  Forward and transposed, with and without bias + ReLU,
    equal to the fp64 product, nothing written outside the output."""
    from pygcn_b200 import _lib

    n = 16384
    gen = torch.Generator(device=dev()).manual_seed(5)
    vals = torch.from_numpy(VALUES).to(dev())
    a = vals[torch.randint(0, len(VALUES), (n, n), generator=gen, device=dev())]
    a *= torch.rand(n, n, generator=gen, device=dev()) < 0.125
    gr = P.Graph.from_torch(a)
    assert gr.dense_route
    a64 = a.double()
    del a
    for f in (300, 260):
        b = torch.randint(-8, 9, (n, f), generator=gen, device=dev()).float()
        bias = torch.randint(-8, 9, (f,), generator=gen, device=dev()).float()
        panel = _panel(b, f, torch.float32)
        for transpose in (False, True):
            ref = ((a64.t() if transpose else a64) @ b.double()).float()
            v = View.__new__(View)
            v.gr, v.flags = gr, 1 if transpose else 0
            for flags, bb, want in ((0, None, ref), (_lib.SPMM_RELU, bias, torch.relu(ref + bias))):
                o = Sentinel(n, f)
                _spmm(P, v, panel, f, o.out, flags, bb)
                o.check(want, "dense f=%d transpose=%s flags=%d" % (f, transpose, flags))


# ------------------------------------------------------------------ column ids at the tag boundary, offsets past 2^32
@pytest.fixture(scope="module")
def wide_graphs(P):
    """4-row CSRs with 2^27 columns (tagged pairs, column 2^27 - 1 present) and 2^27 + 3 (untagged: columns keep bit
    27), no empty row; odd nnz, odd row starts."""
    out = []
    for n_cols in (1 << 27, (1 << 27) + 3):
        cols = [[n_cols - 1, 0, (1 << 26) + 5, (1 << 27) - 1, 12345], [n_cols - 2], [(1 << 27) - 1, 7, n_cols - 1],
                [3 << 25, n_cols - 3]]
        lengths = [len(c) for c in cols]
        c = np.array(sum(cols, []), np.int64)
        vals = np.random.default_rng(n_cols).choice(VALUES, len(c))
        a = _csr(lengths, n_cols, c, vals)
        out.append((a, _graph(P, a)))
    return out


@pytest.mark.parametrize("spmm_kernel", ["auto", "rows", "tma", "group", ("stream", 0)], indirect=True, ids=_kid)
def test_columns_at_the_tag_boundary_and_panel_offsets_past_4gb(P, wide_graphs, spmm_kernel):
    """f = 8 fp32: a forward panel of 2^27 rows is 4 GiB, so gathered byte offsets pass 2^32; every row the CSR does
    not reference is NaN.  Transposed: 2^27 output rows, all but a few of them empty and written as zeros."""
    f = 8
    rs = np.random.default_rng(8)
    for a, gr in wide_graphs:
        used = np.unique(a.indices)
        rows = rs.integers(-8, 9, (len(used), f)).astype(np.float32)
        panel = torch.full((a.shape[1], f), float("nan"), device=dev())
        panel[torch.from_numpy(used).to(dev())] = torch.from_numpy(rows).to(dev())
        local = sp.csr_matrix((a.data, np.searchsorted(used, a.indices), a.indptr), shape=(a.shape[0], len(used)))
        fv = View.__new__(View)
        fv.gr, fv.flags = gr, 0
        o = Sentinel(a.shape[0], f)
        _spmm(P, fv, panel, f, o.out)
        o.check(torch.from_numpy((local @ rows.astype(np.float64)).astype(np.float32)).to(dev()), "forward n_cols=%d" % a.shape[1])
        del panel
        pt = rs.integers(-8, 9, (a.shape[0], f)).astype(np.float32)
        want = (local.T @ pt.astype(np.float64)).astype(np.float32)
        out = torch.full((a.shape[1], f), float("nan"), device=dev())
        fv.flags = 1
        _spmm(P, fv, torch.from_numpy(pt).to(dev()), f, out)
        idx = torch.from_numpy(used).to(dev())
        assert torch.equal(out[idx], torch.from_numpy(want).to(dev())), "transposed n_cols=%d" % a.shape[1]
        out[idx] = 0
        assert not bool(out.ne(0).any()), "transposed n_cols=%d: an unreferenced column is not 0" % a.shape[1]
        del out

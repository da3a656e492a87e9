"""The fp64 tier (graph handles with fp64 values, fp64 SpMM, DMMA products, fp64 column sums, the fp64 layer).

Exact cases: panel and weight entries are dyadic (integers below 2^20 times 2^-30, or small integers), stored values
are in {+-1/4, +-1/2, +-1, +-2}.  Every case asserts that (|A||B|)_ij stays far below 2^53 quanta of its grid, so every
partial sum is exact in any order and the CPU fp64 product is the only correct answer: the check is torch.equal.
Each exact case also fills panel padding with NaN, surrounds the output with a sentinel that must come back bit for
bit, gives the workspace a guard that must stay unchanged (and checks that one byte less is refused), and runs twice
with bit-identical results.
"""
import ctypes

import numpy as np
import pytest
import scipy.sparse as sp
import torch

pytestmark = pytest.mark.gpu

F64 = torch.float64
VALUES = np.array([-2, -1, -0.5, -0.25, 0.25, 0.5, 1, 2], np.float64)
SENTINEL = -12345.0
GUARD = 256
Q = 2.0 ** -30  # quantum of the dyadic panels


def dev():
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def P():
    import pygcn_b200

    assert pygcn_b200._lib.load().gcnb_check_device() == 0, pygcn_b200._lib.last_error()
    return pygcn_b200


def lib():
    from pygcn_b200 import _lib

    return _lib.load()


def check(st, what):
    from pygcn_b200 import _lib

    _lib.check(st, what)


def stream():
    return torch.cuda.current_stream().cuda_stream


def dyadic(rng, shape):
    return rng.integers(-(1 << 20), 1 << 20, size=shape).astype(np.float64) * Q


def assert_exact_bound(a_abs_b_abs, quantum):
    assert float(np.max(a_abs_b_abs, initial=0.0)) / quantum < 2.0 ** 50


# ------------------------------------------------------------------------------------------- structures
def csr_from_lengths(rng, lengths, n_cols):
    rows, cols = [], []
    for r, d in enumerate(lengths):
        rows += [r] * d
        cols += list(rng.integers(0, n_cols, size=d)) if n_cols > 0 else []
    vals = VALUES[rng.integers(0, len(VALUES), size=len(rows))]
    m = sp.coo_matrix((vals, (np.array(rows, np.int64), np.array(cols, np.int64))), shape=(len(lengths), n_cols))
    m = m.tocsr()
    m.sum_duplicates()
    m.sort_indices()
    return m


EDGE_LENGTHS = [0, 1, 2, 7, 8, 9, 15, 16, 17, 31, 32, 33, 63, 64, 65, 1023, 1024, 1025, 2047, 2048, 2049, 3073]


def structures(rng):
    s = {}
    s["bin_edges"] = csr_from_lengths(rng, EDGE_LENGTHS * 2, 4000)
    s["empty_runs"] = csr_from_lengths(rng, [0] * 50 + [3, 0, 0, 1030] + [0] * 40 + [5] * 7 + [0] * 33, 300)
    s["nnz0"] = sp.csr_matrix((17, 9), dtype=np.float64)
    s["one_row"] = csr_from_lengths(rng, [1500], 2000)
    s["rect_wide"] = csr_from_lengths(rng, list(rng.integers(0, 40, size=300)), 70)  # hub columns in A^T: long rows
    s["rect_tall"] = csr_from_lengths(rng, list(rng.integers(0, 5, size=900)) + [1100], 5000)
    return s


def graph_of(P, m):
    t = torch.sparse_csr_tensor(torch.from_numpy(m.indptr.astype(np.int64)), torch.from_numpy(m.indices.astype(np.int64)),
                                torch.from_numpy(m.data.astype(np.float64)), size=m.shape, dtype=F64).to(dev())
    g = P.Graph.from_torch(t)
    assert g.dtype == F64
    return g


def guarded_ws(nbytes):
    buf = torch.empty(nbytes + GUARD, dtype=torch.uint8, device=dev())
    buf[nbytes:] = 0xA5
    return buf


def guard_ok(buf, nbytes):
    return bool((buf[nbytes:] == 0xA5).all())


def panel(rng, rows, f, ld):
    b = torch.full((max(rows, 1), ld), float("nan"), dtype=F64, device=dev())
    vals = dyadic(rng, (rows, f))
    b[:rows, :f] = torch.from_numpy(vals).to(dev())
    return b, vals


def run_spmm(P, g, flags, b, ldb, f, bias=None, mask=None, ld_mask=0, scale=1.0, out=None, ldo=None):
    """gcnb_spmm_f64 into a sentinel-framed output; returns (interior, whole frame, ws ok)."""
    L = lib()
    rows = g.n_cols if flags & 1 else g.n_rows
    ldo = ldo or f + 3
    if out is None:
        out = torch.full((rows + 2, ldo), SENTINEL, dtype=F64, device=dev())
    need = int(L.gcnb_spmm_f64_workspace_bytes(g._h, flags & 1, f))
    ws = guarded_ws(need)
    optr = out.data_ptr() + ldo * 8
    if need > 0:
        assert L.gcnb_spmm_f64(g._h, flags, b.data_ptr(), ldb, f, None if bias is None else bias.data_ptr(),
                               None if mask is None else mask.data_ptr(), ld_mask, scale, optr, ldo, ws.data_ptr(),
                               need - 1, stream()) != 0
    check(L.gcnb_spmm_f64(g._h, flags, b.data_ptr(), ldb, f, None if bias is None else bias.data_ptr(),
                          None if mask is None else mask.data_ptr(), ld_mask, scale, optr, ldo, ws.data_ptr(), need,
                          stream()), "gcnb_spmm_f64")
    torch.cuda.synchronize()
    assert guard_ok(ws, need)
    return out, ldo


def frame_ok(out, rows, f):
    o = out.clone()
    o[1:rows + 1, :f] = SENTINEL
    return bool((o == SENTINEL).all())


# ------------------------------------------------------------------------------------------- SpMM
WIDTHS = [1, 2, 3, 7, 8, 9, 15, 16, 17, 31, 32, 33, 63, 64, 65, 67, 128, 129, 257]


@pytest.mark.parametrize("name", ["bin_edges", "empty_runs", "nnz0", "one_row", "rect_wide", "rect_tall"])
@pytest.mark.parametrize("transpose", [0, 1])
def test_spmm_exact_on_edge_structures(P, name, transpose):
    rng = np.random.default_rng(7)
    m = structures(rng)[name]
    g = graph_of(P, m)
    a = m.T.tocsr() if transpose else m
    for f in WIDTHS:
        for ld in sorted({f, f + (f % 2), f + 2}):  # odd ld: 8-byte path; even: 16-byte path
            b, bv = panel(rng, a.shape[1], f, ld)
            ref = a @ bv
            assert_exact_bound(abs(a) @ np.abs(bv), Q / 4)
            outs = []
            for _ in range(2):
                out, ldo = run_spmm(P, g, transpose, b, ld, f)
                assert frame_ok(out, a.shape[0], f), (name, f, ld)
                outs.append(out)
            got = outs[0][1:a.shape[0] + 1, :f].cpu()
            assert torch.equal(got, torch.from_numpy(ref)), (name, transpose, f, ld)
            assert torch.equal(outs[0], outs[1])


@pytest.mark.parametrize("f", [5, 16, 33, 130])
def test_spmm_epilogues_exact(P, f):
    """bias, ReLU, keep-mask x 2 and accumulate into a strided output, each exact."""
    rng = np.random.default_rng(f)
    m = structures(rng)["empty_runs"]
    g = graph_of(P, m)
    b, bv = panel(rng, m.shape[1], f, f + 1)
    bias_np = dyadic(rng, f)
    bias = torch.from_numpy(bias_np).to(dev())
    mask_np = (rng.random((m.shape[0], f + 3)) < 0.5).astype(np.uint8)
    mask = torch.from_numpy(mask_np).to(dev())
    base = m @ bv
    # bias + relu + mask * 2
    out, ldo = run_spmm(P, g, 2, b, f + 1, f, bias=bias, mask=mask, ld_mask=f + 3, scale=2.0)
    ref = np.where(mask_np[:, :f] != 0, np.maximum(base + bias_np, 0.0) * 2.0, 0.0)
    assert frame_ok(out, m.shape[0], f) and torch.equal(out[1:-1, :f].cpu(), torch.from_numpy(ref))
    # accumulate into a strided output that already holds values
    ldo = f + 5
    prev = dyadic(rng, (m.shape[0], f))
    frame = torch.full((m.shape[0] + 2, ldo), SENTINEL, dtype=F64, device=dev())
    frame[1:-1, :f] = torch.from_numpy(prev).to(dev())
    out, _ = run_spmm(P, g, 4, b, f + 1, f, out=frame, ldo=ldo)
    assert frame_ok(out, m.shape[0], f) and torch.equal(out[1:-1, :f].cpu(), torch.from_numpy(prev + base))


def test_spmm_refuses_fp32_handles(P):
    from pygcn_b200 import _lib

    t = torch.eye(4, device=dev()).to_sparse()
    g = P.Graph.from_torch(t)
    b = torch.zeros(4, 2, dtype=F64, device=dev())
    o = torch.zeros(4, 2, dtype=F64, device=dev())
    st = lib().gcnb_spmm_f64(g._h, 0, b.data_ptr(), 2, 2, None, None, 0, 1.0, o.data_ptr(), 2, None, 0, stream())
    assert st == 1 and "no fp64 values" in _lib.last_error()
    rp = torch.empty(5, dtype=torch.int32, device=dev())
    assert lib().gcnb_graph_export_csr_f64(g._h, 0, rp.data_ptr(), None, None, stream()) == 4


# ------------------------------------------------------------------------------------------- DMMA products
def run_gemm(m, n, k, a, a_rs, a_cs, b, b_rs, b_cs, ldc, bias=None, relu=False):
    L = lib()
    c = torch.full((m + 2, ldc), SENTINEL, dtype=F64, device=dev())
    need = int(L.gcnb_gemm_f64_workspace_bytes(m, n, k))
    ws = guarded_ws(need)
    cp = c.data_ptr() + ldc * 8
    args = (m, n, k, a.data_ptr(), a_rs, a_cs, b.data_ptr(), b_rs, b_cs, cp, ldc)
    if need > 0:
        assert L.gcnb_gemm_f64(*args, ws.data_ptr(), need - 1, stream()) != 0
    if bias is None and not relu:
        check(L.gcnb_gemm_f64(*args, ws.data_ptr(), need, stream()), "gemm_f64")
    else:
        check(L.gcnb_gemm_f64_ex(*args, None if bias is None else bias.data_ptr(), int(relu), ws.data_ptr(), need,
                                 stream()), "gemm_f64_ex")
    torch.cuda.synchronize()
    assert guard_ok(ws, need)
    return c


GEMM_SHAPES = [(1, 1, 1), (63, 31, 15), (64, 32, 16), (65, 33, 17), (64, 64, 0), (200, 65, 513), (130, 130, 64),
               (47, 20, 5000), (602, 256, 3000), (16, 31, 20000), (3, 129, 257)]


@pytest.mark.parametrize("m,n,k", GEMM_SHAPES)
@pytest.mark.parametrize("pattern", ["xw", "xt_ds", "ds_wt"])
def test_dmma_product_exact(P, m, n, k, pattern):
    rng = np.random.default_rng(m * 7 + n * 3 + k)
    A = dyadic(rng, (m, k))
    B = rng.integers(-8, 9, size=(k, n)).astype(np.float64)
    assert_exact_bound(np.abs(A) @ np.abs(B), Q)
    ref = A @ B
    pad = 3
    if pattern == "xw":      # A row-major [m, k] with ld k + pad, B row-major
        ta = torch.full((m, k + pad), float("nan"), dtype=F64, device=dev()); ta[:, :k] = torch.from_numpy(A)
        tb = torch.from_numpy(B).to(dev()).contiguous()
        a_st, b_st = (k + pad, 1), (n, 1)
    elif pattern == "xt_ds":  # A = X^T, X [k, m] with ld m + pad; B row-major
        ta = torch.full((k, m + pad), float("nan"), dtype=F64, device=dev()); ta[:, :m] = torch.from_numpy(A.T)
        tb = torch.from_numpy(B).to(dev()).contiguous()
        a_st, b_st = (1, m + pad), (n, 1)
    else:                     # B = W^T, W [n, k] contiguous
        ta = torch.from_numpy(A).to(dev()).contiguous()
        tb = torch.from_numpy(np.ascontiguousarray(B.T)).to(dev())
        a_st, b_st = (k, 1), (1, k)
    ta = ta if ta.numel() else torch.zeros(1, dtype=F64, device=dev())
    tb = tb if tb.numel() else torch.zeros(1, dtype=F64, device=dev())
    ldc = n + 2
    c1 = run_gemm(m, n, k, ta, *a_st, tb, *b_st, ldc)
    c2 = run_gemm(m, n, k, ta, *a_st, tb, *b_st, ldc)
    assert frame_ok(c1, m, n) and torch.equal(c1, c2)
    assert torch.equal(c1[1:-1, :n].cpu(), torch.from_numpy(ref)), (m, n, k, pattern)
    bias_np = dyadic(rng, n)
    c = run_gemm(m, n, k, ta, *a_st, tb, *b_st, ldc, bias=torch.from_numpy(bias_np).to(dev()), relu=True)
    assert frame_ok(c, m, n) and torch.equal(c[1:-1, :n].cpu(), torch.from_numpy(np.maximum(ref + bias_np, 0.0)))


def test_dmma_runs_only_in_the_fp64_product_kernel():
    import subprocess
    from pygcn_b200 import _lib

    sass = subprocess.run(["cuobjdump", "-sass", _lib.LIB_PATH], capture_output=True, text=True).stdout
    funcs = sass.split("Function : ")
    dmma = [f.split("\n", 1)[0] for f in funcs if "DMMA" in f]
    assert dmma and all("gemm_f64_dmma_kernel" in name for name in dmma), dmma


# ------------------------------------------------------------------------------------------- column sums
@pytest.mark.parametrize("n_rows,f", [(1, 1), (300, 7), (70001, 33), (257, 64)])
def test_colsum_exact_with_signed_zero_mask(P, n_rows, f):
    L = lib()
    rng = np.random.default_rng(n_rows + f)
    gv = dyadic(rng, (n_rows, f))
    yv = rng.integers(-1, 2, size=(n_rows, f)).astype(np.float64)
    yv[rng.random((n_rows, f)) < 0.3] = -0.0
    ld = f + 1
    g = torch.full((n_rows, ld), float("nan"), dtype=F64, device=dev()); g[:, :f] = torch.from_numpy(gv)
    y = torch.from_numpy(yv).to(dev())
    ldgm = f + (f % 2)
    gm = torch.full((n_rows + 2, ldgm), SENTINEL, dtype=F64, device=dev())
    out = torch.full((f + 2,), SENTINEL, dtype=F64, device=dev())
    need = int(L.gcnb_colsum_f64_workspace_bytes(n_rows, f))
    ws = guarded_ws(need)
    args = (n_rows, f, g.data_ptr(), ld, y.data_ptr(), f, gm.data_ptr() + ldgm * 8, ldgm, out.data_ptr() + 8)
    assert L.gcnb_colsum_f64(*args, ws.data_ptr(), need - 1, stream()) != 0
    check(L.gcnb_colsum_f64(*args, ws.data_ptr(), need, stream()), "colsum_f64")
    torch.cuda.synchronize()
    masked = np.where(yv > 0, gv, 0.0)
    assert guard_ok(ws, need)
    assert torch.equal(out[1:-1].cpu(), torch.from_numpy(masked.sum(0)))
    assert out[0].item() == SENTINEL and out[-1].item() == SENTINEL
    assert torch.equal(gm[1:-1, :f].cpu(), torch.from_numpy(masked)) and frame_ok(gm, n_rows, f)


# ------------------------------------------------------------------------------------------- the layer
def layer_case(P, rng, n=600, fin=5, fout=9):
    m = csr_from_lengths(rng, list(rng.integers(0, 12, size=n - 2)) + [1200, 0], n)
    g = graph_of(P, m)
    x = dyadic(rng, (n, fin))
    w = rng.integers(-4, 5, size=(fin, fout)).astype(np.float64)
    b = dyadic(rng, fout)
    G = rng.integers(-8, 9, size=(n, fout)).astype(np.float64)
    return m, g, x, w, b, G


@pytest.mark.parametrize("assoc", ["reference", "aggregate_first"])
@pytest.mark.parametrize("relu", [False, True])
@pytest.mark.parametrize("dropout", [False, True])
@pytest.mark.parametrize("need_dx", [False, True])
def test_layer_exact(P, assoc, relu, dropout, need_dx):
    rng = np.random.default_rng(11)
    m, g, x, w, b, G = layer_case(P, rng, fin=6, fout=9)
    mask_np = (rng.random((m.shape[0], w.shape[1])) < 0.5) if dropout else None
    pre = m @ (x @ w) + b
    assert_exact_bound(abs(m) @ (np.abs(x) @ np.abs(w)) + np.abs(b), Q / 4)
    y = np.maximum(pre, 0.0) if relu else pre
    if dropout:
        y = np.where(mask_np, y * 2.0, 0.0)
    gg = G * (pre > 0) if relu else G
    if dropout:
        gg = np.where(mask_np, gg * 2.0, 0.0)
    results = []
    for _ in range(2):
        xt = torch.from_numpy(x).to(dev()).requires_grad_(need_dx)
        wt = torch.from_numpy(w).to(dev()).requires_grad_()
        bt = torch.from_numpy(b).to(dev()).requires_grad_()
        mk = torch.from_numpy(mask_np).to(dev()) if dropout else None
        out = P.gcn_layer(xt, g, wt, bt, relu=relu, dropout_mask=mk, dropout_p=0.5 if dropout else 0.0, association=assoc)
        out.backward(torch.from_numpy(G).to(dev()))
        results.append((out.detach(), wt.grad, bt.grad, xt.grad))
    out, dw, db, dx = results[0]
    assert torch.equal(out.cpu(), torch.from_numpy(y))
    assert torch.equal(db.cpu(), torch.from_numpy(gg.sum(0)))
    ds = m.T @ gg
    assert torch.equal(dw.cpu(), torch.from_numpy(x.T @ ds))
    if need_dx:
        assert torch.equal(dx.cpu(), torch.from_numpy(ds @ w.T))
    else:
        assert dx is None
    for a, c in zip(results[0], results[1]):
        assert (a is None and c is None) or torch.equal(a, c)


def test_layer_real_valued_bound(P):
    """|ours - ref| <= (len + 2) 2^-53 (|A||B|)_ij on every entry, ref in long double (len = the length of the sum): X W,
    the forward and the transposed SpMM, and the backward products dW = X^T dS (split K) and dX = dS W^T."""
    rng = np.random.default_rng(3)
    n, fin, fout = 3000, 40, 24
    m = csr_from_lengths(rng, list(rng.integers(0, 30, size=n - 1)) + [2500], n)
    m.data = rng.standard_normal(m.nnz)
    g = graph_of(P, m)
    x = rng.standard_normal((n, fin))
    w = rng.standard_normal((fin, fout))
    xw = torch.from_numpy(x).to(dev()) @ torch.from_numpy(w).to(dev())  # any fp64 panel
    xw_ours = P.mm(torch.from_numpy(x).to(dev()), torch.from_numpy(w).to(dev())).cpu().numpy()
    ref_xw = np.einsum("ik,kj->ij", x.astype(np.longdouble), w.astype(np.longdouble))
    bound = (fin + 2) * 2.0 ** -53 * (np.abs(x) @ np.abs(w))
    assert np.all(np.abs(xw_ours - ref_xw) <= bound)
    out = P.spmm(g, xw).cpu().numpy()
    s = xw.cpu().numpy()
    prod = m.data.astype(np.longdouble)[:, None] * s[m.indices].astype(np.longdouble)
    lens = np.diff(m.indptr)
    ref = np.zeros((n, fout), np.longdouble)
    nz = lens > 0
    ref[nz] = np.add.reduceat(prod, m.indptr[:-1][nz], axis=0)
    bound = (lens[:, None] + 2) * 2.0 ** -53 * (abs(m) @ np.abs(s))
    assert np.all(np.abs(out - ref) <= bound)
    # transposed SpMM (the backward of spmm): dS = A^T G
    G = rng.standard_normal((n, fout))
    gt = torch.from_numpy(G).to(dev())
    st = torch.from_numpy(s).to(dev()).requires_grad_()
    (ds,) = torch.autograd.grad(P.spmm(g, st), (st,), gt)
    ds = ds.cpu().numpy()
    mt = m.T.tocsr()
    prod = mt.data.astype(np.longdouble)[:, None] * G[mt.indices].astype(np.longdouble)
    lens = np.diff(mt.indptr)
    ref = np.zeros((n, fout), np.longdouble)
    nz = lens > 0
    ref[nz] = np.add.reduceat(prod, mt.indptr[:-1][nz], axis=0)
    bound = (lens[:, None] + 2) * 2.0 ** -53 * (abs(mt) @ np.abs(G))
    assert np.all(np.abs(ds - ref) <= bound)
    # dW = X^T dS over all n rows (split K) and dX = dS W^T
    dst = torch.from_numpy(ds).to(dev())
    xt = torch.from_numpy(x).to(dev())
    dw = P.mm(xt.t(), dst).cpu().numpy()
    ref = np.einsum("ki,kj->ij", x.astype(np.longdouble), ds.astype(np.longdouble))
    assert np.all(np.abs(dw - ref) <= (n + 2) * 2.0 ** -53 * (np.abs(x).T @ np.abs(ds)))
    dx = P.mm(dst, torch.from_numpy(w).to(dev()).t()).cpu().numpy()
    ref = np.einsum("ik,jk->ij", ds.astype(np.longdouble), w.astype(np.longdouble))
    assert np.all(np.abs(dx - ref) <= (fout + 2) * 2.0 ** -53 * (np.abs(ds) @ np.abs(w).T))


# ------------------------------------------------------------------------------------------- gradcheck
def small_graph(P, rng, n=30, long_row=False):
    lengths = list(rng.integers(0, 5, size=n))
    lengths[3] = 0
    lengths[4] = 0
    if long_row:
        lengths[7] = 2000  # > 1024 distinct columns once duplicates are summed
    m = csr_from_lengths(rng, lengths, n)
    m.data = rng.uniform(0.1, 1.0, m.nnz) * np.sign(m.data)
    return m, graph_of(P, m)


def away_from_kink(P, g, x, w, b, assoc):
    with torch.no_grad():
        pre = P.gcn_layer(x, g, w, b, association=assoc)
    return float(pre.abs().min()) > 1e-4


@pytest.mark.parametrize("assoc", ["reference", "aggregate_first"])
@pytest.mark.parametrize("bias", [False, True])
@pytest.mark.parametrize("relu", [False, True])
def test_gradcheck_layer(P, assoc, bias, relu):
    for seed in range(20):
        rng = np.random.default_rng(seed)
        m, g = small_graph(P, rng)
        x = torch.from_numpy(rng.standard_normal((30, 4))).to(dev()).requires_grad_()
        w = torch.from_numpy(rng.standard_normal((4, 6))).to(dev()).requires_grad_()
        b = torch.from_numpy(rng.standard_normal(6)).to(dev()).requires_grad_() if bias else None
        if not relu or away_from_kink(P, g, x, w, b, assoc):
            break
    assert torch.autograd.gradcheck(lambda x, w, *b: P.gcn_layer(x, g, w, b[0] if b else None, relu=relu, association=assoc),
                                    (x, w) + ((b,) if bias else ()))


def test_gradcheck_dropout_batched_dense_long_spmm_module(P):
    rng = np.random.default_rng(5)
    m, g = small_graph(P, rng)
    x = torch.from_numpy(rng.standard_normal((30, 3))).to(dev()).requires_grad_()
    w = torch.from_numpy(rng.standard_normal((3, 4))).to(dev()).requires_grad_()
    b = torch.from_numpy(rng.standard_normal(4)).to(dev()).requires_grad_()
    mask = torch.from_numpy(rng.random((30, 4)) < 0.6).to(dev())
    assert torch.autograd.gradcheck(lambda x, w, b: P.gcn_layer(x, g, w, b, dropout_mask=mask, dropout_p=0.4), (x, w, b))
    xb = torch.from_numpy(rng.standard_normal((3, 30, 3))).to(dev()).requires_grad_()
    assert torch.autograd.gradcheck(lambda x, w, b: P.gcn_layer(x, g, w, b), (xb, w, b))
    dense = torch.from_numpy(m.toarray()).to(dev())
    assert torch.autograd.gradcheck(lambda x, w, b: P.gcn_layer(x, dense, w, b), (x, w, b))
    ml, gl = small_graph(P, rng, n=3000, long_row=True)
    assert gl.n_long_chunks > 0 and gl.bin_rows[0] > 0
    xl = torch.from_numpy(rng.standard_normal((3000, 2))).to(dev()).requires_grad_()
    wl = torch.from_numpy(rng.standard_normal((2, 3))).to(dev()).requires_grad_()
    assert torch.autograd.gradcheck(lambda x, w: P.gcn_layer(x, gl, w, None), (xl, wl))
    assert torch.autograd.gradcheck(lambda d: P.spmm(g, d), (x,))
    torch.manual_seed(0)
    layer = P.GraphConvolution(3, 4, dropout=0.3).double().to(dev())
    out = layer(x, g)  # training mode: the fused dropout runs in fp64 too
    assert out.dtype == F64 and layer.weight.dtype == F64
    out.sum().backward()
    assert layer.weight.grad.dtype == F64
    layer.eval()
    assert torch.autograd.gradcheck(lambda x: layer(x, g), (x,))


# ------------------------------------------------------------------------------------------- graph build
def test_from_edges_f64_bit_exact(P, golden):
    from oracle import gcn_oracle as O

    cases = []
    gd = golden("cora_pipeline.npz")
    cases.append((gd["edges"][:, 0], gd["edges"][:, 1], int(gd["n"])))
    gen = torch.Generator().manual_seed(1)
    import bench

    s, d = bench.rmat_edges(torch, 1 << 14, 200000, gen, "cpu")
    cases.append((s.numpy(), d.numpy(), 1 << 14))
    for src, dst, n in cases:
        r, c, v = O.edges_to_counts(src, dst, n)
        r, c, v = O.symmetrize_max(r, c, v, n)
        r, c, v = O.add_identity(r, c, v, n)
        r, c, v64 = O.normalize_rows(r, c, v, n)
        ts, td = torch.from_numpy(np.asarray(src, np.int32)).to(dev()), torch.from_numpy(np.asarray(dst, np.int32)).to(dev())
        g64 = P.Graph.from_edges(ts, td, n, dtype=F64)
        g32 = P.Graph.from_edges(ts, td, n)
        rp, col, val = (t.cpu().numpy() for t in g64.csr())
        assert val.dtype == np.float64 and np.array_equal(val.view(np.uint64), v64.view(np.uint64))
        assert np.array_equal(col, c)
        rp32, col32, val32 = (t.cpu().numpy() for t in g32.csr())
        assert np.array_equal(rp, rp32) and np.array_equal(col, col32)
        coo = g64.to_sparse_coo()
        assert coo._values().dtype == F64
        # the fp32 values of the fp64 handle are today's fp32 build
        info_val = torch.empty(g64.nnz, dtype=torch.float32, device=dev())
        rpt = torch.empty(n + 1, dtype=torch.int32, device=dev())
        colt = torch.empty(g64.nnz, dtype=torch.int32, device=dev())
        check(lib().gcnb_graph_export_csr(g64._h, 1, rpt.data_ptr(), colt.data_ptr(), info_val.data_ptr(), stream()), "x")
        t32 = g32.csr(transpose=True)
        assert torch.equal(rpt, t32[0]) and torch.equal(colt, t32[1])
        assert torch.equal(info_val.view(torch.int32), t32[2].view(torch.int32))
        assert np.array_equal(val32.view(np.uint32), v64.astype(np.float32).view(np.uint32))
        t64 = g64.csr(transpose=True)
        assert torch.equal(t64[2].float().view(torch.int32), t32[2].view(torch.int32))


def test_from_coo_f64_keeps_order_and_duplicates(P):
    rng = np.random.default_rng(2)
    nnz = 5000
    row = rng.integers(0, 300, nnz)
    col = rng.integers(0, 200, nnz)
    row[:50], col[:50] = 7, 9  # duplicates
    val = rng.standard_normal(nnz)
    t = torch.sparse_coo_tensor(torch.from_numpy(np.vstack([row, col])), torch.from_numpy(val), (300, 200)).to(dev())
    g = P.Graph.from_torch(t)
    order = np.lexsort((col, row))  # stable (row, col) order
    rp, c, v = (x.cpu().numpy() for x in g.csr())
    assert g.nnz == nnz and np.array_equal(c, col[order]) and np.array_equal(v.view(np.uint64), val[order].view(np.uint64))
    assert np.array_equal(rp, np.searchsorted(row[order], np.arange(301)))
    assert not g.dense_route
    dense = torch.from_numpy(rng.standard_normal((80, 80))).to(dev())  # fully dense: still CSR
    gd = P.Graph.from_torch(dense)
    assert not gd.dense_route and gd.nnz == 6400 and gd.dtype == F64


# ------------------------------------------------------------------------------------------- memory, graphs, routing
def test_cuda_graph_replay_bit_identical(P):
    rng = np.random.default_rng(9)
    m, g, x, w, b, G = layer_case(P, rng, fin=7, fout=12)
    gt = torch.from_numpy(G).to(dev())

    def leaves():
        return [torch.from_numpy(v).to(dev()).requires_grad_() for v in (x, w, b)]

    def step(xt, wt, bt):
        out = P.gcn_layer(xt, g, wt, bt, relu=True)
        dx, dw, db = torch.autograd.grad(out, (xt, wt, bt), gt)
        return out.detach(), dx, dw, db

    eager = [t.clone() for t in step(*leaves())]
    captured = leaves()  # fresh leaves: no autograd node of the eager step stays tied to the default stream
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        step(*captured)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=s):
            static = step(*captured)
    torch.cuda.current_stream().wait_stream(s)
    for _ in range(2):
        graph.replay()
        torch.cuda.synchronize()
        for a, c in zip(eager, static):
            assert torch.equal(a, c)


def test_fp64_step_launches_only_fp64_kernels(P):
    from torch.profiler import ProfilerActivity, profile

    rng = np.random.default_rng(4)
    m, g, x, w, b, G = layer_case(P, rng, fin=20, fout=40)
    xt = torch.from_numpy(x).to(dev()).requires_grad_()
    wt = torch.from_numpy(w).to(dev()).requires_grad_()
    bt = torch.from_numpy(b).to(dev()).requires_grad_()
    gt = torch.from_numpy(G).to(dev())
    torch.cuda.synchronize()
    for assoc in ("reference", "aggregate_first"):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            out = P.gcn_layer(xt, g, wt, bt, relu=True, association=assoc)
            torch.autograd.grad(out, (xt, wt, bt), gt)
            torch.cuda.synchronize()
        names = {e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}
        kernels = {n for n in names if "memcpy" not in n.lower() and "memset" not in n.lower()}
        assert kernels and all("_f64" in n for n in kernels), kernels
        assert any("dmma" in n for n in kernels) and any("spmm_f64" in n for n in kernels)


def test_dtype_rules(P):
    rng = np.random.default_rng(1)
    m, g = small_graph(P, rng)
    x = torch.zeros(30, 3, dtype=F64, device=dev())
    w = torch.zeros(3, 4, dtype=F64, device=dev())
    with pytest.raises(RuntimeError):
        P.gcn_layer(x, g, w.float())
    with pytest.raises(RuntimeError):
        P.gcn_layer(x, g, w, torch.zeros(4, device=dev()))
    adj32 = torch.eye(30, device=dev()).to_sparse()
    with pytest.raises(RuntimeError):
        P.gcn_layer(x, adj32, w)
    with pytest.raises(ValueError):
        P.gcn_layer(x, g, w, precision="tf32x3")
    with pytest.raises(RuntimeError):
        P.spmm(g, x.float())
    with pytest.raises(RuntimeError, match="float32"):
        P.apply_bn(x)


@pytest.mark.parametrize("shape", ["cbg", "reddit", "products"])
def test_full_size_agreement_with_torch_fp64(P, shape):
    """The benchmark's graphs and first-layer shapes (CBG 64 -> 32, Reddit 602 -> 256, products 100 -> 256)."""
    import bench

    wl = bench.WORKLOADS[shape]
    src, dst, n = bench.make_edges(torch, wl, seed=0)
    g = P.Graph.from_edges(src.to(dev()), dst.to(dev()), n, dtype=F64)
    rp, col, val = g.csr()
    a = torch.sparse_csr_tensor(rp.long(), col.long(), val, (n, n))
    fin, fout = wl["dims"][0], wl["dims"][1]
    gen = torch.Generator(device="cuda").manual_seed(0)
    x = torch.randn(n, fin, generator=gen, device=dev(), dtype=F64).requires_grad_()
    w = torch.randn(fin, fout, generator=gen, device=dev(), dtype=F64).requires_grad_()
    b = torch.randn(fout, generator=gen, device=dev(), dtype=F64).requires_grad_()
    G = torch.randn(n, fout, generator=gen, device=dev(), dtype=F64)
    for assoc in ("reference", "aggregate_first"):
        out = P.gcn_layer(x, g, w, b, association=assoc)
        dx, dw, db = torch.autograd.grad(out, (x, w, b), G)
        ref = torch.sparse.mm(a, x @ w) + b
        rdx, rdw, rdb = torch.autograd.grad(ref, (x, w, b), G)
        for o, r in ((out, ref), (dx, rdx), (dw, rdw), (db, rdb)):
            assert float((o.detach() - r.detach()).norm() / r.detach().norm()) <= 1e-12
    del a, g
    torch.cuda.empty_cache()


@pytest.mark.parametrize("agg", [False, True])
@pytest.mark.parametrize("relu,dropout", [(True, False), (False, True), (True, True)])
def test_layer_entry_points_in_exact_workspace(P, agg, relu, dropout):
    """gcnb_layer_forward_f64 / _backward_f64 called directly: workspace of exactly the queried size plus a guard that
    must stay unchanged (one byte less is refused), NaN-filled support / gm / ds panels, sentinel-framed outputs.  No
    bias, ReLU or dropout, n <= 512 and fout > 32: no product splits K, so the queried workspace has no product region
    and the discarded column sums must not be written anywhere."""
    from pygcn_b200 import _lib

    L = lib()
    rng = np.random.default_rng(21)
    n, fin, fout = 300, 6, 64
    m = csr_from_lengths(rng, list(rng.integers(0, 12, size=n - 3)) + [0, 0, 250], n)
    g = graph_of(P, m)
    x = dyadic(rng, (n, fin))
    w = rng.integers(-4, 5, size=(fin, fout)).astype(np.float64)
    G = rng.integers(-8, 9, size=(n, fout)).astype(np.float64)
    mask_np = rng.random((n, fout)) < 0.5 if dropout else None
    ld2 = lambda f: (f + 1) // 2 * 2
    nan = lambda r, c: torch.full((r, c), float("nan"), dtype=F64, device=dev())
    ldx = fin + 2
    xt = nan(n, ldx); xt[:, :fin] = torch.from_numpy(x)
    wt = torch.from_numpy(w).to(dev())
    mk = torch.from_numpy(mask_np.astype(np.uint8)).to(dev()) if dropout else None
    need = int(L.gcnb_layer_f64_workspace_bytes(g._h, fin, fout))
    ws = guarded_ws(need)
    flags = (_lib.LAYER_RELU if relu else 0) | (_lib.LAYER_AGG_FIRST if agg else 0)
    support = nan(n, ld2(fin) if agg else ld2(fout))
    outf = torch.full((n + 2, fout), SENTINEL, dtype=F64, device=dev())
    fwd = lambda wsb: L.gcnb_layer_forward_f64(g._h, xt.data_ptr(), ldx, wt.data_ptr(), None, fin, fout, flags,
                                               None if mk is None else mk.data_ptr(), 2.0, support.data_ptr(),
                                               outf.data_ptr() + fout * 8, ws.data_ptr(), wsb, stream())
    assert fwd(need - 1) == 1 and "workspace too small" in _lib.last_error()
    check(fwd(need), "gcnb_layer_forward_f64")
    torch.cuda.synchronize()
    assert guard_ok(ws, need) and frame_ok(outf, n, fout)
    pre = m @ (x @ w)
    assert_exact_bound(abs(m) @ (np.abs(x) @ np.abs(w)), Q / 4)
    y = np.maximum(pre, 0.0) if relu else pre
    if dropout:
        y = np.where(mask_np, y * 2.0, 0.0)
    assert torch.equal(outf[1:-1].cpu(), torch.from_numpy(y))
    gg = G * (pre > 0) if relu else G
    if dropout:
        gg = np.where(mask_np, gg * 2.0, 0.0)
    gt = torch.from_numpy(G).to(dev())
    gm = nan(n, ld2(fout))
    ds = nan(n, ld2(fin) if agg else ld2(fout))
    dw = torch.full((fin + 2, fout), SENTINEL, dtype=F64, device=dev())
    lddx = fin + 3
    dx = torch.full((n + 2, lddx), SENTINEL, dtype=F64, device=dev())
    bflags = flags | _lib.LAYER_NEED_DX | _lib.LAYER_NEED_DW
    xk, ldk = (support, ld2(fin)) if agg else (xt, ldx)
    bwd = lambda wsb: L.gcnb_layer_backward_f64(
        g._h, xk.data_ptr(), ldk, wt.data_ptr(), gt.data_ptr(), fout, outf.data_ptr() + fout * 8, fin, fout, bflags,
        None if mk is None else mk.data_ptr(), 2.0, gm.data_ptr(), ds.data_ptr(), dw.data_ptr() + fout * 8, None,
        dx.data_ptr() + lddx * 8, lddx, ws.data_ptr(), wsb, stream())
    assert bwd(need - 1) == 1 and "workspace too small" in _lib.last_error()
    check(bwd(need), "gcnb_layer_backward_f64")
    torch.cuda.synchronize()
    assert guard_ok(ws, need) and frame_ok(dw, fin, fout) and frame_ok(dx, n, fin)
    dsr = m.T @ gg
    assert torch.equal(dw[1:-1].cpu(), torch.from_numpy(x.T @ dsr))
    assert torch.equal(dx[1:-1, :fin].cpu(), torch.from_numpy(dsr @ w.T))
    assert torch.equal(gm[:, :fout].cpu(), torch.from_numpy(gg))

"""The column sums (db) and the layer backward against exact references.

gcnb_colsum must return the fp64 column sum rounded to fp32 once.  The gradients are 20-bit values on the 2^-12
quantum, so every fp64 partial sum is exact whatever the order and only the final rounding is left; a kernel that
rounds its block partials to fp32 first differs on many columns.  The adversarial column holds 2^25 and 1 in one
block (warp) and -2^25 in another: its sum is 1, and fp32 block partials give 0.

At layer level, Graph.from_torch builds the handle from a CSR with values in {+-1/4, +-1/2, +-1, +-2}; X, W, G and the
bias are small integers and the dropout scale is 2, so out, dW, dX and db have exactly one fp32 answer.
"""
import pytest
import torch

pytestmark = pytest.mark.gpu

SENTINEL = -12345.0
GUARD = 0xA5


def dev():
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def P():
    import pygcn_b200

    assert pygcn_b200._lib.load().gcnb_check_device() == 0, pygcn_b200._lib.last_error()
    return pygcn_b200


@pytest.fixture(scope="module")
def lib(P):
    return P._lib.load()


def kernels_run(fn):
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        r = fn()
        torch.cuda.synchronize()
    return r, {e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}


def has(names, k):
    return any(k + "<" in n or k + "(" in n for n in names)


def grad_values(gen, rows, cols):
    return (torch.randint(-(1 << 20) + 1, 1 << 20, (rows, cols), generator=gen, device=dev()).double() * 2.0 ** -12).float()


def run_colsum(lib, g, ldg, f, y=None, ldgm=None, out_off=4):
    """gcnb_colsum on g (a [n, ldg] storage, width f), optional ReLU mask y [n, f] and staged copy gm [n, ldgm];
    returns (db, gm, kernel names) after checking the sentinels around db and gm and the workspace guard."""
    n = g.shape[0]
    sp = torch.cuda.current_stream().cuda_stream
    outbuf = torch.full((out_off + f + 8,), SENTINEL, dtype=torch.float32, device=dev())
    out = outbuf[out_off:out_off + f]
    gm = None
    if ldgm is not None:
        gm = torch.full((max(n, 1), ldgm), SENTINEL, dtype=torch.float32, device=dev())
    nbytes = int(lib.gcnb_colsum_workspace_bytes(n, f))
    ws = torch.full((nbytes + 4096,), GUARD, dtype=torch.uint8, device=dev())

    def call():
        return lib.gcnb_colsum(n, f, g.data_ptr(), ldg, y.data_ptr() if y is not None else None, f,
                               gm.data_ptr() if gm is not None else None, ldgm or f, out.data_ptr(), ws.data_ptr(),
                               nbytes, sp)

    from pygcn_b200 import _lib

    st, names = kernels_run(call)
    _lib.check(st, "gcnb_colsum")
    assert bool((ws[nbytes:] == GUARD).all())
    assert bool((outbuf[:out_off] == SENTINEL).all()) and bool((outbuf[out_off + f:] == SENTINEL).all())
    if gm is not None:
        assert bool((gm[:, f:] == SENTINEL).all())
    first = out.clone()
    _lib.check(call(), "gcnb_colsum rerun")
    assert torch.equal(out, first)
    return out, gm, names


def exact_colsum(gv):
    return gv.double().sum(0).float()


@pytest.mark.parametrize("f", [1, 4, 47, 48, 1024, 1025])
@pytest.mark.parametrize("n", [0, 1, 127, 128, 129, 592 * 128 + 1])
@pytest.mark.parametrize("mode", ["plain", "relu", "unaligned"])
def test_colsum(lib, f, n, mode):
    gen = torch.Generator(device=dev()).manual_seed(f * 1000 + n)
    ldg = f + 3 if mode == "relu" else f + 4 - f % 4
    store = torch.full((max(n, 1) * ldg + 4,), float("nan"), dtype=torch.float32, device=dev())
    off = 1 if mode == "unaligned" else 0
    g = store[off:off + n * ldg].view(n, ldg)
    gv = grad_values(gen, n, f)
    g[:, :f] = gv
    y = None
    if mode == "relu":
        y = torch.randint(-2, 3, (n, f), generator=gen, device=dev()).float()
        y[y == 0] = torch.where(torch.rand(y[y == 0].shape, generator=gen, device=dev()) < 0.5, 0.0, -0.0)
        gv = torch.where(y > 0, gv, torch.zeros_like(gv))
    db, gm, names = run_colsum(lib, g, ldg, f, y=y, ldgm=f + 5 if mode == "relu" else None)
    assert torch.equal(db, exact_colsum(gv))
    if gm is not None and n:
        assert torch.equal(gm[:n, :f], gv)
    vec = f % 4 == 0 and f <= 1024 and mode == "plain"
    if n == 0:
        pass
    elif vec:
        assert has(names, "colsum_vec_kernel"), names
    else:
        assert has(names, "colsum_partial_kernel") and (has(names, "reduce_partials_kernel")
                                                         or has(names, "reduce_partials_vec_kernel")), names


def _cancelling(n, f, gen, rows):
    """Small integers, except column 0: zero but for 2^25 at rows[0], 1 at rows[1] and -2^25 at rows[2] (sum 1)."""
    g = torch.randint(-3, 4, (n, f), generator=gen, device=dev()).float()
    g[:, 0] = 0.0
    g[rows[0], 0], g[rows[1], 0], g[rows[2], 0] = 2.0 ** 25, 1.0, -(2.0 ** 25)
    return g


@pytest.mark.parametrize("path", ["vec", "partial"])
@pytest.mark.parametrize("n", [129, 592 * 128 + 1])
def test_colsum_cancellation(lib, path, n):
    gen = torch.Generator(device=dev()).manual_seed(7)
    f = 48 if path == "vec" else 47
    g = _cancelling(n, f, gen, (0, 1, n - 1))
    db, _, names = run_colsum(lib, g, f, f)
    assert has(names, "colsum_vec_kernel" if path == "vec" else "colsum_partial_kernel")
    ref = exact_colsum(g)
    assert float(ref[0]) == 1.0 and float(db[0]) == 1.0, float(db[0])
    assert torch.equal(db, ref)


# ------------------------------------------------------------------ layer level
VALUES = torch.tensor([-2, -1, -0.5, -0.25, 0.25, 0.5, 1, 2])


def _graph(P, n, deg, seed):
    gen = torch.Generator().manual_seed(seed)
    cols = torch.randint(0, n, (n * deg,), generator=gen)
    rows = torch.arange(n).repeat_interleave(deg)
    vals = VALUES[torch.randint(0, 8, (n * deg,), generator=gen)]
    dense = torch.zeros((n, n), dtype=torch.float64)
    dense.index_put_((rows, cols), vals.double(), accumulate=True)  # duplicates add: still on the 2^-2 quantum
    a = dense.to_sparse_csr()
    g = P.Graph.from_torch(torch.sparse_csr_tensor(a.crow_indices(), a.col_indices(), a.values().float(),
                                                   (n, n)).to(dev()))
    return g, dense.to(dev())


def _layer(P, graph, a64, fin, fout, *, relu, mask, need_dx, association, bias_shift=0, g=None, seed=0):
    gen = torch.Generator(device=dev()).manual_seed(seed)
    n = a64.shape[0]
    x = torch.randint(-2, 3, (n, fin), generator=gen, device=dev()).float().requires_grad_(need_dx)
    w = torch.randint(-2, 3, (fin, fout), generator=gen, device=dev()).float().requires_grad_(True)
    b = (torch.randint(-4, 5, (fout,), generator=gen, device=dev()).float() + bias_shift).requires_grad_(True)
    keep = (torch.rand((n, fout), generator=gen, device=dev()) < 0.5) if mask else None
    if g is None:
        g = torch.randint(-2, 3, (n, fout), generator=gen, device=dev()).float()
    # fp64 reference
    pre = a64 @ (x.detach().double() @ w.detach().double()) + b.detach().double()
    y = pre.clamp(min=0) if relu else pre
    if mask:
        y = torch.where(keep, 2 * y, torch.zeros_like(y))
    gm = g.double()
    if mask:
        gm = torch.where(keep, 2 * gm, torch.zeros_like(gm))
    if relu:
        gm = torch.where(y > 0, gm, torch.zeros_like(gm))
    ds = a64.t() @ gm
    ref = {"out": y.float(), "db": gm.sum(0).float(), "dw": (x.detach().double().t() @ ds).float(),
           "dx": (ds @ w.detach().double().t()).float()}
    assert float((x.detach().double().abs().t() @ ds.abs()).max()) < 2.0 ** 20  # dW partial sums < 2^22 quanta of 2^-2

    def run():
        out = P.functional.gcn_layer(x, graph, w, b, relu=relu, dropout_mask=keep, dropout_p=0.5 if mask else 0.0,
                                     association=association)
        out.backward(g)
        torch.cuda.synchronize()
        return out

    out, names = kernels_run(run)
    got = {"out": out.detach(), "db": b.grad.clone(), "dw": w.grad.clone(), "dx": x.grad.clone() if need_dx else None}
    return got, ref, names


@pytest.mark.parametrize("association", ["reference", "aggregate_first"])
@pytest.mark.parametrize("relu", [False, True])
@pytest.mark.parametrize("mask", [False, True])
@pytest.mark.parametrize("need_dx", [False, True])
def test_layer_backward(P, association, relu, mask, need_dx):
    graph, a64 = _graph(P, 3000, 5, 11)
    got, ref, _ = _layer(P, graph, a64, 20, 44, relu=relu, mask=mask, need_dx=need_dx, association=association)
    for key in ("out", "db", "dw") + (("dx",) if need_dx else ()):
        assert torch.equal(got[key], ref[key]), key


def test_layer_fused_db_matches_colsum_route(P):
    """Square, no mask, fin <= 64, fout <= 32, n >= 4096: db rides in the skinny dW kernel.  A ReLU whose y is all
    positive (bias shifted up) forces the colsum route on the same numbers; both must match the exact db and dW."""
    graph, a64 = _graph(P, 4096, 4, 12)
    fused, ref, names = _layer(P, graph, a64, 64, 32, relu=False, mask=False, need_dx=True, association="reference")
    assert has(names, "skinny_tn_kernel") and not has(names, "colsum_vec_kernel") and not has(names, "colsum_partial_kernel")
    coll, ref2, names2 = _layer(P, graph, a64, 64, 32, relu=True, mask=False, need_dx=True, association="reference",
                                bias_shift=4096)
    assert has(names2, "colsum_vec_kernel") or has(names2, "colsum_partial_kernel")
    assert bool((ref2["out"] > 0).all())
    for key in ("db", "dw", "dx"):
        assert torch.equal(fused[key], ref[key]), key
        assert torch.equal(coll[key], ref2[key]), key
    assert torch.equal(fused["db"], coll["db"]) and torch.equal(fused["dw"], coll["dw"])


def test_layer_fused_db_cancellation(P):
    """The adversarial column through the fused route: rows 0 and 1 are one warp's stage, row 8 the next warp's."""
    graph, a64 = _graph(P, 4096, 4, 13)
    gen = torch.Generator(device=dev()).manual_seed(5)
    g = _cancelling(4096, 32, gen, (0, 1, 8))
    x = torch.randint(-2, 3, (4096, 64), generator=gen, device=dev()).float()
    w = torch.randint(-2, 3, (64, 32), generator=gen, device=dev()).float().requires_grad_(True)
    b = torch.zeros(32, device=dev(), requires_grad=True)

    def run():
        P.functional.gcn_layer(x, graph, w, b, association="reference").backward(g)
        torch.cuda.synchronize()

    _, names = kernels_run(run)
    assert has(names, "skinny_tn_kernel") and not has(names, "colsum_vec_kernel")
    ref = g.double().sum(0).float()
    assert float(ref[0]) == 1.0 and float(b.grad[0]) == 1.0, float(b.grad[0])
    assert torch.equal(b.grad, ref)

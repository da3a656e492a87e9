"""Every dense-product route, the column sums and the layer backward, against exact-arithmetic references.

Inputs are built so that every product and every partial sum is exact in fp32 in any summation order: one operand
holds values o * 2^-12 with o odd and 2049 <= |o| <= 4095 (12 significant bits, so both the tf32 `hi` and the `lo` of
the 3xTF32 split are nonzero), the other integers in [-2, 2]; the lo operand is thinned along the reduction so that
max (|A| |B|)_ij <= 2^10, i.e. every partial sum stays below 2^22 quanta of 2^-12 (asserted on every case).  The fp64
product cast to fp32 is then the only correct answer, and the check is torch.equal.  The tcgen05 cases run twice, with
the lo operand on either side, and each asserts that a hi-only product would differ from the exact one on most entries.

Each gemm case also
  * runs once under torch.profiler and asserts which GEMM kernels ran (ROUTES lists one shape per route),
  * fills the operands' padding columns (lda > k, ldb > n, ldx > m) with NaN and C with NaN before the call,
  * surrounds C with a sentinel (ldc > n, a row before and after) that must come back bit for bit,
  * passes exactly gcnb_gemm_workspace_bytes of workspace followed by a guard that must come back unchanged,
  * with one byte less workspace must return an error or the exact answer, guard intact,
  * runs twice and requires bit-identical results.
"""
import pytest
import torch

pytestmark = pytest.mark.gpu

FP32, TF32X3, AUTO = 0, 1, 2
SENTINEL = -12345.0
GUARD = 0xA5
QUANTUM = 2.0 ** -12
BOUND = 2.0 ** 22 * QUANTUM
GEMM_KERNELS = ("skinny_rows_kernel", "skinny_tn_kernel", "gemm_tc_rows_tma_kernel", "gemm_tc_tn_tma_kernel",
                "gemm_fp32_kernel")


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


# ------------------------------------------------------------------ exact inputs
def lo_values(gen, rows, cols, red_dim):
    """12-bit values on the 2^-12 quantum, thinned along the reduction dimension (0 or 1) to <= ~300 per line."""
    length = rows if red_dim == 0 else cols
    o = torch.randint(1024, 2048, (rows, cols), generator=gen) * 2 + 1
    s = torch.randint(0, 2, (rows, cols), generator=gen) * 2 - 1
    keep = torch.rand((rows, cols), generator=gen) < min(1.0, 300.0 / max(length, 1))
    return (o * s * keep).to(torch.float64).mul_(QUANTUM).to(torch.float32)


def int_values(gen, rows, cols, lim=2):
    return torch.randint(-lim, lim + 1, (rows, cols), generator=gen).to(torch.float32)


def tf32_hi(t):
    return (t.view(torch.int32) & -8192).view(torch.float32)  # 0xffffe000: what kind::tf32 reads of a word


def kernels_run(fn):
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        r = fn()
        torch.cuda.synchronize()
    return r, {e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}


def has(names, k):
    return any(k + "<" in n or k + "(" in n for n in names)


def check_kernels(names, expect, absent=()):
    for k in expect:
        assert has(names, k), "expected %s among %s" % (k, sorted(names))
    for k in GEMM_KERNELS:
        if k not in expect:
            assert not has(names, k), "%s ran, the case is for %s (%s)" % (k, expect, sorted(names))
    for k in absent:
        assert not has(names, k), "%s ran (%s)" % (k, sorted(names))


# ------------------------------------------------------------------ one gemm case
class Case:
    def __init__(self, name, m, n, k, expect, layout="rows", b_t=False, prec=TF32X3, lda=None, ldb=None, ldc=None,
                 c_off=4, bias=False, relu=False, absent=(), lo_sides=("a", "b")):
        self.name, self.m, self.n, self.k, self.expect = name, m, n, k, tuple(expect)
        self.layout, self.b_t, self.prec, self.bias, self.relu = layout, b_t, prec, bias, relu
        # default leading dimensions: the next multiple of 4 past the width, so there is always a padding gap
        a_line = k if layout == "rows" else m
        self.lda = lda if lda is not None else a_line + 4 - a_line % 4
        b_line = k if b_t else n
        self.ldb = ldb if ldb is not None else b_line + 4 - b_line % 4
        self.ldc = ldc if ldc is not None else n + 4 - n % 4
        self.c_off, self.absent, self.lo_sides = c_off, tuple(absent), lo_sides

    def __repr__(self):
        return self.name


def _operands(case, lo_side, seed):
    gen = torch.Generator().manual_seed(seed)
    m, n, k = case.m, case.n, case.k
    if lo_side == "a":
        a, b = lo_values(gen, m, k, 1), int_values(gen, k, n)
    else:
        a, b = int_values(gen, m, k), lo_values(gen, k, n, 0)
    bias = int_values(gen, 1, n, 8)[0] if case.bias else None
    return a, b, bias


def _store(logical, ld, transpose):
    """NaN-padded storage of `logical` (rows x cols) with leading dimension ld, stored transposed if asked;
    returns (storage, row stride, column stride) of the logical matrix."""
    src = logical.t() if transpose else logical
    buf = torch.full((src.shape[0], ld), float("nan"), dtype=torch.float32, device=dev())
    buf[:, : src.shape[1]] = src.to(dev())
    return (buf, 1, ld) if transpose else (buf, ld, 1)


def run_gemm_case(lib, case, lo_side, seed=1):
    m, n, k = case.m, case.n, case.k
    a, b, bias = _operands(case, lo_side, seed)
    ad, bd = a.to(dev(), torch.float64), b.to(dev(), torch.float64)
    product = ad @ bd
    if m * n * k:
        assert float((ad.abs() @ bd.abs()).max()) <= BOUND
    if case.prec != FP32 and k > 0 and any(e.startswith("gemm_tc") for e in case.expect):
        ah, bh = (tf32_hi(a), b) if lo_side == "a" else (a, tf32_hi(b))
        hi_only = ah.to(dev(), torch.float64) @ bh.to(dev(), torch.float64)
        frac = float((hi_only != product).double().mean())
        assert frac > 0.5, "hi-only product differs on only %.2f of the entries: the lo path is not tested" % frac
    exact = product + bias.to(dev(), torch.float64) if case.bias else product
    exact = (exact.clamp(min=0) if case.relu else exact).float()

    abuf, a_rs, a_cs = _store(a, case.lda, case.layout != "rows")
    bbuf, b_rs, b_cs = _store(b, case.ldb, case.b_t)
    bias_d = bias.to(dev()) if case.bias else None
    ldc = case.ldc
    base = case.c_off + ldc  # one sentinel row before C
    flat = torch.full((base + (m + 1) * ldc + 16,), SENTINEL, dtype=torch.float32, device=dev())
    c = flat.as_strided((m, n), (ldc, 1), base)
    want = flat.clone()
    want.as_strided((m, n), (ldc, 1), base).copy_(exact)
    nbytes = int(lib.gcnb_gemm_workspace_bytes(m, n, k, case.prec))
    ws = torch.empty((nbytes + 4096,), dtype=torch.uint8, device=dev())
    sp = torch.cuda.current_stream().cuda_stream

    def call(ws_bytes):
        ws.fill_(GUARD)
        c.fill_(float("nan"))
        if case.bias or case.relu:
            return lib.gcnb_gemm_ex(m, n, k, abuf.data_ptr(), a_rs, a_cs, bbuf.data_ptr(), b_rs, b_cs, c.data_ptr(), ldc,
                                    bias_d.data_ptr() if case.bias else None, 1 if case.relu else 0, case.prec,
                                    ws.data_ptr(), ws_bytes, sp)
        return lib.gcnb_gemm(m, n, k, abuf.data_ptr(), a_rs, a_cs, bbuf.data_ptr(), b_rs, b_cs, c.data_ptr(), ldc,
                             case.prec, ws.data_ptr(), ws_bytes, sp)

    from pygcn_b200 import _lib

    st, names = kernels_run(lambda: call(nbytes))
    _lib.check(st, "gemm %s" % case.name)
    check_kernels(names, case.expect, case.absent)
    first = flat.clone()
    assert bool((ws[nbytes:] == GUARD).all()), "write past the workspace size the query returned"
    if not torch.equal(flat, want):
        bad = (c != exact).nonzero()[:5].tolist()
        raise AssertionError("%s lo=%s: C wrong at %s (of %d entries), sentinel changed at %s" % (
            case.name, lo_side, bad, int((c != exact).sum()), (flat != want).nonzero()[:5].flatten().tolist()))
    _lib.check(call(nbytes), "gemm rerun")
    torch.cuda.synchronize()
    assert torch.equal(flat, first), "rerun not bit-identical"
    if nbytes > 0:
        st = call(nbytes - 1)
        torch.cuda.synchronize()
        assert bool((ws[nbytes - 1:] == GUARD).all()), "one byte less workspace: wrote past it"
        if st == 0:
            assert torch.equal(flat, want), "one byte less workspace: neither an error nor the exact answer"
    return names


# ------------------------------------------------------------------ the route table: one row per route
ROUTES = [
    Case("skinny rows", 4097, 32, 16, ["skinny_rows_kernel"], prec=AUTO),
    Case("skinny tn", 16, 32, 4099, ["skinny_tn_kernel", "reduce_partials_vec_kernel"], layout="tn", prec=AUTO),
    Case("skinny tn scalar reduce", 16, 31, 4099, ["skinny_tn_kernel", "reduce_partials_kernel"], layout="tn", prec=AUTO),
    Case("tcgen05 rows", 20000, 64, 36, ["gemm_tc_rows_tma_kernel", "pack_b_kernel"], prec=AUTO),
    Case("tcgen05 tn", 100, 48, 8192, ["gemm_tc_tn_tma_kernel", "reduce_partials_vec_kernel"], layout="tn", prec=AUTO),
    Case("rows on a padded copy", 3600, 47, 602, ["gemm_tc_rows_tma_kernel", "pad_copy_kernel"], prec=AUTO),
    Case("tn on a padded copy", 601, 48, 4096, ["gemm_tc_tn_tma_kernel", "pad_copy_kernel"], layout="tn", prec=AUTO,
         lda=601),
    Case("CUDA-core fp32", 200, 40, 4000, ["gemm_fp32_kernel", "reduce_partials_vec_kernel"], prec=FP32),
    Case("epilogue pass", 100, 40, 20, ["gemm_fp32_kernel", "bias_act_kernel"], prec=AUTO, bias=True, relu=True),
    Case("fused epilogue", 129, 47, 260, ["gemm_tc_rows_tma_kernel"], bias=True, relu=True, absent=["bias_act_kernel"]),
]


@pytest.mark.parametrize("case", ROUTES, ids=repr)
def test_route_table(lib, case):
    for side in case.lo_sides if any(e.startswith("gemm_tc") for e in case.expect) else ("a",):
        run_gemm_case(lib, case, side)


# ------------------------------------------------------------------ tcgen05 rows edges
def _tma_b_resident(n, k):
    """gemm_tc.cu tma_plan(): is the packed B resident in shared memory?"""
    npad = 256 if n >= 256 else -(-n // 32) * 32
    nkb = -(-k // 32)
    budget = 227 * 1024 - 4 * 32 * 36 * 4 - 1024 - 2048
    return nkb * 2 * npad * 128 + 3 * 2 * 128 * 128 <= budget


TC = ["gemm_tc_rows_tma_kernel", "pack_b_kernel"]
ROWS_EDGES = (
    [Case("rows M=%d" % m, m, 33, 36, TC) for m in (1, 31, 32, 33, 127, 128, 129, 148 * 128 + 1)]
    + [Case("rows K=%d" % k, 129, 47, k, TC) for k in (4, 28, 32, 36, 252, 256, 260, 516)]
    + [Case("rows N=%d" % n, 129, n, 36, TC) for n in (1, 4, 31, 32, 33, 47, 255, 256, 257, 513)]
    + [Case("rows B streamed N=32 K=516", 300, 32, 516, TC), Case("rows B streamed N=256 K=256", 300, 256, 256, TC)]
    + [Case("rows B transposed", 129, 47, 36, TC, b_t=True), Case("rows B transposed K=260", 257, 40, 260, TC, b_t=True)]
    + [Case("rows lda=k+28", 129, 33, 36, TC, lda=64)]
    + [Case("rows bias relu K=%d" % k, 300, n, k, TC, bias=True, relu=True, absent=["bias_act_kernel"])
       for k, n in ((36, 47), (260, 33), (516, 256))]
    + [Case("rows ldc%%4=0 aligned N=%d" % n, 129, n, 36, TC, ldc=n + 4 - n % 4 if n % 4 else n + 4, c_off=4)
       for n in (32, 64)]
    + [Case("rows C 4-byte offset N=64", 129, 64, 36, TC, ldc=68, c_off=5),
       Case("rows ldc=65", 129, 64, 36, TC, ldc=65, c_off=4)]
)


def test_rows_edges_cover_both_b_placements():
    res = {_tma_b_resident(c.n, c.k) for c in ROWS_EDGES}
    assert res == {True, False}


@pytest.mark.parametrize("case", ROWS_EDGES, ids=repr)
@pytest.mark.parametrize("side", ["a", "b"])
def test_tcgen05_rows(lib, case, side):
    run_gemm_case(lib, case, side)


# ------------------------------------------------------------------ tcgen05 tn edges
def _tn_splits(m, r):
    """gemm_tc.cu tn_tma_plan(): (splits, rows per split)."""
    mt = -(-m // 128)
    s = max(1, min(148 // mt, -(-r // 128)))
    rps = -(-(-(-r // s)) // 32) * 32
    return -(-r // rps), rps


TN = ["gemm_tc_tn_tma_kernel"]
TN_EDGES = (
    [Case("tn m=%d" % m, m, 48, 1000, TN, layout="tn") for m in (1, 4, 100, 128, 129, 600)]
    + [Case("tn n=%d" % n, 129, n, 1000, TN, layout="tn") for n in (1, 4, 47, 48, 256)]
    + [Case("tn r=%d" % r, 100, 47, r, TN, layout="tn") for r in (32, 96, 128, 129, 4095, 4096, 4097, 16416)]
    + [Case("tn drain r=15000", 600, 32, 15000, TN, layout="tn"),
       Case("tn single split + drain", 9600, 4, 600, TN, layout="tn"),
       Case("tn single split", 300, 33, 128, TN, layout="tn"),
       Case("tn ldx=m+60", 100, 48, 1000, TN, layout="tn", lda=160)]
)


def test_tn_edges_cover_splits_and_drains():
    plans = [_tn_splits(c.m, c.k) for c in TN_EDGES]
    assert any(s == 1 for s, _ in plans) and any(s > 16 for s, _ in plans)
    assert any(s == 1 and rps > 512 for s, rps in plans) and any(s > 1 and rps > 512 for s, rps in plans)


@pytest.mark.parametrize("case", TN_EDGES, ids=repr)
@pytest.mark.parametrize("side", ["a", "b"])
def test_tcgen05_tn(lib, case, side):
    names = run_gemm_case(lib, case, side)
    # a single split writes C directly; many go through workspace and a reduce kernel
    reduced = has(names, "reduce_partials_kernel") or has(names, "reduce_partials_vec_kernel")
    assert reduced == (_tn_splits(case.m, case.k)[0] > 1)


# ------------------------------------------------------------------ padded routes
PAD_EDGES = [
    Case("pad rows k=5", 307693, 65, 5, TC + ["pad_copy_kernel"]),
    Case("pad rows k=47", 64475, 33, 47, TC + ["pad_copy_kernel"]),
    Case("pad rows k=602", 3600, 47, 602, TC + ["pad_copy_kernel"]),
    Case("pad tn m=601", 601, 48, 4096, TN + ["pad_copy_kernel"], layout="tn", lda=601),
    Case("pad tn m=1002", 1002, 33, 3100, TN + ["pad_copy_kernel"], layout="tn", lda=1002),
]


@pytest.mark.parametrize("case", PAD_EDGES, ids=repr)
@pytest.mark.parametrize("side", ["a", "b"])
def test_padded_routes(lib, case, side):
    assert case.m * case.n * case.k >= 1e8
    run_gemm_case(lib, case, side)


# ------------------------------------------------------------------ CUDA-core kernels
SR = ["skinny_rows_kernel"]
SKINNY_ROWS = (
    [Case("skinny rows k=%d n=%d" % (k, n), 4097, n, k, SR, prec=FP32) for k, n in
     ((5, 32), (16, 1), (29, 31), (64, 32), (8, 33), (13, 64), (32, 47))]
    + [Case("skinny rows M=4103 k=47", 4103, 20, 47, SR, prec=FP32),
       Case("skinny rows B transposed", 5000, 33, 30, SR, prec=FP32, b_t=True),
       Case("skinny rows B strided", 4097, 7, 12, SR, prec=FP32, b_t=True, ldb=29)]
)
ST = ["skinny_tn_kernel"]
SKINNY_TN = [Case("skinny tn m=%d n=%d r=%d" % (m, n, r), m, n, r, ST, layout="tn", prec=FP32)
             for m, n, r in ((3, 32, 4099), (8, 1, 4096), (16, 17, 5003), (17, 32, 4097), (32, 8, 8191), (64, 32, 4100),
                             (64, 5, 20001))]
F32 = ["gemm_fp32_kernel"]
FP32_TILES = (
    [Case("fp32 %dx%d" % (m, n), m, n, 100, F32, prec=FP32) for m in (33, 200) for n in (7, 20, 50)]
    + [Case("fp32 split128", 70, 40, 1000, F32, prec=FP32), Case("fp32 split512", 33, 20, 40000, F32, prec=FP32),
       Case("fp32 generic strides", 200, 50, 300, F32, prec=FP32, layout="tn", b_t=True),
       Case("fp32 split generic strides", 50, 30, 3000, F32, prec=FP32, layout="tn", b_t=True),
       Case("fp32 k=0", 5, 7, 0, F32, prec=FP32), Case("fp32 k=0 auto", 70, 40, 0, F32, prec=AUTO)]
)


@pytest.mark.parametrize("case", SKINNY_ROWS + SKINNY_TN + FP32_TILES, ids=repr)
def test_cuda_core_kernels(lib, case):
    names = run_gemm_case(lib, case, "a")
    splits = case.expect == tuple(ST) or (case.name.startswith("fp32 split"))
    if splits:
        assert has(names, "reduce_partials_kernel") or has(names, "reduce_partials_vec_kernel")


def test_reduce_partials_both_kernels(lib):
    v = run_gemm_case(lib, Case("vec", 64, 32, 2000, F32, prec=FP32), "a")
    s = run_gemm_case(lib, Case("scalar", 64, 31, 2000, F32, prec=FP32), "a")
    assert has(v, "reduce_partials_vec_kernel") and has(s, "reduce_partials_kernel")


# ------------------------------------------------------------------ grids past 65535 tiles in y
def test_tn_more_than_65535_m_tiles(P):
    m = 8_400_000  # 65625 tiles of 128
    gen = torch.Generator(device=dev()).manual_seed(3)
    x = torch.randint(-8, 9, (32, m), generator=gen, device=dev()).float()
    y = torch.randint(-8, 9, (32, 4), generator=gen, device=dev()).float()
    for prec in ("tf32x3", "auto"):
        out, names = kernels_run(lambda: P.mm(x.t(), y, precision=prec))
        assert has(names, "gemm_tc_tn_tma_kernel"), sorted(names)
        ref = torch.empty((m, 4), dtype=torch.float32, device=dev())
        for r0 in range(0, m, 1 << 21):
            ref[r0:r0 + (1 << 21)] = (x[:, r0:r0 + (1 << 21)].t().double() @ y.double()).float()
        assert torch.equal(out, ref)
        del out


def test_fp32_more_than_65535_n_tiles(P):
    n = 4_200_000  # 65625 tiles of 64
    gen = torch.Generator(device=dev()).manual_seed(4)
    a = torch.randint(-8, 9, (8, 4), generator=gen, device=dev()).float()
    b = torch.randint(-8, 9, (4, n), generator=gen, device=dev()).float()
    out, names = kernels_run(lambda: P.mm(a, b))
    assert has(names, "gemm_fp32_kernel"), sorted(names)
    assert torch.equal(out, (a.double() @ b.double()).float())

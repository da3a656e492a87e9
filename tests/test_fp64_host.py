"""CPU-side checks of the fp64 entry points: every argument check runs on the host before any launch, so each refusal
is exercised without a GPU, and the workspace sizes follow their plans."""
import ctypes

import pytest


@pytest.fixture(scope="module")
def lib():
    from pygcn_b200 import _lib

    return _lib.load()


def _err():
    from pygcn_b200 import _lib

    return _lib.last_error()


def test_gemm_f64_refusals(lib):
    buf = (ctypes.c_double * 4096)()
    a = ctypes.addressof(buf)
    gemm = lambda m, n, k, pa, pb, pc, ldc, ws, wsb, a_rs=8, b_rs=8: lib.gcnb_gemm_f64(m, n, k, pa, a_rs, 1, pb, b_rs, 1, pc,
                                                                                       ldc, ws, wsb, None)
    assert gemm(0, 8, 8, None, None, None, 8, None, 0) == 0  # empty output: nothing to do
    for call, msg in ((lambda: gemm(-1, 8, 8, a, a, a, 8, None, 0), "negative dimension"),
                      (lambda: gemm(8, 8, 8, a, a, a, 7, None, 0), "ldc < n"),
                      (lambda: gemm(8, 8, 8, None, a, a, 8, None, 0), "null operand"),
                      (lambda: gemm(8, 8, 8, a, a, None, 8, None, 0), "null output"),
                      (lambda: gemm(8, 8, 8, a + 4, a, a, 8, None, 0), "8-byte aligned"),
                      (lambda: gemm(8, 8, 8, a, a, a, 8, None, 0, a_rs=-1), "negative stride"),
                      (lambda: gemm(8, 8, 100000, a, a, a, 8, a, 64), "workspace too small")):
        st = call()
        assert st == 1 and msg in _err(), (st, msg, _err())
    assert lib.gcnb_gemm_f64_ex(8, 8, 8, a, 8, 1, a, 8, 1, a, 8, a + 4, 1, None, 0, None) == 1 and "aligned" in _err()


def test_gemm_f64_workspace_is_the_split_plan(lib):
    # one tile (64 x 32) over 100000 rows: split into 2 * 148 / 1 -> capped at 64 splits of fp64 [m, n] partials
    assert lib.gcnb_gemm_f64_workspace_bytes(16, 32, 100000) == 64 * 16 * 32 * 8
    assert lib.gcnb_gemm_f64_workspace_bytes(100000, 256, 602) == 0   # enough tiles: no split
    assert lib.gcnb_gemm_f64_workspace_bytes(64, 64, 512) == 0        # short reduction: no split
    assert lib.gcnb_gemm_f64_workspace_bytes(0, 8, 8) == 0 and lib.gcnb_gemm_f64_workspace_bytes(8, 8, 0) == 0


def test_colsum_f64_refusals_and_workspace(lib):
    buf = (ctypes.c_double * 4096)()
    a = ctypes.addressof(buf)
    assert lib.gcnb_colsum_f64_workspace_bytes(1, 5) == 5 * 8 + 256
    assert lib.gcnb_colsum_f64_workspace_bytes(10 ** 7, 3) == 512 * 3 * 8 + 256
    cs = lambda n, f, g, ldg, y, gm, out, ws, wsb: lib.gcnb_colsum_f64(n, f, g, ldg, y, f, gm, f, out, ws, wsb, None)
    for call, msg in ((lambda: cs(4, 0, a, 8, None, None, a, a, 4096), "shape out of range"),
                      (lambda: cs(4, 8, a, 8, None, None, None, a, 4096), "null output"),
                      (lambda: cs(4, 8, a, 7, None, None, a, a, 4096), "bad gradient operand"),
                      (lambda: cs(4, 8, a, 8, a, None, a, a, 4096), "bad mask operands"),
                      (lambda: cs(4, 8, a + 4, 8, None, None, a, a, 4096), "8-byte aligned"),
                      (lambda: cs(4, 8, a, 8, None, None, a, a, 8), "workspace too small")):
        st = call()
        assert st == 1 and msg in _err(), (st, msg, _err())


def test_graph_entry_points_refuse_null_handles(lib):
    assert lib.gcnb_spmm_f64(None, 0, None, 8, 8, None, None, 0, 1.0, None, 8, None, 0, None) == 1
    assert "null graph" in _err()
    assert lib.gcnb_layer_forward_f64(None, None, 8, None, None, 8, 8, 0, None, 1.0, None, None, None, 0, None) == 1
    assert "null graph" in _err()
    assert lib.gcnb_layer_backward_f64(None, None, 8, None, None, 8, None, 8, 8, 0, None, 1.0, None, None, None, None,
                                       None, 8, None, 0, None) == 1
    assert "null graph" in _err()
    assert lib.gcnb_layer_f64_workspace_bytes(None, 8, 8) == 0 and lib.gcnb_spmm_f64_workspace_bytes(None, 0, 8) == 0
    assert lib.gcnb_graph_export_csr_f64(None, 0, None, None, None, None) == 1
    out = ctypes.c_void_p()
    assert lib.gcnb_graph_from_coo_f64(-1, 4, 0, None, None, None, None, ctypes.byref(out)) == 1 and not out.value
    assert lib.gcnb_graph_from_dense_f64(4, 4, None, 3, None, None) == 1  # out is null


def test_header_has_keep_f64_flag():
    import os
    import re

    from pygcn_b200 import _lib

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    header = open(os.path.join(root, "include", "gcnb200.h")).read()
    assert int(re.search(r"#define GCNB_BUILD_KEEP_F64 (\d+)", header).group(1)) == _lib.BUILD_KEEP_F64 == 8

"""Accuracy (vs fp64) and time of the tcgen05 "rows" product C = A[M,K] B[K,N] on the layer shapes of the
BASELINE configs.  Run on the GPU box:  python tools/gemm_rows_probe.py [tag]"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import pygcn_b200 as P

dev = torch.device("cuda:0")
torch.manual_seed(0)
tag = sys.argv[1] if len(sys.argv) > 1 else "tcgen05"


def timeit(fn, n=10):
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n * 1e3


SHAPES = [  # (M, N, K, B transposed, what)
    (128, 32, 32, False, "one tile"),
    (333, 7, 16, True, "tiny, N=7"),
    (5000, 47, 100, False, "products last layer (small M)"),
    (3000, 600, 16, False, "N > 256: 3 N tiles"),
    (2708, 16, 1432, False, "Cora L1 (K padded)"),
    (100000, 32, 64, False, "CBG X W"),
    (100000, 64, 32, True, "CBG dX"),
    (232965, 256, 604, False, "Reddit X W (padded K)"),
    (1000000, 256, 100, False, "products L1"),
    (1000000, 256, 256, False, "products L2"),
    (1000000, 47, 256, False, "products L3"),
    (2000000, 128, 128, False, "papers100M"),
]
ok = True
print("[%s]" % tag)
for m, n, k, bt, what in SHAPES:
    a = torch.randn(m, k, device=dev)
    b = torch.randn(n, k, device=dev).t() if bt else torch.randn(k, n, device=dev)
    c = P.mm(a, b, precision="tf32x3")
    rows = torch.randperm(m, device=dev)[:4096]
    ref = a[rows].double() @ b.double()
    e = ((c[rows].double() - ref).abs().max() / ref.abs().max()).item()
    # the tails must be exact too: last rows of the matrix
    tail = slice(max(0, m - 200), m)
    reft = a[tail].double() @ b.double()
    et = ((c[tail].double() - reft).abs().max() / reft.abs().max()).item()
    t = timeit(lambda: P.mm(a, b, precision="tf32x3"))
    gbs = (m * k + k * n + m * n) * 4 / t / 1e3
    print("  %-34s M=%-8d N=%-4d K=%-5d err %.2e tail %.2e | %8.1f us  %6.0f GB/s  %6.1f TFLOP/s(x3)" % (
        what, m, n, k, e, et, t, gbs, 6.0 * m * n * k / t / 1e6))
    ok &= e < 1e-5 and et < 1e-5
    del a, b, c
TSHAPES = [  # (R, M, N, ldy, what):  C[M,N] = X[R,M]^T Y[R,N]
    (32, 128, 32, 32, "one K block"),
    (64, 64, 32, 32, "two K blocks"),
    (4097, 100, 48, 48, "ragged R"),
    (2708, 1432, 16, 16, "Cora dW: 12 M tiles"),
    (100000, 8, 32, 32, "fork dW 8->32"),
    (100000, 64, 32, 32, "CBG dW"),
    (232965, 604, 256, 256, "Reddit dW"),
    (1000000, 100, 256, 256, "products L1 dW"),
    (1000000, 256, 256, 256, "products L2 dW"),
    (1000000, 256, 47, 48, "products L3 dW (N=47, ld 48)"),
    (2000000, 128, 128, 128, "papers100M dW"),
]
for r, m, n, ldy, what in TSHAPES:
    x = torch.randn(r, m, device=dev)
    y = torch.randn(r, ldy, device=dev)[:, :n]
    c = P.mm(x.t(), y, precision="tf32x3")
    ref = torch.zeros(m, n, dtype=torch.float64, device=dev)
    for r0 in range(0, r, 1 << 18):  # fp64 reference in row chunks (bounded memory)
        ref += x[r0:r0 + (1 << 18)].double().t() @ y[r0:r0 + (1 << 18)].double()
    e = ((c.double() - ref).abs().max() / ref.abs().max()).item()
    t = timeit(lambda: P.mm(x.t(), y, precision="tf32x3"))
    gbs = (r * m + r * n) * 4 / t / 1e3
    print("  T %-32s R=%-8d M=%-5d N=%-4d err %.2e | %8.1f us  %6.0f GB/s  %6.1f TFLOP/s(x3)" % (
        what, r, m, n, e, t, gbs, 6.0 * m * n * r / t / 1e6))
    ok &= e < 1e-5
    del x, y, c
print("ALL OK" if ok else "FAILED")
sys.exit(0 if ok else 1)

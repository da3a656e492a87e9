"""Device time of single ops of the layer step (CUDA-graph replay, L2 flushed before each replay): which kernel
serves the narrow products best.  python tools/op_graph_probe.py"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import pygcn_b200 as P
from time_step import dev, graph_time

torch.manual_seed(0)
tiny = torch.zeros(32, 4, device=dev)
w4 = torch.zeros(4, 4, device=dev)
t0 = graph_time(lambda: P.mm(tiny, w4, precision="fp32"))
print("graph replay of one tiny kernel: %.1f us (subtract from the numbers below)" % t0)
for (m, k, n, what) in [(100000, 64, 32, "CBG"), (100000, 32, 32, "fork-like 32->32"), (100000, 8, 32, "fork 8->32"),
                        (233000, 604, 256, "Reddit"), (1000000, 128, 128, "papers (1M rows)")]:
    x = torch.randn(m, k, device=dev)
    w = torch.randn(k, n, device=dev)
    ds = torch.randn(m, n, device=dev)
    for prec in ("auto", "tf32x3"):
        t_xw = graph_time(lambda: P.mm(x, w, precision=prec))
        t_dw = graph_time(lambda: P.mm(x.t(), ds, precision=prec))
        t_dx = graph_time(lambda: P.mm(ds, w.t(), precision=prec))
        by = (m * k + m * n) * 4
        print("  %-18s M=%-8d %3d->%-3d %-7s XW %7.1f us (%5.0f GB/s) | dW %7.1f us (%5.0f GB/s) | dX %7.1f us" % (
            what, m, k, n, prec, t_xw, by / t_xw / 1e3, t_dw, by / t_dw / 1e3, t_dx))

"""fp64 tier against torch's fp64 (cuSPARSE CSR SpMM, cuBLAS DGEMM) on the same tensors, at the benchmark's shapes.

    python tools/fp64_probe.py [--out FILE] [--reps 20]

For CBG (64 -> 32), Reddit (602 -> 256) and the products 3-layer stack (100 -> 256 -> 256 -> 47, ReLU), on the graphs
bench.py generates (fp64 handles, Graph.from_edges(..., dtype=torch.float64)):
  * per-kernel time (CUDA events, median of --reps after warm-up) of the SpMM at the layer's width, X W, dW = X^T dS and
    dX = dS W^T, ours and torch's;
  * the SpMM's algorithmic bytes (int32 col + fp64 val per stored entry, rowptr, the fp64 panel read once, the fp64
    output written once) over its time, as a share of 7.7 TB/s; the DMMA products' FLOP/s;
  * the fwd + bwd step time of the layer (products: of the 3-layer stack), ours and torch's;
  * the norm-wise error of ours against torch's fp64 on out, dW, db and dX.
The card's name and power limit are read in the same run and printed first.  Needs a CUDA device.
"""
import argparse
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402
import pygcn_b200 as P  # noqa: E402

F64 = torch.float64
HBM_BYTES_PER_S = 7.7e12


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # pragma: no cover
        q = "power limit unavailable (%s)" % e
    return "%s, %s" % (name, q)


def timed(fn, reps):
    for _ in range(3):
        fn()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return statistics.median(ts)


def nerr(a, b):
    return float((a.detach() - b.detach()).norm() / b.detach().norm().clamp_min(1e-300))


def graph_for(key):
    src, dst, n = bench.make_edges(torch, bench.WORKLOADS[key], seed=0)
    g = P.Graph.from_edges(src.cuda(), dst.cuda(), n, dtype=F64)
    rp, col, val = g.csr()
    a = torch.sparse_csr_tensor(rp.long(), col.long(), val, (n, n))
    return g, a, n


def kernels(lines, key, g, a, n, fin, fout, reps):
    gen = torch.Generator(device="cuda").manual_seed(1)
    x = torch.randn(n, fin, generator=gen, device="cuda", dtype=F64)
    w = torch.randn(fin, fout, generator=gen, device="cuda", dtype=F64)
    s = torch.randn(n, fout, generator=gen, device="cuda", dtype=F64)
    ours = timed(lambda: P.spmm(g, s), reps)
    ref = timed(lambda: torch.sparse.mm(a, s), reps)
    nbytes = g.nnz * 12 + (n + 1) * 4 + 2 * n * fout * 8
    lines.append("%-9s spmm F=%-3d ours %8.3f ms (%5.1f %% of HBM)   torch sparse.mm %8.3f ms (%5.1f %%)   %.2fx" % (
        key, fout, ours, 100 * nbytes / (ours * 1e-3) / HBM_BYTES_PER_S, ref, 100 * nbytes / (ref * 1e-3) / HBM_BYTES_PER_S,
        ref / ours))
    for what, (ma, mb), flop in (("X W", (x, w), 2.0 * n * fin * fout),
                                 ("X^T dS", (x.t(), s), 2.0 * n * fin * fout),
                                 ("dS W^T", (s, w.t()), 2.0 * n * fin * fout)):
        ours = timed(lambda: P.mm(ma, mb), reps)
        ref = timed(lambda: torch.mm(ma, mb), reps)
        lines.append("%-9s %-7s %d x %d x %d  ours %8.3f ms (%5.2f TFLOP/s)   torch.mm %8.3f ms (%5.2f TFLOP/s)" % (
            key, what, ma.shape[0], mb.shape[1], ma.shape[1], ours, flop / ours * 1e-9, ref, flop / ref * 1e-9))


def stack_step(g, a, n, dims, relu, reps, lines, key):
    gen = torch.Generator(device="cuda").manual_seed(2)
    x = torch.randn(n, dims[0], generator=gen, device="cuda", dtype=F64).requires_grad_()
    params = []
    for fi, fo in zip(dims[:-1], dims[1:]):
        params.append((torch.randn(fi, fo, generator=gen, device="cuda", dtype=F64).div_(fi ** 0.5).requires_grad_(),
                       torch.randn(fo, generator=gen, device="cuda", dtype=F64).requires_grad_()))
    gout = torch.randn(n, dims[-1], generator=gen, device="cuda", dtype=F64)
    leaves = [x] + [t for p in params for t in p]

    def ours():
        h = x
        for w, b in params:
            h = P.gcn_layer(h, g, w, b, relu=relu)
        return [h] + list(torch.autograd.grad(h, leaves, gout))

    def ref():
        h = x
        for w, b in params:
            h = torch.sparse.mm(a, h @ w) + b
            if relu:
                h = torch.relu(h)
        return [h] + list(torch.autograd.grad(h, leaves, gout))

    o, r = ours(), ref()
    names = ["out", "dX"] + [nm for i in range(len(params)) for nm in ("dW%d" % i, "db%d" % i)]
    lines.append("%-9s agreement with torch fp64 (norm-wise): %s" % (
        key, ", ".join("%s %.2e" % (nm, nerr(u, v)) for nm, u, v in zip(names, o, r))))
    t_ours, t_ref = timed(ours, reps), timed(ref, reps)
    lines.append("%-9s step fwd+bwd %s  ours %8.3f ms   torch fp64 %8.3f ms   %.2fx" % (
        key, "->".join(map(str, dims)), t_ours, t_ref, t_ref / t_ours))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--shapes", default="cbg,reddit,products")
    args = ap.parse_args()
    lines = ["card: " + card()]
    report = []
    for key in args.shapes.split(","):
        wl = bench.WORKLOADS[key]
        g, a, n = graph_for(key)
        lines.append("%-9s graph n=%d nnz=%d (fp64 handle, %.1f MB)" % (key, n, g.nnz, g.device_bytes / 1e6))
        kernels(lines, key, g, a, n, wl["dims"][0], wl["dims"][1], args.reps)
        stack_step(g, a, n, wl["dims"], wl["relu"], args.reps, lines, key)
        print("\n".join(lines), flush=True)
        report += lines
        lines = []
        del g, a
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(report) + "\n")


if __name__ == "__main__":
    main()

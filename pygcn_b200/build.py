"""Build libgcnb200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python -m pygcn_b200.build [--force] [--verbose]

The objects and the library land in pygcn_b200/lib/ (git-ignored, but shipped to the
GPU box with the working tree).
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIBDIR, "libgcnb200.so")

SOURCES = ["api.cu", "spmm.cu", "spmm_stream.cu", "gemm_simt.cu", "gemm_skinny.cu", "gemm_tc.cu", "elementwise.cu", "graph_build.cu", "peer.cu", "batchnorm.cu", "dist.cu", "spmm_f64.cu", "gemm_f64.cu"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC",
    "--expt-relaxed-constexpr",
    "-I", os.path.join(ROOT, "include"),
    "-I", CSRC,
]


def _nvcc():
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found: libgcnb200.so cannot be built")
    return exe


def _digest(paths):
    h = hashlib.sha256()
    for p in sorted(paths):
        with open(p, "rb") as f:
            h.update(os.path.relpath(p, ROOT).encode())  # relative: the digest must not depend on where the tree lives
            h.update(f.read())
    h.update(" ".join(NVCC_FLAGS).replace(ROOT, ".").encode())  # (the -I paths are absolute: keep the tree's location out)
    return h.hexdigest()


def _sources():
    return [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]


def _headers():
    hs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    hs.append(os.path.join(ROOT, "include", "gcnb200.h"))
    return hs


def needs_build():
    stamp = os.path.join(LIBDIR, "build.stamp")
    if not (os.path.exists(LIB) and os.path.exists(stamp)):
        return True
    with open(stamp) as f:
        return f.read().strip() != _digest(_sources() + _headers())


def build(force=False, verbose=False):
    """Compile every .cu to an object (in parallel) and link the shared library.  One builder at a time: the ranks of
    a torchrun job that all find a stale library queue on a file lock and the late ones find it fresh."""
    if not force and not needs_build():
        return LIB
    os.makedirs(LIBDIR, exist_ok=True)
    import fcntl

    with open(os.path.join(LIBDIR, ".build.lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and not needs_build():
                return LIB
            return _build_locked(verbose)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)


def _build_locked(verbose):
    nvcc = _nvcc()
    srcs = _sources()

    def compile_one(src):
        obj = os.path.join(LIBDIR, os.path.basename(src)[:-3] + ".o")
        cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s\n%s" % (src, r.stdout, r.stderr))
        if verbose:
            sys.stderr.write(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=min(8, len(srcs))) as ex:
        objs = list(ex.map(compile_one, srcs))
    tmp = LIB + ".tmp.%d" % os.getpid()  # link beside, then rename: a reader never sees a half-written library
    cmd = [nvcc, "-shared", "-o", tmp] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-lcuda", "-ldl"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n%s\n%s" % (r.stdout, r.stderr))
    os.replace(tmp, LIB)
    with open(os.path.join(LIBDIR, "build.stamp"), "w") as f:
        f.write(_digest(srcs + _headers()))
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))

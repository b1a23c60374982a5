"""Build libfenix_knn.so in-tree with nvcc for sm_100a (no JIT cache, no torch extension).

    python -m fenix_b200.csrc.build [--force]

The .so lands next to the package (fenix_b200/libfenix_knn.so); it is git-ignored but
travels to the GPU box with the gpurun snapshot.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.dirname(HERE)
ROOT = os.path.dirname(PKG)
OUT = os.environ.get("FENIX_BUILD_OUT") or os.path.join(PKG, "libfenix_knn.so")   # FENIX_BUILD_OUT: tuning variants
SOURCES = ["fenix_knn.cu"]
DEPS = ["fenix_knn.cu", "common.cuh", "exact_scan.cuh", "direct_scan.cuh", "tc_filter.cuh", "range_search.cuh", "kmeans.cuh",
        os.path.join(ROOT, "include", "fenix_knn.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC,-Wall,-Wno-unused-function",
    "-shared",
    "--expt-relaxed-constexpr",
    "-ldl",
    *os.environ.get("FENIX_NVCC_EXTRA", "").split(),
]


def nvcc_path() -> str:
    cand = os.environ.get("NVCC") or shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(cand):
        raise RuntimeError("nvcc not found; libfenix_knn.so cannot be built")
    return cand


def stale() -> bool:
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    for d in DEPS:
        p = d if os.path.isabs(d) else os.path.join(HERE, d)
        if os.path.getmtime(p) > t:
            return True
    return False


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not stale():
        return OUT
    cmd = [nvcc_path(), *NVCC_FLAGS]
    if verbose:
        cmd += ["-Xptxas", "-v"]
    cmd += [os.path.join(HERE, s) for s in SOURCES] + ["-o", OUT]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
        raise RuntimeError("nvcc failed building libfenix_knn.so")
    if verbose:
        sys.stderr.write(res.stdout + res.stderr)
    return OUT


if __name__ == "__main__":
    path = build(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print(path)

"""Range search against the k-NN search at the same shape (DESIGN.md §4.10), alternating, several runs.

    python scripts/range_bench.py [--only c3,c2,wide] [--runs 3] [--out-dir profiles]

Workloads (synthetic Gaussian rows generated on the device, seeded):
  c3    10M x 768 cosine, 4096 queries; radius = the median 10th-neighbour distance, k-NN k = 10
  c2    1M x 128 L2, 10k queries; radius = the median 100th-neighbour distance, k-NN k = 100
  wide  1M x 128 L2, 256 queries; a radius admitting ~1 % of the rows (candidate lists overflow: prices the scan
        fallback), k-NN k = 100
Per workload: ms per batch (host clock around the call, which ends in a device synchronisation, and the library's
device time), total hits, fallback queries, filter path and operand; GPU name, power limit and SM clock beside them.
Writes profiles/r05_range_<name>.txt."""
from __future__ import annotations

import argparse
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from fenix_b200 import knn  # noqa: E402

WORKLOADS = {
    "c3": dict(n=10_000_000, d=768, nq=4096, metric="cosine", k=10, rank=10),
    "c2": dict(n=1_000_000, d=128, nq=10_000, metric="l2", k=100, rank=100),
    "wide": dict(n=1_000_000, d=128, nq=256, metric="l2", k=100, frac=0.01),
}


def gpu_info() -> str:
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True)
    return out.stdout.strip().splitlines()[0] if out.returncode == 0 and out.stdout.strip() else "unknown GPU"


def make_corpus(ctx, w, seed):
    import torch

    gen = torch.Generator(device="cuda")
    gen.manual_seed(seed)
    c = knn.Corpus(ctx, w["n"], w["d"])
    chunk = 1 << 20
    for a in range(0, w["n"], chunk):
        b = min(w["n"], a + chunk)
        block = torch.randn((b - a, w["d"]), generator=gen, device="cuda", dtype=torch.float32)
        torch.cuda.synchronize()
        c.append_device(block.data_ptr(), b - a)
    c.finalize()
    queries = torch.randn((w["nq"], w["d"]), generator=gen, device="cuda", dtype=torch.float32).cpu().numpy()
    return c, queries


def timed(fn):
    t0 = time.perf_counter()
    out = fn()
    return out, (time.perf_counter() - t0) * 1e3


def run(name: str, w: dict, runs: int, out_dir: str) -> str:
    ctx = knn.Context(0)
    c, queries = make_corpus(ctx, w, seed=sorted(WORKLOADS).index(name) + 1)
    metric, k = w["metric"], w["k"]
    if "rank" in w:
        _, dist = c.search(queries, metric, w["rank"])
        radius = float(np.median(dist[:, w["rank"] - 1]))
        how = f"median {w['rank']}th-neighbour distance"
    else:
        radius = float(np.median([np.quantile(c.distances(q, metric), w["frac"]) for q in queries[:16]]))
        how = f"median {w['frac']:.0%} quantile of 16 distance columns"
    lines = [f"# {name}: {w['n']} x {w['d']} {metric}, {w['nq']} queries; radius {radius:.7g} ({how}); k-NN k = {k}",
             f"# {gpu_info()} (name, power limit, SM clock, max SM clock)"]
    # warm-up: shadows, scratch, CUB's first launches; its hit count sizes the output of the timed calls (one search each)
    cap = int(c.search_range(queries, metric, radius)[0][-1])
    c.search(queries, metric, k)
    for r in range(runs):
        before = c.stats().fallback_queries
        (off, _, _), ms_r = timed(lambda: c.search_range(queries, metric, radius, capacity=cap))
        st = c.stats()
        last_hits = int(off[-1])
        lines.append(f"run {r} range: {ms_r:8.2f} ms host, {st.last_search_ms:8.2f} ms device, filter {st.last_main_kernel_ms:7.2f} ms, "
                     f"hits {last_hits}, fallback queries {st.fallback_queries - before}, path {st.last_path}, operand {st.last_operand}")
        _, ms_k = timed(lambda: c.search(queries, metric, k))
        st = c.stats()
        lines.append(f"run {r} knn:   {ms_k:8.2f} ms host, {st.last_search_ms:8.2f} ms device, filter {st.last_main_kernel_ms:7.2f} ms, "
                     f"path {st.last_path}, operand {st.last_operand}; range / knn {ms_r / ms_k:.2f}")
    lines.append(f"# after the runs: {gpu_info()}")
    c.close()
    ctx.close()
    text = "\n".join(lines) + "\n"
    with open(os.path.join(out_dir, f"r05_range_{name}.txt"), "w") as f:
        f.write(text)
    return text


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--only", default="c3,c2,wide")
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--out-dir", default=os.path.join(ROOT, "profiles"))
    args = ap.parse_args()
    os.makedirs(args.out_dir, exist_ok=True)
    for name in args.only.split(","):
        print(run(name, WORKLOADS[name], args.runs, args.out_dir), flush=True)


if __name__ == "__main__":
    main()

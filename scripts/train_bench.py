"""IVF codebook training (fx_train_codebooks, DESIGN.md §4.11): time per epoch on the device against the host numpy
implementation it replaced.

    python scripts/train_bench.py [--only c3,c3n2,c2] [--epochs 3] [--out-dir profiles]

Workloads (synthetic Gaussian rows generated on the device, seeded):
  c3    10M x 768 cosine, n = 1, k = 1024, batch 4096
  c3n2  10M x 768 cosine, n = 2, k = 64, batch 1024
  c2    1M x 128 L2, n = 1, k = 1024, batch 256 (many small steps: the launch-bound end)
Per workload: seconds per epoch over --epochs epochs after one warm-up epoch (host clock around each library call,
which ends in a device synchronisation; it includes checking and uploading the epoch's positions), the achieved fp64
rate from 2 * N_used * k * D per epoch, and the old host implementation timed on a 200k-row subsample, one epoch,
scaled linearly to N (labelled as scaled). GPU name and power limit are read in the same run.
Writes profiles/r06_train_<name>.txt."""
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
    "c3": dict(n=10_000_000, d=768, metric="cosine", books=1, k=1024, bs=4096),
    "c3n2": dict(n=10_000_000, d=768, metric="cosine", books=2, k=64, bs=1024),
    "c2": dict(n=1_000_000, d=128, metric="l2", books=1, k=1024, bs=256),
}
HOST_ROWS = 200_000


def gpu_info() -> str:
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True)
    return out.stdout.strip().splitlines()[0] if out.returncode == 0 and out.stdout.strip() else "unknown GPU"


def _normalize(x):
    return x / np.maximum(np.linalg.norm(x, axis=-1, keepdims=True), 1e-12)


def _host_distance(u, v, metric):
    if metric == "l2":
        d2 = (u * u).sum(-1)[:, None] - 2.0 * (u @ v.T) + (v * v).sum(-1)[None, :]
        return np.sqrt(np.maximum(d2, 0.0))
    if metric == "cosine":
        return 0.5 - 0.5 * (_normalize(u) @ _normalize(v).T)
    return -(u @ v.T)


def host_epoch(rows, books, bs, metric, rng):
    """One epoch of the host implementation `io.coder.make` used before training moved to the device."""
    n, k = books.shape[:2]
    cosine = metric == "cosine"
    perm = rng.permutation(len(rows))
    step = n * bs
    for lo in range(0, len(perm) // step * step, step):
        sample = rows[np.sort(perm[lo: lo + step])].reshape(n, bs, -1)
        for j in range(n):
            q, v = (_normalize(books[j]), _normalize(sample[j])) if cosine else (books[j], sample[j])
            nearest = np.argmin(_host_distance(v, q, metric), axis=-1)
            total, count = q.copy(), np.ones(k, dtype=np.float32)
            np.add.at(total, nearest, v)
            np.add.at(count, nearest, 1.0)
            q = total / count[:, None]
            books[j] = _normalize(q) if cosine else q
    return books


def run(name, w, epochs, out_dir, info):
    import torch

    n, d, metric, nb, k, bs = w["n"], w["d"], w["metric"], w["books"], w["k"], w["bs"]
    ctx = knn.Context(0)
    corpus = knn.Corpus(ctx, n, d)
    gen = torch.Generator(device="cuda").manual_seed(0)
    chunk = 1_000_000
    for lo in range(0, n, chunk):
        part = torch.randn((min(chunk, n - lo), d), generator=gen, device="cuda", dtype=torch.float32)
        corpus.append_device(part.data_ptr(), part.shape[0])
        torch.cuda.synchronize()
        del part
    corpus.finalize()
    rng = np.random.default_rng(1)
    sel = np.sort(rng.permutation(n)[: nb * k])
    sub_pos = np.sort(rng.choice(n, HOST_ROWS, replace=False))
    # the seed rows and the host subsample: the same seeded chunks generated again, the wanted rows copied to the host
    gen = torch.Generator(device="cuda").manual_seed(0)
    seeds, sub = [], []
    for lo in range(0, n, chunk):
        part = torch.randn((min(chunk, n - lo), d), generator=gen, device="cuda", dtype=torch.float32)
        hi = lo + part.shape[0]
        for want, out in ((sel, seeds), (sub_pos, sub)):
            idx = want[(want >= lo) & (want < hi)] - lo
            if len(idx):
                out.append(part[torch.from_numpy(idx).cuda()].cpu().numpy())
        del part
    books = np.concatenate(seeds).reshape(nb, k, d)
    sub = np.concatenate(sub)
    step = nb * bs
    steps = n // step

    def positions():
        perm = rng.permutation(n)
        return np.sort(perm[: steps * step].reshape(steps, step), axis=1)

    trained = knn.train_codebooks([corpus], metric, books, bs, positions())   # warm-up epoch
    times = []
    for _ in range(epochs):
        pos = positions()
        t0 = time.perf_counter()
        trained = knn.train_codebooks([corpus], metric, trained, bs, pos)
        times.append(time.perf_counter() - t0)
    assert np.isfinite(trained).all()
    flop = 2.0 * steps * step * k * d
    h_books = books.copy()
    t0 = time.perf_counter()
    host_epoch(sub, h_books, bs, metric, np.random.default_rng(2))
    host_s = time.perf_counter() - t0
    lines = [
        f"# r06 train {name}: {n} x {d} {metric}, n_books {nb}, k {k}, batch {bs}; {steps} steps / epoch",
        f"gpu (name, power limit, max SM clock): {info}",
        f"device s/epoch (host clock around fx_train_codebooks, {epochs} epochs after 1 warm-up): "
        + " ".join(f"{t:.3f}" for t in times),
        f"achieved fp64 TFLOP/s (2 N_used k D / epoch): " + " ".join(f"{flop / t / 1e12:.2f}" for t in times),
        f"host numpy (the previous implementation), one epoch on {HOST_ROWS} rows: {host_s:.2f} s; "
        f"SCALED linearly to {n} rows: {host_s * n / HOST_ROWS:.0f} s / epoch (not measured at full size)",
        f"speed-up against the scaled host epoch: {host_s * n / HOST_ROWS / float(np.median(times)):.0f}x",
    ]
    text = "\n".join(lines) + "\n"
    print(text)
    with open(os.path.join(out_dir, f"r06_train_{name}.txt"), "w") as f:
        f.write(text)
    corpus.close()
    ctx.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--only", default=",".join(WORKLOADS))
    ap.add_argument("--epochs", type=int, default=3)
    ap.add_argument("--out-dir", default=os.path.join(ROOT, "profiles"))
    a = ap.parse_args()
    os.makedirs(a.out_dir, exist_ok=True)
    info = gpu_info()
    for name in a.only.split(","):
        run(name, WORKLOADS[name], a.epochs, a.out_dir, info)


if __name__ == "__main__":
    main()

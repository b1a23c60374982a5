#!/usr/bin/env python
"""bench.py - exact k-NN QPS of the B200 path next to the reference's CPU path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config c3] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch of synthetic queries against the resident
corpus. Default workload: BASELINE.json configs[2] "10M x 768 cosine, k=10, 4096-query batch,
row-sharded at 1/2/4/8 B200" - the shape north_star's target is stated on ("exact k-NN at
10M x 768 on 1 B200, near-linear QPS scaling to 8 GPUs"); it fits one GPU (30.7 GB), so the same
total workload runs at every N (strong scaling). Other configs: --config c2|c4|c4s|c5_B.
Launched by torchrun for N > 1 (one rank per GPU, NCCL); rank 0 prints ONE JSON line.

Besides the contract's keys the line carries
  parity  a sample of the TIMED batch re-checked inside the same run, at every N, on the (merged) result rank 0 holds:
          >= 32 queries against the fp64 CUDA-core scan over the whole (sharded) corpus and >= 4 queries against the
          oracle (the reference's per-chunk torch arithmetic + Arrow select_k) over the WHOLE corpus, streamed to the
          host in 65,536-row chunks;
  also    (N = 1, default config) compact lines for the other BASELINE configs that fit one GPU - C2, one C4 shard,
          C5 at batch 1 and 64 - and for SURVEY section 8d's stress inputs at C2 scale (clustered rows, duplicated rows,
          queries drawn from the corpus, 0.1 % rows with 100x the norm), each with its own parity check and
          refined / fallback counters.

--dump-outputs DIR writes what the last timed step returned (see dump_outputs), so that two builds can be compared
output for output: the corpus and the queries depend only on the arguments (seeded), never on the run.
The library is the one build() left next to the package; bench.py compiles and caches nothing in the tree.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CONFIGS = {
    # name: (N rows, D, metric, k, Q, cfg#)
    "c2": dict(n=1_000_000, d=128, metric="l2", k=100, q=10_000, num=2,
               label="SIFT-1M-shape 1M x 128 fp32 L2, k=100, 10k-query batch"),
    "c3": dict(n=10_000_000, d=768, metric="cosine", k=10, q=4096, num=3,
               label="10M x 768 cosine, k=10, 4096-query batch, row-sharded"),
    "c4": dict(n=100_000_000, d=96, metric="inner_product", k=100, q=10_000, num=4,
               label="100M x 96 inner product (Deep-100M shape), k=100, 10k-query batch"),
}
CONFIGS["c1"] = dict(n=100_000, d=128, metric="l2", k=10, q=1, num=1,
                     label="C1 shape: one query per search, exact L2 k=10 over 100k x 128 (the reference's Flight test shape)")
CONFIGS["c4s"] = dict(n=12_500_000, d=96, metric="inner_product", k=100, q=10_000, num=4,
                      label="one 8-GPU shard of C4: 12.5M x 96 inner product, k=100, 10k-query batch")
for _b in (1, 2, 4, 8, 16, 32, 64):
    CONFIGS[f"c5_{_b}"] = dict(n=10_000_000, d=768, metric="cosine", k=10, q=_b, num=5,
                               label=f"latency sweep batch {_b}, k=10 over 10M x 768")
GEN_CHUNK = 65_536  # rows per seeded generation chunk (BASELINE.md §3.1)
STRESS = ("clustered", "duplicates", "queries_from_corpus", "norm_outliers")
DUMP_MAX_BYTES = 64 << 20


def peaks() -> dict:
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        p["_source"] = "measured"
        return p
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "_source": "fallback"}


def ncu_traffic(config: str, world: int):
    """DRAM bytes (read + write) of the dominant kernel per launch, from the committed `ncu --set full` capture of
    this configuration on one GPU (profiles/ncu_traffic.json, written by scripts/summarise_profiles.py), or None."""
    path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if world != 1 or not os.path.exists(path):
        return None, "no single-GPU ncu capture for this configuration"
    rec = json.load(open(path)).get(config)
    if not rec:
        return None, "no single-GPU ncu capture for this configuration"
    return rec["dram_bytes_per_launch"], f"profiles/{rec['capture']} (dram__bytes_read.sum + dram__bytes_write.sum, one launch)"


def query_batch(cfg: dict) -> np.ndarray:
    rng = np.random.default_rng(2000 + cfg["num"])
    return rng.standard_normal((cfg["q"], cfg["d"]), dtype=np.float32)


def workload_config(args, cfg: dict) -> dict:
    """The `config` object: identifies the WORKLOAD only, so both arms (ours / reference) print the same one."""
    corpus_bytes = 4.0 * cfg["n"] * cfg["d"] / max(args.gpus, 1)
    return {
        "workload": f"{args.config}: {cfg['label']}", "n_rows": cfg["n"], "dim": cfg["d"], "metric": cfg["metric"], "k": cfg["k"],
        "queries_per_step": cfg["q"], "precision_mode": "fp32 (exact: bit-exact neighbour ids, distances within 1e-5)",
        "l2_policy": ("the corpus shard of every GPU is larger than L2 (126 MB): no flush needed between steps"
                      if corpus_bytes > 2.5e8 else "the corpus shard fits in L2: steady-state (warm L2) timing"),
    }


# ------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle port of the reference's CPU path, host cores only
# ------------------------------------------------------------------------------------------
def use_all_host_threads() -> int:
    """torchrun exports OMP_NUM_THREADS=1 to every rank; the reference arm is ONE process that owns the host."""
    import pyarrow as pa
    import torch

    n = os.cpu_count() or 1
    try:
        n = len(os.sched_getaffinity(0)) or n
    except Exception:
        pass
    torch.set_num_threads(n)
    pa.set_cpu_count(n)
    return n


def cpu_corpus_sample(cfg: dict, rows: int) -> np.ndarray:
    """First `rows` rows of the synthetic corpus, generated on the host (seed 1000 + cfg#)."""
    out = np.empty((rows, cfg["d"]), dtype=np.float32)
    for ci, lo in enumerate(range(0, rows, GEN_CHUNK)):
        rng = np.random.default_rng([1000 + cfg["num"], ci])
        hi = min(rows, lo + GEN_CHUNK)
        out[lo:hi] = rng.standard_normal((GEN_CHUNK, cfg["d"]), dtype=np.float32)[: hi - lo]
    return out


def time_reference(cfg: dict, steps: int, warmup: int, budget_s: float = 25.0) -> dict:
    """Times oracle.call (the restated fenix.io.index.call: per-chunk torch distance + Arrow
    select_k + take) one query at a time, as the reference serves them, on a bounded row sample;
    per-query cost is linear in N, so QPS at the full N = sample QPS * sample_rows / N."""
    import pyarrow as pa
    import torch

    from oracle import call as oracle_call

    threads = use_all_host_threads()
    sample_rows = min(cfg["n"], max(GEN_CHUNK, int(2.5e8 // cfg["d"])))  # ~1 GB of floats
    corpus = cpu_corpus_sample(cfg, sample_rows)
    batches = []
    for lo in range(0, sample_rows, GEN_CHUNK):
        x = corpus[lo: lo + GEN_CHUNK]
        vec = pa.FixedSizeListArray.from_arrays(pa.array(x.reshape(-1)), list_size=cfg["d"])
        batches.append(pa.record_batch([pa.array(np.arange(lo, lo + len(x), dtype=np.int64)), vec], names=["id", "vector"]))
    table = pa.Table.from_batches(batches)
    queries = query_batch(cfg)
    k = cfg["k"]

    def one(i: int) -> None:
        oracle_call(table, "vector", queries[i % len(queries)], cfg["metric"], select=["id"], maxval=k)

    t0 = time.perf_counter()
    one(0)
    per_query = time.perf_counter() - t0
    q_per_step = max(1, int(budget_s / max(per_query, 1e-6) / max(steps + warmup, 1)))
    q_per_step = min(q_per_step, 64)
    n = 0
    for _ in range(warmup):
        for _ in range(q_per_step):
            one(n); n += 1
    t0 = time.perf_counter()
    for _ in range(steps):
        for _ in range(q_per_step):
            one(n); n += 1
    dt = time.perf_counter() - t0
    sample_qps = steps * q_per_step / dt
    scale = sample_rows / cfg["n"]
    # best case for the CPU: the same arithmetic (oracle.distance = the reference's torch formulas) as ONE batched call
    # over the whole sample instead of one call per chunk and query, plus torch.topk - separates library speed from
    # the reference's per-chunk, per-query overhead (SURVEY.md section 8d, row 3)
    from oracle import distance as oracle_distance
    qb = torch.from_numpy(queries[: min(len(queries), 256)])
    xs = torch.from_numpy(corpus)
    t0 = time.perf_counter()
    torch.topk(oracle_distance(qb, xs, cfg["metric"]), min(k, sample_rows), largest=False)
    best_dt = time.perf_counter() - t0
    best_qps = len(qb) / best_dt * scale
    return dict(
        value=sample_qps * scale, unit="queries/s", cores=torch.get_num_threads(), kind="port",
        sample=(f"{steps} steps x {q_per_step} sequential single-query oracle.call (restated fenix.io.index.call, "
                f"{GEN_CHUNK}-row chunks, select=['id']) on the first {sample_rows} of {cfg['n']} rows; "
                f"measured {sample_qps:.3f} q/s on the sample, scaled by {scale:.4g} (cost linear in N); "
                f"{threads} host threads (torch intra-op + Arrow pool)"),
        ms_per_step=dt / steps * 1e3, host_cpus=os.cpu_count(), arrow_threads=pa.cpu_count(),
        best_case={"value": best_qps, "unit": "queries/s",
                   "what": f"one batched torch call ({len(qb)} queries x {sample_rows} rows, the reference's formulas) + torch.topk, "
                           f"scaled by {scale:.4g}: library speed without the reference's per-chunk, per-query overhead"},
    )


# ------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region (NVML from a thread, ~4 ms period, so
    even a 40 ms region gets samples; falls back to one nvidia-smi query when NVML is unavailable)."""

    REASONS = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}

    def __init__(self, gpu: int) -> None:
        self.gpu = gpu
        self.sm, self.bits, self.max_mhz = [], 0, None
        self._stop = None
        self._thread = None
        self._nvml = None

    def _loop(self, handle) -> None:
        nv = self._nvml
        while not self._stop.is_set():
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(handle, nv.NVML_CLOCK_SM)))
                self.bits |= int(nv.nvmlDeviceGetCurrentClocksEventReasons(handle))
            except Exception:
                break
            self._stop.wait(0.004)

    def start(self) -> None:
        import threading

        try:
            import pynvml as nv

            nv.nvmlInit()
            # honour CUDA_VISIBLE_DEVICES: map the CUDA ordinal to the NVML device through its UUID
            import torch

            uuid = str(torch.cuda.get_device_properties(self.gpu).uuid)
            try:
                handle = nv.nvmlDeviceGetHandleByUUID(("GPU-" + uuid).encode())
            except Exception:
                handle = nv.nvmlDeviceGetHandleByIndex(self.gpu)
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(handle, nv.NVML_CLOCK_SM))
            self._nvml = nv
            self._stop = threading.Event()
            self._thread = threading.Thread(target=self._loop, args=(handle,), daemon=True)
            self._thread.start()
        except Exception:
            self._nvml = None

    def stop(self) -> dict:
        if self._nvml is None:
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.gpu}", "--query-gpu=clocks.sm,clocks.max.sm",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=10).stdout
                a, b = [float(t) for t in out.strip().split(",")[:2]]
                return {"sm_mhz": a, "sm_max_mhz": b, "reasons": ["sampled once after the region (NVML unavailable)"], "samples": 1}
            except Exception:
                return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self._stop.set()
        self._thread.join(timeout=2)
        reasons = sorted(name for name, bit in self.REASONS.items() if self.bits & bit)
        if not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["no samples"], "samples": 0}
        return {"sm_mhz": float(np.median(self.sm)), "sm_max_mhz": self.max_mhz, "reasons": reasons, "samples": len(self.sm)}


# ------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------
def gen_chunk(cfg: dict, ci: int, device, variant: str | None = None):
    """Chunk `ci` (65,536 rows) of the synthetic corpus, generated on the GPU from a seed that depends only on (config,
    chunk) - the content is independent of the world size and of which rank asks. `variant`: a stress input
    (SURVEY.md section 8d) derived from the same rows."""
    import torch

    gen = torch.Generator(device=device)
    gen.manual_seed((1000 + cfg.get("data_num", cfg["num"])) * 1_000_003 + ci)   # data_num: a config that reuses another one's corpus
    block = torch.randn((GEN_CHUNK, cfg["d"]), generator=gen, device=device, dtype=torch.float32)
    if variant == "clustered":
        # the reference tests' generator (tests/test_flight.py:21-22): every batch is shifted by 10 x its first row
        # (batches of 1,024 rows instead of 1,000 keep the 65,536-row chunks self-contained)
        b = block.view(GEN_CHUNK // 1024, 1024, cfg["d"])
        b += 10.0 * b[:, :1, :].clone()
    elif variant == "duplicates":
        # every row appears 4 times (rows 4j .. 4j+3 are copies): ties at every rank, broken by row
        block = block.view(GEN_CHUNK // 4, 4, cfg["d"])[:, :1, :].expand(-1, 4, -1).reshape(GEN_CHUNK, cfg["d"]).contiguous()
    elif variant == "norm_outliers":
        # 0.1 % of the rows carry 100x the norm
        idx = torch.arange(ci % 7, GEN_CHUNK, 1000, device=device)
        block[idx] *= 100.0
    return block


def build_shard(cfg: dict, ctx, lo: int, hi: int, device, variant: str | None = None):
    """Rows [lo, hi) of the synthetic corpus, appended device-to-device chunk by chunk."""
    import torch

    from fenix_b200 import knn

    c = knn.Corpus(ctx, hi - lo, cfg["d"], row_base=lo)
    first, last = lo // GEN_CHUNK, (max(hi, lo + 1) - 1) // GEN_CHUNK
    for ci in range(first, last + 1):
        block = gen_chunk(cfg, ci, device, variant)
        a, b = max(lo, ci * GEN_CHUNK), min(hi, (ci + 1) * GEN_CHUNK)
        if b <= a:
            continue
        piece = block[a - ci * GEN_CHUNK: b - ci * GEN_CHUNK].contiguous()
        torch.cuda.synchronize(device)
        c.append_device(piece.data_ptr(), b - a)
    c.finalize()
    return c


def same_neighbours(got_rows, got_dist, ref_rows, ref_dist, rtol=1e-5, floor=0.0):
    """The parity bar of tests/conftest.py::assert_same_neighbours as a predicate: ids identical after (distance, row)
    ordering - a differing id is accepted only inside a tie band of the reference's own fp32 rounding - and distances
    within rtol relative (absolute floor for GEMM-form cancellation of the reference's L2)."""
    from oracle import canonical

    g_r, g_d = canonical(np.asarray(got_rows), np.asarray(got_dist))
    r_r, r_d = canonical(np.asarray(ref_rows), np.asarray(ref_dist))
    tol = np.maximum(rtol * np.maximum(np.abs(r_d), 1e-30), floor)
    err = np.abs(g_d.astype(np.float64) - r_d.astype(np.float64))
    # relative to the reference distance, or to the noise floor where the reference distance itself is below it (a query
    # that IS a corpus row: both sides compute ~0 from cancelling terms)
    rel = float((err / np.maximum(np.abs(r_d), max(floor, 1e-30))).max()) if len(r_d) else 0.0
    ok_d = bool((err <= tol).all())
    ids_equal = bool(np.array_equal(g_r, r_r))
    ok_ids = ids_equal
    if not ids_equal:
        # only as a permutation / boundary swap among reference distances that tie within the band
        diff = g_r != r_r
        ok_ids = bool((np.abs(r_d[diff] - g_d[diff]) <= 2 * tol[diff]).all()) and \
            (sorted(g_r.tolist()) == sorted(r_r.tolist()) or abs(float(g_d[-1]) - float(r_d[-1])) <= 2 * float(tol[-1]))
    return ok_ids and ok_d, ids_equal, rel


def oracle_topk_streamed(cfg: dict, queries: np.ndarray, device, variant: str | None = None):
    """The reference's arithmetic over the WHOLE corpus on the host: per 65,536-row chunk (regenerated on this GPU from the
    chunk's seed and copied to the host) one `oracle.distance(q, chunk)` call per query - what the reference's per-chunk UDF
    computes (index.py:133-162) - then Arrow's select_k_unstable over the distance column (index.py:165-167)."""
    import pyarrow as pa
    import pyarrow.compute as pc
    import torch

    from oracle import distance as oracle_distance

    use_all_host_threads()
    n, k = cfg["n"], cfg["k"]
    cols = [np.empty(n, dtype=np.float32) for _ in range(len(queries))]
    tq = [torch.from_numpy(np.ascontiguousarray(q)).unsqueeze(0) for q in queries]
    for ci, lo in enumerate(range(0, n, GEN_CHUNK)):
        hi = min(n, lo + GEN_CHUNK)
        chunk = gen_chunk(cfg, ci, device, variant)[: hi - lo].cpu()
        for j, q in enumerate(tq):
            cols[j][lo:hi] = oracle_distance(q, chunk, cfg["metric"]).squeeze(0).numpy()
    out = []
    for j in range(len(queries)):
        table = pa.table({"__ROW__": pa.array(np.arange(n, dtype=np.int64)), "__DISTANCE__": pa.array(cols[j])})
        top = table.take(pc.select_k_unstable(table, min(k, n), [("__DISTANCE__", "ascending")]))
        out.append((top.column("__ROW__").to_numpy(), top.column("__DISTANCE__").to_numpy()))
    return out


def noise_floor(cfg: dict, queries: np.ndarray, max_norm2: float) -> float:
    """Absolute distance floor for the REFERENCE's own fp32 rounding, as in tests/conftest.py::assert_same_neighbours:
    GEMM-form L2 carries ~eps32 (|q|^2 + |x|^2) in d^2 (SURVEY.md 7.3-2); 0.5 - 0.5 cos rounds near 0 / 0.5; an sgemv dot
    product that cancels to ~0 keeps eps32 |q| |x| of accumulation noise."""
    q2 = float((queries.astype(np.float64) ** 2).sum(1).max())
    if cfg["metric"] in ("l2", "euclidean"):
        return 10 * 1e-5 * float(np.sqrt(2.0 ** -22 * (q2 + max_norm2)))
    if cfg["metric"] == "cosine":
        return 2e-7
    return 2.0 ** -22 * float(np.sqrt(q2 * max_norm2))


def parity_block(cfg, search_exact_scan, rows, dist, h_q, device, rank, n_scan=32, n_oracle=4, variant=None, max_norm2=None):
    """Re-check a sample of the timed batch (see the module docstring). `search_exact_scan(queries[m, D]) -> (rows, dist)`
    runs the fp64 scan over the whole (sharded) corpus - collective at N > 1, so every rank calls this function; the
    oracle part runs on rank 0 only. Returns the block on rank 0."""
    n_q = h_q.shape[0]
    pick = np.unique(np.linspace(0, n_q - 1, min(n_scan, n_q)).astype(np.int64))
    t0 = time.perf_counter()
    s_rows, s_dist = search_exact_scan(np.ascontiguousarray(h_q[pick]))
    scan_s = time.perf_counter() - t0
    if rank != 0:
        return None
    # the tensor-core path reranks with the scan's own arithmetic (fp64 accumulation, one rounding): ids and distances are
    # normally bit-equal; where exact terms cancel (distance ~0: a query that is a corpus row) the two fp64 summation
    # orders may differ in the last bits, so the REQUIREMENT is the parity bar with a tight tolerance, bit-equality is reported
    scan_bits = bool(np.array_equal(rows[pick], s_rows) and np.array_equal(dist[pick], s_dist))
    fp64_floor = 4.0 * float(np.sqrt(2.0 ** -52 * ((h_q[pick].astype(np.float64) ** 2).sum(1).max() + (max_norm2 or 1.3 * cfg["d"]))))
    scan_equal = all(same_neighbours(rows[qi], dist[qi], sr, sd, rtol=1e-6, floor=fp64_floor)[0]
                     for qi, sr, sd in zip(pick, s_rows, s_dist))
    o_pick = pick[np.unique(np.linspace(0, len(pick) - 1, min(n_oracle, len(pick))).astype(np.int64))]
    t0 = time.perf_counter()
    ref = oracle_topk_streamed(cfg, h_q[o_pick], device, variant)
    oracle_s = time.perf_counter() - t0
    if max_norm2 is None:
        max_norm2 = 1.3 * cfg["d"]      # N(0,1) rows
    floor = noise_floor(cfg, h_q[o_pick], max_norm2)
    ok_all, ids_all, rel_max = True, True, 0.0
    for (r_rows, r_dist), qi in zip(ref, o_pick):
        ok, ids_equal, rel = same_neighbours(rows[qi], dist[qi], r_rows, r_dist, floor=floor)
        ok_all, ids_all, rel_max = ok_all and ok, ids_all and ids_equal, max(rel_max, rel)
    return {
        "checked_queries": int(len(pick)), "scan_agrees": bool(scan_equal), "scan_ids_and_distances_bit_equal": scan_bits,
        "oracle_queries": int(len(o_pick)), "ids_equal": bool(ids_all), "max_rel_err": rel_max, "within_parity_bar": bool(ok_all),
        "ok": bool(scan_equal and ok_all),
        "how": (f"{len(pick)} queries of the timed batch vs the fp64 CUDA-core scan (FX_PREC_EXACT_SCAN) over the whole corpus, "
                f"same ids, distances within 1e-6 (bit-equality reported); {len(o_pick)} of them vs the oracle (oracle.distance per 65,536-row chunk "
                f"on the host + Arrow select_k_unstable) over all {cfg['n']} rows, ids under (distance, row) order, distances "
                f"within 1e-5 relative"),
        "scan_s": scan_s, "oracle_s": oracle_s,
    }


def roofline_of(cfg_n_shard, n_q_rank, d, k, k_ms, path, clocks, pk):
    """Roofline object of the dominant kernel: algorithmic flops or bytes per launch / CUDA-event kernel time, against the
    measured peak that matches the clock regime of THIS run (burst when the timed region saw no power cap, sustained
    under `sw_power_cap`)."""
    flops = 2.0 * n_q_rank * cfg_n_shard * d
    elem = 2.0 if path == 2 else 4.0     # the bf16 filter streams the bf16 shadow, otherwise the fp32 rows
    bytes_alg = elem * cfg_n_shard * d + 4.0 * n_q_rank * d + 12.0 * n_q_rank * k
    tensor_bound = path in (1, 2) and n_q_rank >= (420 if path == 2 else 210)   # (path 3, the direct scan, reads the fp32 rows once)
    capped = bool(clocks and "sw_power_cap" in (clocks.get("reasons") or []))
    if tensor_bound:
        achieved = flops / (k_ms * 1e-3) / 1e12
        peak = pk["bf16_tflops_sustained"] if capped else pk["bf16_tflops"]
        roof = dict(bound="tensor", achieved=achieved, peak=peak, unit="TFLOP/s", frac=achieved / peak, traffic=None,
                    peak_source=(f"{pk['_source']} bf16 dense, " + ("SUSTAINED (cuBLAS 8192^3 back to back; this run's clock samples show sw_power_cap)"
                                                                     if capped else "BURST (cuBLAS 8192^3 best of 10; no power cap seen in this run's clock samples)")) +
                                ("" if path == 2 else "; this launch issues kind::tf32 MMAs whose nominal rate is half of bf16, so frac <= ~0.5 by construction"),
                    frac_of_burst=achieved / pk["bf16_tflops"], frac_of_sustained=achieved / pk["bf16_tflops_sustained"])
    else:
        achieved = bytes_alg / (k_ms * 1e-3) / 1e9
        peak = pk["hbm_gbs"]
        roof = dict(bound="hbm", achieved=achieved, peak=peak, unit="GB/s", frac=achieved / peak, traffic=None,
                    peak_source=f"{pk['_source']} copy bandwidth")
    roof["algorithmic"] = dict(flops=flops, bytes=bytes_alg, per="launch (one query batch against this rank's shard)")
    return roof


def kernel_name_of(path: int, variant: int) -> str:
    if path == 0:
        return "exact_scan_kernel"
    if path == 3:
        return "knn_direct_kernel (single-launch fp64 scan + in-kernel top-k merge)"
    if path == 1:
        return "knn_tc_filter_kernel<epilogue, tf32> (streaming)"
    if variant & 1:
        return "knn_rq_filter_kernel<epilogue> (resident-query, bf16)"
    return "knn_tc_filter_kernel<epilogue, bf16, pair> (streaming, cta_group::2 CTA pairs)" if variant & 4 \
        else "knn_tc_filter_kernel<epilogue, bf16> (streaming)"


def time_single_gpu(corpus, ctx, cfg, device, steps, warmup, pk, label, variant=None, queries=None, check=True, max_norm2=None,
                    n_scan=16, n_oracle=2):
    """One compact sub-result on ONE GPU (the `also` block): device-resident timing through fx_search_device, kernel time
    from the library's events, parity of a few queries against the fp64 scan and the oracle."""
    import torch

    from fenix_b200 import knn

    metric, k, d = knn.metric_code(cfg["metric"]), cfg["k"], cfg["d"]
    h_q = query_batch(cfg) if queries is None else queries
    n_q = h_q.shape[0]
    d_q = torch.from_numpy(h_q).to(device)
    rows = torch.empty((n_q, k), dtype=torch.int64, device=device)
    dist = torch.empty((n_q, k), dtype=torch.float32, device=device)
    torch.cuda.synchronize(device)
    st0 = corpus.stats()
    for _ in range(warmup):
        corpus.search_device(d_q.data_ptr(), n_q, metric, k, knn.PREC_FP32, rows.data_ptr(), dist.data_ptr())
    sampler = ClockSampler(device.index or 0)
    sampler.start()
    k_ms, s_ms = [], []
    t0 = time.perf_counter()
    for _ in range(steps):
        corpus.search_device(d_q.data_ptr(), n_q, metric, k, knn.PREC_FP32, rows.data_ptr(), dist.data_ptr())
        st = corpus.stats()
        k_ms.append(st.last_main_kernel_ms); s_ms.append(st.last_search_ms)
    torch.cuda.synchronize(device)
    elapsed = time.perf_counter() - t0
    clocks = sampler.stop()
    st1 = corpus.stats()
    n_runs = steps + warmup
    out = {
        "workload": label, "n_rows": cfg["n"], "dim": d, "metric": cfg["metric"], "k": k, "queries_per_step": n_q,
        "ms_per_step": elapsed / steps * 1e3, "value": n_q / (elapsed / steps), "unit": "queries/s", "steps": steps, "warmup": warmup,
        "kernel_ms": float(np.mean(k_ms)), "search_device_ms": float(np.mean(s_ms)),
        "kernel": kernel_name_of(st1.last_path, st1.last_variant), "sample_prepass": bool(st1.last_variant & 2),
        "refined_queries_per_step": (st1.refined_queries - st0.refined_queries) / n_runs,
        "fallback_queries_per_step": (st1.fallback_queries - st0.fallback_queries) / n_runs,
        "clocks": clocks,
    }
    roof = roofline_of(cfg["n"], n_q, d, k, float(np.mean(k_ms)), st1.last_path, clocks, pk)
    out["roofline"] = {key: roof[key] for key in ("bound", "achieved", "peak", "unit", "frac")}
    if check:
        def scan(qs):
            r, dd = corpus.search(qs, cfg["metric"], k, knn.PREC_EXACT_SCAN)
            return r, dd
        pb = parity_block(cfg, scan, rows.cpu().numpy(), dist.cpu().numpy(), h_q, device, 0, n_scan=n_scan, n_oracle=n_oracle,
                          variant=variant, max_norm2=max_norm2)
        out["parity"] = {key: pb[key] for key in ("checked_queries", "scan_agrees", "scan_ids_and_distances_bit_equal", "oracle_queries", "ids_equal",
                                                  "max_rel_err", "within_parity_bar", "ok")}
    return out


def ivf_block(corpus, cfg: dict, device, n_cells=1024, n_probe=8, n_q=256, k=10) -> dict:
    """SURVEY section 8f rank 4 at C2 scale: a batch of IVF searches (coding + probes; here: cells = nearest of 1024 random
    centroids, probes = a query's 8 nearest centroids) as ONE fx_search_cells launch, against the loop of per-query masked
    searches it replaces (the reference's per-query `isin` filter, index.py:119-126), same answers required."""
    import torch

    from fenix_b200 import knn

    gen = torch.Generator(device=device)
    gen.manual_seed(4242)
    cent = torch.randn((n_cells, cfg["d"]), generator=gen, device=device, dtype=torch.float32)
    cells = []
    for ci in range((cfg["n"] + GEN_CHUNK - 1) // GEN_CHUNK):
        block = gen_chunk(cfg, ci, device)[: min(GEN_CHUNK, cfg["n"] - ci * GEN_CHUNK)]
        cells.append(torch.cdist(block, cent).argmin(dim=1).cpu().numpy())
    cell = np.concatenate(cells).astype(np.int64)
    h_q = query_batch(cfg)[:n_q]
    probes = torch.cdist(torch.from_numpy(h_q).to(device), cent).topk(n_probe, dim=1, largest=False).indices.cpu().numpy().astype(np.int32)
    corpus.set_cells(cell)
    sizes = np.bincount(cell, minlength=n_cells)
    probed = float(sizes[probes].sum(1).mean())
    for _ in range(3):
        rows, dist = corpus.search_cells(h_q, cfg["metric"], k, probes)
    t, dev_ms = [], []
    for _ in range(10):
        t0 = time.perf_counter()
        rows, dist = corpus.search_cells(h_q, cfg["metric"], k, probes)
        t.append(time.perf_counter() - t0)
        dev_ms.append(corpus.stats().last_search_ms)
    one = float(np.median(t))
    n_loop, same = 8, True
    masks = [np.isin(cell, probes[i]).astype(np.uint8) for i in range(n_loop)]
    corpus.search(h_q[0], cfg["metric"], k, knn.PREC_FP32, row_mask=masks[0])
    t0 = time.perf_counter()
    for i in range(n_loop):
        r, dd = corpus.search(h_q[i], cfg["metric"], k, knn.PREC_FP32, row_mask=masks[i])
        same = same and np.array_equal(r[0], rows[i]) and np.array_equal(dd[0], dist[i])
    loop = (time.perf_counter() - t0) / n_loop * n_q
    r_s, d_s = corpus.search(h_q[n_loop], cfg["metric"], k, knn.PREC_EXACT_SCAN, row_mask=np.isin(cell, probes[n_loop]).astype(np.uint8))
    same = same and np.array_equal(r_s[0], rows[n_loop]) and np.array_equal(d_s[0], dist[n_loop])
    return {
        "workload": f"batched IVF over the C2 corpus: {n_cells} cells, {n_probe} probes, k={k}, {n_q} queries per call (host buffers in and out)",
        "probed_rows_per_query": probed, "ms_per_step": one * 1e3, "value": n_q / one, "unit": "queries/s",
        "kernel": "knn_direct_kernel<LISTS> (one launch per batch: query q scans the posting lists of its probe cells)",
        "kernel_ms": float(np.mean(dev_ms)),
        "roofline": {"bound": "hbm", "unit": "GB/s", "achieved": probed * cfg["d"] * 4 * n_q / (float(np.mean(dev_ms)) * 1e-3) / 1e9,
                     "note": "bytes of the probed rows (gathered 512-byte rows) / device time of the call incl. its copies"},
        "masked_loop_ms_per_step": loop * 1e3, "masked_loop_note": f"one masked fx_search per query, extrapolated from {n_loop} queries",
        "speedup_over_masked_loop": loop / one,
        "parity": {"checked_queries": n_loop + 1, "ok": bool(same), "how": "bit-equal to the per-query masked searches (tensor-core path) and to a masked fp64 scan"},
    }


def also_block(args, ctx, c3_corpus, device, pk) -> dict:
    """The other BASELINE configs that fit one GPU and SURVEY section 8d's stress inputs, as compact lines (N = 1 only)."""
    import torch

    out = {}
    steps, warmup = 5, 3
    if c3_corpus is not None:
        for b in (1, 64):
            cfg = dict(CONFIGS[f"c5_{b}"], data_num=CONFIGS["c3"]["num"])   # C5 searches the resident C3 corpus
            out[f"c5_{b}"] = time_single_gpu(c3_corpus, ctx, cfg, device, 20, 5, pk, cfg["label"], n_scan=8, n_oracle=1)
    for name in ("c2", "c4s"):
        cfg = dict(CONFIGS[name])
        corpus = build_shard(cfg, ctx, 0, cfg["n"], device)
        out[name] = time_single_gpu(corpus, ctx, cfg, device, steps, warmup, pk, cfg["label"])
        if name == "c2":
            out["ivf_batched"] = ivf_block(corpus, cfg, device)
        corpus.close()
    # C1 shape, one query per search: the latency path. The 51 MB shard is L2-resident in steady state (that IS the
    # serving regime of a shard this small; nothing is flushed between searches and the line says so).
    cfg = dict(CONFIGS["c1"])
    corpus = build_shard(cfg, ctx, 0, cfg["n"], device)
    r = time_single_gpu(corpus, ctx, cfg, device, 200, 20, pk, cfg["label"], n_scan=1, n_oracle=1)
    r["l2_policy"] = "shard (51 MB of fp32 rows) stays L2-resident between searches: steady-state serving of a small shard, not flushed"
    r["roofline"]["note"] = "bytes from L2, not HBM: achieved / HBM peak > 1 is expected; the floor is the L2 read rate"
    h_q = query_batch(cfg)
    o_r = np.empty((1, cfg["k"]), np.int64); o_d = np.empty((1, cfg["k"]), np.float32)
    from fenix_b200 import knn as _knn
    lat = []
    for i in range(520):
        t0 = time.perf_counter()
        corpus.search_raw(h_q.ctypes.data, 1, _knn.metric_code(cfg["metric"]), cfg["k"], _knn.PREC_FP32, o_r.ctypes.data, o_d.ctypes.data)
        lat.append(time.perf_counter() - t0)
    lat = np.array(lat[20:]) * 1e6
    r["e2e_fx_search_us"] = {"p50": float(np.median(lat)), "p99": float(np.percentile(lat, 99)),
                             "what": "host clock around fx_search (pageable host query in, host results out), 500 calls"}
    out["c1"] = r
    corpus.close()
    # stress inputs at C2 scale (L2, k = 100, 10k queries): what the certificate / refinement tiers cost off the
    # friendly i.i.d. Gaussian case
    base = dict(CONFIGS["c2"])
    gauss_ms = out["c2"]["ms_per_step"]
    for variant in STRESS:
        cfg = dict(base)
        corpus = build_shard(cfg, ctx, 0, cfg["n"], device, None if variant == "queries_from_corpus" else variant)
        queries = None
        max_norm2 = None
        if variant == "queries_from_corpus":
            # every query IS a corpus row (distance 0 to itself): rows of chunk 3
            queries = gen_chunk(cfg, 3, device)[: cfg["q"]].cpu().numpy()
        elif variant == "clustered":
            max_norm2 = 130.0 * cfg["d"]
        elif variant == "norm_outliers":
            max_norm2 = 1e4 * 1.3 * cfg["d"]
        r = time_single_gpu(corpus, ctx, cfg, device, steps, warmup, pk, f"stress/{variant}: C2 shape, L2, k=100",
                            variant=None if variant == "queries_from_corpus" else variant, queries=queries, max_norm2=max_norm2)
        r["vs_gaussian_time"] = r["ms_per_step"] / gauss_ms
        out[f"stress_{variant}"] = r
        corpus.close()
    torch.cuda.synchronize(device)
    return out


def dump_outputs(out_dir: str, rows: np.ndarray, dist: np.ndarray) -> None:
    """The search result a caller receives, one line per query of the batch: `neighbour_rows.npy` (global row numbers as
    float64, exact below 2^53; -1 pads), `neighbour_distances.npy` (float32) and `query_index.npy` (float64: which query of
    the batch each line answers). Above DUMP_MAX_BYTES in all, a fixed sample of the queries (seed 0, in batch order)."""
    n_q, k = rows.shape
    per_query = k * (8 + 4) + 8
    index = np.arange(n_q)
    if n_q * per_query > DUMP_MAX_BYTES:
        index = np.sort(np.random.default_rng(0).choice(n_q, DUMP_MAX_BYTES // per_query, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "neighbour_rows.npy"), rows[index].astype(np.float64))
    np.save(os.path.join(out_dir, "neighbour_distances.npy"), dist[index].astype(np.float32))
    np.save(os.path.join(out_dir, "query_index.npy"), index.astype(np.float64))


def run_ours(args, cfg: dict) -> dict:
    import torch
    import torch.distributed as td

    from fenix_b200 import knn
    from fenix_b200.dist import ReplicaSearcher, ShardedSearcher, shard_bounds

    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torchrun --nproc-per-node {args.gpus}")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: the search path has no CPU fallback")
    device = torch.device("cuda", local)
    torch.cuda.set_device(device)
    if world > 1:
        td.init_process_group("nccl", device_id=device)
        td.barrier()

    def barrier():
        if world > 1:
            td.barrier()
        torch.cuda.synchronize(device)

    ctx = knn.Context(local)
    # N > 1: row-shard the corpus, or - small corpora with big batches - replicate it and split the query batch
    par = args.parallelism
    if par == "auto":
        par = "queries" if 8.0 * cfg["n"] * cfg["d"] <= 8e9 and cfg["q"] // max(world, 1) >= 256 else "rows"
    by_queries = par == "queries" and world > 1
    lo, hi = (0, cfg["n"]) if by_queries else shard_bounds(cfg["n"], world, rank)
    t_build = time.perf_counter()
    corpus = build_shard(cfg, ctx, lo, hi, device, args.variant)
    t_build = time.perf_counter() - t_build
    searcher = ReplicaSearcher(corpus) if by_queries else ShardedSearcher(corpus)
    metric, k, n_q, d = knn.metric_code(cfg["metric"]), cfg["k"], cfg["q"], cfg["d"]
    prec = {"fp32": knn.PREC_FP32, "tf32": knn.PREC_TF32, "scan": knn.PREC_EXACT_SCAN}[args.precision]

    h_q = torch.from_numpy(query_batch(cfg)).pin_memory()
    d_q = h_q.to(device)
    h_rows = torch.empty((n_q, k), dtype=torch.int64).pin_memory()
    h_dist = torch.empty((n_q, k), dtype=torch.float32).pin_memory()

    # ---- device-resident timing (value) ----
    for _ in range(args.warmup):
        searcher.search_device(d_q, metric, k, prec)
    sampler = ClockSampler(local)
    barrier()
    if rank == 0:
        sampler.start()
    st0 = corpus.stats()
    kernel_ms, search_ms, xchg_ms = [], [], []
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        rows, dist = searcher.search_device(d_q, metric, k, prec)
        st = corpus.stats()
        kernel_ms.append(st.last_main_kernel_ms)
        search_ms.append(st.last_search_ms)
        xchg_ms.append(st.last_exchange_ms)
    barrier()
    elapsed = time.perf_counter() - t0
    st1 = corpus.stats()
    clocks = sampler.stop() if rank == 0 else None
    launches = st1.kernel_launches - st0.kernel_launches + (args.steps if world > 1 and not by_queries else 0)   # + merge kernels
    fallback = st1.fallback_queries - st0.fallback_queries
    refined = st1.refined_queries - st0.refined_queries

    # ---- end to end with HOST buffers: pinned queries in, pinned results out, copies inside the timed region.
    # N = 1: the reference-facing C-ABI call itself (fx_search on host pointers); N > 1: fx_search_sharded - every rank
    # uploads 1/N of the batch, the slices are all-gathered over NVLink, shard search, candidate all-gather, merge, and the
    # result is read back on rank 0.
    def e2e_step():
        if world == 1:
            corpus.search_raw(h_q.data_ptr(), n_q, metric, k, prec, h_rows.data_ptr(), h_dist.data_ptr())
        else:
            searcher.search_host(h_q, metric, k, prec, h_rows, h_dist, result_rank=0)

    for _ in range(max(1, min(args.warmup, 3))):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        e2e_step()
    barrier()
    e2e_elapsed = time.perf_counter() - t0
    rows_h, dist_h = rows.cpu().numpy(), dist.cpu().numpy()
    if rank == 0:   # the two paths must agree (same kernels, different plumbing)
        assert np.array_equal(h_rows.numpy(), rows_h) and np.array_equal(h_dist.numpy(), dist_h), \
            "e2e result differs from the device-resident result"
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, rows_h, dist_h)

    def rank_max(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=device)
        td.all_reduce(t, op=td.ReduceOp.MAX)
        return float(t.item())

    elapsed = rank_max(elapsed)
    e2e_elapsed = rank_max(e2e_elapsed)
    k_ms = rank_max(float(np.mean(kernel_ms)))
    s_ms = rank_max(float(np.mean(search_ms)))
    x_ms = rank_max(float(np.mean(xchg_ms)))

    # ---- recall of the approximate mode against the exact result ----
    recall = None
    path = st1.last_path            # 0 scan, 1 TF32 filter, 2 bf16 filter
    if args.precision == "fp32" and path >= 1:
        approx = knn.PREC_BF16 if path == 2 else knn.PREC_TF32
        r_t, _ = searcher.search_device(d_q, metric, k, approx)
        a, b = rows_h, r_t.cpu().numpy()
        recall = float(np.mean([len(set(x) & set(y)) / k for x, y in zip(a, b)]))

    # ---- parity of the timed batch, inside this run (collective: every rank takes part in the scan) ----
    parity = None
    if not args.no_parity:
        def scan(qs: np.ndarray):
            tq = torch.from_numpy(qs).to(device)
            r, dd = searcher.search_device(tq, metric, k, knn.PREC_EXACT_SCAN)
            return r.cpu().numpy(), dd.cpu().numpy()
        parity = parity_block(cfg, scan, rows_h, dist_h, h_q.numpy(), device, rank, variant=args.variant,
                              max_norm2={"clustered": 130.0 * d, "norm_outliers": 1.3e4 * d}.get(args.variant))

    out = None
    if rank == 0:
        pk = peaks()
        n_shard = hi - lo
        n_q_rank = -(-n_q // world) if by_queries else n_q     # queries one launch of this rank answers
        variant = int(getattr(st1, "last_variant", 0))
        roof = roofline_of(n_shard, n_q_rank, d, k, k_ms, path, clocks, pk)
        roof["traffic"], roof["traffic_source"] = ncu_traffic(args.config if not (args.rows or args.queries) else "", world)
        roof.update(kernel=kernel_name_of(path, variant), sample_prepass=bool(variant & 2), kernel_ms=k_ms, search_device_ms=s_ms,
                    exchange_ms=x_ms if world > 1 and not by_queries else 0.0)
        out = {
            "metric": "knn_qps", "value": n_q / (elapsed / args.steps), "unit": "queries/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": elapsed / args.steps * 1e3,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32" if args.precision != "tf32" else "tf32", "data": "synthetic",
            "config": workload_config(args, cfg),
            "parallelism": (f"replicated corpus, query batch split x{world}" if by_queries else f"row-shard x{world}"),
            "details": {
                "path": {0: "fp64 exact scan (CUDA cores)", 1: "tcgen05 TF32 filter + fp64 rerank + certificate",
                         2: "tcgen05 bf16-shadow filter + fp64 rerank + certificate"}[path],
                "precision_arg": args.precision,
                "refined_queries": int(refined), "fallback_queries": int(fallback), "corpus_build_s": t_build,
                "exchange": ("none" if world == 1 else
                             "replicated corpus: torch.distributed all-gather of result slices" if by_queries else
                             "fx_search_sharded: the library's own NCCL communicator, all-gather of k x N candidates + merge kernel on the "
                             "search stream, one host synchronisation per search"),
            },
            "clocks": clocks,
            "e2e": {"value": n_q / (e2e_elapsed / args.steps), "unit": "queries/s",
                    "api": "fx_search (C ABI, pinned host buffers)" if world == 1 else
                           ("fenix_b200.dist.ReplicaSearcher.search_host" if by_queries else "fx_search_sharded (C ABI, pinned host buffers)"),
                    "h2d_bytes_per_step": int(h_q.numel() * 4), "d2h_bytes_per_step": int(n_q * k * 12),
                    "h2d_note": "whole job: every rank uploads 1/N of the query batch, the slices are all-gathered over NVLink" if world > 1 else "",
                    "ms_per_step": e2e_elapsed / args.steps * 1e3},
            "gpu_launches": int(launches),
            "roofline": roof,
            # `value` is the slower of the two clocks: the host clock around the K steps (barrier + device synchronise on
            # both sides, max over ranks) also pays the library's host-side work between its kernels; the CUDA-event time
            # is recorded by the library on its own stream around each search (max over ranks, mean over steps)
            "timing": {"value_from": "host clock between device-synchronised barriers, max over ranks",
                       "cuda_event_ms_per_step": s_ms, "host_clock_ms_per_step": elapsed / args.steps * 1e3},
        }
        if parity is not None:
            out["parity"] = parity
        if recall is not None:
            out["approx_mode_recall_at_k"] = {"mode": "bf16" if path == 2 else "tf32", "recall": recall}
        if world == 1 and not args.no_cpu_baseline:
            out["cpu_baseline"] = time_reference(cfg, steps=3, warmup=1, budget_s=20.0)
        if world == 1 and not args.no_also and args.config == "c3" and not (args.rows or args.queries):
            out["also"] = also_block(args, ctx, corpus, device, pk)
    if isinstance(searcher, ShardedSearcher):
        searcher.close()
    corpus.close()
    ctx.close()
    if world > 1:
        td.barrier()
        td.destroy_process_group()
    return out


def run_reference(args, cfg: dict):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return None
    base = time_reference(cfg, steps=args.steps, warmup=args.warmup, budget_s=float(os.environ.get("FENIX_BENCH_BUDGET_S", 120.0)))
    return {
        "impl": "reference", "metric": "knn_qps", "value": base["value"], "unit": "queries/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": base["ms_per_step"],
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, cfg),
        "parallelism": "host cores only (rank 0)",
        "cpu_baseline": {k: base[k] for k in ("value", "unit", "cores", "kind", "sample", "best_case")},
        "e2e": {"value": base["value"], "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--config", default="c3", choices=sorted(CONFIGS))
    ap.add_argument("--precision", default="fp32", choices=["fp32", "tf32", "scan"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the in-run parity block (tuning runs)")
    ap.add_argument("--no-also", action="store_true", help="skip the `also` sub-results (tuning runs)")
    ap.add_argument("--parallelism", default="auto", choices=["auto", "rows", "queries"],
                    help="N > 1: row-shard the corpus, or replicate it and split the query batch (auto: replicate when the "
                         "corpus and its shadows take <= 8 GB and every rank still gets >= 256 queries)")
    ap.add_argument("--variant", default=None, choices=[v for v in STRESS if v != "queries_from_corpus"],
                    help="tuning only: a stress variant of the synthetic corpus (SURVEY.md section 8d)")
    ap.add_argument("--rows", type=int, default=0, help="tuning only: override the corpus row count of the config")
    ap.add_argument("--queries", type=int, default=0, help="tuning only: override the query batch of the config")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the neighbour rows and distances of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs records the GPU path: the reference arm's last step depends on its time budget")
    sys.dont_write_bytecode = True      # the tree may be read-only: nothing is cached in it
    cfg = dict(CONFIGS[args.config])
    if args.rows or args.queries or args.variant:
        cfg["n"] = args.rows or cfg["n"]
        cfg["q"] = args.queries or cfg["q"]
        cfg["label"] += f" [TUNING OVERRIDE rows={cfg['n']} queries={cfg['q']} variant={args.variant}: not a benchmark configuration]"
    out = run_reference(args, cfg) if args.impl == "reference" else run_ours(args, cfg)
    if out is not None:
        print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()

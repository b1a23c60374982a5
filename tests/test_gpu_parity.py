"""GPU parity tests: the CUDA path (through the C ABI) against the oracle and the committed
outputs of the live reference. Bar: neighbour ids bit-exact under (distance, row) order,
distances within 1e-5 relative (BASELINE.json north_star), tolerance written in conftest."""
import os
import socket

import numpy as np
import pyarrow as pa
import pyarrow.compute as pc
import pytest

import fenix_b200 as fenix
from conftest import METRICS, assert_same_neighbours, golden_cases, golden_filter, load_golden, table_of
from fenix_b200 import knn
from oracle import brute_force_f64, canonical, search_rows

pytestmark = pytest.mark.gpu


def client_root(served):
    return served[3]


def free_port():
    """A port no one listens on now: runs of the suite that share a host do not collide."""
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


# "fp32": the library's own routing (a handful of queries over a small shard take the single-launch direct scan);
# "fp32_tc": the same exact mode with the direct scan switched off, so the tensor-core path answers; "scan": the checker
PRECISIONS = {"fp32": knn.PREC_FP32, "fp32_tc": knn.PREC_FP32, "scan": knn.PREC_EXACT_SCAN}


def search_as(ctx, c, prec, queries, metric, k, **kw):
    if prec != "fp32_tc":
        return c.search(queries, metric, k, PRECISIONS[prec], **kw)
    ctx.set_option("FENIX_DIRECT", 0)
    try:
        return c.search(queries, metric, k, PRECISIONS[prec], **kw)
    finally:
        ctx.set_option("FENIX_DIRECT", None)


@pytest.fixture(scope="module")
def ctx(built_library):
    c = knn.Context(0)
    yield c
    c.close()


def make_corpus(ctx, x, row_base=0, pieces=3):
    c = knn.Corpus(ctx, len(x), x.shape[1], row_base=row_base)
    step = max(1, -(-len(x) // pieces))
    for lo in range(0, len(x), step):
        c.append(x[lo: lo + step])
    return c.finalize()


# ---- committed reference outputs ---------------------------------------------------------
@pytest.mark.parametrize("prec", list(PRECISIONS))
@pytest.mark.parametrize("case", [c for c in golden_cases() if c not in ("all_rows", "k_ge_n", "filtered")])
@pytest.mark.parametrize("metric", METRICS)
def test_topk_matches_live_reference_outputs(ctx, case, metric, prec):
    g = load_golden(case)
    corpus, queries, k = g["corpus"], g["queries"], int(g["k"])
    c = make_corpus(ctx, corpus)
    rows, dist = search_as(ctx, c, prec, queries, metric, k)
    for qi in range(len(queries)):
        assert_same_neighbours(rows[qi], dist[qi], g[f"{metric}:{qi}:id"], g[f"{metric}:{qi}:dist"],
                               corpus, queries[qi], metric)
        # our own order is canonical: (distance, row) ascending
        assert np.array_equal(canonical(rows[qi], dist[qi])[0], rows[qi])
    c.close()


@pytest.mark.parametrize("metric", METRICS)
def test_distance_column_matches_reference(ctx, metric):
    g = load_golden("all_rows")
    c = make_corpus(ctx, g["corpus"])
    for qi, q in enumerate(g["queries"]):
        d = c.distances(q, metric)
        ref = g[f"{metric}:{qi}:dist"]  # all rows, table order
        assert np.array_equal(g[f"{metric}:{qi}:id"], np.arange(len(ref)))
        np.testing.assert_allclose(d, ref, rtol=1e-5, atol=2e-6)
    c.close()


@pytest.mark.parametrize("metric", ["l2", "cosine", "dot"])
def test_masked_search_matches_reference_filter(ctx, metric):
    g = load_golden("filtered")
    corpus, k, mod = g["corpus"], int(g["k"]), int(g["filter_mod"])
    mask = (np.arange(len(corpus)) % mod == 0).astype(np.uint8)
    c = make_corpus(ctx, corpus)
    rows, dist = c.search(g["queries"], metric, k, knn.PREC_FP32, row_mask=mask)
    for qi in range(len(g["queries"])):
        assert (rows[qi] % mod == 0).all()
        assert_same_neighbours(rows[qi], dist[qi], g[f"{metric}:{qi}:id"], g[f"{metric}:{qi}:dist"],
                               corpus, g["queries"][qi], metric)
    c.close()


# ---- seeded inputs against the oracle ----------------------------------------------------
@pytest.mark.parametrize("prec", list(PRECISIONS))
@pytest.mark.parametrize("shape", [(20000, 128, 64, 10), (30000, 96, 33, 100), (5000, 768, 16, 10), (4097, 100, 5, 37)])
@pytest.mark.parametrize("metric", ["l2", "cosine", "dot"])
def test_seeded_parity_with_oracle(ctx, shape, metric, prec):
    n, d, nq, k = shape
    rng = np.random.default_rng(n + d)
    corpus = rng.standard_normal((n, d), dtype=np.float32)
    queries = rng.standard_normal((nq, d), dtype=np.float32)
    c = make_corpus(ctx, corpus)
    rows, dist = search_as(ctx, c, prec, queries, metric, k)
    table = table_of(corpus, 4096)
    for qi in range(0, nq, max(1, nq // 6)):  # the oracle is O(N*D) per query
        ref_rows, ref_dist = search_rows(table, "vector", queries[qi], metric, k)
        assert_same_neighbours(rows[qi], dist[qi], ref_rows, ref_dist, corpus, queries[qi], metric)
    want_rows, want_dist = brute_force_f64(corpus, queries, metric, k)
    assert np.array_equal(rows, want_rows)
    np.testing.assert_allclose(dist, want_dist, rtol=2e-6, atol=1e-6)
    c.close()


@pytest.mark.parametrize("prec", list(PRECISIONS))
def test_duplicates_are_ordered_by_row(ctx, prec):
    rng = np.random.default_rng(5)
    corpus = rng.standard_normal((3000, 32), dtype=np.float32)
    corpus[1000:1400] = corpus[17]  # 400 copies of the winner (SURVEY.md 3.1 fact 2)
    c = make_corpus(ctx, corpus)
    for metric in ("l2", "cosine", "dot"):
        rows, dist = search_as(ctx, c, prec, corpus[17], metric, 10)
        want_rows, want_dist = brute_force_f64(corpus, corpus[17], metric, 10)
        assert np.array_equal(rows, want_rows), metric
        np.testing.assert_allclose(dist, want_dist, rtol=2e-6, atol=1e-6)
        if metric == "l2":
            assert rows[0].tolist() == [17] + list(range(1000, 1009)) and (dist[0] == 0).all()
    c.close()


def test_clustered_data_of_reference_tests(ctx):
    """tests/test_flight.py:17-35 data (tight clusters far from the origin) and uniform queries (:104)."""
    rng = np.random.default_rng(11)
    parts = []
    for _ in range(20):
        x = rng.standard_normal((1000, 256), dtype=np.float32)
        parts.append(x + 10 * x[0, :])
    corpus = np.concatenate(parts)
    queries = rng.random((8, 256), dtype=np.float32)
    c = make_corpus(ctx, corpus)
    table = table_of(corpus, 1000)
    for metric in METRICS:
        rows, dist = c.search(queries, metric, 10)
        for qi in range(len(queries)):
            ref_rows, ref_dist = search_rows(table, "vector", queries[qi], metric, 10)
            assert_same_neighbours(rows[qi], dist[qi], ref_rows, ref_dist, corpus, queries[qi], metric)
    c.close()


def test_edge_cases(ctx):
    rng = np.random.default_rng(3)
    corpus = rng.standard_normal((50, 12), dtype=np.float32)
    c = make_corpus(ctx, corpus)
    # k > N: padded with (-1, +inf)
    rows, dist = c.search(corpus[:2], "l2", 64)
    assert (rows[:, 50:] == -1).all() and np.isinf(dist[:, 50:]).all()
    assert sorted(rows[0, :50].tolist()) == list(range(50))
    # zero queries
    r0, d0 = c.search(np.empty((0, 12), np.float32), "l2", 3)
    assert r0.shape == (0, 3)
    with pytest.raises(ValueError):
        c.search(corpus[:1], "l2", 0)
    # any k is served (the reference's select_k_unstable takes any maxval): far beyond N pads
    rows, dist = c.search(corpus[:1], "l2", 5000)
    assert rows.shape == (1, 5000) and sorted(rows[0, :50].tolist()) == list(range(50)) and (rows[0, 50:] == -1).all()
    with pytest.raises(ValueError):
        c.search(np.zeros((1, 5), np.float32), "l2", 3)
    with pytest.raises(knn.FenixKnnError):
        c.append(corpus)  # finalized
    c.close()
    # empty shard
    e = knn.Corpus(ctx, 0, 12).finalize()
    rows, dist = e.search(corpus[:2], "dot", 4)
    assert (rows == -1).all() and np.isinf(dist).all()
    e.close()
    # zero vectors: cosine eps branch gives 0.5
    z = np.zeros((4, 12), np.float32)
    z[1] = 1
    c = make_corpus(ctx, z)
    rows, dist = c.search(np.zeros((1, 12), np.float32), "cosine", 4)
    assert np.allclose(dist, 0.5) and rows[0].tolist() == [0, 1, 2, 3]
    c.close()


def test_row_base_and_sharded_merge_equal_single_shard(ctx):
    """Fake 8-way row sharding on one GPU: shard-local top-k + fx_merge_topk == unsharded search."""
    import torch
    from fenix_b200.dist import shard_bounds

    rng = np.random.default_rng(21)
    corpus = rng.standard_normal((10007, 64), dtype=np.float32)
    corpus[9000] = corpus[12]
    queries = np.concatenate([rng.standard_normal((15, 64), dtype=np.float32), corpus[12:13]])
    k, world = 10, 8
    whole = make_corpus(ctx, corpus)
    want_rows, want_dist = whole.search(queries, "l2", k)
    parts_r, parts_d = [], []
    for r in range(world):
        lo, hi = shard_bounds(len(corpus), world, r)
        s = make_corpus(ctx, corpus[lo:hi], row_base=lo)
        rr, dd = s.search(queries, "l2", k)
        assert rr.min() >= lo and rr.max() < hi
        parts_r.append(rr)
        parts_d.append(dd)
        s.close()
    dev = torch.device("cuda", 0)
    g_rows = torch.from_numpy(np.stack(parts_r)).to(dev)
    g_dist = torch.from_numpy(np.stack(parts_d)).to(dev)
    out_rows = torch.empty((len(queries), k), dtype=torch.int64, device=dev)
    out_dist = torch.empty((len(queries), k), dtype=torch.float32, device=dev)
    torch.cuda.synchronize()
    ctx.merge_topk_device(g_rows.data_ptr(), g_dist.data_ptr(), world, len(queries), k, out_rows.data_ptr(), out_dist.data_ptr())
    assert np.array_equal(out_rows.cpu().numpy(), want_rows)
    assert np.array_equal(out_dist.cpu().numpy(), want_dist)
    whole.close()


@pytest.mark.parametrize("metric", ["l2", "cosine", "dot"])
def test_large_k_runs_in_passes(ctx, metric):
    """k above 2048: the fp64 scan runs in passes of 2048 neighbours, each admitting only keys above the last key of the
    pass before; duplicated rows sit across the pass boundary (ties are broken by row, so the passes still partition)."""
    from oracle import brute_force_f64

    rng = np.random.default_rng(77)
    corpus = rng.standard_normal((9000, 24), dtype=np.float32)
    corpus[4000:4100] = corpus[100:200]          # 100 duplicated rows
    queries = np.concatenate([rng.standard_normal((3, 24), dtype=np.float32), corpus[150:151]])
    c = make_corpus(ctx, corpus)
    for k in (2049, 5000, 9000, 9500):
        rows, dist = c.search(queries, metric, k)
        want_rows, want_dist = brute_force_f64(corpus, queries, metric, k)
        kk = min(k, len(corpus))
        assert np.array_equal(rows[:, :kk], want_rows), (metric, k)
        assert np.allclose(dist[:, :kk], want_dist, rtol=3e-7, atol=3e-6), (metric, k)
        assert (rows[:, kk:] == -1).all()
    c.close()


def test_merge_of_many_long_lists(ctx):
    """lists * k above 8192 entries: the rank merge (no shared-memory limit) equals one unsharded search; k = 1500 over 8
    shards is the case a 1024 < k <= 2048 search hits on an 8-GPU box."""
    import torch
    from fenix_b200.dist import shard_bounds

    rng = np.random.default_rng(31)
    corpus = rng.standard_normal((24_000, 16), dtype=np.float32)
    corpus[20_000:20_050] = corpus[:50]
    queries = np.concatenate([rng.standard_normal((5, 16), dtype=np.float32), corpus[7:8]])
    k, world = 1500, 8
    whole = make_corpus(ctx, corpus)
    want_rows, want_dist = whole.search(queries, "l2", k)
    parts_r, parts_d = [], []
    for r in range(world):
        lo, hi = shard_bounds(len(corpus), world, r)
        s = make_corpus(ctx, corpus[lo:hi], row_base=lo)
        rr, dd = s.search(queries, "l2", k)
        parts_r.append(rr)
        parts_d.append(dd)
        s.close()
    dev = torch.device("cuda", 0)
    g_rows = torch.from_numpy(np.stack(parts_r)).to(dev)
    g_dist = torch.from_numpy(np.stack(parts_d)).to(dev)
    out_rows = torch.empty((len(queries), k), dtype=torch.int64, device=dev)
    out_dist = torch.empty((len(queries), k), dtype=torch.float32, device=dev)
    torch.cuda.synchronize()
    ctx.merge_topk_device(g_rows.data_ptr(), g_dist.data_ptr(), world, len(queries), k, out_rows.data_ptr(), out_dist.data_ptr())
    assert np.array_equal(out_rows.cpu().numpy(), want_rows)
    assert np.array_equal(out_dist.cpu().numpy(), want_dist)
    whole.close()


@pytest.mark.parametrize("metric", ["l2", "cosine", "dot"])
@pytest.mark.parametrize("shape", [(20_000, 256, 300, 10), (50_000, 768, 130, 10), (30_000, 200, 257, 37), (12_345, 448, 129, 100)])
def test_cta_pair_streaming_kernel(ctx, shape, metric):
    """Wide rows (from 7 k-blocks on; narrower ones here by FENIX_TC_PAIR=1) and at least two query tiles take the CTA-pair
    (cta_group::2) streaming kernel: ragged query tiles (the second CTA of a pair holds a near-empty tile), odd widths, a
    row mask, and cosine without the normalised shadow (the multiplicative epilogue) - all against the fp64 scan, a few
    queries against the oracle."""
    from oracle import search_rows

    n, d, nq, k = shape
    rng = np.random.default_rng(n + d)
    corpus = rng.standard_normal((n, d), dtype=np.float32)
    queries = rng.standard_normal((nq, d), dtype=np.float32)
    c = make_corpus(ctx, corpus)
    rows_auto, dist_auto = c.search(queries, metric, k)
    assert bool(c.stats().last_variant & 4) == (d >= 448), "auto: CTA pairs from 7 k-blocks per row on"
    ctx.set_option("FENIX_TC_PAIR", 1)
    rows, dist = c.search(queries, metric, k)
    assert c.stats().last_variant & 4, "expected the CTA-pair kernel"
    assert np.array_equal(rows, rows_auto) and np.array_equal(dist, dist_auto)
    rows_s, dist_s = c.search(queries, metric, k, knn.PREC_EXACT_SCAN)
    assert np.array_equal(rows, rows_s) and np.array_equal(dist, dist_s)
    table = table_of(corpus, 4096)
    for qi in (0, 128, nq - 1):
        ref_rows, ref_dist = search_rows(table, "vector", queries[qi], metric, k)
        assert_same_neighbours(rows[qi], dist[qi], ref_rows, ref_dist, corpus, queries[qi], metric)
    mask = (np.arange(n) % 5 != 1).astype(np.uint8)
    rows_m, dist_m = c.search(queries, metric, k, row_mask=mask)
    assert c.stats().last_variant & 4
    rows_ms, dist_ms = c.search(queries, metric, k, knn.PREC_EXACT_SCAN, row_mask=mask)
    assert np.array_equal(rows_m, rows_ms) and np.array_equal(dist_m, dist_ms)
    if metric == "cosine":
        ctx.set_option("FENIX_NO_NORM_SHADOW", 1)
        try:
            c2 = make_corpus(ctx, corpus)            # a shard that never builds the normalised shadow
            rows_e, dist_e = c2.search(queries, metric, k)
            assert c2.stats().last_variant & 4
            c2.close()
        finally:
            ctx.set_option("FENIX_NO_NORM_SHADOW", None)
        assert np.array_equal(rows_e, rows_s) and np.array_equal(dist_e, dist_s)
    ctx.set_option("FENIX_TC_PAIR", None)
    c.close()


def test_group_search_in_one_process(built_library):
    """fx_group_*: one process owning the devices, an NCCL communicator and a worker thread per device inside the
    library. On a single-GPU box the group has one member (no exchange); with >= 2 GPUs the shards are searched
    concurrently, all-gathered over NVLink and merged on the device."""
    import torch
    from fenix_b200.dist import shard_bounds
    from oracle import brute_force_f64

    n_dev = min(torch.cuda.device_count(), 4)
    rng = np.random.default_rng(55)
    corpus = rng.standard_normal((40_003, 96), dtype=np.float32)
    corpus[30_000] = corpus[11]                      # a cross-shard tie
    queries = np.concatenate([rng.standard_normal((140, 96), dtype=np.float32), corpus[11:12]])
    group = knn.Group(list(range(n_dev)))
    shards = []
    for r in range(n_dev):
        lo, hi = shard_bounds(len(corpus), n_dev, r)
        s = knn.Corpus(group.contexts[r], hi - lo, 96, row_base=lo)
        s.append(corpus[lo:hi])
        shards.append(s.finalize())
    for metric, k in (("l2", 10), ("dot", 100), ("cosine", 1500)):
        rows, dist = group.search(shards, queries, metric, k)
        want_rows, want_dist = brute_force_f64(corpus, queries, metric, k)
        assert np.array_equal(rows, want_rows), (metric, k)
        assert np.allclose(dist, want_dist, rtol=3e-7, atol=3e-6), (metric, k)
    mask = (np.arange(len(corpus)) % 3 != 0).astype(np.uint8)
    rows, dist = group.search(shards, queries, "l2", 10, row_mask=mask)
    live = np.nonzero(mask)[0]
    want_rows, want_dist = brute_force_f64(corpus[live], queries, "l2", 10)
    assert np.array_equal(rows, live[want_rows]) and np.allclose(dist, want_dist, rtol=3e-7, atol=3e-6)
    for s in shards:
        s.close()
    group.close()


@pytest.mark.parametrize("metric", ["l2", "dot"])
def test_norm_outliers_do_not_defeat_the_certificate(ctx, metric):
    """0.1 % of the rows carry 100x the norm. The filter score of a row is a certified UPPER bound of its exact score (the
    row's own error weight rides in the shadow), so the certificate does not depend on the largest norm of the shard:
    no query falls back to the fp64 scan, and the result still equals it."""
    import torch

    n, d, nq, k = 300_000, 128, 700, 100
    g = torch.Generator(device="cuda").manual_seed(99)
    x = torch.randn((n, d), generator=g, device="cuda", dtype=torch.float32)
    x[torch.arange(3, n, 1000, device="cuda")] *= 100.0
    q = torch.randn((nq, d), generator=g, device="cuda", dtype=torch.float32)
    c = knn.Corpus(ctx, n, d)
    torch.cuda.synchronize()
    c.append_device(x.data_ptr(), n)
    c.finalize()
    qh = q.cpu().numpy()
    before = c.stats()
    rows, dist = c.search(qh, metric, k)
    after = c.stats()
    assert after.last_path == 2
    assert after.fallback_queries == before.fallback_queries, "the certificate should hold without the scan"
    assert after.refined_queries - before.refined_queries <= nq // 50
    sub = np.arange(0, nq, 23)
    rows_s, dist_s = c.search(qh[sub], metric, k, knn.PREC_EXACT_SCAN)
    assert np.array_equal(rows[sub], rows_s) and np.array_equal(dist[sub], dist_s)
    if metric == "dot":   # the outliers ARE the nearest neighbours under inner product (100x the dot product)
        assert (rows[:, 0] % 1000 == 3).all()
    c.close()


def test_large_property_checks(ctx):
    """BASELINE-sized shape (1M x 128, k = 100): size-independent properties instead of the oracle:
    planted neighbours are found, results are sorted by (distance, row), sharding is invariant,
    and the tensor-core path agrees with the fp64 scan on a query subset."""
    import torch

    n, d, nq, k = 1_000_000, 128, 256, 100
    g = torch.Generator(device="cuda").manual_seed(1002)
    x = torch.randn((n, d), generator=g, device="cuda", dtype=torch.float32)
    q = torch.randn((nq, d), generator=g, device="cuda", dtype=torch.float32)
    plant = torch.arange(nq, device="cuda") * 3001 + 5
    x[plant] = q + 1e-3 * torch.randn((nq, d), generator=g, device="cuda")  # query i's nearest is row plant[i]
    c = knn.Corpus(ctx, n, d)
    torch.cuda.synchronize()
    c.append_device(x.data_ptr(), n)
    c.finalize()
    qh = q.cpu().numpy()
    rows, dist = c.search(qh, "l2", k)
    assert np.array_equal(rows[:, 0], plant.cpu().numpy())
    assert (np.diff(dist, axis=1) >= 0).all()
    ties = np.diff(dist, axis=1) == 0
    assert (np.diff(rows, axis=1)[ties] > 0).all()
    sub = slice(0, 16)
    rows_s, dist_s = c.search(qh[sub], "l2", k, knn.PREC_EXACT_SCAN)
    assert np.array_equal(rows[sub], rows_s) and np.array_equal(dist[sub], dist_s)
    for metric in ("cosine", "dot"):
        r1, d1 = c.search(qh[sub], metric, 10)
        r2, d2 = c.search(qh[sub], metric, 10, knn.PREC_EXACT_SCAN)
        assert np.array_equal(r1, r2) and np.array_equal(d1, d2)
    c.close()


@pytest.mark.parametrize("metric,dim,k", [("l2", 128, 100), ("dot", 96, 100), ("cosine", 64, 10), ("l2", 100, 10)])
def test_resident_query_kernel_and_sample_prepass(ctx, metric, dim, k):
    """Narrow rows + several query tiles take the resident-query kernel with thresholds from the strided sample
    prepass: same answer as the fp64 scan, the adaptive path (prepass off) and the streaming kernel."""
    import torch

    n, nq = 400_000, 700
    g = torch.Generator(device="cuda").manual_seed(4242 + dim)
    x = torch.randn((n, dim), generator=g, device="cuda", dtype=torch.float32)
    q = torch.randn((nq, dim), generator=g, device="cuda", dtype=torch.float32)
    c = knn.Corpus(ctx, n, dim)
    torch.cuda.synchronize()
    c.append_device(x.data_ptr(), n)
    c.finalize()
    qh = q.cpu().numpy()
    before = c.stats()
    rows, dist = c.search(qh, metric, k)
    after = c.stats()
    assert after.last_path == 2
    assert after.fallback_queries - before.fallback_queries <= 3
    sub = np.arange(0, nq, 37)
    rows_s, dist_s = c.search(qh[sub], metric, k, knn.PREC_EXACT_SCAN)
    assert np.array_equal(rows[sub], rows_s) and np.array_equal(dist[sub], dist_s)
    # the same search through the other kernels (tuning knobs are per-context options; the environment is only read
    # once, at fx_init): adaptive thresholds, the streaming kernels (CTA pairs, one CTA per tile)
    variants = ({"FENIX_TC_PRE": "0"}, {"FENIX_TC_NO_RQ": "1"}, {"FENIX_TC_NO_RQ": "1", "FENIX_TC_PRE": "0"},
                {"FENIX_TC_NO_RQ": "1", "FENIX_TC_PAIR": "1"}, {"FENIX_TC_NO_RQ": "1", "FENIX_TC_PAIR": "1", "FENIX_TC_PRE": "0"})
    for opts in variants:
        for key, value in opts.items():
            ctx.set_option(key, value)
        try:
            rows_e, dist_e = c.search(qh, metric, k)
            variant = c.stats().last_variant
        finally:
            for key in opts:
                ctx.set_option(key, None)
        assert np.array_equal(rows, rows_e) and np.array_equal(dist, dist_e), opts
        if "FENIX_TC_NO_RQ" in opts:
            # (rows this narrow take the one-CTA streaming kernel unless CTA pairs are forced)
            assert (variant & 1) == 0 and bool(variant & 4) == (opts.get("FENIX_TC_PAIR") == "1"), (opts, variant)
    c.close()


@pytest.mark.parametrize("dim", [60, 61, 62, 64, 65, 124, 125, 128, 188, 189, 190, 256])
def test_shadow_geometry_boundaries(ctx, dim):
    """The bf16 shadow keeps -|x|^2/2 (three terms) and the row's error weight in four extra K columns: inside the last
    64-column block when it has room (dim % 64 <= 60), in a separate block per tile otherwise; rows of up to 3 blocks
    take the resident-query kernel.
    Every metric, both kernels (a 300-query and a 40-query batch), against the fp64 scan."""
    import torch

    n, nq, k = 70_000, 300, 10
    g = torch.Generator(device="cuda").manual_seed(1000 + dim)
    x = torch.randn((n, dim), generator=g, device="cuda", dtype=torch.float32)
    x *= (0.5 + torch.rand((n, 1), generator=g, device="cuda"))          # spread the norms: the L2 term matters
    q = torch.randn((nq, dim), generator=g, device="cuda", dtype=torch.float32)
    c = knn.Corpus(ctx, n, dim)
    torch.cuda.synchronize()
    c.append_device(x.data_ptr(), n)
    c.finalize()
    qh = q.cpu().numpy()
    sub = np.arange(0, nq, 11)
    for metric in ("l2", "cosine", "dot"):
        before = c.stats()
        rows, dist = c.search(qh, metric, k)
        st = c.stats()
        blocks = -(-(dim + (4 if metric == "l2" else 0)) // 64)      # 64-column k-blocks the search multiplies
        assert st.last_path == 2 and (st.last_variant & 1) == (1 if blocks <= 3 else 0), (metric, st.last_variant)
        assert st.fallback_queries - before.fallback_queries <= 2
        rows_s, dist_s = c.search(qh[sub], metric, k, knn.PREC_EXACT_SCAN)
        assert np.array_equal(rows[sub], rows_s) and np.array_equal(dist[sub], dist_s), metric
        rows_40, dist_40 = c.search(qh[:40], metric, k)
        assert (c.stats().last_variant & 1) == 0
        assert np.array_equal(rows[:40], rows_40) and np.array_equal(dist[:40], dist_40), metric
    c.close()


@pytest.mark.parametrize("nq,k", [(129, 1), (257, 256), (300, 37)])
def test_resident_query_kernel_edges(ctx, nq, k):
    """Query counts that leave a tile (almost) empty, k = 1 and a large k, and a row mask (the resident-query
    kernel's additive-term variant; masked searches take no prepass) - all against the fp64 scan."""
    import torch

    n, dim = 120_000, 96
    g = torch.Generator(device="cuda").manual_seed(5 + nq)
    x = torch.randn((n, dim), generator=g, device="cuda", dtype=torch.float32)
    q = torch.randn((nq, dim), generator=g, device="cuda", dtype=torch.float32)
    c = knn.Corpus(ctx, n, dim)
    torch.cuda.synchronize()
    c.append_device(x.data_ptr(), n)
    c.finalize()
    qh = q.cpu().numpy()
    mask = (np.random.default_rng(nq).random(n) < 0.4).astype(np.uint8)
    sub = np.unique(np.concatenate([np.arange(0, nq, 17), [nq - 1]]))
    for metric in ("l2", "cosine", "dot"):
        rows, dist = c.search(qh, metric, k)
        # the prepass needs >= 32 sampled tiles at a stride of ~3 K' / 16: k = 256 is too large for this shard
        assert c.stats().last_variant == (3 if k <= 37 else 1), "resident-query kernel expected"
        rows_s, dist_s = c.search(qh[sub], metric, k, knn.PREC_EXACT_SCAN)
        assert np.array_equal(rows[sub], rows_s) and np.array_equal(dist[sub], dist_s), metric
        rows_m, dist_m = c.search(qh, metric, k, knn.PREC_FP32, row_mask=mask)
        assert c.stats().last_variant == 1, "masked: resident-query kernel, no prepass"
        assert mask[rows_m].all()
        rows_ms, dist_ms = c.search(qh[sub], metric, k, knn.PREC_EXACT_SCAN, row_mask=mask)
        assert np.array_equal(rows_m[sub], rows_ms) and np.array_equal(dist_m[sub], dist_ms), metric
    c.close()


def test_sample_prepass_with_an_unrepresentative_sample(ctx):
    """Adversarial layout for the threshold prepass: every sampled tile is filled with copies of the queries, so
    each query's sample threshold lands far above anything the rest of the shard offers and the main pass keeps
    fewer than k candidates. The adaptive re-run (tier 0) must settle those queries exactly."""
    import torch

    n, dim, nq, k = 300_000, 64, 256, 100
    g = torch.Generator(device="cuda").manual_seed(99)
    x = torch.randn((n, dim), generator=g, device="cuda", dtype=torch.float32)
    q = torch.randn((nq, dim), generator=g, device="cuda", dtype=torch.float32)
    # K' = 160 for k = 100 -> the default knobs sample every 30th tile of 128 rows (79 tiles, rank m = 16).
    # Sampled tile j holds 3 q_i for the 128 queries of query tile j % 2: every query owns ~40 sampled blocks whose
    # maximum is 3 |q|^2, so its sample threshold is 3 |q|^2 - and only ~40 < k rows of the shard reach it.
    stride = 30
    for j, t in enumerate(range(0, n // 128, stride)):
        x[t * 128:(t + 1) * 128] = 3.0 * q[(j % 2) * 128:(j % 2) * 128 + 128]
    c = knn.Corpus(ctx, n, dim)
    torch.cuda.synchronize()
    c.append_device(x.data_ptr(), n)
    c.finalize()
    qh = q.cpu().numpy()
    before = c.stats()
    rows, dist = c.search(qh, "dot", k)
    after = c.stats()
    assert after.refined_queries - before.refined_queries >= 64, "the planted sample should defeat most sample thresholds"
    assert after.fallback_queries == before.fallback_queries, "the adaptive re-run should make the fp64 scan unnecessary"
    rows_s, dist_s = c.search(qh, "dot", k, knn.PREC_EXACT_SCAN)
    assert np.array_equal(rows, rows_s) and np.array_equal(dist, dist_s)
    c.close()


@pytest.mark.parametrize("value_type", ["float64", "float16"])
def test_other_float_widths_of_the_vector_column(built_library, value_type, tmp_path):
    """float64 / float16 embedding columns: converted to float32 shards at upload, `__DISTANCE__` typed like the
    column (index.py:153). float64: against the oracle (which, like the reference, computes in float64) at the
    parity bar; float16 (the reference's CPU path has no half cdist): against the fp64 adjudicator."""
    rng = np.random.default_rng(17)
    n, d, k = 6000, 48, 10
    corpus = rng.standard_normal((n, d)).astype(value_type)
    queries = rng.standard_normal((5, d)).astype(value_type)
    vec = pa.FixedSizeListArray.from_arrays(pa.array(corpus.reshape(-1)), d)
    table = pa.table({"id": pa.array(np.arange(n, dtype=np.int64)), "vector": vec})
    root = str(tmp_path)
    fenix.io.table.make(root, "t", table.to_reader())
    try:
        for metric in ("l2", "cosine", "dot"):
            for q in queries:
                res = fenix.io.index.call(root, None, "t", "vector", q, metric=metric, select=["id"], maxval=k)
                assert res.schema.field("__DISTANCE__").type == vec.type.value_type
                got_rows, got_dist = res.column("id").to_numpy(), res.column("__DISTANCE__").to_numpy().astype(np.float64)
                if value_type == "float64":
                    ref_rows, ref_dist = search_rows(table, "vector", q, metric, k)
                    assert_same_neighbours(got_rows, got_dist.astype(np.float32), ref_rows, ref_dist.astype(np.float32),
                                           corpus.astype(np.float32), q.astype(np.float32), metric)
                else:
                    want_rows, want_dist = brute_force_f64(corpus.astype(np.float32), q.astype(np.float32), metric, k)
                    assert np.array_equal(got_rows, want_rows[0])
                    assert np.allclose(got_dist, want_dist[0], rtol=2e-3, atol=2e-3)   # the column type rounds the answer
    finally:
        fenix.io.shards.invalidate(root)


@pytest.mark.parametrize("metric,nq", [("l2", 1), ("cosine", 5), ("dot", 64)])
def test_small_searches_replay_a_cuda_graph(ctx, metric, nq):
    """From its second identical call on a small search (<= 64 queries, no mask) is one captured CUDA graph: call 1 runs
    kernel by kernel, call 2 captures, calls 3+ replay. Every call gets DIFFERENT queries through the same graph and must
    equal the fp64 scan; a bigger search in between (scratch grows) and a knob change both force a re-capture."""
    rng = np.random.default_rng(1234)
    n, d, k = 100_000, 128, 10
    corpus = rng.standard_normal((n, d), dtype=np.float32)
    c = make_corpus(ctx, corpus)
    ctx.set_option("FENIX_DIRECT_MAX_MB", 16)   # (a shard this small would take the direct scan: no graph, nothing to replay)
    launches = []
    for call in range(6):
        q = rng.standard_normal((nq, d), dtype=np.float32)
        if call == 4:
            c.search(rng.standard_normal((700, d), dtype=np.float32), metric, k)      # grows the scratch buffers
        if call == 5:
            ctx.set_option("FENIX_TC_KP", 96)
        before = c.stats().kernel_launches
        rows, dist = c.search(q, metric, k)
        launches.append(c.stats().kernel_launches - before)
        assert c.stats().last_path == 2
        rows_s, dist_s = c.search(q, metric, k, knn.PREC_EXACT_SCAN)
        assert np.array_equal(rows, rows_s) and np.array_equal(dist, dist_s), (metric, nq, call)
    ctx.set_option("FENIX_TC_KP", None)
    assert len(set(launches[1:4])) == 1 and launches[0] == launches[1] + 1, launches   # (call 1 also builds the shadow) the graph runs the plain path's kernels
    # graphs off: same answers
    ctx.set_option("FENIX_GRAPH", 0)
    q = rng.standard_normal((nq, d), dtype=np.float32)
    r0, d0 = c.search(q, metric, k)
    ctx.set_option("FENIX_GRAPH", None)
    for _ in range(3):
        r1, d1 = c.search(q, metric, k)
        assert np.array_equal(r0, r1) and np.array_equal(d0, d1)
    ctx.set_option("FENIX_DIRECT_MAX_MB", None)
    c.close()


def test_each_shadow_is_built_by_the_first_search_that_streams_it(ctx):
    """A shard searched with one metric holds its fp32 rows and ONE bf16 shadow (the normalised rows for cosine, the plain
    rows + augmented columns for L2 / inner product); the second shadow appears only when the other kind of search comes."""
    rng = np.random.default_rng(8)
    n, d = 16_384, 128
    corpus = rng.standard_normal((n, d), dtype=np.float32)
    queries = rng.standard_normal((9, d), dtype=np.float32)    # (<= 8 queries would take the direct scan: no shadow at all)
    c = make_corpus(ctx, corpus)
    rows_bytes = c.stats().device_bytes
    assert rows_bytes == n * (d + 2) * 4                       # rows + the two cached norm terms, no shadow yet
    c.search(queries, "cosine", 5)
    norm_shadow = c.stats().device_bytes - rows_bytes
    assert c.stats().last_path == 2 and norm_shadow == n * d * 2
    c.search(queries, "cosine", 5)
    assert c.stats().device_bytes == rows_bytes + norm_shadow  # nothing more for the same metric
    c.search(queries, "dot", 5)
    plain_shadow = c.stats().device_bytes - rows_bytes - norm_shadow
    assert plain_shadow == n * (d + 64) * 2                    # data blocks + one block per tile for the augmented columns
    c.search(queries, "l2", 5)
    assert c.stats().device_bytes == rows_bytes + norm_shadow + plain_shadow
    c.close()


# ---- the latency path: single-launch direct scan (direct_scan.cuh) ------------------------------------------
@pytest.mark.parametrize("metric", ["l2", "cosine", "dot"])
@pytest.mark.parametrize("shape", [(100_000, 128, 1, 10), (100_000, 128, 8, 10), (20_011, 100, 3, 37), (5_000, 768, 5, 128),
                                   (70_000, 7, 2, 5), (333, 36, 4, 64), (40, 24, 2, 64), (1, 16, 1, 3)])
def test_direct_scan_equals_scan_tensor_path_and_oracle(ctx, shape, metric):
    """<= 8 queries over a small shard are ONE launch per four queries (last_path 3): ids and distances bit-equal to the
    fp64 scan and to the tensor-core path (same fp64 summation order as its rerank), neighbours as the oracle's."""
    n, d, nq, k = shape
    rng = np.random.default_rng(n * 7 + d)
    corpus = rng.standard_normal((n, d), dtype=np.float32)
    queries = rng.standard_normal((nq, d), dtype=np.float32)
    c = make_corpus(ctx, corpus)
    before = c.stats().kernel_launches
    rows, dist = c.search(queries, metric, k)
    st = c.stats()
    assert st.last_path == 3 and st.kernel_launches - before == -(-nq // 4), (st.last_path, st.kernel_launches - before)   # four queries per launch
    rows_s, dist_s = c.search(queries, metric, k, knn.PREC_EXACT_SCAN)
    assert c.stats().last_path == 0
    assert np.array_equal(rows, rows_s) and np.array_equal(dist, dist_s)
    rows_t, dist_t = search_as(ctx, c, "fp32_tc", queries, metric, k)
    assert c.stats().last_path != 3
    assert np.array_equal(rows, rows_t) and np.array_equal(dist, dist_t)
    if n >= k:
        want_rows, want_dist = brute_force_f64(corpus, queries, metric, k)
        assert np.array_equal(rows, want_rows)
        table = table_of(corpus, 4096)
        ref_rows, ref_dist = search_rows(table, "vector", queries[nq - 1], metric, k)
        assert_same_neighbours(rows[nq - 1], dist[nq - 1], ref_rows, ref_dist, corpus, queries[nq - 1], metric)
    else:
        assert (rows[:, n:] == -1).all() and np.isinf(dist[:, n:]).all() and (rows[:, :n] >= 0).all()
    c.close()


def test_direct_scan_masks_duplicates_and_trims(ctx):
    """Row mask, ties broken by row, and a shard large enough per CTA that the candidate buffers are cut back: 300k rows /
    148 CTAs = 2k rows each, ordered so that the rows get closer to query 0 as the row number grows - every row passes the
    running threshold, the worst case for a running top-k."""
    rng = np.random.default_rng(21)
    n, d, k = 300_000, 32, 100
    corpus = rng.standard_normal((n, d), dtype=np.float32)
    queries = rng.standard_normal((3, d), dtype=np.float32)
    far_first = np.argsort(-np.linalg.norm(corpus.astype(np.float64) - queries[0].astype(np.float64), axis=1), kind="stable")
    corpus = np.ascontiguousarray(corpus[far_first])
    corpus[1000:1400] = corpus[-1]                      # 400 copies of the best row
    c = make_corpus(ctx, corpus)
    for metric in ("l2", "dot"):
        rows, dist = c.search(queries, metric, k)
        assert c.stats().last_path == 3
        rows_s, dist_s = c.search(queries, metric, k, knn.PREC_EXACT_SCAN)
        assert np.array_equal(rows, rows_s) and np.array_equal(dist, dist_s), metric
    mask = (rng.random(n) < 0.05).astype(np.uint8)
    mask[:5000] = 0
    rows, dist = c.search(queries, "l2", k, row_mask=mask)
    assert c.stats().last_path == 3 and mask[rows].all()
    rows_s, dist_s = c.search(queries, "l2", k, knn.PREC_EXACT_SCAN, row_mask=mask)
    assert np.array_equal(rows, rows_s) and np.array_equal(dist, dist_s)
    few = np.zeros(n, np.uint8)
    few[[5, 77, 190_000]] = 1
    rows, dist = c.search(queries[:1], "l2", 10, row_mask=few)
    assert sorted(rows[0, :3].tolist()) == [5, 77, 190_000] and (rows[0, 3:] == -1).all() and np.isinf(dist[0, 3:]).all()
    # knobs: off, and the size bound
    ctx.set_option("FENIX_DIRECT", 0)
    c.search(queries, "l2", k)
    assert c.stats().last_path != 3
    ctx.set_option("FENIX_DIRECT", None)
    ctx.set_option("FENIX_DIRECT_MAX_MB", 8)
    c.search(queries, "l2", k)
    assert c.stats().last_path != 3
    ctx.set_option("FENIX_DIRECT_MAX_MB", None)
    # nine queries, or k > 128: the other paths
    c.search(np.repeat(queries, 3, axis=0), "l2", k)
    assert c.stats().last_path != 3
    c.search(queries, "l2", 129)
    assert c.stats().last_path != 3
    c.close()


@pytest.mark.parametrize("shape", [(50_000, 64, 37, 10, 5, 300), (20_000, 200, 3, 100, 40, 64), (30_000, 128, 2, 33, 8, 16),
                                   (5_000, 36, 400, 7, 3, 1000)])
def test_search_cells_equals_per_query_masked_searches(ctx, shape):
    """fx_search_cells (batched IVF in one launch: query q scans the posting lists of its probe cells) against one masked
    fp64 scan per query with the mask the reference would build (`cell isin probes` AND the predicate, index.py:119-126):
    ids and distances bit-equal, short lists padded."""
    n, d, nq, k, n_probe, n_cells = shape
    rng = np.random.default_rng(n + d + nq)
    corpus = rng.standard_normal((n, d), dtype=np.float32)
    queries = rng.standard_normal((nq, d), dtype=np.float32)
    cell = (rng.random(n) ** 2 * n_cells).astype(np.int64)              # uneven cells; some stay empty
    cell[rng.integers(0, n, 5)] = n_cells - 1
    pred = (rng.random(n) < 0.7).astype(np.uint8)
    probes = np.stack([rng.choice(n_cells, n_probe, replace=False) for _ in range(nq)]).astype(np.int32)
    probes[rng.random(probes.shape) < 0.15] = -1                        # unused slots
    c = make_corpus(ctx, corpus)
    assert c.set_cells(cell) == n_cells
    for metric in ("l2", "cosine", "dot"):
        for mask in (None, pred):
            before = c.stats().kernel_launches
            rows, dist = c.search_cells(queries, metric, k, probes, mask)
            assert c.stats().kernel_launches - before == 1
            for qi in range(0, nq, max(1, nq // 12)):
                m_q = np.isin(cell, probes[qi][probes[qi] >= 0]).astype(np.uint8)
                if mask is not None:
                    m_q &= mask
                want_rows, want_dist = c.search(queries[qi], metric, k, knn.PREC_EXACT_SCAN, row_mask=m_q)
                assert np.array_equal(rows[qi], want_rows[0]) and np.array_equal(dist[qi], want_dist[0]), (metric, qi)
                assert (rows[qi] >= 0).sum() == min(k, int(m_q.sum()))
    # a second cell structure replaces the first; errors
    assert c.set_cells(np.zeros(n, np.int64)) == 1
    rows, dist = c.search_cells(queries[:2], "l2", k, np.zeros((2, 1), np.int32))
    want_rows, want_dist = c.search(queries[:2], "l2", k, knn.PREC_EXACT_SCAN)
    assert np.array_equal(rows, want_rows) and np.array_equal(dist, want_dist)
    with pytest.raises(ValueError):
        c.search_cells(queries[:2], "l2", k, np.full((2, 1), 7, np.int32))       # no such cell
    with pytest.raises(NotImplementedError):
        c.search_cells(queries[:2], "l2", 129, np.zeros((2, 1), np.int32))       # k > 128: the caller loops masked searches
    c.close()


def test_tensor_core_path_runs_and_certifies(ctx):
    """fp32 mode must take the tcgen05 path on ordinary data (no silent fallback to the scan) and the
    certificate must hold for (nearly) every query; tf32 mode reports its recall."""
    rng = np.random.default_rng(77)
    corpus = rng.standard_normal((60000, 128), dtype=np.float32)
    queries = rng.standard_normal((300, 128), dtype=np.float32)
    c = make_corpus(ctx, corpus)
    for metric in ("l2", "cosine", "dot"):
        before = c.stats()
        rows, dist = c.search(queries, metric, 10, knn.PREC_FP32)
        after = c.stats()
        assert after.last_path in (1, 2), "tensor-core path not taken"   # 2: bf16-shadow filter (default)
        assert after.fallback_queries - before.fallback_queries <= 3, "certificate fails on gaussian data"
        rows_s, dist_s = c.search(queries, metric, 10, knn.PREC_EXACT_SCAN)
        assert c.stats().last_path == 0
        assert np.array_equal(rows, rows_s) and np.array_equal(dist, dist_s)
        for approx in (knn.PREC_TF32, knn.PREC_BF16):
            rows_t, dist_t = c.search(queries, metric, 10, approx)
            recall = np.mean([len(set(a) & set(b)) / 10 for a, b in zip(rows, rows_t)])
            assert recall >= 0.98, (approx, recall)
    c.close()


@pytest.mark.parametrize("metric", ["l2", "cosine", "dot"])
def test_masked_search_on_tensor_core_path(ctx, metric):
    """Row mask (the device form of index.py:161 filter) folded into the filter epilogue: same answer as the
    masked fp64 scan and as the oracle run on the surviving rows."""
    rng = np.random.default_rng(123)
    corpus = rng.standard_normal((20000, 64), dtype=np.float32)
    queries = rng.standard_normal((70, 64), dtype=np.float32)
    mask = (rng.random(20000) < 0.3).astype(np.uint8)
    mask[:300] = 0
    c = make_corpus(ctx, corpus)
    rows, dist = c.search(queries, metric, 10, knn.PREC_FP32, row_mask=mask)
    assert c.stats().last_path >= 1
    assert mask[rows].all()
    rows_s, dist_s = c.search(queries, metric, 10, knn.PREC_EXACT_SCAN, row_mask=mask)
    assert np.array_equal(rows, rows_s) and np.array_equal(dist, dist_s)
    live = np.nonzero(mask)[0]
    want_rows, want_dist = brute_force_f64(corpus[live], queries, metric, 10)
    assert np.array_equal(rows, live[want_rows])
    # a mask that leaves fewer than k rows: pads, through the fallback tiers
    few = np.zeros(20000, np.uint8)
    few[[5, 77, 19000]] = 1
    rows, dist = c.search(queries[:3], metric, 10, knn.PREC_FP32, row_mask=few)
    assert (np.sort(rows[:, :3], axis=1) == np.array([5, 77, 19000])).all() and (rows[:, 3:] == -1).all()
    c.close()


def test_refinement_pass_settles_ties_and_near_ties(ctx):
    """Duplicates defeat the first-pass certificate (K' equal scores); the preset-threshold refinement pass must
    then produce the exact (distance, row) answer without the full fp64 scan."""
    rng = np.random.default_rng(91)
    corpus = rng.standard_normal((30000, 96), dtype=np.float32)
    corpus[5000:5400] = corpus[17]                    # 400 copies of row 17
    corpus[20000:20050] = corpus[17] + 1e-4           # 50 near-duplicates
    queries = np.concatenate([corpus[17:18], rng.standard_normal((40, 96), dtype=np.float32)])
    c = make_corpus(ctx, corpus)
    for metric in ("l2", "cosine", "dot"):
        before = c.stats()
        rows, dist = c.search(queries, metric, 10, knn.PREC_FP32)
        after = c.stats()
        want_rows, want_dist = c.search(queries, metric, 10, knn.PREC_EXACT_SCAN)
        assert np.array_equal(rows, want_rows) and np.array_equal(dist, want_dist), metric
        assert after.refined_queries - before.refined_queries >= 1, "the duplicate query should need the refinement pass"
        assert after.fallback_queries == before.fallback_queries, "refinement should make the full scan unnecessary here"
    truth_rows, _ = brute_force_f64(corpus, queries[:1], "l2", 10)
    rows, _ = c.search(queries[:1], "l2", 10)
    assert np.array_equal(rows, truth_rows)
    c.close()


@pytest.mark.parametrize("dim", [32, 100, 128, 768])
def test_tf32_error_bound_of_the_certificate(ctx, dim):
    """|filter score - exact score| <= c * |q| * |x| with c = 1.25 * 2^-9 + D * 2^-21 (tc_filter.cuh)."""
    rng = np.random.default_rng(dim)
    corpus = rng.standard_normal((8192, dim), dtype=np.float32) * rng.uniform(0.1, 10, (8192, 1)).astype(np.float32)
    queries = rng.standard_normal((128, dim), dtype=np.float32)
    c = make_corpus(ctx, corpus)
    x = corpus[:256].astype(np.float64)
    q = queries.astype(np.float64)
    qn, xn = np.linalg.norm(q, axis=1)[:, None], np.linalg.norm(x, axis=1)[None, :]
    cerr = 1.25 * 2.0 ** -9 + dim * 2.0 ** -21
    exact = {"dot": q @ x.T, "l2": q @ x.T - 0.5 * xn ** 2, "cosine": (q @ x.T) / np.maximum(xn, 1e-12)}
    scale = {"dot": qn * xn, "l2": qn * xn + 2.0 ** -22 * (0.5 * xn ** 2 + qn * xn), "cosine": qn * np.ones_like(xn)}
    for metric in ("dot", "l2", "cosine"):
        s = c.debug_scores(queries, metric).astype(np.float64)
        ratio = np.abs(s - exact[metric]) / (cerr * scale[metric])
        assert ratio.max() < 0.5, (metric, ratio.max())  # observed ~0.2: the bound has 2x+ headroom
    c.close()


@pytest.mark.parametrize("dim", [64, 768])
def test_bf16_shadow_filter_is_exact_in_fp32_mode(ctx, dim, monkeypatch):
    """With a bf16 shadow the exact mode filters with kind::f16 MMAs; results must not change, and the bf16
    error bound c = 1.1 * 2^-8 + D * 2^-21 must hold for the raw scores."""
    monkeypatch.setenv("FENIX_BF16_SHADOW", "1")
    rng = np.random.default_rng(dim + 5)
    corpus = rng.standard_normal((20000, dim), dtype=np.float32)
    queries = rng.standard_normal((130, dim), dtype=np.float32)
    c = make_corpus(ctx, corpus)
    ctx.set_option("FENIX_DEBUG_BF16", 1)
    try:
        s = c.debug_scores(queries, "dot").astype(np.float64)
    finally:
        ctx.set_option("FENIX_DEBUG_BF16", None)
    q, x = queries[:128].astype(np.float64), corpus[:256].astype(np.float64)
    bound = (1.1 * 2.0 ** -8 + dim * 2.0 ** -21) * np.linalg.norm(q, axis=1)[:, None] * np.linalg.norm(x, axis=1)[None, :]
    assert (np.abs(s - q @ x.T) / bound).max() < 0.6
    for metric in ("l2", "cosine", "dot"):
        rows, dist = c.search(queries, metric, 10, knn.PREC_FP32)
        assert c.stats().last_path == 2   # bf16 filter
        want_rows, want_dist = c.search(queries, metric, 10, knn.PREC_EXACT_SCAN)
        assert np.array_equal(rows, want_rows) and np.array_equal(dist, want_dist), metric
        rows_b, _ = c.search(queries, metric, 10, knn.PREC_BF16)
        assert np.mean([len(set(a) & set(b)) / 10 for a, b in zip(rows, rows_b)]) >= 0.97
    c.close()


# ---- through the reference-facing API ----------------------------------------------------
def test_index_call_matches_oracle_table(ctx, tmp_path):
    rng = np.random.default_rng(9)
    corpus = rng.standard_normal((6000, 64), dtype=np.float32)
    table = table_of(corpus, 1000)
    root = str(tmp_path)
    fenix.io.table.make(root, "test/table", table.to_reader())
    from oracle import call as oracle_call

    q = rng.standard_normal(64)  # float64 target is cast to the column type (index.py:110)
    for metric in METRICS:
        got = fenix.io.index.call(root, None, "test/table", "vector", q, metric=metric, maxval=10)
        want = oracle_call(table, "vector", q, metric, maxval=10)
        assert got.schema == want.schema
        assert_same_neighbours(got.column("id").to_numpy(), got.column("__DISTANCE__").to_numpy(),
                               want.column("id").to_numpy(), want.column("__DISTANCE__").to_numpy(),
                               corpus, q.astype(np.float32), metric)
        # gathered rows are the rows themselves
        ids = got.column("id").to_numpy()
        vec = np.stack(got.column("vector").to_numpy(zero_copy_only=False))
        assert np.array_equal(vec, corpus[ids])
    # maxval None -> all rows, table order; select; filter; multi-source
    got = fenix.io.index.call(root, None, "test/table", "vector", q, metric="l2", select=["id"])
    want = oracle_call(table, "vector", q, "l2", select=["id"])
    assert got.schema == want.schema and got.num_rows == 6000
    assert np.array_equal(got.column("id").to_numpy(), np.arange(6000))
    np.testing.assert_allclose(got.column("__DISTANCE__").to_numpy(), want.column("__DISTANCE__").to_numpy(), rtol=1e-5)
    flt = pc.field("id") >= 5990
    got = fenix.io.index.call(root, None, "test/table", "vector", q, metric="l2", select=["id"], filter=flt, maxval=4)
    want = oracle_call(table, "vector", q, "l2", select=["id"], filter=flt, maxval=4)
    assert sorted(got.column("id").to_pylist()) == sorted(want.column("id").to_pylist())
    got = fenix.io.index.call(root, None, "test/table", "vector", q, metric="l2", select=["id"], filter=flt, maxval=100)
    assert got.column("id").to_pylist() == list(range(5990, 6000))  # <= maxval survivors: table order
    both = fenix.io.index.call(root, None, ["test/table", "test/table"], "vector", q, metric="dot", select=["id"], maxval=6)
    ids = both.column("id").to_pylist()
    assert ids[0::2] == ids[1::2]  # each winner appears once per copy, ordered by (distance, row)
    # cache invalidation: rewriting the table changes the answer
    fenix.io.table.make(root, "test/table", table_of(-corpus, 1000).to_reader())
    flipped = fenix.io.index.call(root, None, "test/table", "vector", q, metric="dot", select=["id"], maxval=1)
    before = oracle_call(table_of(-corpus, 1000), "vector", q, "dot", select=["id"], maxval=1)
    assert flipped.column("id").to_pylist() == before.column("id").to_pylist()


IVF_CASES = sorted(f[len("ivf_"):-len(".npz")] for f in os.listdir(os.path.join(os.path.dirname(__file__), "golden")) if f.startswith("ivf_"))


def _write_reference_coding(root, name, tensor, dim, metric, ksize, nbooks):
    """A codebook file in the reference's own format (coder.py:120-125)."""
    import torch

    path = os.path.join(root, "codings", name + ".torch")
    os.makedirs(os.path.dirname(path), exist_ok=True)
    with open(path, "wb") as f:
        torch.save({"tensor": torch.from_numpy(tensor), "column": pa.list_(pa.float32(), dim),
                    "config": dict(metric=metric, codebook_size=ksize, num_codebooks=nbooks, batch_size=64, num_epochs=2)}, f)


@pytest.mark.parametrize("case", IVF_CASES)
def test_ivf_search_matches_live_reference_outputs(built_library, case, tmp_path):
    """SURVEY.md section 8f rank 4. Given the codebook the live reference trained (fixture), the product must rank
    the probe codes, assign the sidecar codes and answer `index.call(coding=, probes=)` like the reference did."""
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", f"ivf_{case}.npz"))
    root, dim = str(tmp_path), g["corpus"].shape[1]
    metric = str(g["coding_metric"])
    fenix.io.table.make(root, "t", table_of(g["corpus"], int(g["chunk"])).to_reader())
    _write_reference_coding(root, "cb", g["tensor"], dim, metric, int(g["codebook_size"]), int(g["num_codebooks"]))
    try:
        ranked = fenix.io.coder.call(g["queries"], (root, "cb"), None)
        assert ranked.shape == g["ranked"].shape
        top = int(g["probes"].max())
        assert np.array_equal(ranked[:, :top], g["ranked"][:, :top])          # the cells that get probed, in order
        assert np.array_equal(np.sort(ranked, axis=1), np.sort(g["ranked"], axis=1))
        joined = fenix.io.index.make(root, "cb", "t", "vector")
        assert joined.column_names == ["id", "vector", "__CODED_ID__"]
        assert np.array_equal(joined.column("__CODED_ID__").to_numpy(), g["codes"])
        assert [len(c) for c in joined.column("__CODED_ID__").chunks] == [len(c) for c in joined.column("id").chunks]
        flt = golden_filter(int(g["filter_mod"]))
        for qi, q in enumerate(g["queries"]):
            for p in g["probes"]:
                for m in (None, "l2", "cosine", "dot"):
                    res = fenix.io.index.call(root, "cb", "t", "vector", q, metric=m, select=["id"], filter=flt,
                                              maxval=int(g["k"]), probes=int(p))
                    key = f"{m or 'default'}:{qi}:{int(p)}"
                    assert res.column_names == ["id", "__DISTANCE__"]
                    assert_same_neighbours(res.column("id").to_numpy(), res.column("__DISTANCE__").to_numpy(),
                                           g[key + ":id"], g[key + ":dist"], g["corpus"], q, m or metric)
        # the whole query batch in ONE call (batched wire extension; one fx_search_cells launch): per query the answer the
        # live reference gave for that query alone
        for p in g["probes"]:
            for m in (None, "l2", "cosine", "dot"):
                res = fenix.io.index.call(root, "cb", "t", "vector", g["queries"], metric=m, select=["id"], filter=flt,
                                          maxval=int(g["k"]), probes=int(p))
                assert res.column_names == ["id", "__DISTANCE__", "__QUERY__"]
                for qi, q in enumerate(g["queries"]):
                    sel = res.filter(pc.field("__QUERY__") == qi)
                    key = f"{m or 'default'}:{qi}:{int(p)}"
                    assert_same_neighbours(sel.column("id").to_numpy(), sel.column("__DISTANCE__").to_numpy(),
                                           g[key + ":id"], g[key + ":dist"], g["corpus"], q, m or metric)
        # default projection carries the code column, as the joined table does in the reference (index.py:128)
        res = fenix.io.index.call(root, "cb", "t", "vector", g["queries"][0], metric=metric, maxval=3, probes=2)
        assert res.column_names == ["id", "vector", "__CODED_ID__", "__DISTANCE__"]
        assert set(res.column("__CODED_ID__").to_pylist()) <= set(g["ranked"][0, :2].tolist())
    finally:
        fenix.io.coder.drop(root, "cb")
        fenix.io.shards.invalidate(root)


class TestFlightDropIn:
    """The reference's own acceptance test (tests/test_flight.py:42-50, 88-114, 151-154) re-run against
    this package, plus result parity it does not check."""

    VECTOR_SIZE, NUM_VECTORS, BATCH_SIZE = 256, 20_000, 1_000

    @pytest.fixture(scope="class")
    def served(self, tmp_path_factory, built_library):
        root = str(tmp_path_factory.mktemp("fenix"))
        port = free_port()
        server = fenix.Server(root, "127.0.0.1", port)
        rng = np.random.default_rng(42)
        parts = []
        for _ in range(self.NUM_VECTORS // self.BATCH_SIZE):
            x = rng.standard_normal((self.BATCH_SIZE, self.VECTOR_SIZE), dtype=np.float32)
            parts.append(x + 10 * x[0, :])
        corpus = np.concatenate(parts)
        source = table_of(corpus, self.BATCH_SIZE)
        client = fenix.Flight("127.0.0.1", port)
        client.make_table("test/table", source.to_reader())
        yield client, source, corpus, root
        client.remove()
        server.shutdown()

    def test_make_table_roundtrip(self, served):
        client, source, *_ = served
        assert client.read_table("test/table").read_all() == source

    @pytest.mark.parametrize("metric", METRICS)
    def test_search_without_index(self, served, metric):
        client, source, corpus, *_ = served
        target = pc.random(self.VECTOR_SIZE).cast(pa.float32())
        result = client.search(target=target, source="test/table", column="vector", metric=metric, maxval=10)
        assert result.num_rows == 10
        assert result.schema == pa.schema([*source.schema, pa.field("__DISTANCE__", pa.float32())])
        q = target.to_numpy()
        ref_rows, ref_dist = search_rows(source, "vector", q, metric, 10)
        assert_same_neighbours(result.column("id").to_numpy(), result.column("__DISTANCE__").to_numpy(),
                               ref_rows, ref_dist, corpus, q, metric)

    def test_batched_wire_extension(self, served):
        client, source, corpus, *_ = served
        rng = np.random.default_rng(1)
        qs = rng.random((5, self.VECTOR_SIZE), dtype=np.float32)
        out = client.search(qs, "test/table", "vector", "l2", select=["id"], maxval=3)
        assert out.column_names == ["id", "__DISTANCE__", "__QUERY__"] and out.num_rows == 15
        for metric in ("l2", "cosine", "dot"):
            out = client.search(qs, "test/table", "vector", metric, select=["id"], maxval=7)
            assert out.num_rows == 35
            for qi in range(5):
                # every query of the batch against the ORACLE (the reference's own single-query answer), not against
                # this library's single-query path
                sel = out.filter(pc.field("__QUERY__") == qi)
                ref_rows, ref_dist = search_rows(source, "vector", qs[qi], metric, 7)
                assert_same_neighbours(sel.column("id").to_numpy(), sel.column("__DISTANCE__").to_numpy(),
                                       ref_rows, ref_dist, corpus, qs[qi], metric)
        # batched IVF: one probe mask per query, answered on one resident shard
        config = dict(metric="l2", codebook_size=4, num_codebooks=2, batch_size=256, num_epochs=1)
        client.make_index("cbq", "test/table", "vector", config)
        try:
            full = client.search(qs, "test/table", "vector", "l2", coding="cbq", select=["id"], maxval=5, probes=16)
            for qi in range(5):
                sel = full.filter(pc.field("__QUERY__") == qi)
                ref_rows, ref_dist = search_rows(source, "vector", qs[qi], "l2", 5)     # probing every cell = exact search
                assert_same_neighbours(sel.column("id").to_numpy(), sel.column("__DISTANCE__").to_numpy(),
                                       ref_rows, ref_dist, corpus, qs[qi], "l2")
        finally:
            client.drop_index("cbq")

    def test_errors_surface_as_flight_errors(self, served):
        import pyarrow.flight as fl

        client, *_ = served
        with pytest.raises(fl.FlightServerError):
            client.search(np.zeros(self.VECTOR_SIZE, np.float32), "nope", "vector", "l2", maxval=3)
        with pytest.raises(AssertionError):
            client.search(np.zeros(self.VECTOR_SIZE, np.float32), "test/table", "vector", "manhattan")

    def test_make_index_and_ivf_search(self, served):
        """make_index (host k-means + device code assignment) -> search(coding=, probes=): probing every cell equals
        the exact search, probing few cells returns exactly the best rows of those cells."""
        client, source, corpus, *_ = served
        config = dict(metric="l2", codebook_size=4, num_codebooks=2, batch_size=256, num_epochs=1)
        client.make_index("cb", "test/table", "vector", config)
        try:
            joined = client.read_table("test/table", coding="cb", column="vector").read_all()
            assert joined.column_names == ["id", "vector", "__CODED_ID__"]
            codes = joined.column("__CODED_ID__").to_numpy()
            assert codes.min() >= 0 and codes.max() < 16
            q = corpus[123] + np.float32(0.05)
            full = client.search(q, "test/table", "vector", "l2", coding="cb", select=["id"], maxval=10, probes=16)
            exact = client.search(q, "test/table", "vector", "l2", select=["id"], maxval=10)
            assert full.column("id").to_pylist() == exact.column("id").to_pylist()
            few = client.search(q, "test/table", "vector", "l2", coding="cb", select=["id", "__CODED_ID__"], maxval=10, probes=2)
            cells = set(few.column("__CODED_ID__").to_pylist())
            assert 1 <= len(cells) <= 2
            live = np.nonzero(np.isin(codes, list(cells)))[0]
            want_rows, _ = brute_force_f64(corpus[live], q, "l2", 10)
            assert few.column("id").to_pylist() == live[want_rows[0]].tolist()
        finally:
            client.drop_index("cb")
        assert [*fenix.io.index.list(client_root(served))] == []


@pytest.mark.gpu
def test_flight_serves_the_row_sharded_path(built_library, tmp_path, monkeypatch):
    """FENIX_DEVICES lists several GPUs: ONE server process row-shards the table over them and `Server.do_exchange`
    answers through fx_group_search (worker thread + NCCL communicator per device inside the library, candidates
    all-gathered over NVLink, merged on the device). Same answers as the oracle, single-query and batched, with a
    predicate; concurrent clients; a do_put during the searches (the replaced shard set is retired, never closed under
    a running search). Skipped on a single-GPU box."""
    import threading

    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs at least 2 GPUs")
    n_dev = min(torch.cuda.device_count(), 4)
    monkeypatch.setenv("FENIX_DEVICES", ",".join(str(i) for i in range(n_dev)))
    root = str(tmp_path / "served")
    port = free_port()
    server = fenix.Server(root, "127.0.0.1", port)
    client = fenix.Flight("127.0.0.1", port)
    rng = np.random.default_rng(314)
    corpus = rng.standard_normal((30_011, 64), dtype=np.float32)
    source = table_of(corpus, 1000)
    try:
        client.make_table("t", source.to_reader())
        shard = fenix.io.shards.get(root, "t", "vector", fenix.io.shards.load_table(root, "t"))
        assert len(shard.corpora) == n_dev and shard.group is not None
        shard.release()
        qs = rng.standard_normal((9, 64), dtype=np.float32)
        for metric in ("l2", "cosine", "dot"):
            for qi in range(3):
                out = client.search(qs[qi], "t", "vector", metric, select=["id"], maxval=10)
                ref_rows, ref_dist = search_rows(source, "vector", qs[qi], metric, 10)
                assert_same_neighbours(out.column("id").to_numpy(), out.column("__DISTANCE__").to_numpy(), ref_rows, ref_dist,
                                       corpus, qs[qi], metric)
            out = client.search(qs, "t", "vector", metric, select=["id"], maxval=7)
            for qi in range(len(qs)):
                sel = out.filter(pc.field("__QUERY__") == qi)
                ref_rows, ref_dist = search_rows(source, "vector", qs[qi], metric, 7)
                assert_same_neighbours(sel.column("id").to_numpy(), sel.column("__DISTANCE__").to_numpy(), ref_rows, ref_dist,
                                       corpus, qs[qi], metric)
        flt = pc.field("id") > 20_000        # only the last shard(s) hold live rows
        out = client.search(qs[0], "t", "vector", "l2", select=["id"], filter=flt, maxval=5)
        ref_rows, ref_dist = search_rows(source, "vector", qs[0], "l2", 5, filter=flt)
        assert_same_neighbours(out.column("id").to_numpy(), out.column("__DISTANCE__").to_numpy(), ref_rows, ref_dist, corpus, qs[0], "l2")
        # concurrent clients while the table is replaced
        errors, answers = [], []

        def hammer(t):
            try:
                cl = fenix.Flight("127.0.0.1", port)
                for j in range(20):
                    answers.append(cl.search(qs[(t + j) % len(qs)], "t", "vector", "l2", select=["id"], maxval=5).num_rows)
            except BaseException as exc:
                errors.append(exc)

        threads = [threading.Thread(target=hammer, args=(t,)) for t in range(4)]
        for t in threads:
            t.start()
        client.make_table("t", table_of(corpus[:20_000] + np.float32(1.0), 1000).to_reader())
        for t in threads:
            t.join()
        assert not errors, errors[:1]
        assert all(a == 5 for a in answers)
        out = client.search(qs[1], "t", "vector", "l2", select=["id"], maxval=5)
        ref_rows, ref_dist = search_rows(table_of(corpus[:20_000] + np.float32(1.0), 1000), "vector", qs[1], "l2", 5)
        assert_same_neighbours(out.column("id").to_numpy(), out.column("__DISTANCE__").to_numpy(), ref_rows, ref_dist,
                               corpus[:20_000] + np.float32(1.0), qs[1], "l2")
    finally:
        client.remove()
        server.shutdown()
        fenix.io.shards.invalidate(root)

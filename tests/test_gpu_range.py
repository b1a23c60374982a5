"""Exact range search (fx_search_range / Corpus.search_range): every row with d(q, r) <= radius, d the distance
fx_distances reports, each query's hits ordered by (distance, row). Checked against the exact scan's distance column bit
for bit, on the scan path (small shards, overflowed candidate lists, FX_PREC_EXACT_SCAN) and on the tensor-core filter
with thresholds preset from the radius (TF32, bf16 and int8 operands)."""
import ctypes
import os
import socket

import numpy as np
import pyarrow as pa
import pyarrow.compute as pc
import pytest

import fenix_b200 as fenix
from conftest import table_of
from fenix_b200 import knn
from fenix_b200.io.shards import ShardSet

pytestmark = pytest.mark.gpu

METRICS = ("l2", "cosine", "dot")


@pytest.fixture(scope="module")
def ctx(built_library):
    c = knn.Context(0)
    yield c
    c.close()


def make_corpus(ctx, x, row_base=0):
    c = knn.Corpus(ctx, len(x), x.shape[1], row_base=row_base)
    if len(x):
        c.append(x)
    return c.finalize()


def expected(cols, radius, mask=None, row_base=0):
    """CSR of the rows whose distance column entry is <= radius (and unmasked), ordered by (distance, row)."""
    offsets, rows, dist = [0], [], []
    r32 = np.float32(radius)
    for d in cols:
        ok = d <= r32
        if mask is not None:
            ok &= mask.astype(bool)
        r = np.nonzero(ok)[0]
        r = r[np.lexsort((r, d[r]))]
        rows.append(r + row_base)
        dist.append(d[r])
        offsets.append(offsets[-1] + len(r))
    return np.array(offsets, np.int64), np.concatenate(rows).astype(np.int64), np.concatenate(dist).astype(np.float32)


def assert_same(got, want, what=""):
    assert np.array_equal(got[0], want[0]), ("offsets", what)
    assert np.array_equal(got[1], want[1]), ("rows", what)
    assert np.array_equal(got[2].view(np.uint32), want[2].view(np.uint32)), ("distances", what)


@pytest.mark.parametrize("n", [1_000, 50_000, 300_000])
@pytest.mark.parametrize("d", [7, 100, 128, 768])
def test_definition_and_knn_consistency(ctx, d, n):
    """Radii at the 1st, 10th and 100th neighbour distance of three queries, so rows sit exactly on the boundary; the
    first min(k, hits) entries of every query equal the k-NN search's top k."""
    rng = np.random.default_rng(d * 7 + n)
    x = rng.standard_normal((n, d), dtype=np.float32)
    queries = rng.standard_normal((150, d), dtype=np.float32)
    c = make_corpus(ctx, x)
    try:
        for metric in METRICS:
            cols = [c.distances(q, metric) for q in queries]
            rows_k, dist_k = c.search(queries, metric, 10)
            for qi, rank in ((0, 1), (1, 10), (2, 100)):
                radius = float(np.sort(cols[qi])[rank - 1])
                got = c.search_range(queries, metric, radius)
                want = expected(cols, radius)
                assert_same(got, want, (metric, rank))
                st = c.stats()
                assert (st.last_path == 0) if n < 4096 else (st.last_path in (1, 2)), (metric, st.last_path)
                off = got[0]
                for q in range(len(queries)):
                    m = min(10, off[q + 1] - off[q])
                    assert np.array_equal(got[1][off[q]: off[q] + m], rows_k[q, :m]), (metric, q)
                    assert np.array_equal(got[2][off[q]: off[q] + m], dist_k[q, :m]), (metric, q)
            scan = c.search_range(queries, metric, radius, knn.PREC_EXACT_SCAN)
            assert_same(scan, want, (metric, "scan"))
    finally:
        c.close()


def test_paths_agree(ctx, monkeypatch):
    """int8 (cosine, D = 768), bf16 (cosine with FENIX_INT8=0; L2) and TF32 (no shadow) filters give the same result."""
    rng = np.random.default_rng(5)
    n, d = 50_000, 768
    x = rng.standard_normal((n, d), dtype=np.float32)
    queries = rng.standard_normal((40, d), dtype=np.float32)
    c = make_corpus(ctx, x)
    monkeypatch.setenv("FENIX_BF16_SHADOW", "0")
    c_tf32 = make_corpus(ctx, x)
    monkeypatch.delenv("FENIX_BF16_SHADOW")
    try:
        cols = [c.distances(q, "cosine") for q in queries]
        radius = float(np.sort(cols[0])[30])
        want = expected(cols, radius)
        got = c.search_range(queries, "cosine", radius)
        st = c.stats()
        assert st.last_path == 2 and st.last_operand == 2
        assert_same(got, want, "int8")
        ctx.set_option("FENIX_INT8", 0)
        try:
            got = c.search_range(queries, "cosine", radius)
            assert c.stats().last_operand == 1
            assert_same(got, want, "bf16")
        finally:
            ctx.set_option("FENIX_INT8", None)
        got = c_tf32.search_range(queries, "cosine", radius)
        assert c_tf32.stats().last_path == 1
        assert_same(got, want, "tf32")
        cols = [c.distances(q, "l2") for q in queries]
        radius = float(np.sort(cols[1])[30])
        got = c.search_range(queries, "l2", radius)
        assert c.stats().last_operand == 1
        assert_same(got, expected(cols, radius), "l2 bf16")
    finally:
        c.close()
        c_tf32.close()


def test_overflowing_lists_fall_back_to_the_scan(ctx):
    """A radius admitting ~30 % of a 200k-row shard, and +inf: candidate lists overflow, the scan settles the query."""
    rng = np.random.default_rng(9)
    n, d = 200_000, 32
    x = rng.standard_normal((n, d), dtype=np.float32)
    queries = rng.standard_normal((6, d), dtype=np.float32)
    c = make_corpus(ctx, x)
    try:
        for metric in METRICS:
            cols = [c.distances(q, metric) for q in queries]
            for radius in (float(np.quantile(cols[0], 0.3)), float("inf")):
                before = c.stats().fallback_queries
                got = c.search_range(queries, metric, radius)
                assert c.stats().fallback_queries > before, (metric, radius)
                assert_same(got, expected(cols, radius), (metric, radius))
    finally:
        c.close()


@pytest.mark.parametrize("n", [1_000, 60_000])
def test_edge_cases(ctx, n):
    rng = np.random.default_rng(n)
    d = 64
    x = rng.standard_normal((n, d), dtype=np.float32)
    x[10:20] = x[5]                      # duplicates: ten rows at exactly the same distance
    x[30:33] = 0.0                       # zero rows (cosine: eps-clamped norms)
    queries = rng.standard_normal((20, d), dtype=np.float32)
    queries[0] = x[5] + 0.01
    queries[1] = 0.0                     # a zero query
    c = make_corpus(ctx, x)
    mask = (np.arange(n) % 3 != 1).astype(np.uint8)
    mask[12] = 1
    try:
        for metric in METRICS:
            cols = [c.distances(q, metric) for q in queries]
            boundary = float(cols[0][5])     # the duplicates sit exactly on it
            for radius in (boundary, float(np.sort(cols[2])[50])):
                assert_same(c.search_range(queries, metric, radius), expected(cols, radius), (metric, "plain"))
                assert_same(c.search_range(queries, metric, radius, row_mask=mask), expected(cols, radius, mask),
                            (metric, "mask"))
        cols = [c.distances(q, "dot") for q in queries]
        radius = float(np.sort(cols[3])[20])
        assert radius < 0
        assert_same(c.search_range(queries, "dot", radius), expected(cols, radius), "negative radius")
        off, rows, dist = c.search_range(queries[:0], "l2", 1.0)
        assert off.tolist() == [0] and len(rows) == 0 and len(dist) == 0
        with pytest.raises(ValueError):
            c.search_range(queries, "l2", float("nan"))
        with pytest.raises(NotImplementedError):
            c.search_range(queries, "l2", 1.0, knn.PREC_TF32)
    finally:
        c.close()
    empty = make_corpus(ctx, np.zeros((0, d), np.float32))
    try:
        off, rows, dist = empty.search_range(queries, "l2", float("inf"))
        assert off.tolist() == [0] * 21 and len(rows) == 0
    finally:
        empty.close()


def test_capacity(ctx):
    """Too small a capacity: FX_ETRUNC, the offsets of the full result, the output untouched; Python retries once."""
    rng = np.random.default_rng(3)
    n, d = 50_000, 96
    x = rng.standard_normal((n, d), dtype=np.float32)
    queries = rng.standard_normal((9, d), dtype=np.float32)
    c = make_corpus(ctx, x)
    try:
        cols = [c.distances(q, "l2") for q in queries]
        radius = float(np.sort(cols[0])[40])
        want = expected(cols, radius)
        cap = int(want[0][-1]) - 1
        offsets = np.full(10, -7, np.int64)
        rows = np.full(cap, -3, np.int64)
        dist = np.full(cap, 5.0, np.float32)
        lib = knn.load_library()
        code = lib.fx_search_range(c._h, queries.ctypes.data, 9, 0, ctypes.c_float(radius), knn.PREC_FP32, None, cap,
                                   offsets.ctypes.data, rows.ctypes.data, dist.ctypes.data)
        assert code == knn.FX_ETRUNC
        assert np.array_equal(offsets, want[0])
        assert (rows == -3).all() and (dist == 5.0).all()
        assert_same(c.search_range(queries, "l2", radius, capacity=1), want, "retry")
        assert_same(c.search_range(queries, "l2", radius, capacity=0), want, "retry from zero")
    finally:
        c.close()


def test_row_shards_merge_to_the_single_shard_result(ctx):
    rng = np.random.default_rng(11)
    n, d = 90_000, 48
    x = rng.standard_normal((n, d), dtype=np.float32)
    queries = rng.standard_normal((7, d), dtype=np.float32)
    whole = make_corpus(ctx, x)
    bases = [0, 30_000, 31_000]
    parts = [make_corpus(ctx, x[lo:hi], row_base=lo) for lo, hi in zip(bases, bases[1:] + [n])]
    mask = (np.arange(n) % 5 != 0).astype(np.uint8)
    try:
        sharded = ShardSet(dim=d, n_rows=n, corpora=parts, bases=bases)
        for metric in METRICS:
            radius = float(np.sort(whole.distances(queries[0], metric))[200])
            assert_same(sharded.search_range(queries, metric, radius), whole.search_range(queries, metric, radius), metric)
            assert_same(sharded.search_range(queries, metric, radius, row_mask=mask),
                        whole.search_range(queries, metric, radius, row_mask=mask), (metric, "mask"))
    finally:
        whole.close()
        for p in parts:
            p.close()


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def test_flight_end_to_end(built_library, tmp_path):
    rng = np.random.default_rng(21)
    n, d = 20_000, 64
    corpus = rng.standard_normal((n, d), dtype=np.float32)
    source = table_of(corpus, 1_000)
    port = _free_port()
    server = fenix.Server(str(tmp_path), "127.0.0.1", port)
    client = fenix.Flight("127.0.0.1", port)
    try:
        client.make_table("t", source.to_reader())
        ctx = knn.Context(0)
        c = make_corpus(ctx, corpus)
        qs = rng.standard_normal((3, d), dtype=np.float32)
        col0 = c.distances(qs[0], "l2")
        radius = float(np.sort(col0)[25])
        one = client.search_range(qs[0], "t", "vector", "l2", radius)
        assert one.schema == pa.schema([*source.schema, pa.field("__DISTANCE__", pa.float32())])
        want = expected([col0], radius)
        assert np.array_equal(one.column("id").to_numpy(), want[1]) and np.array_equal(one.column("__DISTANCE__").to_numpy(), want[2])
        cols = [c.distances(q, "l2") for q in qs]
        batch = client.search_range(qs, "t", "vector", "l2", radius, select=["id"])
        assert batch.column_names == ["id", "__DISTANCE__", "__QUERY__"]
        want = expected(cols, radius)
        assert np.array_equal(batch.column("id").to_numpy(), want[1])
        assert np.array_equal(batch.column("__QUERY__").to_numpy(), np.repeat(np.arange(3), np.diff(want[0])))
        flt = pc.field("id") >= 7_000
        mask = (source.column("id").to_numpy() >= 7_000).astype(np.uint8)
        filtered = client.search_range(qs, "t", "vector", "l2", radius, select=["id"], filter=flt)
        assert np.array_equal(filtered.column("id").to_numpy(), expected(cols, radius, mask)[1])
        capped = client.search_range(qs, "t", "vector", "l2", radius, select=["id"], maxval=10)
        rows_k, dist_k = c.search(qs, "l2", 10)
        keep = dist_k <= np.float32(radius)
        assert np.array_equal(capped.column("id").to_numpy(), rows_k[keep])
        assert np.array_equal(capped.column("__DISTANCE__").to_numpy(), dist_k[keep])
        c.close()
        ctx.close()
    finally:
        client.remove()
        server.shutdown()


def test_scale_2m_cosine(ctx):
    """2M x 768 cosine, 32 queries, radius at the 50th neighbour of the first: against the scan's distance column."""
    rng = np.random.default_rng(2)
    n, d = 2_000_000, 768
    x = rng.standard_normal((n, d), dtype=np.float32)
    queries = rng.standard_normal((32, d), dtype=np.float32)
    c = make_corpus(ctx, x)
    del x
    try:
        cols = [c.distances(q, "cosine") for q in queries]
        radius = float(np.sort(cols[0])[49])
        got = c.search_range(queries, "cosine", radius)
        assert c.stats().last_operand == 2
        assert_same(got, expected(cols, radius), "2M")
    finally:
        c.close()

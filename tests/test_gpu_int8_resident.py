"""The int8 CTA-pair filter with resident query tiles (FENIX_TC_RESIDENT): each CTA of a pair keeps its whole int8 query
tile in shared memory for a unit and streams only corpus half blocks. Its results must equal the fp64 scan bit for bit,
through every pass that reaches the kernel: the main filter, the sample prepass, masked searches and the preset-threshold
refinement pass."""
import numpy as np
import pytest

from fenix_b200 import knn

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx(built_library):
    c = knn.Context(0)
    yield c
    c.close()


def make_corpus(ctx, x):
    c = knn.Corpus(ctx, len(x), x.shape[1])
    c.append(x)
    return c.finalize()


def search_with(ctx, c, queries, k, opts, **kw):
    for key, value in opts.items():
        ctx.set_option(key, value)
    try:
        before = c.stats()
        rows, dist = c.search(queries, "cosine", k, **kw)
        return rows, dist, before, c.stats()
    finally:
        for key in opts:
            ctx.set_option(key, None)


@pytest.mark.parametrize("d", [200, 384, 768, 1000])
def test_bit_equal_to_the_fp64_scan(ctx, d):
    """300 queries: three query tiles (the second pair holds one tile, the last one ragged); a shard that is not a
    multiple of 256 rows; the default slicing (on 148 SMs: 74 units over 74 pair workers, so no query tile is ever
    reloaded) and forced slices (several units per worker, reloads); a row mask; the sample
    prepass (forced on this small shard by a thin sample); and the refinement pass (K' = 32 flags a quarter of the
    queries or more: a 1200-query batch sends more than one query tile of them through it)."""
    rng = np.random.default_rng(100 + d)
    n, nq, k = 200_000 - 37, 300, 10
    corpus = rng.standard_normal((n, d), dtype=np.float32)
    corpus[150_000:150_040] = corpus[17]               # duplicates: the query near row 17 needs more than k candidates
    queries = rng.standard_normal((nq, d), dtype=np.float32)
    queries[0] = corpus[17] + 0.05 * rng.standard_normal(d).astype(np.float32)
    c = make_corpus(ctx, corpus)
    mask = (np.arange(n) % 4 != 1).astype(np.uint8)
    want = c.search(queries, "cosine", k, knn.PREC_EXACT_SCAN)
    want_m = c.search(queries, "cosine", k, knn.PREC_EXACT_SCAN, row_mask=mask)
    on = {"FENIX_TC_RESIDENT": 1}
    cases = (
        ("default slices", {}),
        ("several units per worker", {"FENIX_TC_SLICES": 90}),
        ("sample prepass", {"FENIX_TC_PRE_SAFETY": 1, "FENIX_TC_PRE_M": 64}),
    )
    for name, opts in cases:
        rows, dist, before, st = search_with(ctx, c, queries, k, {**on, **opts})
        assert st.last_operand == 2 and st.last_resident_queries == 1 and st.last_variant & 4, (name, st)
        assert np.array_equal(rows, want[0]) and np.array_equal(dist, want[1]), name
        assert st.fallback_queries == before.fallback_queries, name
        if name == "sample prepass":
            assert st.last_variant & 2, st
    many = np.concatenate([queries, rng.standard_normal((900, d), dtype=np.float32)])
    want_r = c.search(many, "cosine", k, knn.PREC_EXACT_SCAN)
    rows, dist, before, st = search_with(ctx, c, many, k, {**on, "FENIX_TC_KP": 32, "FENIX_TC_PRE": 0})
    assert st.last_resident_queries == 1 and np.array_equal(rows, want_r[0]) and np.array_equal(dist, want_r[1])
    # more than one query tile of flagged queries: the refinement pass runs through the CTA-pair kernel too
    assert st.refined_queries - before.refined_queries > 128 and st.fallback_queries == before.fallback_queries, st
    rows, dist, _, st = search_with(ctx, c, queries, k, on, row_mask=mask)
    assert st.last_resident_queries == 1 and mask[rows].all()
    assert np.array_equal(rows, want_m[0]) and np.array_equal(dist, want_m[1])
    c.close()


def test_selection(ctx):
    """Auto: where the CTA-pair kernel runs over the int8 shadow (rows from 7 bf16 k-blocks, >= 2 query tiles), the query
    tile leaves room for 4 corpus stages (D <= 1152) and the shard has >= 4M rows. FENIX_TC_RESIDENT=1 takes it wherever
    it fits, =0 never; every choice finds the same rows."""
    import torch

    rng = np.random.default_rng(11)
    for d in (384, 768, 1152, 1280):
        c = make_corpus(ctx, rng.standard_normal((30_000, d), dtype=np.float32))
        q = rng.standard_normal((300, d), dtype=np.float32)
        rows, dist, _, st = search_with(ctx, c, q, 10, {})
        assert st.last_operand == 2 and st.last_resident_queries == 0 and bool(st.last_variant & 4) == (d >= 448), (d, st)
        rows1, dist1, _, st1 = search_with(ctx, c, q, 10, {"FENIX_TC_RESIDENT": 1})
        assert st1.last_resident_queries == (1 if d <= 1152 else 0) and st1.last_variant & 4, (d, st1)
        assert np.array_equal(rows, rows1) and np.array_equal(dist, dist1), d
        c.close()
    n, d = (1 << 22) + 1000, 768
    g = torch.Generator(device="cuda").manual_seed(12)
    x = torch.randn((n, d), generator=g, device="cuda", dtype=torch.float32)
    c = knn.Corpus(ctx, n, d)
    torch.cuda.synchronize()
    c.append_device(x.data_ptr(), n)
    c.finalize()
    del x
    q = rng.standard_normal((300, d), dtype=np.float32)
    rows, dist, _, st = search_with(ctx, c, q, 10, {})
    assert st.last_operand == 2 and st.last_resident_queries == 1 and st.last_variant & 4, st
    rows0, dist0, _, st0 = search_with(ctx, c, q, 10, {"FENIX_TC_RESIDENT": 0})
    assert st0.last_resident_queries == 0 and st0.last_variant & 4, st0
    assert np.array_equal(rows, rows0) and np.array_equal(dist, dist0)
    c.close()


def test_graph_replay_of_single_queries(ctx):
    """Graphs are captured for searches of <= 64 queries, one query tile, which never takes a CTA pair: the forced knob
    changes nothing there, and captured and replayed searches report that and answer as the fp64 scan does."""
    rng = np.random.default_rng(8)
    n, d = 100_000, 768
    c = make_corpus(ctx, rng.standard_normal((n, d), dtype=np.float32))
    q = rng.standard_normal((1, d), dtype=np.float32)
    want = c.search(q, "cosine", 10, knn.PREC_EXACT_SCAN)
    ctx.set_option("FENIX_DIRECT", 0)
    ctx.set_option("FENIX_TC_RESIDENT", 1)
    try:
        for _ in range(4):                             # call 2 captures, calls 3+ replay
            rows, dist = c.search(q, "cosine", 10)
            st = c.stats()
            assert st.last_path == 2 and st.last_operand == 2 and st.last_resident_queries == 0 and not st.last_variant & 4
            assert np.array_equal(rows, want[0]) and np.array_equal(dist, want[1])
    finally:
        ctx.set_option("FENIX_TC_RESIDENT", None)
        ctx.set_option("FENIX_DIRECT", None)
    c.close()

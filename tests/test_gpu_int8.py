"""The int8 filter (operand kind 2): exact cosine searches at small k over wide rows stream an int8 shadow of the
normalised rows with tcgen05 kind::i8 MMAs. Its scores are certified upper bounds of the exact cosine (tc_filter.cuh,
i8_scale), so results must equal the fp64 scan bit for bit."""
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


def quantise(v):
    """The int8 format of a group of vectors (rows of v): normalised rows, the group's scale, the residual norms."""
    v = v.astype(np.float64)
    n = np.maximum(np.linalg.norm(v, axis=1, keepdims=True), 1e-12)
    h = v / n
    m = np.abs(h).max()
    s = np.float32(127.0 / m) if m > 0 else np.float32(1.0)
    t = np.clip(np.rint(h * np.float64(s)), -127, 127)
    return h, s, t, np.linalg.norm(h - t / np.float64(s), axis=1)


def special_rows(rng, d):
    """Tile 0 of the test shards: a zero row, a single-coordinate spike, values at rounding midpoints, Gaussian rest."""
    x = rng.standard_normal((256, d)).astype(np.float32)
    x[3] = 0.0
    x[7] = 0.0
    x[7, d // 2] = 50.0
    x[11] = (np.arange(d) % 7 - 3 + 0.5).astype(np.float32)
    x[12] = 1.0
    return x


@pytest.mark.parametrize("d", [200, 448, 768, 1100])
def test_raw_scores_are_certified_upper_bounds(ctx, d):
    rng = np.random.default_rng(d)
    corpus = rng.standard_normal((8192, d), dtype=np.float32)
    corpus[:256] = special_rows(rng, d)
    queries = rng.standard_normal((128, d), dtype=np.float32)
    queries[5] = 0.0
    queries[9] = corpus[11]
    c = make_corpus(ctx, corpus)
    ctx.set_option("FENIX_INT8", 1)
    try:
        s = c.debug_scores(queries, "cosine").astype(np.float64)
    finally:
        ctx.set_option("FENIX_INT8", None)
    xh, _, _, rx = quantise(corpus[:256])
    e_t = rx.max()
    qh = queries.astype(np.float64) / np.maximum(np.linalg.norm(queries.astype(np.float64), axis=1, keepdims=True), 1e-12)
    bound = np.empty(128)
    for i in range(128):
        _, sq, tq, rq = quantise(queries[i: i + 1])
        bound[i] = np.linalg.norm(tq) / np.float64(sq) * e_t + rq[0]
    exact = qh @ xh.T
    assert (s >= exact - 1e-7).all(), (exact - s).max()
    assert (s <= exact + 2.0 * bound[:, None] + 1e-6).all(), ((s - exact) / bound[:, None]).max()
    assert bound[5] == 0.0 and np.abs(s[5]).max() < 1e-12   # zero query: q~ = 0, a_q = e_q = 0
    c.close()


def test_operand_selection(ctx, monkeypatch):
    rng = np.random.default_rng(3)
    q = rng.standard_normal((300, 256), dtype=np.float32)
    c = make_corpus(ctx, rng.standard_normal((20_000, 256), dtype=np.float32))
    mask = (np.arange(20_000) % 3 != 0).astype(np.uint8)
    for metric, k, kw, want in (("cosine", 10, {}, 2), ("cosine", 16, {}, 2), ("cosine", 17, {}, 1), ("l2", 10, {}, 1),
                                ("dot", 10, {}, 1), ("cosine", 10, {"row_mask": mask}, 2)):
        c.search(q, metric, k, **kw)
        st = c.stats()
        assert st.last_path == 2 and st.last_operand == want, (metric, k, kw.keys(), st.last_operand)
    c.search(q, "cosine", 10, knn.PREC_BF16)
    assert c.stats().last_operand == 1
    ctx.set_option("FENIX_INT8", 0)
    c.search(q, "cosine", 10)
    assert c.stats().last_operand == 1
    ctx.set_option("FENIX_INT8", None)
    c.close()
    narrow = make_corpus(ctx, rng.standard_normal((20_000, 192), dtype=np.float32))
    narrow.search(rng.standard_normal((300, 192), dtype=np.float32), "cosine", 10)
    assert narrow.stats().last_operand == 1            # narrow rows keep the resident-query kernel
    narrow.close()
    ctx.set_option("FENIX_NO_NORM_SHADOW", 1)
    try:
        c2 = make_corpus(ctx, rng.standard_normal((20_000, 256), dtype=np.float32))
        c2.search(q, "cosine", 10)
        assert c2.stats().last_operand == 1
        c2.close()
    finally:
        ctx.set_option("FENIX_NO_NORM_SHADOW", None)
    monkeypatch.setenv("FENIX_BF16_SHADOW", "0")
    c3 = make_corpus(ctx, rng.standard_normal((20_000, 256), dtype=np.float32))
    c3.search(q, "cosine", 10)
    assert c3.stats().last_operand == 0
    c3.close()


@pytest.mark.parametrize("pair", [0, 1])
@pytest.mark.parametrize("d", [256, 768])
def test_bit_equal_to_the_fp64_scan(ctx, d, pair):
    """Forced one-CTA and CTA-pair kernels, sample prepass on and off, a row mask, a ragged last query tile, duplicates
    (the refinement pass) and the spike tile, which must not send any query to the scan."""
    rng = np.random.default_rng(d + pair)
    n, nq, k = 60_000, 300, 10
    corpus = rng.standard_normal((n, d), dtype=np.float32)
    corpus[:256] = special_rows(rng, d)
    corpus[30_000:30_300] = corpus[17]                 # more copies than K': query 0 needs the refinement pass
    queries = rng.standard_normal((nq, d), dtype=np.float32)
    # (a near-copy: an exact copy's distance is 0 up to the fp64 rounding of |q|, which the rerank and the scan sum in
    # different orders)
    queries[0] = corpus[17] + 0.05 * rng.standard_normal(d).astype(np.float32)
    queries[1] = corpus[7] + 0.05 * rng.standard_normal(d).astype(np.float32)   # near the spike row
    c = make_corpus(ctx, corpus)
    mask = (np.arange(n) % 4 != 1).astype(np.uint8)
    want = c.search(queries, "cosine", k, knn.PREC_EXACT_SCAN)
    want_m = c.search(queries, "cosine", k, knn.PREC_EXACT_SCAN, row_mask=mask)
    ctx.set_option("FENIX_INT8", 0)
    bf16 = c.search(queries, "cosine", k)
    ctx.set_option("FENIX_INT8", None)
    assert c.stats().last_operand == 1
    assert np.array_equal(bf16[0], want[0]) and np.array_equal(bf16[1], want[1])
    ctx.set_option("FENIX_TC_PAIR", pair)
    try:
        for pre in (None, 0):
            ctx.set_option("FENIX_TC_PRE", pre)
            before = c.stats()
            rows, dist = c.search(queries, "cosine", k)
            st = c.stats()
            assert st.last_operand == 2 and bool(st.last_variant & 4) == bool(pair), st
            assert np.array_equal(rows, want[0]) and np.array_equal(dist, want[1]), (pre, pair)
            assert st.fallback_queries == before.fallback_queries
            assert st.refined_queries - before.refined_queries >= 1   # the duplicates
            rows, dist = c.search(queries, "cosine", k, row_mask=mask)
            assert np.array_equal(rows, want_m[0]) and np.array_equal(dist, want_m[1]), (pre, pair, "mask")
    finally:
        ctx.set_option("FENIX_TC_PRE", None)
        ctx.set_option("FENIX_TC_PAIR", None)
    c.close()


def test_shadow_sizes(ctx):
    rng = np.random.default_rng(21)
    n, d = 16_384, 300
    c = make_corpus(ctx, rng.standard_normal((n, d), dtype=np.float32))
    q = rng.standard_normal((200, d), dtype=np.float32)
    rows_bytes = c.stats().device_bytes
    c.search(q, "cosine", 10)
    tiles = n // 256
    i8 = tiles * 256 * 128 * 3 + tiles * 8             # three 128-column k-blocks per row, (S_t, E_t) per tile
    assert c.stats().last_operand == 2 and c.stats().device_bytes == rows_bytes + i8
    c.search(q, "cosine", 100)                         # large k: the bf16 normalised shadow joins it
    assert c.stats().last_operand == 1 and c.stats().device_bytes == rows_bytes + i8 + n * 320 * 2
    c.close()


def test_graph_replay_of_single_queries(ctx):
    rng = np.random.default_rng(5)
    n, d = 100_000, 256
    c = make_corpus(ctx, rng.standard_normal((n, d), dtype=np.float32))
    ctx.set_option("FENIX_DIRECT", 0)
    try:
        q = rng.standard_normal((1, d), dtype=np.float32)
        first = c.search(q, "cosine", 10)
        assert c.stats().last_operand == 2
        for _ in range(4):                             # call 2 captures, calls 3+ replay
            rows, dist = c.search(q, "cosine", 10)
            assert c.stats().last_operand == 2
            assert np.array_equal(rows, first[0]) and np.array_equal(dist, first[1])
        other = rng.standard_normal((1, d), dtype=np.float32)
        rows, dist = c.search(other, "cosine", 10)
        want = c.search(other, "cosine", 10, knn.PREC_EXACT_SCAN)
        assert np.array_equal(rows, want[0]) and np.array_equal(dist, want[1])
    finally:
        ctx.set_option("FENIX_DIRECT", None)
    c.close()

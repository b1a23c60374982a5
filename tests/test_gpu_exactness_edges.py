"""The exactness certificate where its error bounds are tight, on exactly summable ("dyadic") data, against the bit-exact
fp64 model of tests/exact_model.py.

* Adversarial rows: true neighbours whose filter score errs downward by as much as the operand allows, and more than K'
  decoys whose exact scores are worse but whose filter scores are higher. The filter ranks them wrongly; only a correct
  bound and certificate recover the answer. Each construction asserts on tile 0 (fx_debug_scores) that it reaches a
  stated fraction of the bound E, and that a certificate built on E/2 would lose the neighbours.
* A magnitude ladder: one shard and its queries scaled by 2^e across the fp32 range (products below FLT_MIN, the bf16
  terms of -|x|^2/2 in the subnormal range, |x|^2 and q.x beyond FLT_MAX). Every path must return the model's rows and
  bits; a route to the scan is fine at the extremes.
* Exact ties at the k-th distance and at the radius across a row_base boundary.
"""
import contextlib

import numpy as np
import pytest

import exact_model as em
from fenix_b200 import knn

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx(built_library):
    c = knn.Context(0)
    yield c
    c.close()


def make_corpus(ctx, x, row_base=0):
    c = knn.Corpus(ctx, len(x), x.shape[1], row_base=row_base)
    c.append(x)
    return c.finalize()


@contextlib.contextmanager
def options(ctx, **kw):
    for k, v in kw.items():
        ctx.set_option(k, v)
    try:
        yield
    finally:
        for k in kw:
            ctx.set_option(k, None)


def assert_topk(got, want, what):
    assert np.array_equal(got[0], want[0]), ("rows", what, np.nonzero((got[0] != want[0]).any(1))[0][:8])
    assert np.array_equal(got[1].view(np.uint32), want[1].view(np.uint32)), ("distances", what)


def assert_csr(got, want, what):
    assert np.array_equal(got[0], want[0]), ("offsets", what)
    assert np.array_equal(got[1], want[1]), ("rows", what)
    assert np.array_equal(got[2].view(np.uint32), want[2].view(np.uint32)), ("distances", what)


def counters(c):
    s = c.stats()
    return s.refined_queries, s.fallback_queries


# ---- how the operands round ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("operand", ["tf32", "bf16"])
def test_operand_rounding_is_within_the_bound_constants(ctx, operand):
    """q = e_0 and rows whose first coordinate walks through one ulp of the operand: the filter score IS the rounded
    coordinate. TF32's constant assumes truncation to 10 bits (error < 2^-10 relative), bf16's round-to-nearest to 8
    significant bits (error <= 2^-8 relative)."""
    d, n = 256, 8192
    x = np.zeros((n, d), np.float32)
    x[:, 1] = 1.0
    j = np.arange(256)
    x[:256, 0] = em.from_ints(np.where(j % 2, -1, 1) * (2 ** 14 + j), -14)
    q = np.zeros((128, d), np.float32)
    q[:, 0] = 1.0
    c = make_corpus(ctx, x)
    with options(ctx, **({"FENIX_DEBUG_BF16": 1} if operand == "bf16" else {})):
        s = c.debug_scores(q, "dot")[0].astype(np.float64)
    c.close()
    exact = x[:256, 0].astype(np.float64)
    rel = np.abs(s - exact) / np.abs(exact)
    bits = 11 if operand == "tf32" else 8
    trunc = np.sign(exact) * np.floor(np.abs(exact) * 2.0 ** (bits - 1)) / 2.0 ** (bits - 1)
    mode = "truncates" if np.array_equal(s, trunc) else "rounds"
    assert mode == ("truncates" if operand == "tf32" else "rounds"), (operand, mode)   # what the constants assume
    assert rel.max() < (2.0 ** -10 if operand == "tf32" else 2.0 ** -8 * (1 + 2.0 ** -7)), (operand, mode, rel.max())
    assert rel.max() > 2.0 ** -(bits + 1), (operand, mode, "the walk must reach the rounding cut")
    print(f"{operand} {mode}: max relative error {rel.max():.3e}")


# ---- adversarial rows at the bound ---------------------------------------------------------------------------------
def plant(rng, operand, d, n, k, n_decoys, spread):
    """Rows 0 .. k-1: true neighbours, every coordinate `a` (the query's too) just short of the operand's rounding cut, so
    that q~.x~ = D loses ~2 ulp/2 (bf16) or ~2 ulp (TF32 truncation) per product. Rows k .. k + n_decoys - 1: decoys, half
    their coordinates 1 + ulp and half 1 - ulp/2, both exact in the operand: filter score D (1 + ulp/4) beats the
    neighbours', exact score a D (1 + ulp/4) loses to theirs (D a^2); in L2 and cosine terms too. The rest: random +-1
    rows (exact, far away), of similar norm, or - spread - mostly 2^-6 of it (the shard's norms spread: the augmented
    inner-product form)."""
    ulp = 2.0 ** -10 if operand == "tf32" else 2.0 ** -7
    cut = ulp if operand == "tf32" else ulp / 2                     # truncation loses up to 1 ulp, rounding 1/2
    a = 1.0 + cut - 2.0 ** -20
    x = np.where(rng.random((n, d)) < 0.5, -1.0, 1.0)
    if spread:
        x[n // 8:] *= 2.0 ** -6
    x[:k] = a
    x[k: k + n_decoys, : d // 2] = 1.0 + ulp
    x[k: k + n_decoys, d // 2:] = 1.0 - ulp / 2
    q = np.full((130, d), a)
    return x.astype(np.float32), q.astype(np.float32)


def plant_normalised(rng, d, n, k, n_decoys):
    """The normalised bf16 shadow stores x^ = x / |x|, so the rounding cut must be met after the normalisation. Rows
    0 .. k-1 (and the query): 254 coordinates u = 1 + 2^-8 - 2^-20 and two u/8; then |x| ~ 15.9 puts x^ just below bf16
    cuts as well (found by a search over such rows on the CPU: 0.89 of the bound). Decoys: 254 ones and two 1/4, whose
    normalised coordinates round upward - cosine 1 - 6e-5, filter score above the neighbours'."""
    u = 1.0 + 2.0 ** -8 - 2.0 ** -20
    row = np.full(d, u)
    row[-2:] = u / 8
    x = np.where(rng.random((n, d)) < 0.5, -1.0, 1.0)
    x[:k] = row
    decoy = np.full(d, 1.0)
    decoy[-2:] = 0.25
    x[k: k + n_decoys] = decoy
    return x.astype(np.float32), np.tile(row, (130, 1)).astype(np.float32)


FORMS = {   # form: (metric, operand kind, options of the search, options of fx_debug_scores)
    "tf32-dot": ("dot", 0, {"FENIX_FP32_FILTER_TF32": 1}, {}),
    "bf16-dot": ("dot", 1, {}, {"FENIX_DEBUG_BF16": 1}),
    "bf16-dot-augmented": ("dot", 1, {}, {"FENIX_DEBUG_BF16": 1}),
    "bf16-l2-augmented": ("l2", 1, {}, {"FENIX_DEBUG_BF16": 1}),
    "bf16-cosine-normalised": ("cosine", 1, {"FENIX_INT8": 0}, {"FENIX_DEBUG_BF16": 1}),
    "bf16-cosine-multiplicative": ("cosine", 1, {"FENIX_INT8": 0, "FENIX_NO_NORM_SHADOW": 1},
                                   {"FENIX_DEBUG_BF16": 1, "FENIX_NO_NORM_SHADOW": 1}),
}


def exact_scores(metric, q, x):
    """The filter's score of each form, in fp64: q.x (dot), q.x - |x|^2/2 (l2), |q| cos (cosine: q . x^)."""
    qq, xx, qx = em.sums(q, x)
    if metric == "dot":
        return qx
    if metric == "l2":
        return qx - 0.5 * xx[None, :]
    return qx / np.maximum(np.sqrt(xx), 1e-12)[None, :]


@pytest.mark.parametrize("form", list(FORMS))
def test_neighbours_at_the_bound_are_recovered(ctx, form):
    """k = 10, 100 decoys (> K' + 1). Sharpness on tile 0 (fx_debug_scores): the forms with an error bound E = c |q| max|x|
    (cosine: c |q|) must show (a) the neighbours' filter error reaching >= 0.6 of E and (c) their filter score below
    s(d_k) - E/2, so that a certificate on half the bound would lose them; the augmented forms carry the allowance in the
    score, which (b) must stay an upper bound while the rounding (a, c) uses more than half of it. Then the search must
    return the model's answer bit for bit, settled by the refinement tier."""
    metric, kind, opts, dbg = FORMS[form]
    rng = np.random.default_rng(7)
    d, n, k = 256, 8192, 10
    if form == "bf16-cosine-normalised":
        x, q = plant_normalised(rng, d, n, k, 100)
    else:
        x, q = plant(rng, "tf32" if kind == 0 else "bf16", d, n, k, 100, form == "bf16-dot-augmented")
    assert em.summable(21, 21, d)
    c = make_corpus(ctx, x)
    with options(ctx, **dbg):
        s = c.debug_scores(q, metric)[0].astype(np.float64)
    exact = exact_scores(metric, q[:1], x[:256])[0]
    nq, xm = np.sqrt(em.sums(q[:1], x)[0][0]), np.sqrt(em.sums(q[:1], x)[1].max())
    s_k = np.sort(exact)[::-1][k - 1]
    assert s_k == exact[0] and (exact[k: k + 100] < s_k).all() and (s[k: k + 100] > s[:k].max()).all()
    if form.endswith("augmented"):
        # u |x| (u = c |q|) rides in the score: it must stay an upper bound (b), and the rounding must use more than
        # half of the allowance (a, c): an allowance of half the size would leave the score below the exact one
        allowance = em.c_err(d, 1) * nq * np.sqrt(em.sums(q[:1], x[:k])[1])
        frac = 1.0 - ((s[:k] - exact[:k]) / allowance).min()
        assert (s[:k] >= exact[:k] - 1e-6 * np.abs(exact[:k])).all(), (s[:k] - exact[:k]).min()    # (b)
        assert frac >= 0.6, frac                                                                  # (a), (c)
    else:
        e = em.c_err(d, kind) * nq * (1.0 if metric == "cosine" else xm)
        frac = (exact[:k] - s[:k]).max() / e
        assert 0.6 <= frac <= 1.0, (form, frac)                                   # (a)
        assert (s[:k] < s_k - e / 2).all(), form                                  # (c)
    print(f"{form}: filter error / E = {frac:.3f}")
    want = em.topk(em.distances(q, x, metric), k)
    before = counters(c)
    with options(ctx, **opts):
        got = c.search(q, metric, k)
    st = c.stats()
    assert st.last_operand == kind, st
    assert_topk(got, want, (form, counters(c), before))
    refined, fallback = np.subtract(counters(c), before)
    assert refined >= 1 and fallback == 0, (refined, fallback)   # tier 1 settles the queries the first pass flags
    c.close()


def test_tiers_on_adversarial_rows(ctx):
    """The bf16 construction, settled by each tier: (0) with fewer decoys than K' the certificate passes near the bound
    and no counter moves; (1) more than 1024 exact copies at the k-th distance overflow tier 1 into the fp64 scan
    (fallback_queries moves); (2) a masked search over the same rows; (3) the resident-query kernel (D <= 192, 256
    queries) and the streaming one (FENIX_TC_NO_RQ) on the construction."""
    rng = np.random.default_rng(11)
    d, n, k = 128, 16384, 10
    x, q = plant(rng, "bf16", d, n, k, 20, False)
    q = np.concatenate([q, q])[:256]
    c = make_corpus(ctx, x)
    before = counters(c)
    assert_topk(c.search(q, "dot", k), em.topk(em.distances(q, x, "dot"), k), "certificate")
    assert counters(c) == before and c.stats().last_variant & 1, c.stats()      # resident-query kernel, no tier
    x[20:120] = x[20]
    x[4000:5100] = x[0]
    c.close()
    c = make_corpus(ctx, x)
    D = em.distances(q, x, "dot")
    before = counters(c)
    assert_topk(c.search(q, "dot", k), em.topk(D, k), "ties")
    assert c.stats().last_variant & 1, c.stats()
    assert counters(c)[1] > before[1], "more than 1024 rows at the k-th distance go to the scan"
    mask = (np.arange(n) % 3 != 0).astype(np.uint8)
    assert_topk(c.search(q, "dot", k, row_mask=mask), em.topk(D, k, mask=mask), "mask")
    with options(ctx, FENIX_TC_NO_RQ=1):
        assert_topk(c.search(q, "dot", k), em.topk(D, k), "streaming kernel")
        assert c.stats().last_variant & 1 == 0, c.stats()
    c.close()


# ---- int8: tiles whose (S_t, E_t) differ sharply -------------------------------------------------------------------
def int8_shard(rng, d):
    """8192 + 100 rows (33 tiles, the last ragged). Neighbour tiles 0, 1 (odd: the second CTA of a pair) and 32 (the
    last): row 0 a one-hot spike (S_t = 127), rows 1 - 4 the neighbours, the rest random dyadic rows. A neighbour t has
    coordinates +-119/16 and +-135/16 with |t| = 126.8, so 127 t^ sits 0.448 of a grid step above the int8 grid point,
    toward sign(q_i): the residual is aligned with q^ and sets the tile's E_t (~0.056). Decoy tiles 2 and 31: dense +-1
    rows with sign(q) and 1 - 4 signs flipped - on the int8 grid (E_t ~ 0), cosine 0.97 - 0.99. With the right
    (S_t, E_t) a neighbour's upper bound (~1) beats every decoy; with E_t = 0 it drops to ~0.94, below all 512 decoys
    (more than K' = 256), and the certificate would pass on the decoys. The query: t itself."""
    n = 32 * 256 + 100
    sign = np.where(rng.random(d) < 0.5, -1.0, 1.0)
    mag = np.where(np.arange(d) < 135, 119 / 16, 135 / 16)
    t = (sign * mag).astype(np.float32)
    x = em.dyadic(rng, (n, d), 8, -6)
    for tile in (0, 1, 32):
        x[tile * 256] = 0.0
        x[tile * 256, 0] = 1.0
        x[tile * 256 + 1: tile * 256 + 5] = t
    for tile in (2, 31):
        blk = np.tile(sign, (256, 1))
        for r in range(256):
            blk[r, rng.choice(d, 1 + r % 4, replace=False)] *= -1
        x[tile * 256: (tile + 1) * 256] = blk.astype(np.float32)
    q = em.dyadic(rng, (300, d), 8, -4)
    q[0] = t
    assert em.summable(8, 8, d)
    return x, q


def test_int8_construction_is_sharp(ctx):
    """Tile 0 of the int8 shard: the neighbours' upper bounds (b) stay above the exact cosine, and their aligned residuals
    use (a) >= 0.6 of the allowance a_q E_t + e_q, so (c) half of it would leave the bound below the exact cosine."""
    rng = np.random.default_rng(3)
    x, q = int8_shard(rng, 256)
    _, e_t = em.i8_tiles(x)
    assert e_t[[0, 1, 32]].min() > 100 * e_t[[2, 31]].max() and len(x) % 256 == 100
    c = make_corpus(ctx, x)
    with options(ctx, FENIX_INT8=1):
        s = c.debug_scores(q, "cosine")[0, 1:5].astype(np.float64)
    c.close()
    qq, xx, qx = em.sums(q[:1], x[1:5])
    exact = qx[0] / (np.sqrt(qq[0]) * np.sqrt(xx))
    _, a_q, e_q = em.i8_query(q[0])
    allowance = a_q * e_t[0] + e_q
    frac = 1.0 - ((s - exact) / allowance).min()
    assert (s >= exact - 1e-6).all(), (s - exact).min()           # (b)
    assert frac >= 0.6, frac                                      # (a), (c)
    print(f"int8: residual share of the allowance = {frac:.3f}")


@pytest.mark.parametrize("pair,resident", [(0, 0), (1, 0), (1, 1)])
@pytest.mark.parametrize("pre", [None, 0])
def test_int8_tiles_beyond_tile_0(ctx, pair, resident, pre):
    rng = np.random.default_rng(3)
    x, q = int8_shard(rng, 256)
    c = make_corpus(ctx, x)
    want = em.topk(em.distances(q, x, "cosine"), 10)
    assert set(want[0][0]) == {1, 2, 3, 4, 257, 258, 259, 260, 8193, 8194}
    with options(ctx, FENIX_TC_PAIR=pair, FENIX_TC_RESIDENT=resident, FENIX_TC_PRE=pre):
        got = c.search(q, "cosine", 10)
    st = c.stats()
    assert st.last_operand == 2 and bool(st.last_variant & 4) == bool(pair) and st.last_resident_queries == resident, st
    assert_topk(got, want, (pair, resident, pre))
    c.close()


# ---- range search at the radius ------------------------------------------------------------------------------------
@pytest.mark.parametrize("metric,radius_rank,opts,operand", [
    ("l2", 5, {}, 1), ("dot", 0, {}, 1), ("cosine", 5, {}, 2), ("cosine", 5, {"FENIX_INT8": 0}, 1),
    ("l2", 5, {"FENIX_FP32_FILTER_TF32": 1}, 0), ("dot", 0, {"FENIX_FP32_FILTER_TF32": 1}, 0), ("l2", None, {}, 1)])
def test_range_rows_at_the_radius(ctx, metric, radius_rank, opts, operand):
    """Dyadic rows, the bf16 construction's neighbours planted, radius = a row's exact distance: every row at the radius
    is returned, none one fp32 ulp beyond it, on each operand the range path selects (int8 and the normalised bf16
    shadow for cosine, the augmented bf16 shadow, TF32). radius_rank None: an L2 radius of 0 with exact duplicates of
    the query."""
    rng = np.random.default_rng(5)
    d, n = 256, 8192
    x, q = plant(rng, "bf16", d, n, 10, 100, False)
    q = np.concatenate([q[:2], em.dyadic(rng, (128, d), 8, -8)])
    x[5000:5003] = q[2]
    c = make_corpus(ctx, x)
    D = em.distances(q, x, metric)
    radius = 0.0 if radius_rank is None else float(np.sort(D[0])[radius_rank])
    with options(ctx, **opts):
        for r in (radius, float(np.nextafter(np.float32(radius), np.float32(np.inf)))):
            got = c.search_range(q, metric, r)
            assert c.stats().last_operand == operand, c.stats()
            assert_csr(got, em.range_csr(D, r), (metric, r, opts, counters(c)))
        if metric == "dot":
            r = float(np.sort(D[0])[20])
            assert r < 0
            assert_csr(c.search_range(q, metric, r), em.range_csr(D, r), "negative radius")
    c.close()


# ---- the magnitude ladder ------------------------------------------------------------------------------------------
LADDER = (-75, -70, -66, -64, -62, -60, -56, -30, 0, 30, 56, 58, 60, 61, 62)


@pytest.fixture(scope="module")
def ladder_data():
    rng = np.random.default_rng(2)
    n, d, nq = 8192, 256, 130
    x = em.dyadic(rng, (n, d), 10, -10)
    q = em.dyadic(rng, (nq, d), 10, -10)
    q[:20] = x[100:120] + em.dyadic(rng, (20, d), 3, -10)
    assert em.summable(11, 11, d)
    return x, q


@pytest.mark.parametrize("metric", ["l2", "cosine", "dot"])
def test_magnitude_ladder(ctx, ladder_data, metric):
    """Coordinates of magnitude up to 2^e: products cross FLT_MIN near e = -63 and vanish below e = -75; the -|x|^2/2
    terms go subnormal below e ~ -59; |x|^2 and the near-copies' q.x pass FLT_MAX at e = 61 / 62."""
    x0, q0 = ladder_data
    k, n = 10, len(x0)
    probes = np.tile(np.arange(4, dtype=np.int32), (len(q0), 1))
    log = []
    for e in LADDER:
        x, q = em.scaled(x0, e), em.scaled(q0, e)
        c = make_corpus(ctx, x)
        c.set_cells(np.arange(n) % 4)
        D = em.distances(q, x, metric)
        want = em.topk(D, k)
        runs = (("tc", {}, lambda: c.search(q, metric, k)),
                ("tf32", {"FENIX_FP32_FILTER_TF32": 1}, lambda: c.search(q, metric, k)),
                ("scan", {}, lambda: c.search(q, metric, k, knn.PREC_EXACT_SCAN)),
                ("direct", {}, lambda: c.search(q[:1], metric, k)),
                ("cells", {}, lambda: c.search_cells(q, metric, k, probes)))
        for label, opts, fn in runs:
            before = counters(c)
            with options(ctx, **opts):
                got = fn()
            st = c.stats()
            what = (e, label, f"path {st.last_path} operand {st.last_operand}", "refined/fallback",
                    np.subtract(counters(c), before))
            log.append(what)
            m = len(got[0])
            assert_topk(got, (want[0][:m], want[1][:m]), what)
        col = c.distances(q[3], metric)
        assert np.array_equal(col.view(np.uint32), D[3].view(np.uint32)), (e, "distances")
        radius = float(np.sort(D[1])[20])
        before = counters(c)
        assert_csr(c.search_range(q, metric, radius), em.range_csr(D, radius),
                   (e, "range", c.stats().last_path, np.subtract(counters(c), before)))
        c.close()
    print("\n".join(str(w) for w in log))


def test_products_beyond_flt_max_with_finite_norms(ctx):
    """Inner product, |q| ~ 2^133, rows of norm ~ 16: |x|^2 and max|x| are finite, but q.x overflows fp32 in the filter's
    products and sums. The certificate must not trust the scores, however small the bound constant makes E look."""
    rng = np.random.default_rng(9)
    d, n = 256, 8192
    x = em.dyadic(rng, (n, d), 6, -14)
    q = em.scaled(np.abs(em.dyadic(rng, (130, d), 6, -6)), 125)
    x[50, : d // 2] = 1.0                      # 16-term chunks of q.x pass +FLT_MAX, then -FLT_MAX
    x[50, d // 2:] = -0.984375
    x[51:60] = 9 / 2048                        # decoys: a little worse than row 50
    c = make_corpus(ctx, x)
    for metric in ("dot", "l2", "cosine"):
        D = em.distances(q, x, metric)
        assert_topk(c.search(q, metric, 10), em.topk(D, 10), metric)
        r = float(np.sort(D[0])[3])
        assert_csr(c.search_range(q, metric, r), em.range_csr(D, r), (metric, "range"))
    c.close()


# ---- subnormal products ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("operand", ["tf32", "bf16"])
def test_subnormal_products_stay_within_the_bound(ctx, operand):
    """Coordinates m 2^-74 (|m| < 2^8, normal floats): every product lies in [2^-148, 2^-132), below FLT_MIN. The filter
    score may lose such products, but by no more than the bound's absolute term c_abs (tc_c_abs); whether the tensor cores
    kept them exactly is printed."""
    rng = np.random.default_rng(13)
    d = 768
    x = np.abs(em.dyadic(rng, (8192, d), 8, -74))
    q = np.abs(em.dyadic(rng, (128, d), 8, -74))
    c = make_corpus(ctx, x)
    with options(ctx, **({"FENIX_DEBUG_BF16": 1} if operand == "bf16" else {})):
        s = c.debug_scores(q, "dot").astype(np.float64)
    c.close()
    exact = em.sums(q, x[:256])[2]
    c_abs = 2.0 * (d + 8) * 2.0 ** -126
    assert (np.abs(s - exact) <= c_abs).all(), np.abs(s - exact).max() / c_abs
    print(f"{operand}: subnormal products kept exactly: {bool(np.array_equal(s, exact))}")


# ---- ties across a shard boundary ----------------------------------------------------------------------------------
def test_ties_across_a_row_base_boundary(ctx):
    """Six exact copies at the k-th distance (k = 4) and at the radius, three on each side of a row_base boundary: the
    lowest global rows win the k-NN merge (fx_merge_topk) and the device group's search (two GPUs or more), and
    ShardSet.search_range returns every copy in (distance, row) order."""
    import torch

    from fenix_b200.io.shards import ShardSet

    rng = np.random.default_rng(4)
    d, n, k = 64, 10000, 4
    x = em.dyadic(rng, (n, d), 8, -8)
    q = em.dyadic(rng, (16, d), 8, -8)
    ties = [40, 4990, 4999, 5000, 5001, 9990]
    x[ties] = q[0] * 0.5
    D = em.distances(q, x, "l2")
    want = em.topk(D, k)
    assert list(want[0][0]) == ties[:k]
    shards = [make_corpus(ctx, x[:5000]), make_corpus(ctx, x[5000:], row_base=5000)]
    parts = [s.search(q, "l2", k) for s in shards]
    dev = torch.device("cuda", 0)
    g_rows = torch.from_numpy(np.stack([p[0] for p in parts])).to(dev)
    g_dist = torch.from_numpy(np.stack([p[1] for p in parts])).to(dev)
    out_rows = torch.empty((len(q), k), dtype=torch.int64, device=dev)
    out_dist = torch.empty((len(q), k), dtype=torch.float32, device=dev)
    torch.cuda.synchronize()
    ctx.merge_topk_device(g_rows.data_ptr(), g_dist.data_ptr(), 2, len(q), k, out_rows.data_ptr(), out_dist.data_ptr())
    assert_topk((out_rows.cpu().numpy(), out_dist.cpu().numpy()), want, "merge")
    radius = float(D[0, 40])
    sset = ShardSet(dim=d, n_rows=n, corpora=shards, bases=[0, 5000])
    assert_csr(sset.search_range(q, "l2", radius), em.range_csr(D, radius), "ShardSet.search_range")
    for s in shards:
        s.close()
    if torch.cuda.device_count() >= 2:
        group = knn.Group([0, 1])
        try:
            parts = [knn.Corpus(group.contexts[i], 5000, d, row_base=5000 * i) for i in range(2)]
            for i, p in enumerate(parts):
                p.append(x[5000 * i: 5000 * (i + 1)])
                p.finalize()
            assert_topk(group.search(parts, q, "l2", k), want, "group")
        finally:
            group.close()

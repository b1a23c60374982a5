"""CPU tests of the bit-exact fp64 model (tests/exact_model.py) and of the build's dependency list."""
import math
import os
import re

import numpy as np
import pytest

import exact_model as em
from oracle import brute_force_f64

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def dyadic_pair(seed, d=256, bits=12, exp=-12):
    rng = np.random.default_rng(seed)
    return em.dyadic(rng, (40, d), bits, exp), em.dyadic(rng, (500, d), bits, exp)


def test_dyadic_sums_are_order_independent():
    q, x = dyadic_pair(1, d=768, bits=20, exp=-20)
    assert em.summable(20, 20, 768) and not em.summable(24, 24, 768)
    rng = np.random.default_rng(0)
    for i, j in ((0, 0), (3, 17), (39, 499)):
        p = q[i].astype(np.float64) * x[j].astype(np.float64)
        want = float(p.sum())
        assert math.fsum(p) == want
        for _ in range(5):
            perm = rng.permutation(len(p))
            assert float(np.cumsum(p[perm])[-1]) == want
            assert float(sum(p[perm[::-1]].tolist())) == want
    assert em.exact_sums_ok(q, x)


@pytest.mark.parametrize("metric", ["l2", "cosine", "dot"])
def test_model_agrees_with_the_oracle(metric):
    q, x = dyadic_pair(2)
    rows, dist = brute_force_f64(x, q, metric, 10)
    want_rows, want_dist = em.topk(em.distances(q, x, metric), 10)
    assert np.array_equal(rows, want_rows)
    assert np.array_equal(dist.view(np.uint32), want_dist.view(np.uint32))


def test_ties_are_true_ties():
    q, x = dyadic_pair(3)
    x[[7, 70, 300]] = x[5]
    for metric in ("l2", "cosine", "dot"):
        d = em.distances(q, x, metric)
        assert d[0, 5] == d[0, 7] == d[0, 70] == d[0, 300]
        rows, dist = em.topk(d, 500)
        r = list(rows[0])
        assert r.index(5) < r.index(7) < r.index(70) < r.index(300)   # equal distances: ascending rows
        same = np.nonzero(d[0] == d[0, 5])[0]
        qq, xx, qx = em.sums(q[:1], x[same])
        assert len(set(qx[0].tolist())) == 1 and len(set(xx.tolist())) == 1   # the tie is exact, not a rounding


def test_powers_of_two_scaling():
    q, x = dyadic_pair(4, bits=10, exp=-10)
    base = {m: em.distances(q, x, m) for m in ("l2", "cosine", "dot")}
    for e in (-30, -5, 7, 30):
        qs, xs = em.scaled(q, e), em.scaled(x, e)
        assert np.array_equal(em.distances(qs, xs, "l2"), (base["l2"].astype(np.float64) * 2.0 ** e).astype(np.float32))
        assert np.array_equal(em.distances(qs, xs, "cosine"), base["cosine"])
        assert np.array_equal(em.distances(qs, xs, "dot"), (base["dot"].astype(np.float64) * 2.0 ** (2 * e)).astype(np.float32))
    # beyond the fp32 range: -|x|^2 overflows to -inf; such distances tie and are ordered by row
    xs = em.scaled(x, 62)
    d = em.distances(xs[[7, 3]], xs, "dot")
    assert np.isneginf(d[0, 7]) and np.isneginf(d[1, 3])
    rows, dist = em.topk(d, 500)
    ninf = np.nonzero(np.isneginf(d[0]))[0]
    assert np.array_equal(rows[0, :len(ninf)], ninf) and np.isneginf(dist[0, :len(ninf)]).all()
    # below the fp32 range: cosine's norms clamp to 1e-12, every distance is 0.5 - a tiny term
    d = em.distances(em.scaled(q, -75), em.scaled(x, -75), "cosine")
    assert (d == np.float32(0.5)).all()


def test_range_and_masked_expectations():
    q, x = dyadic_pair(5)
    d = em.distances(q, x, "l2")
    r = float(np.sort(d[0])[9])
    off, rows, dist = em.range_csr(d, r)
    assert off[1] - off[0] >= 10 and (dist[: off[1]] <= np.float32(r)).all()
    assert np.all(np.diff(dist[: off[1]]) >= 0)
    mask = (np.arange(len(x)) % 2).astype(np.uint8)
    off_m, rows_m, _ = em.range_csr(d, r, mask=mask)
    assert set(rows_m.tolist()) <= set(np.nonzero(mask)[0].tolist())
    rows_k, dist_k = em.topk(d[:, :5], 8)
    assert (rows_k[:, 5:] == -1).all() and np.isinf(dist_k[:, 5:]).all()
    rows_k, _ = em.topk(d, 10, mask=mask, row_base=1000)
    assert (rows_k % 2 == 1).all() and rows_k.min() >= 1000


def test_int8_tile_model():
    rng = np.random.default_rng(6)
    d = 256
    ternary = em.ternary(rng, 256, d, 64)
    spike = (np.round(rng.standard_normal((256, d)) * 64) / 64).astype(np.float32)
    spike[:, 0] = 40.0
    s, e = em.i8_tiles(np.concatenate([ternary, spike, ternary[:100]]))
    assert len(s) == 3 and e[0] < 1e-12 and e[2] < 1e-12 and e[1] > 1e-3
    assert s[1] < s[0]
    sq, aq, eq = em.i8_query(ternary[0])
    assert eq < 1e-12 and abs(aq - 1.0) < 1e-12


def test_build_lists_every_included_header():
    """Every quoted #include reachable from fenix_knn.cu is in build.DEPS, so editing any of them rebuilds the library."""
    from fenix_b200.csrc import build

    deps = {os.path.normpath(d if os.path.isabs(d) else os.path.join(build.HERE, d)) for d in build.DEPS}
    todo, seen = [os.path.join(build.HERE, s) for s in build.SOURCES], set()
    while todo:
        path = os.path.normpath(todo.pop())
        if path in seen:
            continue
        seen.add(path)
        with open(path) as f:
            for name in re.findall(r'^\s*#\s*include\s+"([^"]+)"', f.read(), re.M):
                todo.append(os.path.join(os.path.dirname(path), name))
    assert seen - deps == set()
    assert os.path.join(build.HERE, "direct_scan.cuh") in seen

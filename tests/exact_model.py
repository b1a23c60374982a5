"""Bit-exact fp64 model of the distances the library reports, for exactly summable ("dyadic") data.

Every exact path (the fp64 scan, the finish kernels' 8-lane rerank, the direct scan, the IVF cells search) sums fp64
products of fp32 coordinates, each in its own order. On data whose coordinates are m * 2^s with bounded integers m
(max|m_q| * max|m_x| * D < 2^52, and the same for the squares) every such sum is an exact integer multiple of a power of
two, so every order gives the same bits, and a numpy restatement of `finish_distance` (csrc/common.cuh) predicts each
reported distance bit for bit:

  l2      sqrt(max((qq - 2 qx) + xx, 0))
  cosine  0.5 - 0.5 * (qx / (max(sqrt(qq), 1e-12) * max(sqrt(xx), 1e-12)))
  dot     -qx

then one rounding to float32 and + 0.0. Where nvcc may contract to an FMA the product is by a power of two (2 qx,
0.5 t), exact in fp64, so the FMA and the separate operations round alike.

The module also models the int8 shadow's format per 256-row tile (to_i8_tiled_kernel): the tile's scale S_t, its
residual bound E_t and every row's residual, so that constructions can be checked on the CPU before they run.
"""
from __future__ import annotations

import math

import numpy as np

METRIC = {"l2": 0, "euclidean": 0, "cosine": 1, "dot": 2, "inner_product": 2}
TILE = 256          # corpus rows per filter tile (TC_BN) and per int8 scale
F32_MAX = float(np.finfo(np.float32).max)


# ---- dyadic data --------------------------------------------------------------------------------------------------
def dyadic(rng, shape, bits, exp=0):
    """float32 array m * 2^exp with integers |m| < 2^bits (bits <= 24: exact in float32 at any normal scale)."""
    assert 1 <= bits <= 24
    m = rng.integers(-(2 ** bits - 1), 2 ** bits, size=shape)
    return from_ints(m, exp)


def from_ints(m, exp=0):
    """float32(m * 2^exp), asserting that the conversion is exact."""
    v = np.ldexp(np.asarray(m, dtype=np.float64), exp)
    x = v.astype(np.float32)
    assert np.array_equal(x.astype(np.float64), v), "not representable in float32"
    return x


def ternary(rng, n, dim, nnz):
    """n rows with exactly nnz coordinates +-1 and zeros elsewhere: one norm, so a tile of them sits on the int8 grid
    (E_t ~ 0)."""
    x = np.zeros((n, dim), np.float32)
    for r in range(n):
        x[r, rng.choice(dim, nnz, replace=False)] = rng.choice((-1.0, 1.0), nnz)
    return x


def summable(q_bits, x_bits, dim):
    """True when every fp64 sum of D products of such coordinates (q.x, q.q, x.x) is exact in any order."""
    b = max(q_bits, x_bits)
    return (2 ** (q_bits + x_bits)) * dim < 2 ** 52 and (2 ** (2 * b)) * dim < 2 ** 52


def scaled(x, e):
    """x * 2^e, exactly (asserts that no coordinate leaves float32's range or loses bits)."""
    v = np.ldexp(np.asarray(x, dtype=np.float64), e)
    y = v.astype(np.float32)
    assert np.array_equal(y.astype(np.float64), v), f"2^{e} scaling is not exact in float32"
    return y


# ---- the exact sums and finish_distance ----------------------------------------------------------------------------
def sums(queries, corpus):
    """(qq[Q], xx[N], qx[Q, N]) in fp64. On dyadic data these are exact, whatever the summation order."""
    q = np.atleast_2d(np.asarray(queries, dtype=np.float64))
    x = np.asarray(corpus, dtype=np.float64)
    return (q * q).sum(1), (x * x).sum(1), q @ x.T


def finish_distance(metric, qq, xx, qx):
    """numpy float64 restatement of fx::finish_distance: the same operations in the same order, one rounding to fp32."""
    m = METRIC[metric] if isinstance(metric, str) else metric
    qq, xx, qx = (np.asarray(v, dtype=np.float64) for v in (qq, xx, qx))
    with np.errstate(over="ignore", invalid="ignore"):
        if m == 0:
            d2 = (qq - 2.0 * qx) + xx
            d = np.sqrt(np.where(d2 > 0.0, d2, 0.0))
        elif m == 1:
            nq = np.maximum(np.sqrt(qq), 1e-12)
            nx = np.maximum(np.sqrt(xx), 1e-12)
            d = 0.5 - 0.5 * (qx / (nq * nx))
        else:
            d = -qx
        return d.astype(np.float32) + np.float32(0.0)


def distances(queries, corpus, metric):
    """float32 distance matrix [Q, N], bit for bit what every exact path reports (dyadic data)."""
    qq, xx, qx = sums(queries, corpus)
    return finish_distance(metric, qq[:, None], xx[None, :], qx)


def exact_sums_ok(queries, corpus):
    """Checks on the CPU that the data are summable: shuffled-order and math.fsum sums equal the numpy ones bit for
    bit on a sample of pairs (used by the model's own tests)."""
    q = np.atleast_2d(np.asarray(queries, dtype=np.float64))
    x = np.asarray(corpus, dtype=np.float64)
    rng = np.random.default_rng(0)
    for i, j in zip(rng.integers(0, len(q), 8), rng.integers(0, len(x), 8)):
        p = q[i] * x[j]
        want = float(p.sum())
        if math.fsum(p) != want:
            return False
        for _ in range(3):
            if float(np.add.reduce(p[rng.permutation(len(p))])) != want:
                return False
    return True


# ---- expected results ----------------------------------------------------------------------------------------------
def topk(dist, k, mask=None, row_base=0):
    """(rows[Q, k], dist[Q, k]) by (distance, row), padded with (-1, +inf); masked rows (mask == 0) excluded."""
    dist = np.atleast_2d(dist)
    n_q, n = dist.shape
    live = np.arange(n) if mask is None else np.nonzero(np.asarray(mask).astype(bool))[0]
    rows = np.full((n_q, k), -1, np.int64)
    out = np.full((n_q, k), np.inf, np.float32)
    for i in range(n_q):
        d = dist[i, live]
        order = live[np.lexsort((live, d))][:k]
        rows[i, :len(order)] = order + row_base
        out[i, :len(order)] = dist[i, order]
    return rows, out


def range_csr(dist, radius, mask=None, row_base=0):
    """(offsets[Q + 1], rows, dist) of every row with distance <= float32(radius), each query's hits by (distance,
    row): the layout of Corpus.search_range."""
    r32 = np.float32(radius)
    offsets, rows, out = [0], [], []
    for d in np.atleast_2d(dist):
        ok = d <= r32
        if mask is not None:
            ok &= np.asarray(mask).astype(bool)
        r = np.nonzero(ok)[0]
        r = r[np.lexsort((r, d[r]))]
        rows.append(r + row_base)
        out.append(d[r])
        offsets.append(offsets[-1] + len(r))
    return (np.array(offsets, np.int64), np.concatenate(rows).astype(np.int64),
            np.concatenate(out).astype(np.float32))


# ---- the int8 shadow's format (to_i8_tiled_kernel / knn_qprep_i8_kernel) -------------------------------------------
def unit_rows(v):
    """x^ = x * (1 / max(|x|, 1e-12)): the kernels multiply by the fp64 inverse norm."""
    v = np.atleast_2d(np.asarray(v, dtype=np.float64))
    inv = 1.0 / np.maximum(np.sqrt((v * v).sum(1)), 1e-12)
    return v * inv[:, None]


def i8_group(v):
    """The int8 format of a group of rows (one corpus tile, or one query): (x^, S, x~, residual norms)."""
    h = unit_rows(v)
    m = np.abs(h).max()
    s = np.float32(127.0 / m) if m > 0 else np.float32(1.0)
    t = np.clip(np.rint(h * np.float64(s)), -127, 127)
    return h, s, t, np.sqrt(((h - t * (1.0 / np.float64(s))) ** 2).sum(1))


def i8_tiles(corpus):
    """Per 256-row tile: S_t (float32) and E_t (the largest residual norm, fp64; the kernel rounds it up to fp32)."""
    n = len(corpus)
    st, et = [], []
    for lo in range(0, n, TILE):
        _, s, _, r = i8_group(corpus[lo: lo + TILE])
        st.append(s)
        et.append(r.max())
    return np.array(st, np.float32), np.array(et)


def i8_query(q):
    """(S_q, a_q = |q~| / S_q, e_q = |q^ - q~/S_q|) of one query."""
    _, s, t, r = i8_group(q)
    return s, float(np.linalg.norm(t[0]) / np.float64(s)), float(r[0])


# ---- filter error bounds (tc_filter.cuh: tc_c_err, tc_c_add) ---------------------------------------------------------
def c_err(dim, kind):
    """|filter - exact| <= c |q| |x| for the TF32 (kind 0) and bf16 (kind 1) operands."""
    prod = 1.25 * 2.0 ** -9 if kind == 0 else 1.10 * 2.0 ** -7
    return prod + dim * 2.0 ** -21

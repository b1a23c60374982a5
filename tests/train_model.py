"""numpy restatement of one mini-batch k-means step of IVF codebook training (fx_train_codebooks, io.coder.make).

Assignment: every sample row takes the codeword with the smallest fp32 distance, ties to the lowest codeword. The sums
qq, xx and qx are fp64 sums of fp32 products in ascending coordinate order, as the kernel forms them; each product of
two fp32 values is exact in fp64, so the sums here have the kernel's bits on any data, and `exact_model.finish_distance`
turns them into the distance.
Update: fp64 sum of the old codeword, then its rows in sample order (np.add.at adds in index order), one fp64 division
by 1 + count, one rounding to fp32. Cosine normalises the old codeword and the rows first and the mean after, in fp64.
"""
from __future__ import annotations

import numpy as np

from exact_model import finish_distance


def seq_sums(a, b, fast=False):
    """(aa[R], bb[K], ab[R, K]): fp64 sums over the coordinates in ascending order (`fast`: numpy's own order, which
    can differ in the last bits, for checks with a tolerance)."""
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    if fast:
        return (a * a).sum(1), (b * b).sum(1), a @ b.T
    aa, bb, ab = np.zeros(len(a)), np.zeros(len(b)), np.zeros((len(a), len(b)))
    for d in range(a.shape[1]):
        aa += a[:, d] * a[:, d]
        bb += b[:, d] * b[:, d]
        ab += a[:, d, None] * b[None, :, d]
    return aa, bb, ab


def assign(rows, book, metric, fast=False):
    """(nearest codeword[R], squared row norms[R])."""
    xx, cc, xc = seq_sums(rows, book, fast)
    dist = finish_distance(metric, xx[:, None], cc[None, :], xc)
    return np.argmin(dist, axis=1), xx


def _unit(v, nn):
    return v / np.maximum(np.sqrt(nn), 1e-12)[:, None]


def step(books, rows_of, positions, batch, metric, fast=False):
    """One step for every codebook: `rows_of(pos)` gives the fp32 rows at global positions. Returns new books and the
    assignments [n, batch]."""
    books = np.array(books, np.float32)
    cosine = metric == "cosine"
    nearest = []
    for j in range(books.shape[0]):
        x = rows_of(positions[j * batch: (j + 1) * batch])
        a, xx = assign(x, books[j], metric, fast)
        nearest.append(a)
        c = books[j].astype(np.float64)
        v = x.astype(np.float64)
        if cosine:
            c = _unit(c, (c * c).sum(1))
            v = _unit(v, xx)
        total = c.copy()
        np.add.at(total, a, v)
        count = np.ones(len(c))
        np.add.at(count, a, 1.0)
        m = total / count[:, None]
        if cosine:
            m = _unit(m, (m * m).sum(1))
        books[j] = m.astype(np.float32)
    return books, np.stack(nearest)


def epoch(books, rows_of, positions, batch, metric, fast=False):
    """Every step of one call: positions [n_steps, n * batch]."""
    for s in range(len(positions)):
        books, _ = step(books, rows_of, positions[s], batch, metric, fast)
    return books


def epoch_positions(rng, n_rows, n_books, batch):
    """The per-step sorted positions `coder.make` draws for one epoch (remainder dropped)."""
    step_rows = n_books * batch
    perm = rng.permutation(n_rows)
    steps = n_rows // step_rows
    return np.sort(perm[: steps * step_rows].reshape(steps, step_rows), axis=1)

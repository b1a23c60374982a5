"""Metric arithmetic seam `distance(u, v, metric)` and the IVF codebooks (`Config`, `make`, `load`, `call`).

Mirrors fenix.io.coder (src/fenix/io/coder/coder.py): same metric names and conventions (Euclidean
distance WITH sqrt; 0.5 - 0.5*cos with eps 1e-12; negated dot; ValueError on an unknown name), same
on-disk codebook format (`<root>/codings/<name>.torch`, a torch-pickled dict {tensor (n, k, D), column type,
config}), same composite-code convention: a vector's code is the rank of its (codeword_0, .., codeword_{n-1})
combination in the k^n product space, codebook 0 most significant (coder.py:171-181).

Where the arithmetic runs: every vector-to-codeword distance (`distance`, the probe ranking of `call`, the code
assignment behind `io.index.make`) is computed by libfenix_knn on the device against a small resident shard
holding the codewords; the host only adds n distances per composite code and ranks k^n sums (coder.py:171-186).
Codebook TRAINING (`make`, coder.py:93-127: mini-batch k-means) runs on the device too: the host draws the seeds and
the per-epoch permutations, and every epoch is one `fx_train_codebooks` call over the column's resident shards.
"""
from __future__ import annotations

import os
import threading
from typing import Iterator, Optional, Sequence, TypedDict

import numpy as np
import pyarrow as pa

from .. import knn
from . import shards as _shards

LOCATION: str = "codings"


def distance(u, v, metric: str):
    """Distances between every row of `u` (U x D) and every row of `v` (V x D) -> (U x V).

    Accepts numpy arrays or CPU torch tensors and returns the same kind."""
    code = knn.metric_code(metric)
    as_tensor = type(u).__module__.startswith("torch")
    un = np.ascontiguousarray(u.detach().cpu().numpy() if as_tensor else np.asarray(u), dtype=np.float32)
    vn = v.detach().cpu().numpy() if type(v).__module__.startswith("torch") else np.asarray(v)
    vn = np.ascontiguousarray(vn, dtype=np.float32)
    if un.ndim != 2 or vn.ndim != 2 or un.shape[1] != vn.shape[1]:
        raise ValueError(f"distance expects (U,D) and (V,D), got {un.shape} and {vn.shape}")
    corpus = knn.Corpus(_shards.context(_shards.devices()[0]), vn.shape[0], vn.shape[1])
    try:
        corpus.append(vn)
        corpus.finalize()
        out = np.stack([corpus.distances(row, code) for row in un]) if len(un) else np.empty((0, vn.shape[0]), np.float32)
    finally:
        corpus.close()
    if as_tensor:
        import torch

        return torch.from_numpy(out)
    return out


class Config(TypedDict):
    metric: str
    codebook_size: int
    num_codebooks: int
    batch_size: int
    num_epochs: int


class Coding(TypedDict):
    tensor: np.ndarray      # (num_codebooks, codebook_size, D) float32
    column: pa.DataType
    config: Config


_codings: dict[tuple, tuple] = {}     # (root, name) -> (file signature, Coding, device shards of the codebooks)
_codings_lock = threading.Lock()
_codings_gates: dict[tuple, threading.Lock] = {}   # one build per key at a time


def path_of(root: str, name: str) -> str:
    return os.path.join(root, LOCATION, name + ".torch")


def _read(path: str) -> Coding:
    import torch

    with open(path, "rb") as f:
        raw = torch.load(f, map_location="cpu", weights_only=False)   # the reference's own format (coder.py:73-74)
    tensor = raw["tensor"]
    tensor = tensor.detach().cpu().numpy() if hasattr(tensor, "detach") else np.asarray(tensor)
    return {"tensor": np.ascontiguousarray(tensor, dtype=np.float32), "column": raw["column"], "config": dict(raw["config"])}


def load(root: str, name: str) -> Coding:
    """Codebook `name` (coder.py:68-90), cached per file version together with its device shards."""
    return _entry(root, name)[1]


def _entry(root: str, name: str) -> tuple:
    path = path_of(root, name)
    st = os.stat(path)
    sig = (st.st_mtime_ns, st.st_size)
    key = (os.path.abspath(root), name)
    with _codings_lock:
        hit = _codings.get(key)
        if hit is not None and hit[0] == sig:
            return hit
        gate = _codings_gates.setdefault(key, threading.Lock())
    with gate:   # single-flight: concurrent first uses of a coding share one build
        with _codings_lock:
            hit = _codings.get(key)
            if hit is not None and hit[0] == sig:
                return hit
        coding = _read(path)
        books = [_book_shard(coding["tensor"][j]) for j in range(coding["tensor"].shape[0])]
        with _codings_lock:
            # a replaced entry is only dropped, never closed here: threads still ranking codes against its books hold
            # references, and the device shards are freed when the last one lets go (Corpus.__del__)
            _codings[key] = fresh = (sig, coding, books)
    return fresh


def forget(root: Optional[str] = None, name: Optional[str] = None) -> None:
    """Drop cached codings (and with them the device shards of their codebooks): all, those under `root`, or one."""
    root = os.path.abspath(root) if root is not None else None
    with _codings_lock:
        for key in [k for k in _codings if (root is None or k[0] == root) and (name is None or k[1] == name)]:
            _codings.pop(key)


def _book_shard(codewords: np.ndarray) -> knn.Corpus:
    corpus = knn.Corpus(_shards.context(_shards.devices()[0]), codewords.shape[0], codewords.shape[1])
    corpus.append(np.ascontiguousarray(codewords, dtype=np.float32))
    corpus.finalize()
    return corpus


def _codeword_distances(books: Sequence[knn.Corpus], vectors: np.ndarray, metric: str) -> np.ndarray:
    """(T, n, k) distances of every vector to every codeword, computed on the device (one resident shard per
    codebook; the distance-column kernel gives the reference-convention distance of a query to every row)."""
    code = knn.metric_code(metric)
    return np.stack([np.stack([b.distances(v, code) for b in books]) for v in vectors])


def composite_sums(d: np.ndarray) -> np.ndarray:
    """(T, n, k) codeword distances -> (T, k^n) summed distance of every composite code, codebook 0 most
    significant (coder.py:171-181), accumulated in float32 in codebook order like the reference."""
    t, n, k = d.shape
    out = np.zeros((t, 1), dtype=np.float32)
    for j in range(n):
        out = (out[:, :, None] + d[:, j, None, :].astype(np.float32)).reshape(t, -1)
    return out


def call(target, coding, maxval: Optional[int] = None):
    """Composite codes of `target` ranked by summed codeword distance, best first (coder.py:143-194):
    all k^n of them, or the `maxval` best. Accepts what the reference accepts (ndarray / Tensor / Arrow array /
    Table) and answers in kind (ndarray / Tensor / ListArray<int64>)."""
    as_tensor = type(target).__module__.startswith("torch")
    as_numpy = isinstance(target, np.ndarray)
    if isinstance(coding, tuple):
        _sig, coding, books = _entry(*coding)
        owned = False
    else:
        books = [_book_shard(np.asarray(coding["tensor"][j])) for j in range(len(coding["tensor"]))]
        owned = True
    try:
        metric = coding["config"]["metric"]
        if isinstance(target, pa.Table):
            target = target.column(coding["column"]).combine_chunks()   # as coder.py:161 (the stored column TYPE keys the lookup there too)
        if isinstance(target, pa.ChunkedArray):
            target = target.combine_chunks()
        if isinstance(target, pa.Array):
            target = _shards.chunk_rows(target)
        if as_tensor:
            target = target.detach().cpu().numpy()
        vectors = np.ascontiguousarray(np.atleast_2d(np.asarray(target)), dtype=np.float32)
        sums = composite_sums(_codeword_distances(books, vectors, metric))
        if maxval is not None:
            part = np.argpartition(sums, min(maxval, sums.shape[1]) - 1, axis=1)[:, :maxval]
            order = np.take_along_axis(part, np.argsort(np.take_along_axis(sums, part, axis=1), axis=1, kind="stable"), axis=1)
        else:
            order = np.argsort(sums, axis=1, kind="stable")
        order = order.astype(np.int64)
    finally:
        if owned:
            for b in books:
                b.close()
    if as_tensor:
        import torch

        return torch.from_numpy(order)
    if as_numpy:
        return order
    return pa.array(iter(order), type=pa.list_(pa.int64()))


def assign(root: str, name: str, vectors: np.ndarray) -> np.ndarray:
    """Composite code of every row of `vectors` (the `call(x, coding, 1)[0]` of index.py:49-51): the nearest
    codeword per codebook is one k = 1 search of the rows against that codebook's resident shard."""
    _sig, coding, books = _entry(root, name)
    k = int(coding["config"]["codebook_size"])
    code = np.zeros(len(vectors), dtype=np.int64)
    if len(vectors) == 0:
        return code
    q = np.ascontiguousarray(vectors, dtype=np.float32)
    for b in books:
        rows, _dist = b.search(q, coding["config"]["metric"], 1)
        code = code * k + rows[:, 0]
    return code


def _seed_rows(column: pa.ChunkedArray, sel: np.ndarray) -> np.ndarray:
    """Rows at the ascending global positions `sel` of a vector column, read from its chunks."""
    bounds = np.cumsum([0] + [len(c) for c in column.chunks])
    which = np.searchsorted(bounds, sel, side="right") - 1
    out = np.empty((len(sel), column.type.list_size), dtype=np.float32)
    for w in np.unique(which):
        hit = which == w
        out[hit] = _shards.chunk_rows(column.chunks[w])[sel[hit] - bounds[w]]
    return out


def make(root: str, name: str, source, column: str, config: Config, rng: Optional[np.random.Generator] = None) -> Coding:
    """Train codebook `name` on `column` of `source` (coder.py:93-127): n codebooks of k codewords seeded with
    random rows, then `num_epochs` passes of mini-batch k-means in which every codeword moves to the mean of itself
    and the batch vectors assigned to it (coder.py:53-65, `index_reduce(.., "mean")` counts the old codeword).

    The host draws the seeds and every epoch's permutation from `rng` (default: unseeded, like the reference's); the
    epochs run on the device against the column's resident shards (`knn.train_codebooks`, one call per epoch)."""
    import torch

    knn.metric_code(config["metric"])
    data = _shards.load_table(root, source)
    n, k, bs = int(config["num_codebooks"]), int(config["codebook_size"]), int(config["batch_size"])
    total = data.num_rows
    if total < n * k:
        raise ValueError(f"{total} rows cannot seed {n} codebooks of {k} codewords")
    rng = np.random.default_rng() if rng is None else rng
    vectors = data.column(column)
    books = _seed_rows(vectors, np.sort(rng.permutation(total)[: n * k])).reshape(n, k, -1)
    step = n * bs
    with _shards.get(root, source, column, data) as shard:
        for _ in range(int(config["num_epochs"])):
            perm = rng.permutation(total)
            steps = total // step
            positions = np.sort(perm[: steps * step].reshape(steps, step), axis=1)
            books = knn.train_codebooks(shard.corpora, config["metric"], books, bs, positions)
    path = path_of(root, name)
    os.makedirs(os.path.dirname(path), exist_ok=True)
    with open(path, "wb") as f:
        torch.save({"tensor": torch.from_numpy(np.ascontiguousarray(books)), "column": vectors.type,
                    "config": dict(config)}, f)
    return load(root, name)


def list(root: str) -> Iterator[str]:
    base = os.path.join(root, LOCATION)
    for dirpath, _dirs, files in os.walk(base):
        for f in sorted(files):
            if f.endswith(".torch"):
                yield os.path.relpath(os.path.join(dirpath, f), base).removesuffix(".torch")


def drop(root: str, name: str) -> None:
    path = path_of(root, name)
    if os.path.exists(path):
        os.unlink(path)
    forget(root, name)

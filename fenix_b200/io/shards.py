"""Device-resident corpus shards: the Arrow -> pinned host -> HBM handoff.

Replaces fenix.io.torch.from_arrow (src/fenix/io/torch/torch.py:6-10), which re-wraps the
mmap'd values buffer of every chunk on every query, with a copy made ONCE per table version:
each record batch's FixedSizeList values buffer is handed (zero-copy numpy view) to
fx_corpus_append, which stages it through a pinned ring and DMAs it into the shard.
The cache is keyed on (root, sources, column) and validated against (mtime_ns, size) of the
backing files, so do_put / drop-table / remove invalidate it (SURVEY.md §5, §8f rank 2).
"""
from __future__ import annotations

import functools
import os
import threading
from dataclasses import dataclass, field
from typing import Optional, Sequence

import numpy as np
import pyarrow as pa

from .. import knn
from . import table as _table

_lock = threading.Lock()
_contexts: dict[int, knn.Context] = {}
_groups: dict[tuple, knn.Group] = {}
_cache: dict[tuple, "ShardSet"] = {}
_building: dict[tuple, threading.Lock] = {}   # one upload per key at a time (single-flight)


def devices() -> list[int]:
    """CUDA devices the in-process server shards over (FENIX_DEVICES="0,1,..."; default "0")."""
    spec = os.environ.get("FENIX_DEVICES", "0")
    return [int(tok) for tok in spec.split(",") if tok.strip() != ""]


def context(device: int) -> knn.Context:
    with _lock:
        ctx = _contexts.get(device)
        if ctx is None:
            ctx = _contexts[device] = knn.Context(device)
        return ctx


def group(device_ids: Sequence[int]) -> knn.Group:
    """The process-wide device group for this device list (fx_group_create: contexts + NCCL communicators + a worker
    thread per device inside the library). One per distinct list; lives as long as the process."""
    key = tuple(int(d) for d in device_ids)
    with _lock:
        g = _groups.get(key)
        if g is None:
            g = _groups[key] = knn.Group(list(key))
        return g


def chunk_rows(chunk: pa.FixedSizeListArray) -> np.ndarray:
    """Zero-copy (rows, D) float32 view of one chunk's values buffer.

    Unlike torch.py:8-10 (`.values`, which ignores a slice offset) the chunk's offset is
    honoured; validity bitmaps are ignored exactly as the reference does.
    """
    typ = chunk.type
    if not pa.types.is_fixed_size_list(typ):
        raise TypeError(f"vector column must be FixedSizeList<float32>[D], got {typ}")
    d = typ.list_size
    vals = chunk.values.to_numpy(zero_copy_only=True)
    lo = chunk.offset * d
    rows = vals[lo: lo + len(chunk) * d].reshape(len(chunk), d)
    if typ.value_type == pa.float32():
        return rows
    if typ.value_type in (pa.float16(), pa.float64()):
        # shards are float32 (north_star); other float widths are converted once, at upload. The reference computes
        # in the column's own type (index.py:133-159), so float64 columns agree to float32 rounding, not bit for bit.
        return rows.astype(np.float32)
    raise NotImplementedError(f"embedding columns must be float16 / float32 / float64 (got {typ.value_type})")


@dataclass
class ShardSet:
    """Row-sharded device copy of one vector column (one Corpus per device).

    Lifetime: request threads LEASE a set for the duration of a search (`with shard.lease():`); `retire()` - called when
    the table changes or the cache drops the entry - closes it at once when idle, otherwise when the last lease is
    returned. A set is never closed under a running search (the C library additionally validates every corpus handle,
    include/fenix_knn.h fx_corpus_destroy)."""

    dim: int
    n_rows: int
    corpora: list[knn.Corpus] = field(default_factory=list)
    bases: list[int] = field(default_factory=list)
    signature: tuple = ()
    group: Optional[knn.Group] = None      # >= 2 devices: the in-library device group that runs the exchange
    _users: int = 0
    _retired: bool = False
    _guard: threading.Lock = field(default_factory=threading.Lock)
    # batched IVF: the coding whose cells the (single) corpus currently holds as its inverted index + the sorted composite
    # codes behind the dense cell numbers; `_cells_lock` spans "install the cells, then search them" (io/index.py)
    _cells: Optional[tuple] = None
    _cells_lock: threading.Lock = field(default_factory=threading.Lock)

    # ---- leases ----
    def lease(self) -> "ShardSet":
        with self._guard:
            if self._retired and not self.corpora:
                raise RuntimeError("shard set is closed")
            self._users += 1
        return self

    def release(self) -> None:
        with self._guard:
            self._users -= 1
            close_now = self._retired and self._users == 0
        if close_now:
            self._close()

    def __enter__(self) -> "ShardSet":
        return self

    def __exit__(self, *exc) -> None:
        self.release()

    def retire(self) -> None:
        """No new searches; free the device memory as soon as the running ones are done."""
        with self._guard:
            self._retired = True
            close_now = self._users == 0
        if close_now:
            self._close()

    def close(self) -> None:
        self.retire()

    def _close(self) -> None:
        for c in self.corpora:
            c.close()
        self.corpora = []

    # ---- search ----
    def search(self, queries: np.ndarray, metric: str, k: int, precision: int = knn.PREC_FP32,
               row_mask: Optional[np.ndarray] = None) -> tuple[np.ndarray, np.ndarray]:
        if len(self.corpora) == 1:
            return self.corpora[0].search(queries, metric, k, precision, row_mask)
        # one process, several devices: fx_group_search - every device searches its shard concurrently (worker threads
        # inside the library), the k x W candidates are all-gathered over NVLink and merged on the device
        return self.group.search(self.corpora, queries, metric, k, precision, row_mask)

    def search_range(self, queries: np.ndarray, metric: str, radius: float, precision: int = knn.PREC_FP32,
                     row_mask: Optional[np.ndarray] = None) -> tuple[np.ndarray, np.ndarray, np.ndarray]:
        """Every row within `radius` of each query: (offsets[Q + 1], rows, dist) in CSR form, each query's hits ordered
        by (distance, row). Several devices: each shard in turn (as `distances`), the lists merged on the host."""
        if len(self.corpora) == 1:
            return self.corpora[0].search_range(queries, metric, radius, precision, row_mask)
        n_q = np.atleast_2d(np.asarray(queries)).shape[0]
        qids, rows, dists = [], [], []
        for c, base in zip(self.corpora, self.bases):
            part_mask = None if row_mask is None else row_mask[base: base + c.n_rows]
            off, r, d = c.search_range(queries, metric, radius, precision, part_mask)
            qids.append(np.repeat(np.arange(n_q, dtype=np.int64), np.diff(off)))
            rows.append(r)
            dists.append(d)
        qid, row, dist = np.concatenate(qids), np.concatenate(rows), np.concatenate(dists)
        order = np.lexsort((row, dist, qid))
        offsets = np.zeros(n_q + 1, dtype=np.int64)
        np.cumsum(np.bincount(qid, minlength=n_q), out=offsets[1:])
        return offsets, row[order], dist[order]

    def distances(self, query: np.ndarray, metric: str) -> np.ndarray:
        parts = [c.distances(query, metric) for c in self.corpora]
        return parts[0] if len(parts) == 1 else np.concatenate(parts)


def from_chunks(column: pa.ChunkedArray, device_ids: Optional[Sequence[int]] = None) -> ShardSet:
    """Upload a FixedSizeList<float32>[D] column, row-sharded contiguously over the devices."""
    typ = column.type
    if not pa.types.is_fixed_size_list(typ):
        raise TypeError(f"vector column must be FixedSizeList<float32>[D], got {typ}")
    if typ.value_type not in (pa.float16(), pa.float32(), pa.float64()):
        raise NotImplementedError(f"embedding columns must be float16 / float32 / float64 (got {typ.value_type})")
    dim, n = typ.list_size, len(column)
    devs = list(device_ids) if device_ids is not None else devices()
    world = max(1, len(devs))
    per = -(-n // world) if n else 0
    shard = ShardSet(dim=dim, n_rows=n)
    ctxs = [context(devs[0])] if world == 1 else None
    if world > 1:
        shard.group = group(devs)
        ctxs = shard.group.contexts
    for r in range(world):
        lo, hi = min(n, r * per), min(n, (r + 1) * per)      # trailing shards of a tiny table are empty
        shard.bases.append(lo)
        shard.corpora.append(knn.Corpus(ctxs[r], max(hi - lo, 0), dim, row_base=lo))
    pos = 0
    for chunk in column.chunks:
        rows = chunk_rows(chunk)
        done = 0
        while done < len(rows):
            r = min(pos // per, world - 1) if per else 0
            room = shard.bases[r] + shard.corpora[r].capacity - pos
            take = min(room, len(rows) - done)
            shard.corpora[r].append(rows[done: done + take])
            done += take
            pos += take
    for c in shard.corpora:
        c.finalize()
    return shard


@functools.lru_cache(maxsize=256)
def _abs(root: str) -> str:
    return os.path.abspath(root)


@functools.lru_cache(maxsize=1024)
def _path(root: str, name: str) -> str:
    return _table.path_of(root, name)


def _signature(root: str, names: Sequence[str]) -> tuple:
    """Version of the backing files: (name, mtime, size) each - one stat per file and request."""
    sig = []
    for n in names:
        st = os.stat(_path(root, n))
        sig.append((n, st.st_mtime_ns, st.st_size))
    return tuple(sig)


_tables: dict[tuple, tuple] = {}


def load_table(root: str, source: str | Sequence[str], with_signature: bool = False):
    """`io.table.load` with the parsed (memory-mapped, zero-copy) Table cached per file version: the
    reference re-maps and re-parses the IPC stream on every search (index.py:93-97, ~3.5 % of its query
    time at 100 chunks, more with many chunks)."""
    names = (source,) if isinstance(source, str) else tuple(source)
    key = (_abs(root), names)
    sig = _signature(root, names)
    with _lock:
        hit = _tables.get(key)
    if hit is None or hit[0] != sig:
        table = _table.load(root, source)
        with _lock:
            _tables[key] = (sig, table)
    else:
        table = hit[1]
    return (table, sig) if with_signature else table


def get(root: str, source: str | Sequence[str], column: str, table: pa.Table, signature: Optional[tuple] = None) -> ShardSet:
    """LEASED shard set for `column` of the named table(s): `with shards.get(...) as shard:` (or release() it). Uploads
    on first use - one upload per key however many request threads miss at once (single-flight); a set replaced by a
    newer table version is retired, not closed under the searches still running on it."""
    names = (source,) if isinstance(source, str) else tuple(source)
    key = (_abs(root), names, column, tuple(devices()))
    sig = _signature(root, names) if signature is None else signature   # (`signature`: the one load_table just took)
    with _lock:
        hit = _cache.get(key)
        if hit is not None and hit.signature == sig:
            return hit.lease()
        gate = _building.setdefault(key, threading.Lock())
    with gate:
        with _lock:   # somebody else may have finished the upload while this thread waited at the gate
            hit = _cache.get(key)
            if hit is not None and hit.signature == sig:
                return hit.lease()
        fresh = from_chunks(table.column(column))
        fresh.signature = sig
        with _lock:
            old = _cache.get(key)
            _cache[key] = fresh
            leased = fresh.lease()
    if old is not None:
        old.retire()
    return leased


def warm(root: str, spec: Optional[str] = None) -> list[str]:
    """Upload shards ahead of the first search: `spec` (default: $FENIX_WARM) = "table:column,table2:column2,...".
    A table without ":column" warms every FixedSizeList<float> column. Returns what was uploaded. Called by the server
    at start-up and after every do_put (SURVEY.md section 5 / 8f rank 2)."""
    spec = os.environ.get("FENIX_WARM", "") if spec is None else spec
    done = []
    for item in [tok.strip() for tok in spec.split(",") if tok.strip()]:
        name, _, column = item.partition(":")
        try:
            table = load_table(root, name)
        except (FileNotFoundError, OSError):
            continue
        columns = [column] if column else vector_columns(table)
        for col in columns:
            get(root, name, col, table).release()
            done.append(f"{name}:{col}")
    return done


def vector_columns(table: pa.Table) -> list[str]:
    return [f.name for f in table.schema
            if pa.types.is_fixed_size_list(f.type) and f.type.value_type in (pa.float16(), pa.float32(), pa.float64())]


def invalidate(root: Optional[str] = None, name: Optional[str] = None) -> None:
    """Drop cached shards (all, those under `root`, or those that include table `name`)."""
    root = os.path.abspath(root) if root is not None else None
    with _lock:
        doomed = [k for k in _cache if (root is None or k[0] == root) and (name is None or name in k[1])]
        victims = [_cache.pop(k) for k in doomed]
        for k in [k for k in _tables if (root is None or k[0] == root) and (name is None or name in k[1])]:
            _tables.pop(k)
    for v in victims:
        v.retire()

"""Search orchestration: the drop-in seam `io.index.call`, plus the IVF sidecars (`make`, `load`, `list`, `drop`).

Mirrors fenix.io.index.call (src/fenix/io/index/index.py:81-170): same arguments, same result schema (select columns + `__DISTANCE__` typed as the
column's value type), same `maxval` edge cases (None or >= row count returns every row in
table order with the distance attached, index.py:165), same filter-before-distance semantics
(index.py:161). What changes is where the arithmetic runs: the per-chunk Arrow UDF ->
torch.cdist -> select_k_unstable chain (index.py:133-168) is replaced by one call into
libfenix_knn against a device-resident shard set; only the k winning rows are gathered on the
host. Result rows are ordered by (distance, row position) - the reference's order among equal
distances is unspecified ("unstable").

The IVF branch (`coding` + `probes`, index.py:113-126) is the same search with one more predicate: the rows
whose `__CODED_ID__` (sidecar written by `make`, index.py:38-66) is among the query's `probes` best composite
codes. The codes are ranked by `io.coder.call` (codeword distances on the device), the predicate becomes the row
mask of the masked exact search - no filtered copy of the corpus is made, unlike index.py:161.
"""
from __future__ import annotations

from typing import Sequence

import numpy as np
import pyarrow as pa
import pyarrow.compute as pc

import os

from .. import knn
from . import arrow as _arrow
from . import coder as _coder
from . import shards as _shards
from . import table as _table
from .batcher import MicroBatcher

_batcher = MicroBatcher()

CODE_COL: str = "__CODED_ID__"
DIST_COL: str = "__DISTANCE__"
QUERY_COL: str = "__QUERY__"
LOCATION: str = "indexes"


def _distance_array(dist: np.ndarray, value_type: pa.DataType) -> pa.Array:
    """`__DISTANCE__` is typed like the column's values (index.py:153)."""
    if value_type == pa.float16():
        return pa.array(dist.astype(np.float16), type=value_type)
    return pa.array(dist, type=value_type)


_bounds_cache: dict[int, tuple] = {}   # id(table) -> (table, {column name: chunk bounds}); tables are the cached, immutable ones


def _chunk_bounds(data: pa.Table, name: str) -> np.ndarray:
    hit = _bounds_cache.get(id(data))
    if hit is None or hit[0] is not data:
        if len(_bounds_cache) >= 16:
            _bounds_cache.clear()
        hit = _bounds_cache[id(data)] = (data, {})
    bounds = hit[1].get(name)
    if bounds is None:
        bounds = hit[1][name] = np.cumsum([0] + [len(c) for c in data.column(name).chunks])
    return bounds


def _chunk_views(data: pa.Table, name: str):
    """Zero-copy numpy views of the column's chunks (1-D for primitive values, (rows, D) for fixed-size lists of them),
    cached with the chunk bounds; None when the column cannot be viewed (nulls, strings, nested types)."""
    _chunk_bounds(data, name)
    slot = _bounds_cache[id(data)][1]
    key = ("views", name)
    if key in slot:
        return slot[key]
    col = data.column(name)
    typ = col.type
    views = None
    try:
        if pa.types.is_fixed_size_list(typ) and (pa.types.is_floating(typ.value_type) or pa.types.is_integer(typ.value_type)):
            d = typ.list_size
            if all(c.null_count == 0 and c.values.null_count == 0 for c in col.chunks):
                views = [c.values.to_numpy(zero_copy_only=True)[c.offset * d: (c.offset + len(c)) * d].reshape(len(c), d) for c in col.chunks]
        elif pa.types.is_floating(typ) or pa.types.is_integer(typ):
            if all(c.null_count == 0 for c in col.chunks):
                views = [c.to_numpy(zero_copy_only=True) for c in col.chunks]
    except (pa.ArrowInvalid, pa.ArrowNotImplementedError, ValueError):
        views = None
    slot[key] = views
    return views


def take_rows(data: pa.Table, columns: Sequence[str], rows: np.ndarray) -> pa.Table:
    """`data.select(columns).take(rows)` (index.py:163-166) for a FEW rows of a table with MANY chunks: every row is
    resolved to its chunk by bisection over chunk bounds cached per table and gathered there (one-row slices, one
    concatenation per column). pyarrow's Table.take walks - and for nested columns concatenates - all chunks of every
    column first: 4.7 ms per query for the 10 winning rows of a 100k x 128 table in 100 record batches when the vector
    column is returned, 0.2 ms even for the id column alone, against 0.1 ms for the search itself."""
    rows = np.asarray(rows, dtype=np.int64)
    sub = data.select(columns)
    if data.num_rows == 0 or len(rows) == 0 or len(rows) > 256 or len(rows) * 8 > data.num_rows:
        return sub.take(pa.array(rows, type=pa.int64()))
    out = []
    for name in columns:
        col = data.column(name)
        if col.num_chunks <= 4:
            out.append(col.take(pa.array(rows, type=pa.int64())).combine_chunks())
            continue
        bounds = _chunk_bounds(data, name)
        which = np.searchsorted(bounds, rows, side="right") - 1
        local = rows - bounds[which]
        views = _chunk_views(data, name)
        if views is not None:
            # numeric columns: gather straight out of the chunks' buffers (a tenth of the cost of ten one-row slices)
            if views[0].ndim == 2:
                vals = np.stack([views[c][i] for c, i in zip(which.tolist(), local.tolist())])
                out.append(pa.FixedSizeListArray.from_arrays(pa.array(vals.reshape(-1), type=col.type.value_type), col.type.list_size))
            else:
                vals = np.fromiter((views[c][i] for c, i in zip(which.tolist(), local.tolist())), dtype=views[0].dtype, count=len(rows))
                out.append(pa.array(vals, type=col.type))
            continue
        out.append(pa.concat_arrays([col.chunk(int(c)).slice(int(i), 1) for c, i in zip(which, local)]))
    return pa.Table.from_arrays(out, schema=sub.schema)


def _is_tensor(x) -> bool:
    return type(x).__module__.startswith("torch") and hasattr(x, "numpy")


def coerce_target(target, dim: int) -> np.ndarray:
    """Query -> float32 array of shape (Q, dim).

    The reference accepts ChunkedArray / Array / Tensor / ndarray / FixedSizeListScalar and casts
    to the column's value type (index.py:101-111). 2-D input (Q queries per call) is this
    build's wire extension; the reference raises on it.
    """
    if isinstance(target, pa.ChunkedArray):
        target = target.combine_chunks()
    if isinstance(target, pa.FixedSizeListScalar):
        target = target.values
    if isinstance(target, pa.FixedSizeListArray):
        flat = target.values.to_numpy(zero_copy_only=False)
        lo = target.offset * target.type.list_size
        target = flat[lo: lo + len(target) * target.type.list_size].reshape(len(target), target.type.list_size)
    elif isinstance(target, pa.Array):
        target = target.to_numpy(zero_copy_only=False)
    if _is_tensor(target):
        target = target.detach().cpu().numpy()
    q = np.asarray(target)
    if q.ndim == 1:
        q = q.reshape(1, -1)
    if q.ndim != 2 or q.shape[1] != dim:
        raise pa.ArrowInvalid(f"target has shape {tuple(np.asarray(target).shape)}; the column holds vectors of size {dim}")
    return np.ascontiguousarray(q, dtype=np.float32)


def _row_mask(data: pa.Table, column: str, filter: pc.Expression) -> np.ndarray:
    """Evaluate the predicate on the host over the scalar columns -> byte mask over rows."""
    n = data.num_rows
    probe = data.drop_columns([column]).append_column("__ROW__", pa.array(np.arange(n, dtype=np.int64)))
    try:
        kept = probe.filter(filter).column("__ROW__")
    except (pa.ArrowInvalid, KeyError):
        # the predicate references the vector column itself
        kept = data.append_column("__ROW__", pa.array(np.arange(n, dtype=np.int64))).filter(filter).column("__ROW__")
    mask = np.zeros(n, dtype=np.uint8)
    mask[kept.to_numpy()] = 1
    return mask


def call(
    root: str,
    coding: str | None,
    source: str | Sequence[str] | pa.Table,
    column: str,
    target,
    metric: str | None = None,
    select: Sequence[str] | None = None,
    filter: pc.Expression | None = None,
    maxval: int | None = None,
    probes: int | None = None,
    precision: int = knn.PREC_FP32,
    radius: float | None = None,
) -> pa.Table:
    """`radius` (this build's extension): every row within that distance of the target, ordered by (distance, row); with
    `maxval` as well, at most maxval of them (the exact k-NN, rows beyond the radius dropped)."""
    if metric is not None:
        knn.metric_code(metric)  # ValueError on unknown names, as coder.py:50
    if radius is not None:
        radius = float(radius)
        if radius != radius:
            raise ValueError("radius is NaN")
        if coding is not None or probes is not None:
            raise NotImplementedError("range search (radius) over an IVF coding is not supported")
    if isinstance(source, pa.Table):
        data = source
        shard = _shards.from_chunks(data.column(column))
        owned = True
    else:
        base, sig = _shards.load_table(root, source, with_signature=True)   # raises like table.load when the file is missing
        shard = _shards.get(root, source, column, base, sig)
        # with a coding the table carries its `__CODED_ID__` sidecar column (index.py:93-95)
        data = load(root, coding, source, column) if coding is not None else base
        owned = False

    try:
        typ = data.schema.field(column).type
        queries = coerce_target(target, typ.list_size)
        batched = queries.shape[0] != 1 or _batched_input(target)

        probe_codes = None
        if coding is not None and probes is not None:
            code = _coder.load(root, coding)                       # index.py:113-117
            if metric is None:
                metric = code["config"]["metric"]
            probe_codes = _coder.call(queries, (root, coding), int(probes))   # (Q, probes) composite codes, best first
        if metric is None:
            raise AssertionError("metric is required")
        knn.metric_code(metric)  # ValueError on unknown names, as coder.py:50

        out_cols = [*select] if select is not None else data.column_names
        mask = _row_mask(data, column, filter) if filter is not None else None
        if radius is not None:
            return _range(shard, data, out_cols, typ, queries, batched, metric, radius, maxval, mask, precision)

        if probe_codes is not None and batched:
            # Batched IVF: every query has its own probe cells, i.e. its own row mask (index.py:113-126 per query).
            codes = data.column(CODE_COL).to_numpy()
            # One launch for the batch when the shard is on one device and the shape fits (k <= 128, <= 512 probes): the
            # shard keeps its rows grouped by cell and query q scans only the posting lists of its probe codes.
            # (a table passed in directly has no cached shard: grouping its rows by cell would be paid on every call)
            fast = None if owned and queries.shape[0] < 16 else _search_cells(
                shard, _cells_key(root, coding, source, column), codes, queries, metric, maxval, probe_codes, mask, precision)
            if fast is not None:
                rows, dist = fast
                keep = rows.reshape(-1) >= 0
                out = take_rows(data, out_cols, rows.reshape(-1)[keep])
                out = out.append_column(DIST_COL, _distance_array(dist.reshape(-1)[keep], typ.value_type))
                qid = np.repeat(np.arange(rows.shape[0], dtype=np.int32), rows.shape[1])[keep]
                return out.append_column(QUERY_COL, pa.array(qid, type=pa.int32())).combine_chunks()
            # otherwise: the shard, the predicate mask and the code column are prepared once; each query is one masked
            # search on the resident shard.
            parts = []
            for qi in range(queries.shape[0]):
                cell = np.isin(codes, probe_codes[qi]).astype(np.uint8)
                m_q = cell if mask is None else (mask & cell)
                n_live = int(m_q.sum())
                k = n_live if maxval is None else min(int(maxval), n_live)
                if k < 1:
                    continue
                r_q, d_q = shard.search(queries[qi: qi + 1], metric, k, precision, m_q)
                keep = r_q[0] >= 0
                one = take_rows(data, out_cols, r_q[0][keep])
                one = one.append_column(DIST_COL, _distance_array(d_q[0][keep], typ.value_type))
                parts.append(one.append_column(QUERY_COL, pa.array(np.full(one.num_rows, qi, dtype=np.int32))))
            if not parts:
                empty = data.select(out_cols).slice(0, 0).append_column(DIST_COL, pa.array([], type=typ.value_type))
                return empty.append_column(QUERY_COL, pa.array([], type=pa.int32())).combine_chunks()
            return pa.concat_tables(parts).combine_chunks()

        if probe_codes is not None and mask is None and maxval is not None and not owned:
            # one query, no predicate: the probed cells' sizes say whether more than maxval rows survive; if so the search
            # reads just those cells' rows (fx_search_cells) instead of building an N-byte mask on the host and passing
            # over the whole shard
            fast = _search_cells(shard, _cells_key(root, coding, source, column), data.column(CODE_COL).to_numpy(), queries, metric,
                                 maxval, probe_codes, None, precision, more_than=int(maxval))
            if fast is not None:
                rows, dist = fast
                keep = rows[0] >= 0
                out = take_rows(data, out_cols, rows[0][keep])
                return out.append_column(DIST_COL, _distance_array(dist[0][keep], typ.value_type)).combine_chunks()

        if probe_codes is not None:
            # `__CODED_ID__ isin(probe codes)` AND the caller's predicate (index.py:119-126)
            cell = np.isin(data.column(CODE_COL).to_numpy(), probe_codes[0]).astype(np.uint8)
            mask = cell if mask is None else (mask & cell)
        n_live = int(mask.sum()) if mask is not None else data.num_rows

        if not batched and (maxval is None or n_live <= maxval):
            # every (surviving) row, table order, distance attached (index.py:162-165)
            dist = shard.distances(queries[0], metric)
            out = data.select(out_cols).append_column(DIST_COL, _distance_array(dist, typ.value_type))
            if mask is not None:
                out = out.filter(pa.array(mask.view(np.bool_)))
            return out.combine_chunks()

        k = n_live if maxval is None else min(int(maxval), n_live)
        if k < 1:
            empty = data.select(out_cols).slice(0, 0).append_column(DIST_COL, pa.array([], type=typ.value_type))
            if batched:
                empty = empty.append_column(QUERY_COL, pa.array([], type=pa.int32()))
            return empty.combine_chunks()
        if not batched and mask is None and not owned and _batcher.enabled:
            # concurrent single-query RPCs against the same table/metric/k share one pass over the corpus
            key = (id(shard), metric, k, precision)
            r1, d1 = _batcher.submit(key, queries[0], lambda qs: shard.search(qs, metric, k, precision, None))
            rows, dist = r1[None, :], d1[None, :]
        else:
            rows, dist = shard.search(queries, metric, k, precision, mask)

        keep = rows.reshape(-1) >= 0
        flat_rows = rows.reshape(-1)[keep]
        out = take_rows(data, out_cols, flat_rows)
        out = out.append_column(DIST_COL, _distance_array(dist.reshape(-1)[keep], typ.value_type))
        if batched:
            qid = np.repeat(np.arange(rows.shape[0], dtype=np.int32), rows.shape[1])[keep]
            out = out.append_column(QUERY_COL, pa.array(qid, type=pa.int32()))
        return out.combine_chunks()
    finally:
        if owned:
            shard.close()
        else:
            shard.release()   # the lease taken by shards.get


def _range(shard, data: pa.Table, out_cols, typ, queries: np.ndarray, batched: bool, metric: str, radius: float, maxval,
           mask, precision) -> pa.Table:
    """Rows within `radius` of each query, ordered by (distance, row): the range search, or with `maxval` the exact k-NN
    (k = min(maxval, surviving rows)) cut at the radius."""
    n_q = queries.shape[0]
    if maxval is None:
        offsets, rows, dist = shard.search_range(queries, metric, radius, precision, mask)
        qid = np.repeat(np.arange(n_q, dtype=np.int32), np.diff(offsets))
    else:
        n_live = int(mask.sum()) if mask is not None else data.num_rows
        k = min(int(maxval), n_live)
        if k < 1:
            rows, dist, qid = np.zeros(0, np.int64), np.zeros(0, np.float32), np.zeros(0, np.int32)
        else:
            r, d = shard.search(queries, metric, k, precision, mask)
            keep = (r >= 0) & (d <= np.float32(radius))   # the radius as the library sees it (one float32)
            rows, dist = r[keep], d[keep]
            qid = np.repeat(np.arange(n_q, dtype=np.int32), k).reshape(n_q, k)[keep]
    out = take_rows(data, out_cols, rows)
    out = out.append_column(DIST_COL, _distance_array(dist, typ.value_type))
    if batched:
        out = out.append_column(QUERY_COL, pa.array(qid, type=pa.int32()))
    return out.combine_chunks()


def _cells_key(root: str, coding: str, source, column: str) -> tuple:
    """Identity of the code column an inverted index was built from: the coding's name and the version (mtime, size) of
    every sidecar file - `make_index` under the same name replaces the cells."""
    if isinstance(source, pa.Table):
        return (coding, id(source))
    names = [source] if isinstance(source, str) else [*source]
    sig = []
    for one in names:
        try:
            st = os.stat(sidecar_path(root, coding, one, column))
            sig.append((one, st.st_mtime_ns, st.st_size))
        except OSError:
            sig.append((one, None, None))
    return (coding, tuple(sig))


def _search_cells(shard, coding, codes: np.ndarray, queries: np.ndarray, metric: str, maxval, probe_codes: np.ndarray,
                  mask, precision, more_than: int | None = None):
    """fx_search_cells for an IVF search, or None when the one-launch path does not apply (several devices, maxval None or
    > 128, too many probes, an approximate precision mode; `more_than`: the first query's probed cells hold no more rows
    than that - the caller then returns every surviving row instead, index.py:162-165)."""
    if len(shard.corpora) != 1 or maxval is None or int(maxval) < 1 or precision != knn.PREC_FP32:
        return None
    corpus = shard.corpora[0]
    if corpus.n_rows == 0 or corpus.n_rows != len(codes):
        return None
    with shard._cells_lock:
        cells = shard._cells
        if cells is None or cells[0] != coding:
            uniq, dense = np.unique(codes, return_inverse=True)      # composite codes present in the sidecar -> 0 .. n_cells - 1
            corpus.set_cells(dense)
            cells = shard._cells = (coding, uniq, np.bincount(dense, minlength=len(uniq)))
        uniq = cells[1]
        # probe codes -> dense cell numbers; codes no row carries and repeated codes become -1
        pc_ = np.asarray(probe_codes, dtype=np.int64)
        pos_c = np.minimum(np.searchsorted(uniq, pc_), len(uniq) - 1)
        dense_p = np.where(uniq[pos_c] == pc_, pos_c, -1).astype(np.int32)
        srt = np.sort(dense_p, axis=1)
        if ((srt[:, 1:] == srt[:, :-1]) & (srt[:, 1:] >= 0)).any():
            for qi in range(dense_p.shape[0]):
                _, first = np.unique(dense_p[qi], return_index=True)
                dup = np.ones(dense_p.shape[1], dtype=bool)
                dup[first] = False
                dense_p[qi, dup] = -1
        if more_than is not None and int(cells[2][dense_p[0][dense_p[0] >= 0]].sum()) <= more_than:
            return None
        try:
            return corpus.search_cells(queries, metric, min(int(maxval), corpus.n_rows), dense_p, mask)
        except NotImplementedError:
            return None


def _batched_input(target) -> bool:
    if isinstance(target, pa.ChunkedArray):
        return pa.types.is_fixed_size_list(target.type)
    if isinstance(target, pa.FixedSizeListArray):
        return True
    if isinstance(target, np.ndarray) or _is_tensor(target):
        return target.ndim == 2
    return False


# ---- IVF sidecars (index.py:19-78): <root>/indexes/<source>/<column>/<coding>.arrow, one int64 column ----------
def sidecar_path(root: str, name: str, source: str, column: str) -> str:
    return os.path.join(root, LOCATION, source, column, name + ".arrow")


def load(root: str, name: str, source, column: str) -> pa.Table:
    """The source table(s) with the `__CODED_ID__` column of coding `name` attached (index.py:19-35)."""
    if isinstance(source, str):
        _coder.load(root, name)
        return _table.join(_shards.load_table(root, source), _arrow.load(sidecar_path(root, name, source, column)), axis=1)
    if not isinstance(source, Sequence):
        raise AssertionError("source must be a table name or a sequence of names")
    return _table.join(*(load(root, name, one, column) for one in source))


def make(root: str, name: str, source, column: str) -> pa.Table:
    """Assign every row of `column` its composite code under coding `name` and write the sidecar, one record batch
    per record batch of the source (index.py:38-66). The assignment runs on the device (`io.coder.assign`)."""
    if isinstance(source, str):
        _coder.load(root, name)
        table = _shards.load_table(root, source)

        def batches():
            for chunk in table.column(column).chunks:
                yield pa.record_batch([pa.array(_coder.assign(root, name, _shards.chunk_rows(chunk)))], names=[CODE_COL])

        _arrow.make(sidecar_path(root, name, source, column),
                    pa.RecordBatchReader.from_batches(pa.schema({CODE_COL: pa.int64()}), batches()))
        return load(root, name, source, column)
    if not isinstance(source, Sequence):
        raise AssertionError("source must be a table name or a sequence of names")
    return _table.join(*(make(root, name, one, column) for one in source))


def list(root: str):
    base = os.path.join(root, LOCATION)
    for dirpath, _dirs, files in os.walk(base):
        for f in sorted(files):
            if f.endswith(".arrow"):
                yield os.path.relpath(os.path.join(dirpath, f), base).removesuffix(".arrow")


def drop(root: str, name: str, source: str, column: str) -> None:
    path = sidecar_path(root, name, source, column)
    if os.path.exists(path):
        os.unlink(path)

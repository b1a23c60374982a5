"""ctypes binding of libfenix_knn.so (C ABI declared in include/fenix_knn.h).

This module is the only place Python touches the CUDA path. There is deliberately no CPU
fallback: if the shared library is missing, or no B200 is visible, the calls raise.

Reference seam this replaces: fenix.io.coder.distance + pc.select_k_unstable
(src/fenix/io/coder/coder.py:38-50, src/fenix/io/index/index.py:162-168).
"""
from __future__ import annotations

import ctypes
import os
import threading
import weakref
from dataclasses import dataclass
from typing import Optional

import numpy as np

__all__ = [
    "FenixKnnError", "Context", "Corpus", "Comm", "Group", "Stats", "METRICS", "metric_code",
    "PREC_FP32", "PREC_TF32", "PREC_BF16", "PREC_EXACT_SCAN", "load_library", "library_path", "COMM_ID_BYTES",
    "train_codebooks",
]

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_NAME = "libfenix_knn.so"
COMM_ID_BYTES = 128
ABI_VERSION = 6

FX_OK = 0
FX_EINVAL, FX_ECUDA, FX_ENOMEM, FX_ESTATE, FX_EUNSUP = -1, -2, -3, -4, -5
FX_ETRUNC = -6   # fx_search_range: output capacity too small, out_offsets holds the sizes needed
PREC_FP32, PREC_TF32, PREC_BF16, PREC_EXACT_SCAN = 0, 1, 2, 3

# the five names accepted by the reference (flight.py:254, coder.py:39,42,47) -> 3 forms
METRICS = {"l2": 0, "euclidean": 0, "cosine": 1, "dot": 2, "inner_product": 2}

# every symbol include/fenix_knn.h declares (tests check the library exports all of them)
ABI_SYMBOLS = (
    "fx_init", "fx_shutdown", "fx_corpus_create", "fx_corpus_append", "fx_corpus_append_device",
    "fx_corpus_finalize", "fx_corpus_destroy", "fx_search", "fx_search_device", "fx_distances",
    "fx_merge_topk", "fx_get_stats", "fx_debug_scores", "fx_last_error", "fx_abi_version", "fx_set_option",
    "fx_comm_unique_id", "fx_comm_init_rank", "fx_comm_destroy", "fx_search_sharded", "fx_search_sharded_device",
    "fx_group_create", "fx_group_size", "fx_group_ctx", "fx_group_search", "fx_group_destroy",
    "fx_corpus_set_cells", "fx_search_cells", "fx_search_range", "fx_train_codebooks",
)


class FenixKnnError(RuntimeError):
    """A libfenix_knn call failed (message comes from fx_last_error())."""

    def __init__(self, code: int, message: str) -> None:
        super().__init__(f"[fenix_knn {code}] {message}")
        self.code = code


def metric_code(metric: str) -> int:
    try:
        return METRICS[metric]
    except KeyError:
        # same failure type as the reference's server side (coder.py:50)
        raise ValueError(f"unknown metric {metric!r}") from None


class _FxStats(ctypes.Structure):
    _fields_ = [
        ("n_rows", ctypes.c_int64), ("dim", ctypes.c_int32), ("pitch", ctypes.c_int32),
        ("device_bytes", ctypes.c_int64), ("searches", ctypes.c_int64), ("queries", ctypes.c_int64),
        ("fallback_queries", ctypes.c_int64), ("refined_queries", ctypes.c_int64), ("kernel_launches", ctypes.c_int64),
        ("last_search_ms", ctypes.c_double), ("last_main_kernel_ms", ctypes.c_double),
        ("last_path", ctypes.c_int32), ("last_variant", ctypes.c_int32), ("last_exchange_ms", ctypes.c_double),
        ("last_operand", ctypes.c_int32), ("last_resident_queries", ctypes.c_int32),
    ]


@dataclass(frozen=True)
class Stats:
    n_rows: int
    dim: int
    pitch: int
    device_bytes: int
    searches: int
    queries: int
    fallback_queries: int
    refined_queries: int
    kernel_launches: int
    last_search_ms: float
    last_main_kernel_ms: float
    last_path: int
    last_variant: int = 0
    last_exchange_ms: float = 0.0
    last_operand: int = 0          # filter operand of the last search: 0 fp32 / TF32, 1 bf16, 2 int8
    last_resident_queries: int = 0 # 1: int8 CTA-pair filter with resident query tiles


_lib_lock = threading.Lock()
_lib: Optional[ctypes.CDLL] = None


def library_path() -> str:
    return os.environ.get("FENIX_KNN_LIB", os.path.join(_HERE, _LIB_NAME))


def load_library() -> ctypes.CDLL:
    """dlopen libfenix_knn.so and declare the prototypes. Raises if it has not been built."""
    global _lib
    with _lib_lock:
        if _lib is not None:
            return _lib
        path = library_path()
        if not os.path.exists(path):
            raise FenixKnnError(
                FX_ESTATE,
                f"{path} not found: build it with `python -m fenix_b200.csrc.build` "
                "(there is no CPU fallback for the search path)",
            )
        lib = ctypes.CDLL(path)
        vp, i32, i64 = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64
        lib.fx_abi_version.restype = ctypes.c_int
        lib.fx_last_error.restype = ctypes.c_char_p
        lib.fx_init.argtypes = [ctypes.c_int, ctypes.POINTER(vp)]
        lib.fx_shutdown.argtypes = [vp]
        lib.fx_corpus_create.argtypes = [vp, i64, i32, i32, i64, ctypes.POINTER(vp)]
        lib.fx_corpus_append.argtypes = [vp, vp, i64]
        lib.fx_corpus_append_device.argtypes = [vp, vp, i64]
        lib.fx_corpus_finalize.argtypes = [vp]
        lib.fx_corpus_destroy.argtypes = [vp]
        lib.fx_search.argtypes = [vp, vp, i64, i32, i32, i32, vp, vp, vp]
        lib.fx_search_device.argtypes = [vp, vp, i64, i32, i32, i32, vp, vp, vp]
        lib.fx_distances.argtypes = [vp, vp, i32, vp]
        lib.fx_merge_topk.argtypes = [vp, vp, vp, i32, i64, i32, vp, vp]
        lib.fx_get_stats.argtypes = [vp, ctypes.POINTER(_FxStats)]
        lib.fx_debug_scores.argtypes = [vp, vp, i64, i32, vp]
        lib.fx_set_option.argtypes = [vp, ctypes.c_char_p, ctypes.c_char_p]
        lib.fx_comm_unique_id.argtypes = [vp]
        lib.fx_comm_init_rank.argtypes = [vp, vp, i32, i32, ctypes.POINTER(vp)]
        lib.fx_comm_destroy.argtypes = [vp]
        lib.fx_search_sharded.argtypes = [vp, vp, vp, i64, i32, i32, i32, vp, vp, vp]
        lib.fx_search_sharded_device.argtypes = [vp, vp, vp, i64, i32, i32, i32, vp, vp, vp]
        lib.fx_group_create.argtypes = [ctypes.POINTER(i32), i32, ctypes.POINTER(vp)]
        lib.fx_group_size.argtypes = [vp]
        lib.fx_group_ctx.argtypes = [vp, i32]
        lib.fx_group_search.argtypes = [vp, ctypes.POINTER(vp), vp, i64, i32, i32, i32, vp, vp, vp]
        lib.fx_group_destroy.argtypes = [vp]
        lib.fx_corpus_set_cells.argtypes = [vp, vp, i64, vp, i64]
        lib.fx_search_cells.argtypes = [vp, vp, i64, i32, i32, vp, i32, vp, vp, vp]
        lib.fx_search_range.argtypes = [vp, vp, i64, i32, ctypes.c_float, i32, vp, i64, vp, vp, vp]
        lib.fx_train_codebooks.argtypes = [ctypes.POINTER(vp), i32, i32, i32, i32, i32, vp, i64, vp]
        for name in ABI_SYMBOLS:
            fn = getattr(lib, name)
            if name not in ("fx_last_error", "fx_group_ctx"):
                fn.restype = ctypes.c_int
        lib.fx_last_error.restype = ctypes.c_char_p
        lib.fx_group_ctx.restype = vp
        _lib = lib
        return lib


def _check(lib: ctypes.CDLL, code: int) -> None:
    if code == FX_OK:
        return
    msg = (lib.fx_last_error() or b"").decode(errors="replace")
    if code == FX_EINVAL:
        raise ValueError(f"[fenix_knn {code}] {msg}")
    if code == FX_EUNSUP:
        raise NotImplementedError(f"[fenix_knn {code}] {msg}")
    if code == FX_ENOMEM:
        raise MemoryError(f"[fenix_knn {code}] {msg}")
    raise FenixKnnError(code, msg)


_nccl_preloaded = False


def preload_nccl() -> None:
    """Make libnccl.so.2 resolvable for the library's dlopen: a process that imported torch has it already; a bare
    server loads the copy bundled with the nvidia-nccl wheel (FENIX_NCCL_LIB overrides, see fenix_knn.h)."""
    global _nccl_preloaded
    if _nccl_preloaded or os.environ.get("FENIX_NCCL_LIB"):
        return
    _nccl_preloaded = True
    try:
        import importlib.util

        spec = importlib.util.find_spec("nvidia.nccl")
        for base in (spec.submodule_search_locations if spec is not None else ()):
            path = os.path.join(base, "lib", "libnccl.so.2")
            if os.path.exists(path):
                ctypes.CDLL(path, mode=ctypes.RTLD_GLOBAL)
                return
    except Exception:
        pass  # the library's own dlopen reports what is missing


class Context:
    """One CUDA device (streams + scratch). Thread-safe: searches on one context serialise."""

    def __init__(self, device: int = 0, _borrowed: Optional[int] = None) -> None:
        self._lib = load_library()
        self._h = ctypes.c_void_p()
        self.device = int(device)
        self._corpora: "weakref.WeakSet[Corpus]" = weakref.WeakSet()
        self._owned = _borrowed is None
        if _borrowed is not None:      # a context owned by a Group (fx_group_ctx)
            self._h = ctypes.c_void_p(_borrowed)
        else:
            _check(self._lib, self._lib.fx_init(self.device, ctypes.byref(self._h)))

    def set_option(self, name: str, value: Optional[object]) -> None:
        """Tuning knob by the name of its environment variable (read once at fx_init); None restores the default."""
        _check(self._lib, self._lib.fx_set_option(self._h, name.encode(), None if value is None else str(value).encode()))

    def close(self) -> None:
        """Shut the context down. Shards still alive on it are destroyed first: the C ABI requires every corpus to be
        destroyed before its context (a corpus handle outliving fx_shutdown would point at freed state)."""
        if getattr(self, "_h", None) is not None and self._h:
            for corpus in list(getattr(self, "_corpora", ())):
                corpus.close()
            if self._owned:
                self._lib.fx_shutdown(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self) -> None:  # pragma: no cover - best effort
        try:
            self.close()
        except Exception:
            pass

    def merge_topk_device(self, d_rows: int, d_dist: int, n_lists: int, n_q: int, k: int,
                          d_out_rows: int, d_out_dist: int) -> None:
        """Merge per-shard device lists (raw device pointers) into the global top-k."""
        _check(self._lib, self._lib.fx_merge_topk(self._h, d_rows, d_dist, n_lists, n_q, k, d_out_rows, d_out_dist))


def cells_csr(cell_of_row: np.ndarray) -> tuple[np.ndarray, np.ndarray]:
    """Inverted index of a dense cell assignment: (rows grouped by cell - ascending row inside a cell - as int32,
    offsets[n_cells + 1] of every cell's slice as int64), the layout fx_corpus_set_cells takes."""
    cells = np.ascontiguousarray(cell_of_row, dtype=np.int64)
    if cells.size and cells.min() < 0:
        raise ValueError("cell numbers must be >= 0")
    n_cells = int(cells.max()) + 1 if cells.size else 0
    inv = np.argsort(cells, kind="stable").astype(np.int32)
    off = np.zeros(n_cells + 1, dtype=np.int64)
    if n_cells:
        np.cumsum(np.bincount(cells, minlength=n_cells), out=off[1:])
    return inv, off


def train_codebooks(shards: "list[Corpus]", metric: str | int, books: np.ndarray, batch: int,
                    positions: np.ndarray) -> np.ndarray:
    """One epoch of mini-batch k-means on the device (fx_train_codebooks): `books` (n, k, D) float32 codewords, trained
    on the rows of the contiguous row shards `shards` (shard 0's device trains). `positions` (n_steps, n * batch) holds
    global row positions, ascending within a step; step s trains codebook j on positions[s, j*batch:(j+1)*batch].
    Returns the trained codewords (a new array)."""
    m = metric if isinstance(metric, int) else metric_code(metric)
    out = np.array(books, dtype=np.float32, order="C", copy=True)
    if out.ndim != 3:
        raise ValueError(f"books must be (n_books, k, dim), got shape {out.shape}")
    pos = np.ascontiguousarray(positions, dtype=np.int64)
    if pos.ndim != 2 or pos.shape[1] != out.shape[0] * int(batch):
        raise ValueError(f"positions must be (n_steps, {out.shape[0]} * batch), got shape {pos.shape}")
    if not shards:
        raise ValueError("no shards")
    if any(c.dim != out.shape[2] for c in shards):
        raise ValueError(f"codewords have {out.shape[2]} coordinates, the shards {[c.dim for c in shards]}")
    lib = shards[0]._lib
    handles = (ctypes.c_void_p * len(shards))(*[c._h for c in shards])
    _check(lib, lib.fx_train_codebooks(handles, len(shards), m, out.shape[0], out.shape[1], int(batch), pos.ctypes.data,
                                       pos.shape[0], out.ctypes.data))
    return out


class Corpus:
    """A device-resident row shard of a corpus (float32, row-major)."""

    def __init__(self, ctx: Context, capacity_rows: int, dim: int, row_base: int = 0) -> None:
        self._lib = ctx._lib
        self.ctx = ctx
        self.dim = int(dim)
        self.capacity = int(capacity_rows)
        self.row_base = int(row_base)
        self._h = ctypes.c_void_p()
        self._finalized = False
        _check(self._lib, self._lib.fx_corpus_create(ctx._h, self.capacity, self.dim, 0, self.row_base, ctypes.byref(self._h)))
        ctx._corpora.add(self)

    # ---- ingest ----
    def append(self, rows: np.ndarray) -> None:
        """Append row-major float32 rows from host memory (e.g. an Arrow values buffer view)."""
        rows = np.asarray(rows)
        if rows.dtype != np.float32:
            raise TypeError(f"corpus rows must be float32, got {rows.dtype}")
        if rows.ndim == 1:
            if rows.size % self.dim:
                raise ValueError("flat row buffer is not a multiple of dim")
            rows = rows.reshape(-1, self.dim)
        if rows.ndim != 2 or rows.shape[1] != self.dim:
            raise ValueError(f"expected (*, {self.dim}) rows, got {rows.shape}")
        if not rows.flags.c_contiguous:
            rows = np.ascontiguousarray(rows)
        _check(self._lib, self._lib.fx_corpus_append(self._h, rows.ctypes.data, rows.shape[0]))

    def append_device(self, device_ptr: int, n_rows: int) -> None:
        _check(self._lib, self._lib.fx_corpus_append_device(self._h, device_ptr, int(n_rows)))

    def finalize(self) -> "Corpus":
        _check(self._lib, self._lib.fx_corpus_finalize(self._h))
        self._finalized = True
        return self

    # ---- search ----
    def search(self, queries: np.ndarray, metric: str | int, k: int, precision: int = PREC_FP32,
               row_mask: Optional[np.ndarray] = None) -> tuple[np.ndarray, np.ndarray]:
        """k-NN of each query row. Returns (rows[int64, Q x k], dist[float32, Q x k]) ordered by
        (distance, row); short lists are padded with (-1, +inf)."""
        m = metric if isinstance(metric, int) else metric_code(metric)
        q = np.asarray(queries)
        if q.ndim == 1:
            q = q.reshape(1, -1)
        if q.ndim != 2 or q.shape[1] != self.dim:
            raise ValueError(f"expected queries of shape (*, {self.dim}), got {q.shape}")
        q = np.ascontiguousarray(q, dtype=np.float32)
        n_q = q.shape[0]
        k = int(k)
        out_rows = np.empty((n_q, max(k, 0)), dtype=np.int64)
        out_dist = np.empty((n_q, max(k, 0)), dtype=np.float32)
        mask_ptr = None
        if row_mask is not None:
            row_mask = np.ascontiguousarray(row_mask, dtype=np.uint8)
            if row_mask.shape != (self.n_rows,):
                raise ValueError(f"row_mask must have shape ({self.n_rows},), got {row_mask.shape}")
            mask_ptr = row_mask.ctypes.data
        _check(self._lib, self._lib.fx_search(self._h, q.ctypes.data, n_q, m, k, int(precision), mask_ptr,
                                              out_rows.ctypes.data, out_dist.ctypes.data))
        return out_rows, out_dist

    def search_range(self, queries: np.ndarray, metric: str | int, radius: float, precision: int = PREC_FP32,
                     row_mask: Optional[np.ndarray] = None,
                     capacity: Optional[int] = None) -> tuple[np.ndarray, np.ndarray, np.ndarray]:
        """Every row within `radius` of each query (distance <= radius, inclusive). Returns (offsets[int64, Q + 1],
        rows[int64], dist[float32]) in CSR form: query q's hits are rows[offsets[q]:offsets[q + 1]], ordered by
        (distance, row). `precision` is PREC_FP32 or PREC_EXACT_SCAN (the result is exact either way).

        The result size is unknown before the search: the first call uses `capacity` (default: 64 hits per query) and,
        when the hits do not fit, the library reports the sizes needed and the search runs a SECOND time into buffers
        of that size."""
        m = metric if isinstance(metric, int) else metric_code(metric)
        radius = float(radius)
        if radius != radius:
            raise ValueError("radius is NaN")
        q = np.asarray(queries)
        if q.ndim == 1:
            q = q.reshape(1, -1)
        if q.ndim != 2 or q.shape[1] != self.dim:
            raise ValueError(f"expected queries of shape (*, {self.dim}), got {q.shape}")
        q = np.ascontiguousarray(q, dtype=np.float32)
        n_q = q.shape[0]
        mask_ptr = None
        if row_mask is not None:
            row_mask = np.ascontiguousarray(row_mask, dtype=np.uint8)
            if row_mask.shape != (self.n_rows,):
                raise ValueError(f"row_mask must have shape ({self.n_rows},), got {row_mask.shape}")
            mask_ptr = row_mask.ctypes.data
        offsets = np.zeros(n_q + 1, dtype=np.int64)
        cap = 64 * n_q if capacity is None else int(capacity)
        for attempt in range(2):
            rows = np.empty(cap, dtype=np.int64)
            dist = np.empty(cap, dtype=np.float32)
            code = self._lib.fx_search_range(self._h, q.ctypes.data, n_q, m, radius, int(precision), mask_ptr, cap,
                                             offsets.ctypes.data, rows.ctypes.data, dist.ctypes.data)
            if code != FX_ETRUNC or attempt == 1:
                break
            cap = int(offsets[-1])   # the sizes the first search reported
        _check(self._lib, code)
        total = int(offsets[-1])
        return offsets, rows[:total], dist[:total]

    def search_raw(self, q_ptr: int, n_q: int, metric: int, k: int, precision: int,
                   out_rows_ptr: int, out_dist_ptr: int, mask_ptr: Optional[int] = None) -> None:
        """fx_search on caller-owned HOST buffers (pinned buffers are DMA'd directly)."""
        _check(self._lib, self._lib.fx_search(self._h, q_ptr, n_q, metric, k, precision, mask_ptr, out_rows_ptr, out_dist_ptr))

    def search_device(self, d_q_ptr: int, n_q: int, metric: int, k: int, precision: int,
                      d_out_rows_ptr: int, d_out_dist_ptr: int, d_mask_ptr: Optional[int] = None) -> None:
        """fx_search_device: everything stays in HBM (raw device pointers)."""
        _check(self._lib, self._lib.fx_search_device(self._h, d_q_ptr, n_q, metric, k, precision, d_mask_ptr,
                                                     d_out_rows_ptr, d_out_dist_ptr))

    def search_sharded_raw(self, comm: "Comm", q_ptr: int, n_q: int, metric: int, k: int, precision: int,
                           out_rows_ptr: Optional[int], out_dist_ptr: Optional[int], mask_ptr: Optional[int] = None,
                           on_device: bool = False) -> None:
        """fx_search_sharded / fx_search_sharded_device: COLLECTIVE over the ranks of `comm` (query all-gather, shard
        search, candidate all-gather, merge and result copy on one stream, one host synchronisation)."""
        fn = self._lib.fx_search_sharded_device if on_device else self._lib.fx_search_sharded
        _check(self._lib, fn(self._h, comm._h, q_ptr, n_q, metric, k, precision, mask_ptr, out_rows_ptr, out_dist_ptr))

    # ---- batched IVF (index.py:113-126 for a whole query batch): rows grouped by cell, one launch per batch ----
    def set_cells(self, cell_of_row: np.ndarray) -> int:
        """Give the shard its inverted index: `cell_of_row[r]` = dense cell number (0 .. n_cells - 1) of local row r.
        Returns n_cells."""
        cells = np.ascontiguousarray(cell_of_row, dtype=np.int64)
        if cells.shape != (self.n_rows,):
            raise ValueError(f"cell_of_row must have shape ({self.n_rows},), got {cells.shape}")
        inv, off = cells_csr(cells)
        n_cells = len(off) - 1
        _check(self._lib, self._lib.fx_corpus_set_cells(self._h, inv.ctypes.data, inv.size, off.ctypes.data, n_cells))
        return n_cells

    def search_cells(self, queries: np.ndarray, metric: str | int, k: int, probes: np.ndarray,
                     row_mask: Optional[np.ndarray] = None) -> tuple[np.ndarray, np.ndarray]:
        """Exact k-NN of every query among the rows of the cells it probes (`probes[q]`: cell numbers, -1 = unused, no
        duplicates), ANDed with `row_mask`. One launch for the batch; NotImplementedError for shapes it does not take."""
        m = metric if isinstance(metric, int) else metric_code(metric)
        q = np.ascontiguousarray(np.atleast_2d(np.asarray(queries)), dtype=np.float32)
        if q.shape[1] != self.dim:
            raise ValueError(f"expected queries of shape (*, {self.dim}), got {q.shape}")
        pr = np.ascontiguousarray(np.atleast_2d(np.asarray(probes)), dtype=np.int32)
        if pr.shape[0] != q.shape[0]:
            raise ValueError(f"expected one probe list per query, got {pr.shape} for {q.shape[0]} queries")
        n_q, k = q.shape[0], int(k)
        out_rows = np.empty((n_q, max(k, 0)), dtype=np.int64)
        out_dist = np.empty((n_q, max(k, 0)), dtype=np.float32)
        mask_ptr = None
        if row_mask is not None:
            row_mask = np.ascontiguousarray(row_mask, dtype=np.uint8)
            if row_mask.shape != (self.n_rows,):
                raise ValueError(f"row_mask must have shape ({self.n_rows},), got {row_mask.shape}")
            mask_ptr = row_mask.ctypes.data
        _check(self._lib, self._lib.fx_search_cells(self._h, q.ctypes.data, n_q, m, k, pr.ctypes.data, pr.shape[1], mask_ptr,
                                                    out_rows.ctypes.data, out_dist.ctypes.data))
        return out_rows, out_dist

    def distances(self, query: np.ndarray, metric: str | int) -> np.ndarray:
        """Distance of one query to every row (the reference's maxval=None branch)."""
        m = metric if isinstance(metric, int) else metric_code(metric)
        q = np.ascontiguousarray(np.asarray(query).reshape(-1), dtype=np.float32)
        if q.size != self.dim:
            raise ValueError(f"expected a query of {self.dim} values, got {q.size}")
        out = np.empty(self.n_rows, dtype=np.float32)
        _check(self._lib, self._lib.fx_distances(self._h, q.ctypes.data, m, out.ctypes.data))
        return out

    def debug_scores(self, queries: np.ndarray, metric: str | int) -> np.ndarray:
        """Raw tensor-core filter scores, first 128 queries x first 256 rows (diagnostics)."""
        m = metric if isinstance(metric, int) else metric_code(metric)
        q = np.ascontiguousarray(np.atleast_2d(queries), dtype=np.float32)
        out = np.zeros((128, 256), dtype=np.float32)
        _check(self._lib, self._lib.fx_debug_scores(self._h, q.ctypes.data, q.shape[0], m, out.ctypes.data))
        return out

    # ---- introspection ----
    def stats(self) -> Stats:
        s = _FxStats()
        _check(self._lib, self._lib.fx_get_stats(self._h, ctypes.byref(s)))
        return Stats(**{f: getattr(s, f) for f, _ in _FxStats._fields_})

    @property
    def n_rows(self) -> int:
        return self.stats().n_rows

    def close(self) -> None:
        if getattr(self, "_h", None) is not None and self._h:
            if self.ctx._h:   # the context destroys its shards when it is closed first
                self._lib.fx_corpus_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self) -> None:  # pragma: no cover - best effort
        try:
            self.close()
        except Exception:
            pass


class Comm:
    """This rank's membership in a group of row shards (one NCCL communicator owned by the library).

    One process per GPU: rank 0 calls `Comm.unique_id()`, the 128 bytes are broadcast by any means (torch.distributed,
    a file, a socket) and every rank constructs `Comm(ctx, id, world, rank)` - collectively."""

    def __init__(self, ctx: Context, unique_id: bytes, world: int, rank: int) -> None:
        if len(unique_id) != COMM_ID_BYTES:
            raise ValueError(f"unique id must be {COMM_ID_BYTES} bytes")
        preload_nccl()
        self._lib = ctx._lib
        self.ctx, self.world, self.rank = ctx, int(world), int(rank)
        self._h = ctypes.c_void_p()
        buf = ctypes.create_string_buffer(bytes(unique_id), COMM_ID_BYTES)
        _check(self._lib, self._lib.fx_comm_init_rank(ctx._h, buf, self.world, self.rank, ctypes.byref(self._h)))

    @staticmethod
    def unique_id() -> bytes:
        preload_nccl()
        lib = load_library()
        buf = ctypes.create_string_buffer(COMM_ID_BYTES)
        _check(lib, lib.fx_comm_unique_id(buf))
        return buf.raw

    def close(self) -> None:
        if getattr(self, "_h", None) is not None and self._h:
            if self.ctx._h:
                self._lib.fx_comm_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self) -> None:  # pragma: no cover - best effort
        try:
            self.close()
        except Exception:
            pass


class Group:
    """ONE process owning several devices (the Flight server's deployment): a context, an NCCL communicator and a
    worker thread per device, all inside the library (fx_group_*). Shard i of a corpus lives on `contexts[i]`."""

    def __init__(self, devices: "list[int]") -> None:
        preload_nccl()
        self._lib = load_library()
        self.devices = [int(d) for d in devices]
        self._h = ctypes.c_void_p()
        arr = (ctypes.c_int32 * len(self.devices))(*self.devices)
        _check(self._lib, self._lib.fx_group_create(arr, len(self.devices), ctypes.byref(self._h)))
        self.contexts = [Context(d, _borrowed=self._lib.fx_group_ctx(self._h, i)) for i, d in enumerate(self.devices)]

    def search(self, shards: "list[Corpus]", queries: np.ndarray, metric: str | int, k: int, precision: int = PREC_FP32,
               row_mask: Optional[np.ndarray] = None) -> tuple[np.ndarray, np.ndarray]:
        """Global k-NN over the row shards (contiguous, in order): every device searches its shard, candidates are
        all-gathered over NVLink and merged on the device; queries and results are host arrays."""
        m = metric if isinstance(metric, int) else metric_code(metric)
        if len(shards) != len(self.devices):
            raise ValueError(f"expected {len(self.devices)} shards, got {len(shards)}")
        q = np.ascontiguousarray(np.atleast_2d(np.asarray(queries)), dtype=np.float32)
        if q.shape[1] != shards[0].dim:
            raise ValueError(f"expected queries of shape (*, {shards[0].dim}), got {q.shape}")
        n_q, k = q.shape[0], int(k)
        out_rows = np.empty((n_q, max(k, 0)), dtype=np.int64)
        out_dist = np.empty((n_q, max(k, 0)), dtype=np.float32)
        mask_ptr = None
        if row_mask is not None:
            row_mask = np.ascontiguousarray(row_mask, dtype=np.uint8)
            mask_ptr = row_mask.ctypes.data
        handles = (ctypes.c_void_p * len(shards))(*[c._h for c in shards])
        _check(self._lib, self._lib.fx_group_search(self._h, handles, q.ctypes.data, n_q, m, k, int(precision), mask_ptr,
                                                    out_rows.ctypes.data, out_dist.ctypes.data))
        return out_rows, out_dist

    def close(self) -> None:
        if getattr(self, "_h", None) is not None and self._h:
            for ctx in self.contexts:
                ctx.close()           # destroys the shards still alive on it; the group owns the context itself
            self._lib.fx_group_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self) -> None:  # pragma: no cover - best effort
        try:
            self.close()
        except Exception:
            pass

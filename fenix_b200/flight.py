"""Arrow Flight server + client with the reference's wire format for the search path.

Mirrors src/fenix/flight.py: `Server.do_exchange` (flight.py:62-77) unpickles the command
dict {coding, source, column, metric, select, filter, maxval, probes}, reads the single
`target` column of the request stream and answers with one table; `Flight.search`
(flight.py:242-288) is byte-compatible with the reference client, so either side can be
swapped independently. do_put / do_get / drop-table / remove are restated because the device
shard cache must be invalidated when a table changes. IVF actions (make-coder / make-index / drop-index) are
served: codebook training on the host at ingest time, code assignment and probe ranking on the device.

NOTE (inherited, documented in SURVEY.md §5): commands are pickles - only expose the port to
trusted clients.

Wire extension (reference raises on these inputs, so it is free to define): a 2-D ndarray /
Tensor or a FixedSizeListArray target sends Q queries in one RPC; the answer then carries an
extra `__QUERY__: int32` column and holds k rows per query, grouped by query.
"""
from __future__ import annotations

import functools
import os
import threading
import pickle
import shutil
from dataclasses import dataclass
from typing import Iterator, Sequence

import numpy as np
import pyarrow as pa
import pyarrow.compute as pc
import pyarrow.flight as fl

from . import io

METRICS: frozenset[str] = frozenset({"cosine", "dot", "inner_product", "l2", "euclidean"})


class Server(fl.FlightServerBase):
    def __init__(self, root: str, host: str = "0.0.0.0", port: int = 9001) -> None:
        self.root = os.path.abspath(root)
        self.grpc = f"grpc://{host}:{port}"
        self._view: dict = {}  # per-server do_get options (set-*/del-* actions), as the reference keeps them
        super().__init__(location=self.grpc)
        # FENIX_WARM="table:column,...": device shards of those columns are uploaded before the first request
        if os.environ.get("FENIX_WARM"):
            io.shards.warm(self.root)
        elif os.environ.get("FENIX_EAGER_INIT", "1") != "0":
            # CUDA context + library initialisation (2 - 3 s on a fresh process) happen behind the server's start-up instead
            # of inside the first do_put / search. No usable device: the request that needs one reports it.
            def _init_devices() -> None:
                try:
                    devs = io.shards.devices()
                    if len(devs) > 1:
                        io.shards.group(devs)       # one process, several devices: contexts + NCCL communicators
                    else:
                        io.shards.context(devs[0])
                except Exception:
                    pass

            threading.Thread(target=_init_devices, name="fenix-init", daemon=True).start()

    def get_flight_info(self, ctx, descriptor):
        raise NotImplementedError()

    def list_flights(self, ctx, criteria):
        raise NotImplementedError()

    # ---- tables --------------------------------------------------------------------------
    def do_put(self, ctx, descriptor, reader, writer) -> None:
        name = descriptor.path[0].decode()
        io.table.make(self.root, name, reader.to_reader())
        # Upload at ingest: the table's vector columns go to the device(s) now (rows + norms + bf16 shadow), so the first
        # search after a do_put does not pay for the upload. FENIX_UPLOAD_ON_PUT=0 restores the lazy behaviour.
        if os.environ.get("FENIX_UPLOAD_ON_PUT", "1") != "0":
            try:
                io.shards.warm(self.root, name)
            except Exception:   # no usable device now: the search that needs it will say so
                pass

    def do_get(self, ctx, ticket):
        names = ticket.ticket.decode().split(":")
        if "coding" in self._view and "column" in self._view:
            data = io.index.load(self.root, self._view["coding"], names, self._view["column"])
        else:
            data = io.table.load(self.root, names)
        if "filter" in self._view:
            data = data.filter(self._view["filter"])
        if "select" in self._view:
            data = data.select(self._view["select"])
        return fl.GeneratorStream(data.schema, data.to_reader())

    # ---- search (the hot path) -----------------------------------------------------------
    def do_exchange(self, ctx, descriptor, reader, writer) -> None:
        config = pickle.loads(descriptor.command)
        config["target"] = reader.read_all().column("target").combine_chunks()
        config["filter"] = pickle.loads(config["filter"])
        data = io.index.call(self.root, **config)
        writer.begin(data.schema)
        writer.write_table(data)

    # ---- actions -------------------------------------------------------------------------
    def do_action(self, ctx, action):
        config = pickle.loads(action.body.to_pybytes())
        kind = action.type
        if kind == "make-coder":
            io.coder.make(self.root, **config)
        elif kind == "make-index":
            io.index.make(self.root, **config)
        elif kind == "drop-table":
            io.table.drop(self.root, **config)
        elif kind == "drop-index":
            # the codebook and every sidecar written under its name (flight.py:92-100 of the reference)
            io.coder.drop(self.root, **config)
            for path in [*io.index.list(self.root)]:
                parts = path.split(os.sep)
                if len(parts) >= 3 and parts[-1] == config["name"]:
                    io.index.drop(self.root, parts[-1], os.sep.join(parts[:-2]), parts[-2])
        elif kind == "remove":
            io.shards.invalidate(self.root)
            io.coder.forget(self.root)
            shutil.rmtree(self.root)
        elif kind.startswith("set-") and kind[4:] in ("coding", "column", "filter", "select"):
            self._view[kind[4:]] = config[kind[4:]]
        elif kind.startswith("del-") and kind[4:] in ("coding", "column", "filter", "select"):
            self._view.pop(kind[4:], None)
        else:
            raise ValueError(f"unknown action {kind!r}")
        return iter(())


@dataclass(frozen=True)
class Flight:
    host: str = "0.0.0.0"
    port: int = 9001

    @functools.cached_property
    def conn(self) -> fl.FlightClient:
        return fl.connect(f"grpc://{self.host}:{self.port}")

    def __del__(self) -> None:
        if "conn" in self.__dict__:
            self.conn.close()

    def _act(self, kind: str, body: dict) -> None:
        # draining the result stream surfaces server-side failures to the caller
        for _ in self.conn.do_action(fl.Action(kind, pickle.dumps(body))):
            pass

    def make_table(self, name: str, data: pa.RecordBatchReader) -> "Flight":
        writer, _ = self.conn.do_put(fl.FlightDescriptor.for_path(name), data.schema)
        with writer:
            for batch in data:
                writer.write_batch(batch)
        return self

    def read_table(self, source: str | Sequence[str], coding: str | None = None, column: str | None = None,
                   select: Sequence[str] | None = None, filter: pc.Expression | None = None) -> pa.RecordBatchReader:
        if coding is not None and column is not None:
            self._act("set-coding", {"coding": coding})
            self._act("set-column", {"column": column})
        if select is not None:
            self._act("set-select", {"select": select})
        if filter is not None:
            self._act("set-filter", {"filter": filter})
        ticket = fl.Ticket(source if isinstance(source, str) else ":".join(source))
        try:
            return self.conn.do_get(ticket).to_reader()
        finally:
            for opt in ("coding", "column", "select", "filter"):
                self._act(f"del-{opt}", {})

    def drop_table(self, name: str) -> "Flight":
        self._act("drop-table", {"name": name})
        return self

    def make_index(self, name: str, source, column: str, config) -> "Flight":
        self._act("make-coder", {"name": name, "source": source, "column": column, "config": config})
        return self.sync_index(name, source, column)

    def sync_index(self, name: str, source, column: str) -> "Flight":
        self._act("make-index", {"name": name, "source": source, "column": column})
        return self

    def drop_index(self, name: str) -> "Flight":
        self._act("drop-index", {"name": name})
        return self

    def search(self, target, source: str | Sequence[str], column: str, metric: str, coding: str | None = None,
               select: Sequence[str] | None = None, filter: pc.Expression | None = None,
               maxval: int | None = None, probes: int | None = None) -> pa.Table:
        assert metric in METRICS
        return self._exchange(target, {
            "coding": coding, "source": source, "column": column, "metric": metric, "select": select,
            "filter": pickle.dumps(filter), "maxval": maxval, "probes": probes,
        })

    def search_range(self, target, source: str | Sequence[str], column: str, metric: str, radius: float,
                     select: Sequence[str] | None = None, filter: pc.Expression | None = None,
                     maxval: int | None = None) -> pa.Table:
        """Every row within `radius` of the target (distance <= radius), ordered by (distance, row); with `maxval`, at
        most that many, nearest first. The command is `search`'s plus a "radius" key, so requests without one stay
        byte-identical to the reference client's."""
        assert metric in METRICS
        return self._exchange(target, {
            "coding": None, "source": source, "column": column, "metric": metric, "select": select,
            "filter": pickle.dumps(filter), "maxval": maxval, "probes": None, "radius": float(radius),
        })

    def _exchange(self, target, config: dict) -> pa.Table:
        command = pickle.dumps(config)
        if type(target).__module__.startswith("torch"):
            target = target.numpy()
        if isinstance(target, np.ndarray):
            if target.ndim == 2:  # wire extension: Q queries in one RPC
                target = pa.FixedSizeListArray.from_arrays(pa.array(np.ascontiguousarray(target).reshape(-1)), target.shape[1])
            else:
                target = pa.array(target)
        request = pa.table({"target": target})
        writer, reader = self.conn.do_exchange(fl.FlightDescriptor.for_command(command))
        with writer:
            writer.begin(request.schema)
            writer.write_table(request)
            writer.done_writing()
            return reader.read_all()

    def remove(self) -> "Flight":
        self._act("remove", {})
        return self

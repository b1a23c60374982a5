"""Range search (radius) without a GPU: the Flight command's wire format and the argument errors `io.index.call` raises
before any device work."""
import pickle

import numpy as np
import pyarrow as pa
import pytest

import fenix_b200 as fenix
from fenix_b200 import knn


def _capture_command(method="search", **kw):
    seen = {}

    class FakeWriter:
        def __enter__(self):
            return self

        def __exit__(self, *a):
            return False

        def begin(self, schema):
            pass

        def write_table(self, t):
            pass

        def done_writing(self):
            pass

    class FakeReader:
        def read_all(self):
            return pa.table({"ok": [1]})

    class FakeConn:
        def do_exchange(self, descriptor):
            seen["descriptor"] = descriptor
            return FakeWriter(), FakeReader()

        def close(self):
            pass

    client = fenix.Flight()
    client.__dict__["conn"] = FakeConn()
    getattr(client, method)(np.arange(4, dtype=np.float32), "s", "vector", "l2", select=["id"], **kw)
    return seen["descriptor"].command


def test_radius_travels_only_when_set():
    keys = {"coding", "source", "column", "metric", "select", "filter", "maxval", "probes"}
    plain = pickle.loads(_capture_command(maxval=7))
    assert set(plain) == keys
    cmd = pickle.loads(_capture_command("search_range", radius=0.25))
    assert set(cmd) == keys | {"radius"}
    assert cmd["radius"] == 0.25 and cmd["maxval"] is None and cmd["coding"] is None and cmd["probes"] is None
    with_k = pickle.loads(_capture_command("search_range", radius=1, maxval=3))
    assert with_k["radius"] == 1.0 and with_k["maxval"] == 3
    # without the radius, the range command is the plain one
    del with_k["radius"]
    assert with_k == {**plain, "maxval": 3}


def test_nan_radius_is_value_error_before_any_device_work(tmp_path, monkeypatch):
    def no_device(*a, **k):
        raise AssertionError("device work before the argument check")

    monkeypatch.setattr(fenix.io.shards, "get", no_device)
    monkeypatch.setattr(fenix.io.shards, "from_chunks", no_device)
    with pytest.raises(ValueError):
        fenix.io.index.call(str(tmp_path), None, "t", "vector", np.zeros(4), metric="l2", radius=float("nan"))


def test_radius_with_a_coding_is_not_implemented(tmp_path, monkeypatch):
    def no_device(*a, **k):
        raise AssertionError("device work before the argument check")

    monkeypatch.setattr(fenix.io.shards, "get", no_device)
    monkeypatch.setattr(fenix.io.shards, "from_chunks", no_device)
    with pytest.raises(NotImplementedError):
        fenix.io.index.call(str(tmp_path), "cbq", "t", "vector", np.zeros(4), metric="l2", probes=4, radius=1.0)
    with pytest.raises(NotImplementedError):
        fenix.io.index.call(str(tmp_path), None, "t", "vector", np.zeros(4), metric="l2", probes=4, radius=1.0)


def test_abi_declares_the_range_search():
    assert "fx_search_range" in knn.ABI_SYMBOLS and knn.ABI_VERSION == 6 and knn.FX_ETRUNC == -6

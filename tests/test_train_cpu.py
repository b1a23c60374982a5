"""IVF codebook training without a GPU: the C symbol is declared and exported, `coder.make` rejects too few rows before
any device work, and the per-step positions it hands the library follow the sampling of the reference."""
import ctypes
import re

import numpy as np
import pytest

import fenix_b200 as fenix
import train_model as tm
from conftest import table_of
from fenix_b200 import knn
from test_abi import HEADER


def test_symbol_declared_and_exported_with_abi_6(built_library):
    text = re.sub(r"/\*.*?\*/", "", open(HEADER).read(), flags=re.S)
    assert re.search(r"\bfx_train_codebooks\s*\(", text)
    assert "#define FX_ABI_VERSION 6" in open(HEADER).read()
    assert "fx_train_codebooks" in knn.ABI_SYMBOLS and knn.ABI_VERSION == 6
    assert hasattr(ctypes.CDLL(built_library), "fx_train_codebooks")


def test_too_few_rows_is_value_error_before_any_device_work(tmp_path, monkeypatch):
    def no_device(*a, **k):
        raise AssertionError("device work before the argument check")

    monkeypatch.setattr(fenix.io.shards, "get", no_device)
    monkeypatch.setattr(fenix.io.shards, "from_chunks", no_device)
    x = np.zeros((20, 4), np.float32)
    fenix.io.table.make(str(tmp_path), "t", table_of(x, 8).to_reader())
    config = dict(metric="l2", codebook_size=7, num_codebooks=3, batch_size=4, num_epochs=1)
    with pytest.raises(ValueError):
        fenix.io.coder.make(str(tmp_path), "cb", "t", "vector", config)


class FakeShardSet:
    corpora = ["shard"]

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.released = True


def test_positions_handed_to_the_library(tmp_path, monkeypatch):
    x = np.arange(1030 * 3, dtype=np.float32).reshape(1030, 3)
    fenix.io.table.make(str(tmp_path), "t", table_of(x, 100).to_reader())
    calls = []

    def fake_train(shards, metric, books, batch, positions):
        calls.append((shards, metric, books.copy(), batch, positions.copy()))
        return books + 1

    monkeypatch.setattr(fenix.io.shards, "get", lambda *a, **k: FakeShardSet())
    monkeypatch.setattr(fenix.knn, "train_codebooks", fake_train)
    monkeypatch.setattr(fenix.io.coder, "load", lambda root, name: name)
    n, k, bs = 2, 5, 60
    config = dict(metric="cosine", codebook_size=k, num_codebooks=n, batch_size=bs, num_epochs=3)
    fenix.io.coder.make(str(tmp_path), "cb", "t", "vector", config, rng=np.random.default_rng(7))
    ref = np.random.default_rng(7)
    seeds = x[np.sort(ref.permutation(1030)[: n * k])].reshape(n, k, 3)
    assert len(calls) == 3
    for e, (shards, metric, books, batch, positions) in enumerate(calls):
        assert shards == ["shard"] and metric == "cosine" and batch == bs
        assert np.array_equal(books, seeds + e)
        want = tm.epoch_positions(ref, 1030, n, bs)
        assert positions.shape == (1030 // (n * bs), n * bs)           # the 1030 % 120 remainder is dropped
        assert np.array_equal(positions, want)
        assert (np.diff(positions, axis=1) > 0).all()                  # sorted within every step: codebook j's
                                                                       # sample is the j-th run of bs of them

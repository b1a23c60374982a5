"""IVF codebook training on the device (fx_train_codebooks / knn.train_codebooks / io.coder.make), checked against the
numpy restatement in train_model.py: bit for bit for L2 and inner product, within 4 ulp for cosine."""
import ctypes

import numpy as np
import pytest

import fenix_b200 as fenix
import train_model as tm
from conftest import table_of
from exact_model import dyadic
from fenix_b200 import knn

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx(built_library):
    c = knn.Context(0)
    yield c
    c.close()


def corpus(ctx, x, row_base=0):
    c = knn.Corpus(ctx, len(x), x.shape[1], row_base=row_base)
    c.append(np.ascontiguousarray(x))
    return c.finalize()


def steps(rng, n_rows, n_books, batch, n_steps, row_base=0):
    """n_steps sorted samples of n_books * batch distinct positions each."""
    return np.stack([np.sort(rng.choice(n_rows, n_books * batch, replace=False)) for _ in range(n_steps)]) + row_base


def seeds(rng, x, n_books, k):
    return x[np.sort(rng.permutation(len(x))[: n_books * k])].reshape(n_books, k, -1)


@pytest.mark.parametrize("metric", ["l2", "dot"])
@pytest.mark.parametrize("dim,n_books,k,batch", [
    (7, 1, 4, 13), (7, 2, 37, 101), (96, 2, 256, 300), (96, 1, 37, 77), (768, 1, 2048, 130), (768, 2, 4, 65),
])
def test_bit_exact_on_dyadic_data(ctx, metric, dim, n_books, k, batch):
    rng = np.random.default_rng(dim * 1000 + k + batch)
    base = 1000
    n = max(n_books * k, 3 * n_books * batch) + 17
    x = dyadic(rng, (n, dim), 4)
    c = corpus(ctx, x, row_base=base)
    rows_of = lambda pos: x[pos - base]
    books = seeds(rng, x, n_books, k)
    want = books
    got = books
    for ep in range(3):
        pos = steps(rng, n, n_books, batch, 2, base)
        got = knn.train_codebooks([c], metric, got, batch, pos)
        want = tm.epoch(want, rows_of, pos, batch, metric)
        assert got.tobytes() == want.tobytes(), f"epoch {ep}"
    c.close()


def test_cosine_close_to_the_restatement(ctx):
    rng = np.random.default_rng(5)
    centres = rng.standard_normal((16, 96)).astype(np.float32) * 8
    x = (centres[rng.integers(0, 16, 4000)] + rng.standard_normal((4000, 96)).astype(np.float32)).astype(np.float32)
    c = corpus(ctx, x)
    books = np.stack([x[np.sort(rng.choice(4000, 16, replace=False))]])
    pos = steps(rng, 4000, 1, 500, 3)
    old = books
    for s in range(3):   # the restatement's assignments are the k = 1 search's on these well-separated clusters
        b = corpus(ctx, old[0])
        rows, _ = b.search(x[pos[s]], "cosine", 1)
        b.close()
        old, want_a = tm.step(old, lambda p: x[p], pos[s], 500, "cosine")
        assert np.array_equal(rows[:, 0], want_a[0])
    got = knn.train_codebooks([c], "cosine", books, 500, pos)
    ulp = np.abs(got.view(np.int32).astype(np.int64) - old.view(np.int32).astype(np.int64))
    assert ulp.max() <= 4, ulp.max()
    assert np.allclose(np.linalg.norm(got.astype(np.float64), axis=-1), 1.0, atol=1e-6)
    c.close()


def test_ties_go_to_the_lowest_codeword(ctx):
    x = np.array([[0, 0], [2, 0], [1, 0], [1, 0], [5, 5]], np.float32)
    c = corpus(ctx, x)
    for metric in ("l2", "dot"):
        books = np.array([[[0, 0], [0, 0], [2, 0], [2, 0]]], np.float32)   # duplicated codewords
        pos = np.arange(5)[None]
        got = knn.train_codebooks([c], metric, books, 5, pos)
        want = tm.epoch(books, lambda p: x[p], pos, 5, metric)
        assert got.tobytes() == want.tobytes(), metric
        a, _ = tm.assign(x, books[0], metric)
        if metric == "l2":   # rows 2, 3 sit halfway between codewords 0/1 and 2/3: codeword 0 wins
            assert a.tolist() == [0, 2, 0, 0, 2]
    c.close()


@pytest.mark.parametrize("metric", ["l2", "cosine", "dot"])
def test_assignment_matches_a_k1_search(ctx, metric):
    """A one-step epoch on dyadic data (every summation order gives the same distances): the trainer's assignment is
    the k = 1 search's nearest codeword, and the update moves each codeword to the predicted mean."""
    rng = np.random.default_rng(11)
    x = dyadic(rng, (3000, 32), 6)
    c = corpus(ctx, x)
    books = seeds(rng, x, 1, 50)
    pos = steps(rng, 3000, 1, 1000, 1)
    got = knn.train_codebooks([c], metric, books, 1000, pos)
    b = corpus(ctx, books[0])
    rows, _ = b.search(x[pos[0]], metric, 1)
    want, a = tm.step(books, lambda p: x[p], pos[0], 1000, metric)
    assert np.array_equal(rows[:, 0], a[0])
    if metric == "cosine":
        ulp = np.abs(got.view(np.int32).astype(np.int64) - want.view(np.int32).astype(np.int64))
        assert ulp.max() <= 4
    else:
        assert got.tobytes() == want.tobytes()
    b.close()
    c.close()


def test_deterministic_and_edges(ctx):
    rng = np.random.default_rng(3)
    x = rng.standard_normal((5000, 64)).astype(np.float32)
    c = corpus(ctx, x)
    books = seeds(rng, x, 2, 100)
    pos = steps(rng, 5000, 2, 700, 3)
    for metric in ("l2", "cosine", "dot"):
        a = knn.train_codebooks([c], metric, books, 700, pos)
        b = knn.train_codebooks([c], metric, books, 700, pos)
        assert a.tobytes() == b.tobytes(), metric
    # no steps: untouched
    assert knn.train_codebooks([c], "l2", books, 700, pos[:0]).tobytes() == books.tobytes()
    # k = 1: the one codeword becomes the mean of itself and the sample
    one = books[:1, :1]
    got = knn.train_codebooks([c], "l2", one, 10, pos[:1, :10])
    assert got.tobytes() == tm.epoch(one, lambda p: x[p], pos[:1, :10], 10, "l2").tobytes()
    # a codeword no row picks stays as it was
    far = books[:1, :3].copy()
    far[0, 2] = 1e6
    got = knn.train_codebooks([c], "l2", far, 50, pos[:1, :50])
    assert got[0, 2].tobytes() == far[0, 2].tobytes()
    c.close()


def test_argument_errors(ctx):
    rng = np.random.default_rng(4)
    x = rng.standard_normal((200, 8)).astype(np.float32)
    c = corpus(ctx, x, row_base=100)
    books = np.stack([x[:4]])
    lib = knn.load_library()
    good = np.arange(100, 110, dtype=np.int64)[None]
    cases = {
        "outside below": np.arange(99, 109)[None], "outside above": np.arange(291, 301)[None],
        "not ascending": good[:, ::-1].copy(),
    }
    for what, pos in cases.items():
        with pytest.raises(ValueError):
            knn.train_codebooks([c], "l2", books, 10, pos)
    with pytest.raises(ValueError):                          # k < 1
        knn.train_codebooks([c], "l2", books[:, :0], 10, good)
    with pytest.raises(ValueError):                          # batch < 1
        knn.train_codebooks([c], "l2", books, 0, good[:, :0])
    with pytest.raises(ValueError):                          # dims differ
        knn.train_codebooks([c], "l2", np.zeros((1, 4, 9), np.float32), 10, good)
    other = corpus(ctx, x[:50], row_base=0)                  # not contiguous with c
    with pytest.raises(ValueError):
        knn.train_codebooks([c, other], "l2", books, 10, good)
    handles = (ctypes.c_void_p * 1)(c._h)
    out = books.copy()
    assert lib.fx_train_codebooks(None, 1, 0, 1, 4, 10, good.ctypes.data, 1, out.ctypes.data) == knn.FX_EINVAL
    assert lib.fx_train_codebooks(handles, 1, 0, 1, 4, 10, None, 1, out.ctypes.data) == knn.FX_EINVAL
    assert lib.fx_train_codebooks(handles, 1, 0, 1, 4, 10, good.ctypes.data, 1, None) == knn.FX_EINVAL
    assert lib.fx_train_codebooks(handles, 1, 0, 0, 4, 10, good.ctypes.data, 1, out.ctypes.data) == knn.FX_EINVAL
    assert lib.fx_train_codebooks(handles, 1, 7, 1, 4, 10, good.ctypes.data, 1, out.ctypes.data) == knn.FX_EINVAL
    assert out.tobytes() == books.tobytes()
    # the shard still works afterwards
    assert knn.train_codebooks([c], "l2", books, 10, good).shape == books.shape
    other.close()
    c.close()


def test_row_shards_equal_one_shard(ctx):
    import torch

    rng = np.random.default_rng(8)
    x = dyadic(rng, (6000, 48), 5)
    whole = corpus(ctx, x)
    parts = [corpus(ctx, x[:2500]), corpus(ctx, x[2500:], row_base=2500)]
    books = seeds(rng, x, 2, 40)
    pos = steps(rng, 6000, 2, 900, 3)
    for metric in ("l2", "cosine"):
        one = knn.train_codebooks([whole], metric, books, 900, pos)
        two = knn.train_codebooks(parts, metric, books, 900, pos)
        assert one.tobytes() == two.tobytes(), metric
    if torch.cuda.device_count() >= 2:
        ctx1 = knn.Context(1)
        remote = [parts[0], corpus(ctx1, x[2500:], row_base=2500)]
        two = knn.train_codebooks(remote, "cosine", books, 900, pos)
        assert two.tobytes() == one.tobytes()   # `one`: the cosine result on the whole shard
        remote[1].close()
        ctx1.close()
    for p in parts + [whole]:
        p.close()


def test_coder_make_end_to_end(built_library, tmp_path):
    root = str(tmp_path)
    rng = np.random.default_rng(21)
    x = dyadic(rng, (4099, 24), 5)
    fenix.io.table.make(root, "t", table_of(x, 1000).to_reader())
    config = dict(metric="l2", codebook_size=8, num_codebooks=2, batch_size=300, num_epochs=2)
    coding = fenix.io.coder.make(root, "cb", "t", "vector", config, rng=np.random.default_rng(99))
    ref = np.random.default_rng(99)
    want = x[np.sort(ref.permutation(len(x))[:16])].reshape(2, 8, -1)
    for _ in range(2):
        want = tm.epoch(want, lambda p: x[p], tm.epoch_positions(ref, len(x), 2, 300), 300, "l2")
    assert coding["tensor"].tobytes() == want.tobytes()
    fenix.io.coder.forget()
    assert fenix.io.coder.load(root, "cb")["tensor"].tobytes() == want.tobytes()
    fenix.io.index.make(root, "cb", "t", "vector")
    q = x[:3] + np.float32(0.25)
    for qi in range(3):
        got = fenix.io.index.call(root, "cb", "t", "vector", q[qi], metric="l2", maxval=10, probes=64)
        exact = fenix.io.index.call(root, None, "t", "vector", q[qi], metric="l2", maxval=10)
        assert got.column("id").to_pylist() == exact.column("id").to_pylist()


def test_scale_2m_768_cosine(ctx):
    rng = np.random.default_rng(2)
    n, dim, k, bs = 2_000_000, 768, 1024, 4096
    x = rng.standard_normal((n, dim), dtype=np.float32)
    c = corpus(ctx, x)
    books = seeds(rng, x, 1, k)
    pos = steps(rng, n, 1, bs, 5)
    got = knn.train_codebooks([c], "cosine", books, bs, pos)
    want = tm.epoch(books, lambda p: x[p], pos, bs, "cosine", fast=True)
    ulp = np.abs(got.view(np.int32).astype(np.int64) - want.view(np.int32).astype(np.int64))
    assert ulp.max() <= 4, ulp.max()
    full = tm.epoch_positions(rng, n, 1, bs)
    got = knn.train_codebooks([c], "cosine", books, bs, full)
    assert np.isfinite(got).all()
    assert np.allclose(np.linalg.norm(got.astype(np.float64), axis=-1), 1.0, atol=1e-6)
    c.close()

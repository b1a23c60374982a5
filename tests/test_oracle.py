"""CPU tests: the oracle restatement against the committed outputs of the live reference."""
import numpy as np
import pytest
import torch

from conftest import METRICS, golden_cases, golden_filter, load_golden, table_of
from oracle import brute_force_f64, call, canonical, distance, search_rows
from oracle.fenix_oracle import _cdist_mm

# torch threads of the run that recorded the ref_*.npz outputs (tests/golden/PROVENANCE.txt)
GOLDEN_TORCH_THREADS = 8


@pytest.fixture
def golden_torch_threads():
    """MKL divides an sgemm's work by the intra-op thread count, so the last bits of a distance depend on that count
    (D = 100 differs at 1, 2 or 4 threads): replay the recorded calls with the count they ran with."""
    before = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_TORCH_THREADS)
    yield
    torch.set_num_threads(before)


@pytest.mark.parametrize("shape", [(1, 1000, 128), (1, 1000, 256), (1, 513, 100), (4, 2000, 96), (30, 40, 8)])
def test_l2_restatement_is_bitwise_torch_cdist(shape):
    u_rows, v_rows, d = shape
    g = torch.Generator().manual_seed(u_rows * 7 + d)
    u = torch.randn(u_rows, d, generator=g)
    v = torch.randn(v_rows, d, generator=g) + 3
    assert torch.equal(torch.cdist(u, v), _cdist_mm(u, v))
    assert torch.equal(torch.cdist(u, v), distance(u, v, "l2"))


def test_unknown_metric_raises_value_error():
    with pytest.raises(ValueError):
        distance(torch.zeros(1, 4), torch.zeros(2, 4), "manhattan")


@pytest.mark.parametrize("case", golden_cases())
@pytest.mark.parametrize("metric", METRICS)
def test_oracle_reproduces_live_reference(case, metric, golden_torch_threads):
    """ids and distances bit-identical to what fenix.io.index.call returned, in its own order."""
    g = load_golden(case)
    table = table_of(g["corpus"], int(g["chunk"]))
    k = None if int(g["k"]) < 0 else int(g["k"])
    flt = golden_filter(int(g["filter_mod"]))
    for qi, q in enumerate(g["queries"]):
        out = call(table, "vector", q, metric, select=["id"], filter=flt, maxval=k)
        assert out.column_names == ["id", "__DISTANCE__"]
        ref_id, ref_dist = g[f"{metric}:{qi}:id"], g[f"{metric}:{qi}:dist"]
        got_id, got_dist = out.column("id").to_numpy(), out.column("__DISTANCE__").to_numpy()
        # same library routines at the same call sites -> same bits; order of exact ties may differ
        # only through pyarrow's heap, which is the same code here
        assert np.array_equal(canonical(got_id, got_dist)[0], canonical(ref_id, ref_dist)[0])
        assert np.array_equal(np.sort(got_dist), np.sort(ref_dist))


@pytest.mark.parametrize("metric", ["l2", "cosine", "dot"])
def test_fp64_adjudicator_agrees_with_reference_outputs(metric):
    g = load_golden("gauss")
    for qi, q in enumerate(g["queries"]):
        rows, dist = brute_force_f64(g["corpus"], q, metric, int(g["k"]))
        ref_rows, ref_dist = canonical(g[f"{metric}:{qi}:id"], g[f"{metric}:{qi}:dist"])
        assert np.array_equal(rows[0], ref_rows)
        np.testing.assert_allclose(dist[0], ref_dist, rtol=1e-5, atol=1e-6)


def test_search_rows_matches_id_column():
    g = load_golden("clustered")
    table = table_of(g["corpus"], int(g["chunk"]))
    rows, dist = search_rows(table, "vector", g["queries"][0], "l2", 10)
    assert np.array_equal(rows, g["l2:0:id"])
    assert np.array_equal(dist, g["l2:0:dist"])


def test_schema_and_maxval_edges():
    g = load_golden("all_rows")
    table = table_of(g["corpus"], int(g["chunk"]))
    out = call(table, "vector", g["queries"][0], "l2")
    assert out.num_rows == table.num_rows
    assert out.column_names == ["id", "vector", "__DISTANCE__"]
    assert np.array_equal(out.column("id").to_numpy(), np.arange(table.num_rows))  # table order, unsorted

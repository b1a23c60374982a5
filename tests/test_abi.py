"""CPU tests of the C-ABI boundary: the library builds, loads and exports what the header
declares; argument errors are reported the documented way; without a GPU every compute entry
point fails loudly (no CPU fallback)."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from fenix_b200 import knn

HEADER = os.path.join(ROOT, "include", "fenix_knn.h")


def declared_symbols():
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(fx_[a-z_0-9]+)\s*\(", text)))


def test_header_symbols_are_exported(built_library):
    lib = ctypes.CDLL(built_library)
    names = declared_symbols()
    assert set(names) == set(knn.ABI_SYMBOLS), (names, knn.ABI_SYMBOLS)
    for name in names:
        assert hasattr(lib, name), f"{name} declared in include/fenix_knn.h but not exported"


def test_abi_version_and_no_torch_dependency(built_library):
    lib = knn.load_library()
    assert lib.fx_abi_version() == knn.ABI_VERSION
    out = subprocess.run(["ldd", built_library], capture_output=True, text=True).stdout
    assert "torch" not in out and "c10" not in out  # plain C ABI, no torch types behind it


def test_sass_is_sm100a(built_library):
    from fenix_b200.csrc.build import nvcc_path

    # the toolkit that built the library, whether or not its bin/ is on PATH
    cuobjdump = os.path.join(os.path.dirname(os.path.realpath(nvcc_path())), "cuobjdump")
    out = subprocess.run([cuobjdump, "-lelf", built_library], capture_output=True, text=True).stdout
    assert "sm_100a" in out, out


def _has_gpu():
    try:
        import torch

        return torch.cuda.is_available()
    except Exception:
        return False


@pytest.mark.skipif(_has_gpu(), reason="checks the no-GPU failure mode")
def test_fails_loudly_without_gpu(built_library):
    with pytest.raises(knn.FenixKnnError) as err:
        knn.Context(0)
    assert "no CPU fallback" in str(err.value)


@pytest.mark.skipif(_has_gpu(), reason="checks the no-GPU failure mode")
def test_index_call_has_no_cpu_fallback(built_library, tmp_path):
    import fenix_b200 as fenix
    from conftest import table_of

    corpus = np.random.default_rng(0).standard_normal((64, 8), dtype=np.float32)
    fenix.io.table.make(str(tmp_path), "t", table_of(corpus, 32).to_reader())
    with pytest.raises(knn.FenixKnnError):
        fenix.io.index.call(str(tmp_path), None, "t", "vector", corpus[0], metric="l2", maxval=3)


def build_c_demo(built_library, out_dir) -> str:
    """gcc examples/knn_demo.c against include/fenix_knn.h and the built library: a plain-C host, no Python, no torch."""
    exe = os.path.join(str(out_dir), "knn_demo")
    lib_dir = os.path.dirname(built_library)
    cmd = ["gcc", "-O2", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "examples", "knn_demo.c"),
           "-L", lib_dir, "-lfenix_knn", f"-Wl,-rpath,{lib_dir}", "-Wl,--allow-shlib-undefined", "-lm", "-o", exe]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    return exe


def test_c_host_compiles_against_the_header(built_library, tmp_path):
    exe = build_c_demo(built_library, tmp_path)
    if not _has_gpu():
        # without a device the C host fails the documented way: FX_ECUDA from fx_init, message from fx_last_error
        res = subprocess.run([exe], capture_output=True, text=True)
        assert res.returncode == 2 and "no CPU fallback" in res.stderr, (res.returncode, res.stderr)


@pytest.mark.gpu
def test_c_host_runs_and_matches_its_brute_force(built_library, tmp_path):
    res = subprocess.run([build_c_demo(built_library, tmp_path)], capture_output=True, text=True, timeout=300)
    assert res.returncode == 0 and "KNN DEMO OK" in res.stdout, (res.stdout[-2000:], res.stderr[-2000:])
    assert "path 3" in res.stdout and "path 2" in res.stdout       # the direct scan for one query, the tcgen05 filter for the batch


def test_null_arguments_are_einval(built_library):
    lib = knn.load_library()
    assert lib.fx_init(0, None) == knn.FX_EINVAL
    assert b"NULL" in lib.fx_last_error()
    assert lib.fx_corpus_finalize(None) == knn.FX_EINVAL
    assert lib.fx_search(None, None, 1, 0, 1, 0, None, None, None) == knn.FX_EINVAL
    assert lib.fx_get_stats(None, None) == knn.FX_EINVAL


def test_metric_names_match_reference():
    assert set(knn.METRICS) == {"cosine", "dot", "inner_product", "l2", "euclidean"}
    assert knn.metric_code("euclidean") == knn.metric_code("l2")
    assert knn.metric_code("dot") == knn.metric_code("inner_product")
    with pytest.raises(ValueError):
        knn.metric_code("manhattan")

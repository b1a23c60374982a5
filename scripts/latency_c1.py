"""In-process latency of a single-query search on the C1 shape (100k x 128, L2, k = 10): `io.index.call` (the seam),
`shard.search` (host glue + C ABI) and the raw C-ABI call on pre-allocated buffers, with the CUDA-graph replay of small
searches on and off; plus the 10M x 768 batch-1 search (C5) when --c5 is given."""
import ctypes, os, sys, tempfile, time
import numpy as np, pyarrow as pa
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from fenix_b200 import io as fio, knn

N, D, K = 100_000, 128, 10
rng = np.random.default_rng(1)
corpus = rng.standard_normal((N, D), dtype=np.float32)
batches = [pa.record_batch([pa.array(np.arange(lo, lo + 1000, dtype=np.int64)), pa.FixedSizeListArray.from_arrays(pa.array(corpus[lo:lo+1000].reshape(-1)), D)], names=["id", "vector"]) for lo in range(0, N, 1000)]
root = tempfile.mkdtemp()
fio.table.make(root, "c1", pa.Table.from_batches(batches).to_reader())
qs = rng.standard_normal((300, D), dtype=np.float32)


def timeit(fn, n=300):
    for i in range(5):
        fn(i)
    t = []
    for i in range(n):
        t0 = time.perf_counter(); fn(i); t.append(time.perf_counter() - t0)
    t = np.array(t) * 1e6
    return f"p50 {np.median(t):8.1f} us  p99 {np.percentile(t, 99):8.1f} us"


data = fio.shards.load_table(root, "c1")
shard = fio.shards.get(root, "c1", "vector", data)
c = shard.corpora[0]
out_rows = np.empty((1, K), np.int64); out_dist = np.empty((1, K), np.float32)
m = knn.metric_code("l2")


def raw(i):
    c.search_raw(qs[i % 300].ctypes.data, 1, m, K, knn.PREC_FP32, out_rows.ctypes.data, out_dist.ctypes.data)


def report(title):
    print(f"--- {title}")
    print("index.call select=[id]    ", timeit(lambda i: fio.index.call(root, None, "c1", "vector", qs[i % 300], metric="l2", select=["id"], maxval=K)))
    print("index.call default select ", timeit(lambda i: fio.index.call(root, None, "c1", "vector", qs[i % 300], metric="l2", maxval=K)))
    print("shard.search              ", timeit(lambda i: shard.search(qs[i % 300: i % 300 + 1], "l2", K)))
    print("fx_search (raw C ABI)     ", timeit(raw, 1000))
    st0 = c.stats(); raw(0); st = c.stats()
    print(f"device time of the last search {st.last_search_ms * 1e3:.1f} us, main kernel {st.last_main_kernel_ms * 1e3:.1f} us, "
          f"path {st.last_path}, variant {st.last_variant}, launches/search {st.kernel_launches - st0.kernel_launches}")


# the library's own routing: a single query over a 51 MB shard is ONE launch (direct_scan.cuh, path 3)
report("default routing (single-launch direct scan)")
for b in (2, 4, 8):
    o_r = np.empty((b, K), np.int64); o_d = np.empty((b, K), np.float32)
    print(f"fx_search, {b} queries        ", timeit(lambda i: c.search_raw(qs[i % 290:].ctypes.data, b, m, K, knn.PREC_FP32, o_r.ctypes.data, o_d.ctypes.data), 500),
          f" device {c.stats().last_search_ms * 1e3:.1f} us path {c.stats().last_path}")
c.ctx.set_option("FENIX_DIRECT", 0)
for graph in (1, 0):
    c.ctx.set_option("FENIX_GRAPH", graph)
    report(f"FENIX_DIRECT=0: tensor-core pipeline, CUDA graph replay of small searches {'on' if graph else 'off'}")
c.ctx.set_option("FENIX_GRAPH", None)
c.ctx.set_option("FENIX_DIRECT", None)
shard.release()

if "--c5" in sys.argv:
    import torch
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import bench
    cfg = dict(bench.CONFIGS["c5_1"], data_num=bench.CONFIGS["c3"]["num"])
    ctx = fio.shards.context(0)
    dev = torch.device("cuda", 0)
    big = bench.build_shard(cfg, ctx, 0, cfg["n"], dev)
    q5 = rng.standard_normal((300, cfg["d"]), dtype=np.float32)
    m5 = knn.metric_code(cfg["metric"])
    for graph in (1, 0):
        ctx.set_option("FENIX_GRAPH", graph)
        for b in (1, 8, 64):
            o_r = np.empty((b, K), np.int64); o_d = np.empty((b, K), np.float32)
            print(f"C5 batch {b:2d}, graph {'on ' if graph else 'off'}: fx_search ",
                  timeit(lambda i: big.search_raw(q5[(i * b) % 200:].ctypes.data, b, m5, K, knn.PREC_FP32, o_r.ctypes.data, o_d.ctypes.data), 100),
                  f" device {big.stats().last_search_ms * 1e3:.1f} us")
    ctx.set_option("FENIX_GRAPH", None)
    big.close()

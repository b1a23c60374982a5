import numpy as np, sys, os
sys.path.insert(0, os.getcwd())
from fenix_b200 import knn
rng = np.random.default_rng(1)
x = rng.standard_normal((100_000, 128), dtype=np.float32)
ctx = knn.Context(0); c = knn.Corpus(ctx, len(x), 128); c.append(x); c.finalize()
q = rng.standard_normal((8, 128), dtype=np.float32)
for nq in (1, 2, 4, 8):
    for _ in range(5):
        r, d = c.search(q[:nq], "l2", 10)
    rs, ds = c.search(q[:nq], "l2", 10, knn.PREC_EXACT_SCAN)
    ctx.set_option("FENIX_DIRECT", 0)
    rt, dt = c.search(q[:nq], "l2", 10)
    ctx.set_option("FENIX_DIRECT", None)
    for _ in range(3):
        c.search(q[:nq], "l2", 10)
    print(nq, "queries: kernel", round(c.stats().last_search_ms * 1e3, 1), "us; == scan", np.array_equal(r, rs) and np.array_equal(d, ds),
          "== tensor path", np.array_equal(r, rt) and np.array_equal(d, dt))
ctx.set_option("FENIX_DEBUG_DIRECT", 1)
for i in range(3):
    c.search(q[:1], "l2", 10)
c.search(q[:4], "l2", 10)
ctx.set_option("FENIX_DEBUG_DIRECT", None)

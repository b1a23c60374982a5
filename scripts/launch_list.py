"""Launch list of one search: every kernel of the library that one `fx_search` of a bench.py configuration launches, with
its device time (torch.profiler, CUDA activities) and its share of the search's kernel time.

    python scripts/launch_list.py [--config c3] [--warm 2]

The corpus and the query batch are bench.py's (seeded). `--warm` searches run first (shadow build, plan, module load), so
the profiled search is a steady-state one. Prints a table; the card, its power limit and the SM clock are on the last line.
"""
import argparse
import collections
import os
import re
import subprocess
import sys

sys.dont_write_bytecode = True
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402
from torch.profiler import ProfilerActivity, profile  # noqa: E402

import bench  # noqa: E402
from fenix_b200 import knn  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="c3", choices=sorted(bench.CONFIGS))
    ap.add_argument("--warm", type=int, default=2)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("launch_list.py profiles a GPU; none is visible")
    cfg = dict(bench.CONFIGS[args.config])
    dev = torch.device("cuda", 0)
    ctx = knn.Context(0)
    corpus = bench.build_shard(cfg, ctx, 0, cfg["n"], dev)
    q = bench.query_batch(cfg)
    for _ in range(args.warm):
        corpus.search(q, cfg["metric"], cfg["k"])
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        corpus.search(q, cfg["metric"], cfg["k"])
        torch.cuda.synchronize()
    st = corpus.stats()
    tot, cnt = collections.Counter(), collections.Counter()
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA and "fx::" in e.name:
            k = re.sub(r"\(.*", "", e.name).replace("void ", "")
            tot[k] += getattr(e, "device_time", None) or e.cuda_time
            cnt[k] += 1
    all_us = sum(tot.values())
    print(f"# one {args.config} search ({cfg['n']} x {cfg['d']} {cfg['metric']}, k = {cfg['k']}, {len(q)} queries) after "
          f"{args.warm} warm-up searches: kernels of the library, device time (torch.profiler)")
    print(f"# last_variant {st.last_variant}, last_resident_queries {st.last_resident_queries}, last_operand {st.last_operand}, "
          f"refined {st.refined_queries}, scanned {st.fallback_queries} (over all searches of this shard)")
    for k, us in tot.most_common():
        print(f"{100 * us / all_us:6.2f}%  {us / 1e3:9.3f} ms  {cnt[k]:3d} launches  {k}")
    print(f"# total {all_us / 1e3:.3f} ms of kernel time")
    smi = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    print(f"# gpu: {smi}")
    corpus.close()
    ctx.close()


if __name__ == "__main__":
    main()

"""int8 against bf16 shadow filter for exact cosine (k = 10, 4096 queries, Gaussian rows), and the K' sweep that sets
TC_KP_I8 (tc_filter.cuh).

    python scripts/int8_ab.py widths [--rows 1000000] [--dims 256,384,512,768,1024]
    python scripts/int8_ab.py kp [--rows 10000000,1250000] [--ks 10,16] [--kps 128,160,192,224,256,320]

widths: for each row width, the bf16 and the int8 filter (FENIX_INT8=0 / 1) through the CTA-pair and the one-CTA streaming
kernel (FENIX_TC_PAIR=1 / 0), and for int8 also the CTA-pair kernel with resident query tiles (FENIX_TC_RESIDENT=1; the
two others run with it off): the main filter kernel's time (mean of 4 searches after 2 warm-up searches), its rate and
share of the data sheet's dense int8 peak (ops = 2 Q N D, bytes = N D of the int8 shadow), the queries refined and sent to
the fp64 scan per search, and the SM clock / power limit read right after the runs.
kp: refined and scanned queries per search of the int8 filter at D = 768 for each forced K' (FENIX_TC_KP). TC_KP_I8 is the
smallest K' that refines at most 0.5 % of the batch and scans none.
"""
import argparse
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from fenix_b200 import knn  # noqa: E402

INT8_PEAK_TOPS = 4500.0   # B200 data sheet, dense int8, per GPU (1000 W card)
NQ = 4096


def gpu_state():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,clocks.sm,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return out[0] if out else "?"


def make_shard(ctx, n, d, seed):
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(seed)
    c = knn.Corpus(ctx, n, d)
    step = 500_000
    for lo in range(0, n, step):
        m = min(step, n - lo)
        x = torch.randn((m, d), generator=g, device=dev)
        torch.cuda.synchronize()
        c.append_device(x.data_ptr(), m)
        del x
    c.finalize()
    return c, torch.randn((NQ, d), generator=g, device=dev)


def run(ctx, c, q, k, reps=4, warm=2):
    nq = q.shape[0]
    rows = torch.empty((nq, k), dtype=torch.int64, device=q.device)
    dist = torch.empty((nq, k), dtype=torch.float32, device=q.device)
    ts = []
    before = c.stats()
    for i in range(warm + reps):
        c.search_device(q.data_ptr(), nq, knn.metric_code("cosine"), k, knn.PREC_FP32, rows.data_ptr(), dist.data_ptr())
        if i >= warm:
            ts.append(c.stats().last_main_kernel_ms)
    st = c.stats()
    n_s = warm + reps
    return (float(np.mean(ts)), st, (st.refined_queries - before.refined_queries) / n_s,
            (st.fallback_queries - before.fallback_queries) / n_s, rows.clone())


def widths(args):
    ctx = knn.Context(0)
    for d in [int(v) for v in args.dims.split(",")]:
        c, q = make_shard(ctx, args.rows, d, d)
        ops = 2.0 * NQ * args.rows * d
        ref = None
        for op, i8 in (("bf16", 0), ("int8", 1)):
            ctx.set_option("FENIX_INT8", i8)
            kernels = (("pair", 1, 0), ("one-CTA", 0, 0)) if i8 == 0 else (("resident", 1, 1), ("pair", 1, 0), ("one-CTA", 0, 0))
            for kern, pair, res in kernels:
                ctx.set_option("FENIX_TC_PAIR", pair)
                ctx.set_option("FENIX_TC_RESIDENT", res)
                ms, st, refd, fb, rows = run(ctx, c, q, 10)
                same = "-" if ref is None else str(torch.equal(rows, ref))
                ref = rows if ref is None else ref
                tops = ops / ms / 1e9
                print(f"D={d} N={args.rows} {op:4s} {kern:8s} kernel {ms:8.3f} ms  {tops:7.0f} TOPS  {tops / INT8_PEAK_TOPS:.3f} of int8 peak"
                      f"  {args.rows * d / ms / 1e9:6.2f} TB/s int8 bytes  operand {st.last_operand} variant {st.last_variant}"
                      f" resident {st.last_resident_queries}  refined {refd:.1f} scanned {fb:.1f} per search  same ids {same}", flush=True)
        ctx.set_option("FENIX_TC_PAIR", None)
        ctx.set_option("FENIX_TC_RESIDENT", None)
        ctx.set_option("FENIX_INT8", None)
        print(f"  gpu: {gpu_state()}", flush=True)
        c.close()
    ctx.close()


def kp_sweep(args):
    ctx = knn.Context(0)
    for n in [int(v) for v in args.rows.split(",")]:
        c, q = make_shard(ctx, n, 768, 7)
        for k in [int(v) for v in args.ks.split(",")]:
            for kp in [int(v) for v in args.kps.split(",")]:
                ctx.set_option("FENIX_TC_KP", kp)
                ms, st, refd, fb, _ = run(ctx, c, q, k, reps=3, warm=1)
                print(f"N={n} k={k} K'={kp}: kernel {ms:8.3f} ms  refined {refd:.1f} ({100 * refd / NQ:.2f} %) scanned {fb:.1f}"
                      f" per search of {NQ}  operand {st.last_operand} variant {st.last_variant}", flush=True)
            ctx.set_option("FENIX_TC_KP", None)
        print(f"  gpu: {gpu_state()}", flush=True)
        c.close()
    ctx.close()


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("what", choices=["widths", "kp"])
    ap.add_argument("--rows", default=None)
    ap.add_argument("--dims", default="256,384,512,768,1024")
    ap.add_argument("--ks", default="10,16")
    ap.add_argument("--kps", default="128,160,192,224,256,320")
    a = ap.parse_args()
    if a.what == "widths":
        a.rows = int(a.rows or 1_000_000)
        widths(a)
    else:
        a.rows = a.rows or "10000000,1250000"
        kp_sweep(a)

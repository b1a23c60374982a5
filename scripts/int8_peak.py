"""Measured dense int8 tensor-core rate of one GPU: torch._int_mm (cuBLASLt, int8 x int8 -> int32) on n x n x n.

    python scripts/int8_peak.py [--n 8192] [--seconds 3]

burst: best of 10 single calls (CUDA events) right after a short warm-up, while the clock is still high. sustained:
back-to-back calls for --seconds, total ops over total device time, once the card has settled at its power limit. Both
print the median SM clock sampled during the region (NVML, bench.ClockSampler), and the line names the card, its power
limit and the kernel cuBLASLt ran (torch.profiler), so that one can tell whether it reached the tcgen05 int8 path.
Prints one JSON line. The "fraction of the int8 peak" figures in DESIGN.md are quoted against `sustained_tops` and
`burst_tops` of this script, with the data sheet's 4500 TOPS (dense, 1000 W card) beside them.
"""
import argparse
import json
import os
import subprocess
import sys

sys.dont_write_bytecode = True
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from bench import ClockSampler  # noqa: E402

DATASHEET_TOPS = 4500.0


def card() -> str:
    out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    return out or "?"


def kernel_names(a, b) -> list:
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        torch._int_mm(a, b)
        torch.cuda.synchronize()
    return sorted({e.key for e in prof.key_averages() if e.device_type == torch.autograd.DeviceType.CUDA})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=8192)
    ap.add_argument("--seconds", type=float, default=3.0)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("int8_peak.py measures a GPU; none is visible")
    n = args.n
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(0)
    a = torch.randint(-127, 128, (n, n), generator=g, device=dev, dtype=torch.int8)
    b = torch.randint(-127, 128, (n, n), generator=g, device=dev, dtype=torch.int8).t()   # column-major B, as cuBLASLt wants it
    ops = 2.0 * n * n * n
    for _ in range(3):
        torch._int_mm(a, b)
    torch.cuda.synchronize()

    sampler = ClockSampler(0)
    sampler.start()
    best = float("inf")
    for _ in range(10):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        torch._int_mm(a, b)
        e1.record()
        e1.synchronize()
        best = min(best, e0.elapsed_time(e1))
    burst_clk = sampler.stop()

    per = max(1, int(args.seconds * 1e3 / best))
    torch._int_mm(a, b)
    torch.cuda.synchronize()
    sampler = ClockSampler(0)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(per):
        torch._int_mm(a, b)
    e1.record()
    e1.synchronize()
    sust_ms = e0.elapsed_time(e1) / per
    sust_clk = sampler.stop()

    burst_tops, sust_tops = ops / best / 1e9, ops / sust_ms / 1e9
    print(json.dumps({
        "what": f"torch._int_mm {n}^3 int8 -> int32", "card": card(), "kernels": kernel_names(a, b),
        "burst_ms": round(best, 4), "burst_tops": round(burst_tops, 1), "burst_clock": burst_clk,
        "sustained_ms": round(sust_ms, 4), "sustained_calls": per, "sustained_tops": round(sust_tops, 1), "sustained_clock": sust_clk,
        "datasheet_tops": DATASHEET_TOPS, "burst_of_datasheet": round(burst_tops / DATASHEET_TOPS, 3),
        "sustained_of_datasheet": round(sust_tops / DATASHEET_TOPS, 3),
    }), flush=True)


if __name__ == "__main__":
    main()

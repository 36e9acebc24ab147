"""
gbm_smart_lev's per-step series: the running log-return sum (method="sum") against the chain (the default).

  1e6 investors x 500 steps on both grids of the GBM script (-1..1 / 0.2 and 0.2..2 / 0.2) and x 2000 steps
  on the first; fp32 (float32 x) and under a float64 default (float64 x).  chain and sum alternate, --reps
  runs each after a warm-up; the best run counts.  Then one profiled run of engine.gbm_series_sum per dtype:
  device time of its kernels by part (S dump, select, moments, the rest: LOG sweep / final chain and row
  statistics) from torch.profiler, and the routed leverage count.

Writes one JSON document (stdout, or --out): wall time per run (host clock around work that ends in a device
synchronise), investor-steps/s, the device name and its power limit read in the same run.

    python tools/bench_gbm_series.py --reps 3 --out results/bench_gbm_series.json
"""
import argparse
import json
import math
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from rlmd_b200 import engine, lev_exp  # noqa: E402
from tools.bench_fp64 import device_power_limit_w, timed  # noqa: E402

GRIDS = {"op": (-1.0, 1.0, 0.2, 0.05, math.sqrt(0.2)), "snp": (0.2, 2.0, 0.2, 0.0540025395205692, 0.1897916175617430)}
# kernel-name prefixes: each part holds its pass kernels and their resolve kernels
PARTS = (("dump", "gbm_sum_chunk_kernel"), ("select", "sum_select_"), ("moments", "sum_moment_"))


def split(x, lev, top, dtype):
    """Device time (ms) per part of one gbm_series_sum call, from the profiler's kernel records."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        _, _, routed = engine.gbm_series_sum(lev, lev, 100.0, top, x, dtype=dtype)
        torch.cuda.synchronize()
    out = {"dump": 0.0, "select": 0.0, "moments": 0.0, "other": 0.0}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if t <= 0:
            continue
        part = next((p for p, k in PARTS if k in e.key), "other")
        out[part] += t / 1e3
    return out, int(routed.sum())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--investors", type=int, default=1_000_000)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_gbm_series needs a CUDA device")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    n = a.investors
    top = max(1, int(n * 1e-4))
    res = {"device": torch.cuda.get_device_name(dev), "power_limit_w": device_power_limit_w(0), "investors": n,
           "top": top, "timing": "host clock around each call, device synchronised before and after; chain and sum "
           "alternate, the first call of each configuration is a warm-up and not reported; split_ms: kernel device "
           "time from torch.profiler, one run - dump: gbm_sum_chunk_kernel; select: sum_select_kernel and "
           "sum_select_resolve_kernel (six levels); moments: sum_moment_kernel and sum_moment_resolve_kernel (two "
           "passes); other: everything else (LOG sweep / final fp64 chain, row statistics of data_T, the chain "
           "series of unrouted leverages, the fp64 state pass, memsets)", "cases": []}
    for grid, h in (("op", 500), ("snp", 500), ("op", 2000)):
        lo_, hi_, inc, mu, sigma = GRIDS[grid]
        g = torch.Generator(device=dev).manual_seed(h)
        x32 = ((mu - sigma ** 2 / 2) + sigma * torch.randn((n, h), generator=g, device=dev)).float()
        for dtype in (torch.float32, torch.float64):
            x = x32 if dtype == torch.float32 else x32.double()
            lev = np.asarray(lev_exp.param_range(lo_, hi_, inc), dtype=np.float32 if dtype == torch.float32
                             else np.float64)

            def run(method):
                old = torch.get_default_dtype()
                torch.set_default_dtype(dtype)
                try:
                    return lev_exp.gbm_smart_lev(dev, x, n, h, top, 100.0, lo_, hi_, inc, method=method)
                finally:
                    torch.set_default_dtype(old)

            case = {"grid": grid, "steps": h, "points": len(lev), "dtype": str(dtype).replace("torch.", ""),
                    "seconds": {"chain": [], "sum": []}}
            for m in ("chain", "sum"):
                timed(lambda: run(m))
            for _ in range(a.reps):
                for m in ("chain", "sum"):
                    t, _ = timed(lambda: run(m))
                    case["seconds"][m].append(t)
            best = {m: min(v) for m, v in case["seconds"].items()}
            case["best_seconds"] = best
            case["investor_steps_per_s"] = {m: n * h / t for m, t in best.items()}
            case["speedup"] = best["chain"] / best["sum"]
            case["split_ms"], case["routed"] = split(x, lev, top, dtype)
            res["cases"].append(case)
            print(json.dumps(case), file=sys.stderr)
            del x
        del x32
        torch.cuda.empty_cache()

    text = json.dumps(res, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()

"""
coin_smart_lev's per-step series: the up-move count lattice (method="counts") against the chain (the default).

  C1's smart size (1e6 investors x 3e3 flips, the 10-point grid 0.1..1.0, top = 1e-4 N), fp32 and under a
  float64 default, over the same uint8 codes; counts and chain alternating, --reps runs each after a warm-up.
  Then one instrumented run per dtype: CUDA events around each part of engine.coin_series_counts (the
  histogram pass, the statistics, the final-time chain and its row statistics, the chain series of the
  leverages that keep it) and the routed leverage count.

Writes one JSON document (stdout, or --out): wall time per run (host clock around work that ends in a device
synchronise), path-steps/s (grid points x investors x steps per second), the device name and its power limit
read in the same run.

    python tools/bench_coin_lattice.py --reps 3 --out results/bench_coin_lattice.json
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from rlmd_b200 import engine, lev_exp  # noqa: E402
from tools.bench_fp64 import device_power_limit_w, timed  # noqa: E402


def split(codes, dtype, top):
    """Per-part device time (ms) of one coin_series_counts call, restated part by part as it runs them."""
    n, h = codes.shape
    fp64 = dtype == torch.float64
    lev = (lev_exp._grid64 if fp64 else lev_exp._grid)(0.1, 1.0, 0.1, 0.5, -0.4)
    f = (lev_exp.coin_factor_table64 if fp64 else lev_exp.coin_factor_table)(lev, 0.5, -0.4)
    ev = {}

    def mark(name):
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        ev[name] = e

    mark("start")
    if fp64:
        engine.lev_final_f64("discrete", f, 100.0, top, codes)
    else:
        data_T = engine.lev_sweep("discrete", f, 100.0, outcomes=codes, mode="chain")["data_T"]
        engine.rowstats(data_T, top)
    mark("final_chain")
    k = torch.empty(n, dtype=torch.int32, device=codes.device)
    hist, kmin, kmax = engine.coin_lattice_count(codes, 0, h, k)
    mark("count")
    _, fails = engine.coin_lattice_stats(hist, kmin, kmax, 0, f, 100.0, top, n, dtype=dtype)
    mark("stats")
    rest = np.flatnonzero(fails.cpu().numpy() != 0)
    mark("route")
    if rest.size:
        engine.lev_series("discrete", f[rest], lev[rest], 100.0, top, outcomes=codes, dtype=dtype)
    mark("chain_series")
    torch.cuda.synchronize()
    names = list(ev)
    out = {b: ev[a].elapsed_time(ev[b]) for a, b in zip(names, names[1:]) if b != "route"}
    out["chain_series"] = ev["route"].elapsed_time(ev["chain_series"])
    return out, int(len(lev) - rest.size)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--investors", type=int, default=1_000_000)
    ap.add_argument("--steps", type=int, default=3000)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_coin_lattice needs a CUDA device")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    n, h = a.investors, a.steps
    top = max(1, int(n * 1e-4))
    g = len(lev_exp.param_range(0.1, 1.0, 0.1))
    res = {"device": torch.cuda.get_device_name(dev), "power_limit_w": device_power_limit_w(0),
           "investors": n, "steps": h, "grid": g, "top": top,
           "timing": "host clock around each call, device synchronised before and after; the first call of each "
           "configuration is a warm-up and not reported; split: CUDA events around each part, one run",
           "runs": [], "split_ms": {}, "routed": {}}
    codes = engine.lev_draw("discrete", n, h, seed=420, probs=(0.5, 0.5))

    def coin(dtype, method):
        old = torch.get_default_dtype()
        torch.set_default_dtype(dtype)
        try:
            return lev_exp.coin_smart_lev(dev, codes, n, h, top, 100.0, 0.5, -0.4, 0.1, 1.0, 0.1, method=method)
        finally:
            torch.set_default_dtype(old)

    configs = [(d, m) for d in (torch.float32, torch.float64) for m in ("chain", "counts")]
    for d, m in configs:
        timed(lambda: coin(d, m))
    for rep in range(a.reps):
        for d, m in configs:
            t, (data, _) = timed(lambda: coin(d, m))
            assert data.dtype == d
            res["runs"].append({"what": "coin_smart_lev", "method": m, "dtype": str(d).replace("torch.", ""),
                                "rep": rep, "seconds": t, "path_steps_per_s": g * n * h / t})
            del data
    for d in (torch.float32, torch.float64):
        name = str(d).replace("torch.", "")
        split(codes, d, top)
        res["split_ms"][name], res["routed"][name] = split(codes, d, top)
    best = {}
    for r in res["runs"]:
        key = r["dtype"] + "_" + r["method"]
        best[key] = min(best.get(key, float("inf")), r["seconds"])
    res["best_seconds"] = best
    res["speedup"] = {d: best[d + "_chain"] / best[d + "_counts"] for d in ("float32", "float64")}

    text = json.dumps(res, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()

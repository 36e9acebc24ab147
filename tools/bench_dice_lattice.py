"""
dice_smart_lev / dice_sh_smart_lev's per-step series: the count-tuple lattice (method="tuples") against the chain
(the default).

  The scripts' sizes - dice_smart_lev at 1e6 investors x 5e3 steps, dice_sh_smart_lev at 1e6 x 2e3, top = 1e-4 N -
  each at its script's 10-point grid and at 64 leverages over the same range (the chain's cost grows with the grid,
  the lattice's barely does), over the same uint8 codes; chain and tuples alternating, --reps runs each after a
  warm-up.  Then one instrumented run per configuration: CUDA events around each part of
  engine.dice_series_tuples (the bounds pass, the count passes, the statistics, the final-time chain and its row
  statistics, the chain series of the leverages that keep it) and the routed leverage count.

Writes one JSON document (stdout, or --out): wall time per run (host clock around work that ends in a device
synchronise), path-steps/s (grid points x investors x steps per second), the device name and its power limit
read in the same run.

    python tools/bench_dice_lattice.py --reps 3 --out results/bench_dice_lattice.json
"""
import argparse
import contextlib
import io
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from rlmd_b200 import engine, lev_exp  # noqa: E402
from tools.bench_fp64 import device_power_limit_w, timed  # noqa: E402

SH = (-1.0, 5.0, -1.0)
CONFIGS = [
    # (function, steps, grid (low, high) , grid points)
    ("dice_smart_lev", 5000, (0.1, 1.0), 10),
    ("dice_smart_lev", 5000, (0.1, 1.0), 64),
    ("dice_sh_smart_lev", 2000, (0.73, 1.0), 10),
    ("dice_sh_smart_lev", 2000, (0.73, 1.0), 64),
]


def grid(lo, hi, g):
    """The script's grid at 10 points (param_range with its increment), else g points evenly over [lo, hi]."""
    if g == 10:
        return lev_exp._grid(lo, hi, round((hi - lo) / 9, 2), 0.5, -0.5)
    return np.linspace(lo, hi, g).astype(np.float32)


def factors(fn, lev):
    if fn == "dice_smart_lev":
        return lev_exp.dice_factor_table(lev, 0.5, -0.5, 0.05)
    return lev_exp.dice_sh_factor_table(lev, 0.5, -0.5, 0.05, *SH)


def split(codes, f, top):
    """Per-part device time (ms) of one dice_series_tuples call, restated part by part as it runs them."""
    n, h = codes.shape
    ms = {"final_chain": 0.0, "bounds": 0.0, "count": 0.0, "stats": 0.0, "chain_series": 0.0}

    def part(name, fn):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = fn()
        b.record()
        b.synchronize()
        ms[name] += a.elapsed_time(b)
        return out

    part("final_chain", lambda: engine.rowstats(engine.lev_sweep("discrete", f, 100.0, outcomes=codes,
                                                                 mode="chain")["data_T"], top))
    ab = torch.empty((2, n), dtype=torch.int32, device=codes.device)
    bounds = part("bounds", lambda: engine.dice_lattice_bounds(codes, 0, h, ab))
    offsets, chunks = engine.dice_lattice_plan(bounds.cpu().numpy(), 256 << 20)
    off = torch.as_tensor(offsets, device=codes.device)
    hist = torch.empty(max(c for _, _, c in chunks), dtype=torch.int32, device=codes.device)
    fails = torch.zeros(f.shape[0], dtype=torch.int32, device=codes.device)
    for t0, t1, cells in chunks:
        hs = part("count", lambda: engine.dice_lattice_count(codes, t0, t1, ab, bounds[:, t0:t1], off[t0:t1], cells,
                                                             hist=hist))
        part("stats", lambda: engine.dice_lattice_stats(hs, bounds[:, t0:t1], off[t0:t1], t0, f, 100.0, top, n,
                                                        fails=fails))
    rest = np.flatnonzero(fails.cpu().numpy() != 0)
    if rest.size:
        part("chain_series", lambda: engine.lev_series("discrete", f[rest], f[rest, 0], 100.0, top, outcomes=codes))
    box_cells = int(sum(c for _, _, c in chunks))
    return ms, int(f.shape[0] - rest.size), len(chunks), box_cells


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--investors", type=int, default=1_000_000)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_dice_lattice needs a CUDA device")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    n = a.investors
    top = max(1, int(n * 1e-4))
    res = {"device": torch.cuda.get_device_name(dev), "power_limit_w": device_power_limit_w(0), "investors": n,
           "top": top, "probs": [1 / 6, 1 / 6, 2 / 3],
           "timing": "host clock around each call, device synchronised before and after; the first call of each "
           "configuration is a warm-up and not reported; split: CUDA events around each part, one run after a "
           "warm-up of the same parts", "configs": []}
    for fn, h, (lo, hi), g in CONFIGS:
        codes = engine.lev_draw("discrete", n, h, seed=420, probs=(1 / 6, 1 / 6, 2 / 3))
        lev = grid(lo, hi, g)
        f = factors(fn, lev)

        def run(method):
            # the public route: lev_series / dice_series_tuples through the shim's own _series
            with contextlib.redirect_stdout(io.StringIO()):
                if fn == "dice_smart_lev" and g == 10:
                    return lev_exp.dice_smart_lev(dev, codes, n, h, top, 100.0, 0.5, -0.5, 0.05, lo, hi,
                                                  round((hi - lo) / 9, 2), method=method)
                if fn == "dice_sh_smart_lev" and g == 10:
                    return lev_exp.dice_sh_smart_lev(dev, codes, n, h, top, 100.0, 0.5, -0.5, 0.05, *SH, lo, hi,
                                                     round((hi - lo) / 9, 2), method=method)
            return engine.lev_series("discrete", f, lev, 100.0, top, outcomes=codes, method=method)

        cfg = {"function": fn, "steps": h, "grid": g, "lev": [float(x) for x in lev], "runs": []}
        for m in ("chain", "tuples"):
            timed(lambda: run(m))
        for rep in range(a.reps):
            for m in ("chain", "tuples"):
                t, (data, _) = timed(lambda: run(m))
                assert data.shape == (g, 13, h - 1)
                cfg["runs"].append({"method": m, "rep": rep, "seconds": t, "path_steps_per_s": g * n * h / t})
                del data
        split(codes, f, top)
        cfg["split_ms"], cfg["routed"], cfg["chunks"], cfg["box_cells"] = split(codes, f, top)
        best = {m: min(r["seconds"] for r in cfg["runs"] if r["method"] == m) for m in ("chain", "tuples")}
        cfg["best_seconds"] = best
        cfg["speedup"] = best["chain"] / best["tuples"]
        cfg["count_pass_investor_steps_per_s"] = n * h / (cfg["split_ms"]["count"] * 1e-3)
        res["configs"].append(cfg)
        print(json.dumps({k: cfg[k] for k in ("function", "steps", "grid", "best_seconds", "speedup", "split_ms",
                                             "routed")}), flush=True)
        del codes

    text = json.dumps(res, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()

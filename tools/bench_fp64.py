"""
Throughput of the float64 leverage path (the reference run under a float64 default dtype).

  coin_smart_lev at C1's smart size (1e6 investors x 3e3 steps, the 10-point grid 0.1..1.0),
      fp64 and fp32 over the same uint8 codes, alternating;
  the GBM fp64 series (engine.lev_series_f64) at 1e6 x 1e3 over fp64 x, 10 grid points.

Writes one JSON document (stdout, or --out): wall time per run (host clock around work that ends in a
device synchronise), path-steps/s (grid points x investors x steps per second), the algorithmic bytes per
path-step (bytes_per_path_step below), the device name and its power limit read in the same run.

    python tools/bench_fp64.py --reps 3 --out results/bench_fp64.json
"""
import argparse
import contextlib
import io
import json
import math
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from rlmd_b200 import engine, lev_exp  # noqa: E402


def bytes_per_path_step(kind: str, dtype: torch.dtype, g: int) -> float:
    """
    HBM bytes the series moves per (grid point, investor, step): the dump of the wealth after the step
    (written once) and read by every pass of the row statistics (4 passes of 4 B in fp32, 8 passes of
    8 B in fp64), plus the outcome read shared by the grid points of one launch (uint8 codes / fp32 x once
    per grid; fp64 chain: once per tile of 8 (discrete) or 4 (GBM) points).
    """
    if dtype == torch.float64:
        pt = 8 if kind == "discrete" else 4
        outcome = (1.0 if kind == "discrete" else 8.0) * math.ceil(g / pt) / g
        return 8.0 + 8 * 8.0 + outcome
    return 4.0 + 4 * 4.0 + (1.0 if kind == "discrete" else 4.0) / g


def device_power_limit_w(index: int):
    try:
        import pynvml

        pynvml.nvmlInit()
        return pynvml.nvmlDeviceGetEnforcedPowerLimit(pynvml.nvmlDeviceGetHandleByIndex(index)) / 1000.0
    except Exception:
        pass
    try:
        out = subprocess.check_output(["nvidia-smi", "-i", str(index), "--query-gpu=power.limit",
                                       "--format=csv,noheader,nounits"], text=True)
        return float(out.strip().splitlines()[0])
    except Exception:
        return None


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    with contextlib.redirect_stdout(io.StringIO()):
        r = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--investors", type=int, default=1_000_000)
    ap.add_argument("--coin-steps", type=int, default=3000)
    ap.add_argument("--gbm-steps", type=int, default=1000)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_fp64 needs a CUDA device")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    n = a.investors
    top = max(1, int(n * 1e-4))
    res = {"device": torch.cuda.get_device_name(dev), "power_limit_w": device_power_limit_w(0),
           "investors": n, "top": top, "timing": "host clock around each call, device synchronised before and "
           "after; the first call of each configuration is a warm-up and not reported", "runs": []}

    # coin: fp32 and fp64 over the same codes, alternating
    h = a.coin_steps
    codes = engine.lev_draw("discrete", n, h, seed=420, probs=(0.5, 0.5))
    g = len(lev_exp.param_range(0.1, 1.0, 0.1))

    def coin(dtype):
        old = torch.get_default_dtype()
        torch.set_default_dtype(dtype)
        try:
            return lev_exp.coin_smart_lev(dev, codes, n, h, top, 100.0, 0.5, -0.4, 0.1, 1.0, 0.1)
        finally:
            torch.set_default_dtype(old)

    for dtype in (torch.float32, torch.float64):
        timed(lambda: coin(dtype))
    for rep in range(a.reps):
        for dtype in (torch.float32, torch.float64):
            t, (data, _) = timed(lambda: coin(dtype))
            assert data.dtype == dtype
            res["runs"].append({"what": "coin_smart_lev", "dtype": str(dtype).replace("torch.", ""), "rep": rep,
                                "grid": g, "steps": h, "seconds": t, "path_steps_per_s": g * n * h / t,
                                "bytes_per_path_step": bytes_per_path_step("discrete", dtype, g)})
            del data
    del codes
    torch.cuda.empty_cache()

    # GBM fp64 series from fp64 x
    h = a.gbm_steps
    gen = torch.Generator(device=dev).manual_seed(420)
    x = 0.036 + 0.19 * torch.randn((n, h), generator=gen, dtype=torch.float64, device=dev)
    lev = np.asarray(lev_exp.param_range(0.2, 2.0, 0.2), dtype=np.float64)

    def gbm():
        return engine.lev_series_f64("gbm", lev, lev, 100.0, top, x)

    timed(gbm)
    for rep in range(a.reps):
        t, (data, _) = timed(gbm)
        res["runs"].append({"what": "lev_series_f64 gbm", "dtype": "float64", "rep": rep, "grid": len(lev),
                            "steps": h, "seconds": t, "path_steps_per_s": len(lev) * n * h / t,
                            "bytes_per_path_step": bytes_per_path_step("gbm", torch.float64, len(lev))})
        del data

    text = json.dumps(res, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()

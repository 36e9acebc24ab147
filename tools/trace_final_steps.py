"""
A torch.profiler trace of a few steps of bench.py's flagship workload (dice, 1e6 investors x 1e4 steps as
2-bit codes, 20 leverages, top 100, one GPU, depth 1, timing events on as in the bench), and per step the
kernels' start and end on the device: whether the count kernel of step i+1 starts before step i's
tally_select_kernel ends (programmatic dependent launch, DESIGN.md §4.1).

    python tools/trace_final_steps.py OUT.json [--steps 6]

Tracing slows the host; the times it prints are not bench values.
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from rlmd_b200 import engine, lev_exp  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out")
    ap.add_argument("--steps", type=int, default=6)
    a = ap.parse_args()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    lev = np.asarray(lev_exp.param_range(*bench.GRID), dtype=np.float32)
    table = lev_exp.dice_factor_table(lev, *bench.RETURNS)
    oc = engine.lev_draw("discrete", bench.N_INVESTORS, bench.HORIZON, seed=420, probs=bench.PROBS, device=dev,
                         packed=True)
    pipe = engine.FinalSweepPipeline("discrete", table, bench.V0, bench.TOP, device=dev)
    pipe.timing = True
    for _ in range(5):
        pipe.submit(oc)
    pipe.synchronize()
    acts = [torch.profiler.ProfilerActivity.CPU, torch.profiler.ProfilerActivity.CUDA]
    with torch.profiler.profile(activities=acts) as prof:
        for _ in range(a.steps):
            pipe.submit(oc)
        pipe.synchronize()
    prof.export_chrome_trace(a.out)
    ev = json.load(open(a.out))["traceEvents"]
    kern = sorted((e for e in ev if e.get("cat") == "kernel"), key=lambda e: e["ts"])
    rows = [(e["name"].split("<")[0].split("(")[0].replace("void ", "").replace("b200::", ""), e["ts"],
             e["ts"] + e["dur"]) for e in kern]
    t0 = rows[0][1] if rows else 0.0
    for name, s, e in rows:
        print(f"{name:32s} start {s - t0:9.1f} us  end {e - t0:9.1f} us  ({e - s:6.1f} us)")
    sel = [r for r in rows if r[0] == "tally_select_kernel"]
    cnt = [r for r in rows if r[0] == "log_discrete_packed_kernel"]
    steps = [(sel[i][2], cnt[i + 1][1]) for i in range(min(len(sel), len(cnt) - 1))]   # (select i end, count i+1 start)
    print(json.dumps({"count_next_starts_before_select_ends_us": [round(e - s, 1) for e, s in steps],
                      "step_us": [round(cnt[i + 1][2] - cnt[i][2], 1) for i in range(len(cnt) - 1)]}))


if __name__ == "__main__":
    main()

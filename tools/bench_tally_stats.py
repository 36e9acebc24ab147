"""Statistics part of one tally step (finalize + statistics) timed with CUDA events, for select-kernel shapes:
B200_SELECT_CLUSTER=.. B200_SELECT_CACHE=.. python tools/bench_tally_stats.py [n_investors]"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from rlmd_b200 import engine, lev_exp, tally
n, h = int(sys.argv[1]) if len(sys.argv) > 1 else 1_000_000, 10_000
lev = np.asarray(lev_exp.param_range(0.05, 1.0, 0.05), np.float32)
f = lev_exp.dice_factor_table(lev, 0.5, -0.5, 0.05)
oc = engine.lev_draw("discrete", n, h, seed=420, probs=(1/6, 1/6, 2/3), packed=True)
t = tally.FinalTally(n)
ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
reps = 30
for radix in (False, True):      # the log-wealth route (default), then the radix route (B200_LEV_FLAG_RADIX_SELECT)
    tt = np.zeros(3)
    for it in range(reps + 3):
        ev[0].record(); t.add(oc, 3); ev[1].record(); t.finalize(); ev[2].record()
        st = t.stats(f, 100.0, h, n_total=n, top=100, radix_select=radix); ev[3].record()
        torch.cuda.synchronize()
        if it >= 3:
            tt += [ev[i].elapsed_time(ev[i + 1]) * 1e3 for i in range(3)]
    print(os.environ.get("B200_SELECT_CLUSTER"), os.environ.get("B200_SELECT_CACHE"), "radix" if radix else "log-wealth",
          "count/finalize/stats us:", (tt / reps).round(1), t.info()["bins"], "radix-route grid points:", t.info()["radix_route"])

"""Per-phase clock stamps of tally_select_kernel (library built with -DB200_TALLY_DEBUG)."""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from rlmd_b200 import engine, lev_exp, tally
n, h = 1_000_000, 10_000
lev = np.asarray(lev_exp.param_range(0.05, 1.0, 0.05), np.float32)
f = lev_exp.dice_factor_table(lev, 0.5, -0.5, 0.05)
oc = engine.lev_draw("discrete", n, h, seed=420, probs=(1/6, 1/6, 2/3), packed=True)
t = tally.FinalTally(n)
names = {
    "log-wealth": ["start", "zero+sync+wealth loop (exp, sums, histogram)", "push+sums+sync", "resolve (scan, 4 bins)+sync",
                   "gather loop+extremes", "sums+sync", "sort candidates+split+sync", "pass3 loop", "block sums", "sync"],
    "radix": ["start", "wealth+zero+sync", "pass0 loop", "push+sums+sync", "resolve0+read", "pass1 loop", "pass1 push",
              "sync", "resolve1..p2 start", "pass2 loop", "pass2 push", "sums,resolve2,read", "pass3 loop", "block sums",
              "sync"],
}
for route in ("log-wealth", "radix"):
    for it in range(3):
        t.add(oc, 3); t.finalize(); st = t.stats(f, 100.0, h, n_total=n, top=100, radix_select=route == "radix")
    torch.cuda.synchronize()
    w = t.ws[16:64].cpu().numpy()
    nm = names[route]
    for off, tag in ((0, "g=0"), (24, "g=last")):
        s = w[off:off + 24]; s = s[s != 0]
        d = np.diff(s)
        print(route, tag, "total cycles", s[-1] - s[0], [(nm[i + 1] if i + 1 < len(nm) else "?", int(x)) for i, x in enumerate(d)])
    print(t.info())

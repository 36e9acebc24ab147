"""The count kernel's SM-scaling curve: the final-time count sweep of bench.py's headline (1e6 investors x 1e4
dice rolls at 2 bits, tally sink) timed by CUDA events on k SMs, each k a green context (a per-process SM
partition; torch.cuda.GreenContext).  A sweep that still runs at the HBM rate on ~90 SMs can leave the rest to
the tally statistics beside it.

    python tools/bench_count_sms.py [--sms 148,120,100,88,60,16] [--out profiles/rNN_count_sms.json]

k = 16 is the check that the library's launches run inside the green context at all: on 16 of 148 SMs the
sweep must take well over twice as long as on all of them ("inside_green_context" in the output).
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    out = {}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        out["name"], out["power_limit"], out["sm_max_clock"] = [s.strip() for s in q.split(",")]
    except Exception as e:  # noqa: BLE001 - the numbers still stand without the card line
        out["error"] = repr(e)
    return out


def sm_clock_mhz():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=clocks.sm", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        return float(q)
    except Exception:  # noqa: BLE001
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--investors", type=int, default=1_000_000)
    ap.add_argument("--horizon", type=int, default=10_000)
    ap.add_argument("--sms", default="148,120,100,88,60,16")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=2, help="passes over the SM list (the spread across passes)")
    ap.add_argument("--label", default="")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch

    from rlmd_b200 import engine
    from rlmd_b200.tally import FinalTally

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    n, h = args.investors, args.horizon
    outcomes = engine.lev_draw("discrete", n, h, seed=420, probs=(1 / 6, 1 / 6, 2 / 3), device=dev, packed=True)
    nbytes = n * ((h + 3) // 4)
    tally = FinalTally(n, device=dev)

    def sweep():
        tally.rows = 0              # the table keeps counting the same rows; only the host bookkeeping is reset
        tally.add(outcomes, 3)

    def timed(stream):
        with torch.cuda.stream(stream):
            for _ in range(3):
                sweep()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            for _ in range(args.reps):
                sweep()
            b.record(stream)
        b.synchronize()
        return a.elapsed_time(b) / args.reps

    sms = [int(s) for s in args.sms.split(",")]
    contexts = {k: torch.cuda.GreenContext.create(num_sms=k, device_id=0) for k in sms}
    rows = {k: [] for k in sms}
    clocks = []
    for _ in range(args.rounds):
        for k in sms:
            gc = contexts[k]
            gc.set_context()
            try:
                rows[k].append(timed(gc.Stream()))
            finally:
                gc.pop_context()
            clocks.append(sm_clock_mhz())
    tally.finalize()
    torch.cuda.synchronize()

    curve = []
    for k in sms:
        best = min(rows[k])
        curve.append({"sms": k, "ms": rows[k], "best_ms": best, "tb_per_s": nbytes / (best * 1e-3) / 1e12})
    full = max(sms)
    ratio = min(rows[min(sms)]) / min(rows[full])
    res = {
        "tool": "tools/bench_count_sms.py", "label": args.label,
        "workload": f"log_discrete_packed_kernel<3, tally> over {n} x {h} 2-bit codes ({nbytes / 1e9:.2f} GB), "
                    f"CUDA events over {args.reps} launches per point, {args.rounds} passes over the SM list",
        "card": card(), "sm_mhz_samples": clocks,
        "inside_green_context": {"ms_ratio_fewest_to_most_sms": ratio, "sms": [min(sms), full],
                                 "holds": ratio > 2.0},
        "curve": curve,
    }
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()

"""
The count-lattice per-step series on investor shards - coin_series_counts(..., group=) and
dice_series_tuples(..., group=) - against the chain series (lev_series(..., group=)) over the same shards.
Weak scaling: --investors per GPU (default 1e6), one process per GPU, NCCL (a one-rank group on one GPU, so the
sharded walk and its collectives run there too).

  coin at C1's smart size: H = 3e3, G = 10 (l = 0.1 .. 1.0), top = 1e-4 N
  dice at the script's size: H = 5e3, G = 10 (l = 0.1 .. 1.0), top = 100

Per shape: a warm-up of each method, then --reps rounds alternating the sharded lattice call and the chain series
(world 1: also the one-GPU call without a group); the time of a call is the slowest rank's, host clock around
work that ends in a device synchronise, ranks lined up by a barrier before each call.  Then one instrumented run
restating the sharded walk part by part (CUDA events, slowest rank): count (the count passes; dice: and the bounds
pass), exchange (the all-reduces of the bounds / band and histograms), stats (this rank's slice of the steps and
the all-gather), chain_fallback (the sharded lev_series of unrouted leverages), data_T (the final-time chain and
its sharded row statistics).  Rank 0 writes one JSON document with the card, power limit and SM clocks.

  python tools/bench_lattice_sharded.py --out results/lattice_sharded_n1.json
  python -m torch.distributed.run --nproc-per-node 8 tools/bench_lattice_sharded.py --out ...
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from rlmd_b200 import engine, lev_exp, sharding  # noqa: E402

SHAPES = [("coin", 3000, None), ("dice", 5000, 100)]     # (kind, steps, top; None: 1e-4 of the investors)


def card(index):
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, sm_max, sm = [s.strip() for s in q.splitlines()[0].split(",")]
        return {"name": name, "power_limit": power, "sm_max_clock": sm_max, "sm_clock": sm}
    except Exception as e:  # noqa: BLE001 - the numbers still stand without the card line
        return {"name": torch.cuda.get_device_name(), "error": repr(e)}


def inputs(kind):
    lev = np.asarray(lev_exp.param_range(0.1, 1.0, 0.1), dtype=np.float32)
    if kind == "coin":
        return lev, lev_exp.coin_factor_table(lev, 0.5, -0.4), (0.5, 0.5)
    return lev, lev_exp.dice_factor_table(lev, 0.5, -0.5, 0.05), (1 / 6, 1 / 6, 2 / 3)


def slowest(x, group):
    t = torch.tensor([x], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
    return float(t.item())


def timed(fn, group):
    dist.barrier(group=group)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return slowest(time.perf_counter() - t0, group), out


def split(kind, codes, f, lev, top, n_total, group):
    """Per-part device ms of one sharded call, restated as coin_series_counts / dice_series_tuples run them."""
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    n, h = codes.shape
    dev = codes.device
    ms = {"count": 0.0, "exchange": 0.0, "stats": 0.0, "chain_fallback": 0.0, "data_T": 0.0}

    def part(name, fn):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = fn()
        b.record()
        b.synchronize()
        ms[name] += a.elapsed_time(b)
        return out

    part("data_T", lambda: engine.rowstats(engine.lev_sweep("discrete", f, 100.0, outcomes=codes, mode="chain")
                                           ["data_T"], top, n_total=n_total, group=group))
    fails = torch.zeros(f.shape[0], dtype=torch.int32, device=dev)
    cells_total = 0
    if kind == "coin":
        tc = min(h, (256 << 20) // (4 * (h + 1)))
        k = torch.empty(n, dtype=torch.int32, device=dev)
        for t0 in range(0, h, tc):
            t1 = min(h, t0 + tc)
            hs, lo, hi = part("count", lambda: engine.coin_lattice_count(codes, t0, t1, k))
            part("exchange", lambda: (dist.all_reduce(hs, group=group),
                                      dist.all_reduce(lo, op=dist.ReduceOp.MIN, group=group),
                                      dist.all_reduce(hi, op=dist.ReduceOp.MAX, group=group)))
            cells_total += hs.numel()
            s0, cnt = sharding.shard_range(t1 - t0, world, rank)
            part("stats", lambda: sharding.gather_steps(engine.coin_lattice_stats(
                hs[s0:s0 + cnt], lo[s0:s0 + cnt], hi[s0:s0 + cnt], t0 + s0, f, 100.0, top, n_total, fails=fails)[0],
                t1 - t0, group))
    else:
        ab = torch.empty((2, n), dtype=torch.int32, device=dev)
        bounds = part("count", lambda: engine.dice_lattice_bounds(codes, 0, h, ab))

        def reduce_bounds():
            lo, hi = bounds[0::2].contiguous(), bounds[1::2].contiguous()
            dist.all_reduce(lo, op=dist.ReduceOp.MIN, group=group)
            dist.all_reduce(hi, op=dist.ReduceOp.MAX, group=group)
            return torch.stack([lo[0], hi[0], lo[1], hi[1]])

        bounds = part("exchange", reduce_bounds)
        offsets, chunks = engine.dice_lattice_plan(bounds.cpu().numpy(), 256 << 20)
        off = torch.as_tensor(offsets, device=dev)
        hist = torch.empty(max(c for _, _, c in chunks), dtype=torch.int32, device=dev)
        for t0, t1, cells in chunks:
            hs = part("count", lambda: engine.dice_lattice_count(codes, t0, t1, ab, bounds[:, t0:t1], off[t0:t1],
                                                                 cells, hist=hist))
            part("exchange", lambda: dist.all_reduce(hs, group=group))
            cells_total += cells
            s0, cnt = sharding.shard_range(t1 - t0, world, rank)
            a = t0 + s0
            part("stats", lambda: sharding.gather_steps(engine.dice_lattice_stats(
                hs, bounds[:, a:a + cnt], off[a:a + cnt], a, f, 100.0, top, n_total, fails=fails)[0], t1 - t0, group))
    dist.all_reduce(fails, group=group)
    rest = np.flatnonzero(fails.cpu().numpy() != 0)
    if rest.size:
        part("chain_fallback", lambda: engine.lev_series("discrete", f[rest], lev[rest], 100.0, top, outcomes=codes,
                                                         n_total=n_total, group=group))
    return {k: slowest(v, group) for k, v in ms.items()}, int(f.shape[0] - rest.size), 4 * cells_total


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--investors", type=int, default=1_000_000, help="per GPU")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--kinds", default="coin,dice")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_lattice_sharded needs a CUDA device")
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if "RANK" not in os.environ:
        os.environ.update(RANK="0", WORLD_SIZE="1", MASTER_ADDR="127.0.0.1", MASTER_PORT="29531")
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    group = dist.group.WORLD
    world, rank = dist.get_world_size(), dist.get_rank()
    n = a.investors
    res = {"tool": "tools/bench_lattice_sharded.py", "gpus": world, "investors_per_gpu": n,
           "exchange": os.environ.get("RLMD_B200_EXCHANGE", "p2p"), "cards": [], "shapes": [],
           "timing": "host clock around each call (device synchronised, ranks barriered), slowest rank; warm-up "
           "not reported; split: CUDA events around each part of one restated run, slowest rank per part"}
    for kind, h, top in SHAPES:
        if kind not in a.kinds.split(","):
            continue
        top = top or max(1, int(n * world * 1e-4))
        lev, f, probs = inputs(kind)
        codes = engine.lev_draw("discrete", n, h, seed=17, investor_offset=rank * n, probs=probs)
        lattice = engine.coin_series_counts if kind == "coin" else engine.dice_series_tuples
        calls = {"sharded": lambda: lattice(f, lev, 100.0, top, codes, group=group),
                 "chain": lambda: engine.lev_series("discrete", f, lev, 100.0, top, outcomes=codes,
                                                    n_total=n * world, group=group)}
        if world == 1:
            calls["one_gpu"] = lambda: lattice(f, lev, 100.0, top, codes)
        for fn in calls.values():
            timed(fn, group)
        runs, clocks = {m: [] for m in calls}, []
        for _ in range(a.reps):
            for m, fn in calls.items():
                t, out = timed(fn, group)
                runs[m].append(t)
                del out
            clocks.append(card(local).get("sm_clock"))
        routed = lattice(f, lev, 100.0, top, codes, group=group)[2]
        ms, n_routed, hist_bytes = split(kind, codes, f, lev, top, n * world, group)
        cfg = {"kind": kind, "steps": h, "grid": int(f.shape[0]), "top": top, "runs_s": runs,
               "best_s": {m: min(v) for m, v in runs.items()}, "routed": int(routed.sum()),
               "split_routed": n_routed, "split_ms": ms, "histogram_bytes_per_rank": hist_bytes,
               "exchange_share": ms["exchange"] / sum(ms.values()), "sm_clock_samples": clocks}
        res["shapes"].append(cfg)
        if rank == 0:
            print(json.dumps({k: cfg[k] for k in ("kind", "best_s", "split_ms", "exchange_share", "routed")}),
                  flush=True)
        del codes
        torch.cuda.empty_cache()
    cards = [None] * world
    dist.all_gather_object(cards, card(local), group=group)
    res["cards"] = cards
    if rank == 0:
        text = json.dumps(res, indent=1)
        if a.out:
            os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
            with open(a.out, "w") as fh:
                fh.write(text + "\n")
        print(text)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()

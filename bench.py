#!/usr/bin/env python
"""
bench.py - headline benchmark of the leverage-sweep hot path (contract in the
task prompt; BASELINE.json metric "investor-steps/sec (leverage sweep)").

Workload (BASELINE.json configs[1]): lev/dice_roll.py's trinary die-roll sweep,
1e6 investors x 1e4 steps per GPU, the script's final-time grid
param_range(0.05, 1.00, 0.05) = 20 leverages, top = 100.  One "step" is one
pass of the `dice_fixed_final_lev` hot path over one synthetic outcome array:
    count kernel (log-domain sweep; its sink is the tally of outcome-count tuples)
    -> distinct tuples -> the reference's 12 summary statistics per leverage
    (weighted exact order statistics, fp64 moments); `--stats rows` runs the
    general path instead (data_T[20,N] -> 4-pass radix-select row statistics).
`value`: the outcome array is resident in HBM in the engine's packed format (2
bits per roll, `--format packed2`, the default; `--format u8` = one byte per
roll): the sweep is bound by the one read of that array, so its size is the cost.
`e2e`: the REFERENCE'S ENTRY POINT called the way lev/dice_roll.py:147-150 calls
it - rlmd_b200.lev_exp.dice_fixed_final_lev(device, outcomes, ...) with
`outcomes` an int64 [N,H] HOST tensor (pinned), stdout captured: chunked H2D of the
int64 array, ingest kernel, statistics, the printed text - PCIe-bound at 8 bytes
per roll.  The same call on uint8 / 2-bit host arrays is reported next to it.
On one GPU steps run strictly one after the other (sweep, then its statistics);
across GPUs the statistics of step i - mostly the exchange's latency - run beside
the sweep of step i+1 (engine.FinalSweepPipeline's defaults; `other_depth` reports
the other setting, `--pipeline` / `--no-pipeline` force one).
With N GPUs (one process per GPU, torchrun) every rank owns its own 1e6
investors (weak scaling); the only cross-GPU traffic is one exchange of the
ranks' distinct-tuple lists per step over NVLink peer memory.

`--workload gbm` (BASELINE.json configs[3], the north star's target): one step =
lev/gbm.py's gbm_fixed_final_lev on 1.25e7 investors x 1e4 steps per GPU (1e8
over 8 GPUs), outcomes drawn on the device (Philox4x32-10 + Box-Muller), 10
leverages, WITH the 12 statistics per leverage and the growth-rate summaries
(valid-run count, mean / median / 5th percentile) over all shards.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Prints ONE JSON line.  `--impl reference` times the reference's own CPU
implementation of the same path (torch-CPU port, all host threads) on a bounded
sample of the same workload.  `--dump-outputs DIR` writes what the last timed step
returned to its caller as DIR/<name>.npy (float64, non-finite entries 0) and
DIR/<name>_nonfinite.npy (which entries were inf / nan): `stats` [G,12], and for
`--workload gbm` also `growth`.  The inputs depend only on the arguments, so two
builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_INVESTORS = 1_000_000
HORIZON = 10_000
TOP = 100
GRID = (0.05, 1.00, 0.05)
RETURNS = (0.5, -0.5, 0.05)
PROBS = (1 / 6, 1 / 6, 2 / 3)
V0 = 100.0
METRIC = "investor-steps/sec (leverage sweep)"
UNIT = "investor-steps/s"
WORKLOAD = "lev/dice_roll.py dice_fixed_final_lev: 1e6 investors x 1e4 steps per GPU, 20 leverages, top 100"
GBM_WORKLOAD = ("lev/gbm.py gbm_fixed_final_lev: 1.25e7 investors x 1e4 steps per GPU (1e8 over 8 GPUs), "
                "10 leverages, top 1e-4 N, on-device Philox outcomes")
GBM_GRID = (-1.0, 1.0, 0.2)
GBM_SIGMA = 0.2 ** 0.5
GBM_MEAN = 0.05 - 0.2 / 2


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)), "measured"
        except Exception:
            pass
    return {"hbm_gbs": 6650.0}, "fallback"


# ------------------------------------------------------------------ CPU arm
def host_threads():
    """All host threads the CPU arm may use (torchrun exports OMP_NUM_THREADS=1: undo that for rank 0)."""
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def cpu_reference_step(n_s, h, workload="dice"):
    """One pass of the torch-CPU port over a fresh [n_s, h] outcome array in the reference's dtype."""
    import torch

    from oracle import lev_ref_port as port

    gen = torch.Generator().manual_seed(420)
    top = max(1, int(n_s * 1e-4))
    if workload == "gbm":
        x = (GBM_MEAN + GBM_SIGMA * torch.randn((n_s, h), generator=gen)).to(torch.float32)
        t0 = time.perf_counter()
        rows, levs = port.fixed_final("gbm", x, top, V0, None, GBM_GRID)
        dt = time.perf_counter() - t0
        assert len(rows) == 10
        return dt
    u = torch.rand((n_s, h), generator=gen)
    outcomes = torch.where(u < PROBS[0], 0, torch.where(u < PROBS[0] + PROBS[1], 1, 2)).to(torch.int64)
    del u
    t0 = time.perf_counter()
    rows, levs = port.fixed_final("dice", outcomes, top, V0, RETURNS, GRID)
    dt = time.perf_counter() - t0
    assert len(rows) == 20
    return dt


def run_reference(args):
    import torch

    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    torch.set_num_threads(host_threads())
    cores = torch.get_num_threads()
    h = HORIZON
    # size the per-step sample so that the whole K+W run ends within ~2.5 minutes
    probe = cpu_reference_step(200, h, args.workload)
    rate = 200 / probe  # investors per second at this horizon and grid
    budget = 150.0 / max(1, args.steps + args.warmup)
    n_s = int(max(200, min(args.ref_sample, rate * budget)))
    for _ in range(args.warmup):
        cpu_reference_step(n_s, h, args.workload)
    ts = [cpu_reference_step(n_s, h, args.workload) for _ in range(args.steps)]
    total = sum(ts)
    value = n_s * h * args.steps / total
    per_gpu = "1.25e7" if args.workload == "gbm" else "1e6"
    sample = (f"{n_s} investors x {h} steps per step (of the {per_gpu} x 1e4 per-GPU workload), "
              f"{10 if args.workload == 'gbm' else 20} leverages, torch-CPU ops on {cores} threads")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": GBM_WORKLOAD if args.workload == "gbm" else WORKLOAD, "sample": sample},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


def measure_cpu_baseline(args, torch):
    """The bounded CPU sample beside the GPU number (rank 0 only; all host threads)."""
    torch.set_num_threads(host_threads())
    n_s = args.cpu_sample if args.workload != "gbm" else max(2000, args.cpu_sample // 2)
    dt = cpu_reference_step(n_s, HORIZON, args.workload)
    fn = "gbm_fixed_final_lev" if args.workload == "gbm" else "dice_fixed_final_lev"
    return {
        "value": n_s * HORIZON / dt, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
        "sample": f"{n_s} investors x {HORIZON} steps, {10 if args.workload == 'gbm' else 20} leverages: torch-CPU "
                  f"port of {fn} (oracle/lev_ref_port.py), {dt:.1f} s",
    }


# ------------------------------------------------------------- clock sampler
class ClockSampler(threading.Thread):
    def __init__(self, index, period=0.005):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._halt = threading.Event()
        self.ok = False
        self.mark = 0
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def sample(self):
        if not self.ok:
            return
        nv = self.nv
        try:
            self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
            mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(
                nv, "nvmlDeviceGetCurrentClocksEventReasons") else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
            names = {
                0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown",
                0x4: "sw_power_cap", 0x80: "hw_power_brake_slowdown",
            }
            for bit, name in names.items():
                if mask & bit:
                    self.reasons.add(name)
        except Exception:
            pass

    def run(self):
        while not self._halt.is_set():
            self.sample()
            time.sleep(self.period)

    def begin_timed(self):
        self.mark = len(self.samples)

    def stop(self):
        self._halt.set()
        self.join(timeout=1)
        import statistics

        timed = self.samples[self.mark:]
        return {
            "sm_mhz": statistics.median(self.samples) if self.samples else None,
            "sm_max_mhz": self.max_mhz,
            "reasons": sorted(self.reasons),
            "samples": len(self.samples),
            "samples_in_timed_region": len(timed),
            "sm_mhz_timed_region": statistics.median(timed) if timed else None,
            "note": "sampled every 5 ms from the last warm-up steps (same kernels, same load) to the end of the "
                    "timed region",
        }


def dump_outputs(out_dir, **arrays):
    """
    --dump-outputs: each array as <out_dir>/<name>.npy in float64 with its non-finite entries set to 0, and
    <name>_nonfinite.npy saying what stood there: 0 finite, 1 +inf, 2 -inf, 3 nan.  The statistics follow
    the reference's fp32 arithmetic, so wealth that overflows fp32 turns means into inf and std_mean into nan;
    split like this every file is finite and two runs compare entry by entry (nan never equals nan).
    """
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a, dtype=np.float64)
        code = np.select([np.isposinf(a), np.isneginf(a), np.isnan(a)], [1.0, 2.0, 3.0], 0.0)
        np.save(os.path.join(out_dir, name + ".npy"), np.where(code == 0, a, 0.0))
        np.save(os.path.join(out_dir, name + "_nonfinite.npy"), code)


def physical_gpu_index(local_rank):
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local_rank])
        except Exception:
            return local_rank
    return local_rank


# ------------------------------------------------- the metric's other clauses
def _event_time(torch, fn, warm, reps):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) * 1e-3 / reps


def _max_over_ranks(torch, dist, dev, world, values):
    if world == 1:
        return [float(v) for v in values]
    t = torch.tensor(values, dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return [float(x) for x in t]


# lane-instructions per investor-step of log_gbm_philox_kernel (SASS count, DESIGN.md section 4) and the measured
# FP32/INT issue peak of a B200 at 1965 MHz (profiles/r01_microbench_pipes.jsonl: FFMA 3.5965e13 lane-instr/s)
GBM_INSTR_PER_STEP = 19.2
ISSUE_PEAK = 3.5965e13


def gbm_roofline(per_gpu_rate, launch_ms):
    ach = per_gpu_rate * GBM_INSTR_PER_STEP
    return {"bound": "issue", "kernel": "log_gbm_philox_kernel", "achieved": ach / 1e12, "peak": ISSUE_PEAK / 1e12,
            "unit": "T lane-instr/s", "frac": ach / ISSUE_PEAK, "traffic": None, "avg_launch_ms": launch_ms,
            "instr_per_investor_step": GBM_INSTR_PER_STEP,
            "peak_source": "measured FFMA issue rate, tools/microbench.cu (profiles/r01_microbench_pipes.jsonl); "
                           "the kernel's 2 MUFU per step also bound it at 2.3e12 steps/s (XU pipe 0.5 warp-instr/clk/SM)"}


def run_secondary(torch, dist, engine, lev_exp, np, dev, rank, world, hbm_peak, skip_gbm=False):
    """
    Side numbers for the other clauses of BASELINE.json's metric, outside the timed
    region of the headline (every rank runs them; times are the max over ranks):
    * C4: GBM leverage sweep kernel alone, on-device Philox draws, 1.25e7 investors x 1e4 steps
      per GPU (the whole step with statistics is `--workload gbm`);
    * C5: n-step replay sampling, batch 256 from a full 1e6 buffer (per call, graph replay,
      and 16384 mini-batches per launch), and the fused collector (env step + append + sample).
    """
    from rlmd_b200 import collector, envs
    from rlmd_b200.replay_torch import ReplayBufferTorch

    out = {}
    n_g, h = 12_500_000, HORIZON
    times = []
    if not skip_gbm:
        levg = np.asarray(lev_exp.param_range(*GBM_GRID), np.float32)
        buf = torch.empty((len(levg), n_g), dtype=torch.float32, device=dev)
        t = _event_time(torch, lambda: engine.lev_sweep(
            "gbm", levg, V0, n_investors=n_g, horizon=h, seed=420, investor_offset=rank * n_g, log_mean=GBM_MEAN,
            sigma=GBM_SIGMA, mode="log", out_data_T=buf, device=dev), 1, 3)
        del buf
        times.append(t)
    # C1: the coin of lev/coin_flip.py (1e6 investors x 3e3 flips, 20 leverages) at ONE bit per flip, every rank
    # its own replica (no exchange): count kernel -> tally -> statistics, like the headline
    n_c, h_c = 1_000_000, 3_000
    levc = np.asarray(lev_exp.param_range(0.05, 1.0, 0.05), np.float32)
    coin = engine.lev_draw("discrete", n_c, h_c, seed=421, investor_offset=rank * n_c, probs=(0.5, 0.5), packed=True,
                           bits=1, device=dev)
    cpipe = engine.FinalSweepPipeline("discrete", lev_exp.coin_factor_table(levc, 0.5, -0.4), V0, max(1, n_c // 10_000),
                                      device=dev, depth=1)
    coin_idx = len(times)
    times.append(_event_time(torch, lambda: cpipe.submit(coin), 5, 200))
    cpipe.synchronize()
    del coin, cpipe
    mem, batch = 1_000_000, 256
    rs = np.random.RandomState(0)
    ends = np.cumsum(rs.randint(5, 61, size=mem // 5))
    done = np.zeros(mem, dtype=bool)
    done[ends[ends < mem] - 1] = True
    base = len(times)
    BULK = 16384
    for nstep in (1, 5, 10):
        inputs = {"gpu": str(dev), "input_dims": (5,), "num_actions": 1, "mini_batch_size": batch, "discount": 0.99,
                  "multi_steps": nstep, "r_abs_zero": None, "dynamics": "M", "buffer": mem, "n_cumsteps": mem}
        rb = ReplayBufferTorch(inputs)
        st = torch.randn((mem, 5), dtype=torch.float64, device=dev)
        rb.store_batch(st, st[:, :1], 1 + 0.01 * st[:, 0], st, torch.as_tensor(done, device=dev))
        t1 = _event_time(torch, lambda: rb.sample_exp(), 5, 50)
        # bulk: BULK mini-batches per launch (one kernel: the block that draws a mini-batch gathers it); a launch of
        # 1024 x 256 samples takes less GPU time than the eager call's ~33 us of host work, so it says nothing
        # about the kernels
        tk = _event_time(torch, lambda: rb.sample_many(BULK), 2, 10)
        idx_k = rb.sample_many(BULK)[0].reshape(-1).clone()        # the same samples with the slots supplied:
        tgat = _event_time(torch, lambda: rb.sample_many(BULK, batches=idx_k), 2, 10)   # the gather kernel alone
        del idx_k
        tg = None
        if hasattr(rb, "capture_sampler"):
            run = rb.capture_sampler()
            tg = _event_time(torch, run, 5, 200)
        times += [t1, tk, tg if tg is not None else 0.0, tgat]
        del rb, st
    env = envs.Coin_InvA(1, n_envs=1, seed=1, device=dev)
    col = collector.Collector(env, 100_000, {"mini_batch_size": batch, "discount": 0.99, "multi_steps": 5,
                                             "r_abs_zero": None, "dynamics": "M"}, seed=2)
    act = torch.full((1, 1), 0.4, dtype=torch.float64, device=dev)
    run = col.capture(act, k=1)
    tc = _event_time(torch, run, 20, 2000)
    times.append(tc)
    times = _max_over_ranks(torch, dist, dev, world, times)
    if not skip_gbm:
        t = times[0]
        out["gbm_philox_sweep"] = {
            "value": world * n_g * h / t, "unit": UNIT, "ms_per_launch": t * 1e3,
            "workload": "lev/gbm.py final-time sweep kernel alone (no statistics), Philox4x32-10 + Box-Muller on "
                        "device, 1.25e7 investors x 1e4 steps per GPU, 10 leverages",
            "roofline": gbm_roofline(n_g * h / t, t * 1e3),
        }
    tcoin = times[coin_idx]
    out["coin_final_sweep_c1"] = {
        "value": n_c * h_c / tcoin, "unit": UNIT, "per_gpu": True, "ms_per_step": tcoin * 1e3,
        "workload": "lev/coin_flip.py coin_fixed_final_lev's sweep: 1e6 investors x 3e3 flips, 20 leverages, outcomes "
                    "resident as 1-bit codes (375 MB), count kernel -> tally of count tuples -> 12 statistics per leverage",
        "roofline": {"bound": "hbm", "kernel": "log_discrete_packed_kernel<2, tally sink, 1 bit> + statistics",
                     "achieved": n_c * h_c / 8 / tcoin / 1e9, "peak": hbm_peak, "unit": "GB/s",
                     "frac": n_c * h_c / 8 / tcoin / 1e9 / hbm_peak, "traffic": None,
                     "note": "whole step: ~58 us to read 375 MB of codes at the HBM peak + the statistics of the <= 3001 "
                             "count tuples (compaction + cluster select, latency-bound)"},
    }
    ns = (1, 5, 10)
    bytes_per_sample = {1: 106, 5: 114 + 4 * 4, 10: 114 + 4 * 9}   # SURVEY section 8(d)
    bulk = {n: BULK * batch / times[base + 4 * i + 1] for i, n in enumerate(ns)}
    gath = {n: BULK * batch / times[base + 4 * i + 3] for i, n in enumerate(ns)}
    out["replay_nstep_sampling"] = {
        "unit": "samples/s", "buffer": mem, "batch": batch, "per_gpu": True,
        "per_call": {str(n): batch / times[base + 4 * i] for i, n in enumerate(ns)},
        "per_call_us": {str(n): times[base + 4 * i] * 1e6 for i, n in enumerate(ns)},
        "graph_replay_us": {str(n): times[base + 4 * i + 2] * 1e6 for i, n in enumerate(ns)
                            if times[base + 4 * i + 2] > 0},
        "bulk_batches_per_launch": BULK,
        "bulk_draw_and_gather": {str(n): bulk[n] for n in ns},
        "bulk_gather_only": {str(n): gath[n] for n in ns},
        "roofline": {str(n): {"bound": "hbm", "kernel": "replay_draw_gather_kernel (gather_only: replay_gather_bulk_kernel)",
                              "achieved": bulk[n] * bytes_per_sample[n] / 1e9, "peak": hbm_peak, "unit": "GB/s",
                              "frac": bulk[n] * bytes_per_sample[n] / 1e9 / hbm_peak, "traffic": None,
                              "algorithmic_bytes_per_sample": bytes_per_sample[n],
                              "gather_only": {"achieved": gath[n] * bytes_per_sample[n] / 1e9,
                                              "frac": gath[n] * bytes_per_sample[n] / 1e9 / hbm_peak},
                              "note": "draw + gather of 16384 x 256 samples in one launch (distinct slots per mini-batch: "
                                      "Philox + a shared-memory hash set; the drawing block gathers); gather_only: the "
                                      "same samples with the slots supplied.  Random 20-byte rows of a 52 MB buffer: "
                                      "L2-resident, sector-amplified"}
                     for n in ns},
    }
    out["collector_graph_coin_invA"] = {
        "unit": "env-steps/s", "n_envs": 1, "value": 1 / times[-1], "us_per_step_store_sample": times[-1] * 1e6,
        "note": "one CUDA-graph replay = env step + replay append + 5-step sample of 256",
    }
    return out


# ------------------------------------------------------------------ GPU arm
def init_dist(torch, dist):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (rlmd_b200 has no CPU path)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    group = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        group = dist.group.WORLD
    return world, rank, local_rank, dev, group


def timed_steps(torch, dist, world, local_rank, args, step, after):
    """W warm-up steps, then exactly K timed steps between barrier + synchronize on both sides;
    device time by CUDA events, max over ranks.  The clock sampler runs from the warm-up on."""
    warm = max(args.warmup, 3)
    sampler = ClockSampler(physical_gpu_index(local_rank))
    for _ in range(warm):
        step(None)
    after()
    torch.cuda.synchronize()
    sampler.start()
    # the same steps again under the sampler for >= 0.25 s (not timed): clocks under THIS load
    t0 = time.perf_counter()
    extra = 0
    while time.perf_counter() - t0 < 0.25 and not os.environ.get("RLMD_BENCH_NO_BURN"):   # (profiling runs skip it)
        for _ in range(10):
            step(None)
        after()
        torch.cuda.synchronize()
        extra += 10
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    sampler.begin_timed()
    t_start, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_start.record()
    for i in range(args.steps):
        step(i)
    after()
    t_end.record()
    sampler.sample()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    clocks = sampler.stop()
    return t_start.elapsed_time(t_end) * 1e-3, clocks, warm + extra


def run_gpu(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    from rlmd_b200 import engine, lev_exp

    if args.workload == "gbm":
        return run_gpu_gbm(args)
    world, rank, local_rank, dev, group = init_dist(torch, dist)
    peaks, peak_kind = load_peaks()
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))

    n, h = args.investors, HORIZON
    lev = np.asarray(lev_exp.param_range(*GRID), dtype=np.float32)
    table = lev_exp.dice_factor_table(lev, *RETURNS)
    g = table.shape[0]
    top_total = TOP * world
    n_total = n * world

    # synthetic outcomes of this rank's investors, resident in HBM (2.5 GB >> 126 MB L2:
    # every step streams the whole array from DRAM again)
    packed = args.format == "packed2"
    outcomes = engine.lev_draw("discrete", n, h, seed=420, investor_offset=rank * n, probs=PROBS, device=dev,
                               packed=packed)
    row_bytes = (h + 3) // 4 if packed else h            # algorithmic bytes per investor row
    # depth 1: every sweep waits for the previous step's statistics, so a step is sweep -> statistics, one after
    # the other (--pipeline: the statistics of step i run beside the sweep of step i+1)
    depth = 2 if args.pipeline else 1 if args.no_pipeline else None       # None: the engine's default
    pipe = engine.FinalSweepPipeline("discrete", table, V0, top_total, device=dev, group=group, n_total=n_total,
                                     depth=depth, statistics=args.stats)
    depth = pipe.depth
    pipe.timing = True
    stats_holder = {}
    ev = [None] * args.steps
    cur = torch.cuda.current_stream()

    def step(i):
        stats_holder["s"] = pipe.submit(outcomes)
        if i is not None:
            ev[i] = pipe.last_sweep

    def after():
        cur.wait_stream(pipe.sweep_stream)
        cur.wait_stream(pipe.stats_stream)

    elapsed, clocks, warm_done = timed_steps(torch, dist, world, local_rank, args, step, after)
    pipe.synchronize()          # raises if the tally overflowed / a peer timed out
    sweep_s = sum(a.elapsed_time(b) for a, b in ev) * 1e-3 / args.steps
    elapsed, sweep_s = _max_over_ranks(torch, dist, dev, world, [elapsed, sweep_s])
    value = n_total * h * args.steps / elapsed
    stats = stats_holder["s"].cpu().numpy()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, stats=stats)

    # the other statistics path on the same outcomes, once: the two must agree
    other = engine.FinalSweepPipeline("discrete", table, V0, top_total, device=dev, group=group, n_total=n_total,
                                      depth=1, statistics="rows" if args.stats == "tally" else "tally")
    ref_stats = other.submit(outcomes)
    other.synchronize()
    ref_stats = ref_stats.cpu().numpy()
    fin = np.isfinite(ref_stats) & (ref_stats != 0)
    agree = {"order_statistics_identical": bool(np.array_equal(stats[:, 9:12], ref_stats[:, 9:12])),
             "max_rel_diff_moments": float(np.max(np.abs(stats[fin] - ref_stats[fin]) / np.abs(ref_stats[fin])))}
    # the pipelined rate and, for comparison, the other statistics path at depth 1
    extra_rates = {}
    for name, p in (("other_depth", None), ("other_stats_path", other)):
        if args.no_secondary:
            break
        if p is None:
            p = engine.FinalSweepPipeline("discrete", table, V0, top_total, device=dev, group=group,
                                          n_total=n_total, depth=3 - depth, statistics=args.stats)
        for _ in range(3):
            p.submit(outcomes)
        p.synchronize()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(args.steps):
            p.submit(outcomes)
        cur.wait_stream(p.sweep_stream)
        cur.wait_stream(p.stats_stream)
        b.record()
        torch.cuda.synchronize()
        dtp, = _max_over_ranks(torch, dist, dev, world, [a.elapsed_time(b) * 1e-3])
        extra_rates[name] = {"value": n_total * h * args.steps / dtp, "unit": UNIT,
                             "ms_per_step": 1e3 * dtp / args.steps, "statistics": p.statistics, "depth": p.depth}
        p.synchronize()
    del other

    # the count kernel alone (nothing beside it), after the timed region
    if args.stats == "tally":
        def alone_fn():      # the count kernel with the tally as its sink (host row bookkeeping reset each time)
            pipe.tallies[0].rows = 0
            pipe.tallies[0].add(outcomes, 3)
    else:
        alone_fn = lambda: engine.lev_sweep("discrete", table, V0, outcomes=outcomes, mode="log",   # noqa: E731
                                            out_data_T=pipe.data_T[0])
    alone_s = _event_time(torch, alone_fn, 2, 20)
    if args.stats == "tally":
        pipe.tallies[0].finalize()      # empties the table the repeats filled
        torch.cuda.synchronize()
    alone_s, = _max_over_ranks(torch, dist, dev, world, [alone_s])
    if args.stats == "tally":
        # count kernel, compaction, [merge, mark, unique,] select (profiles/r02_launches_final.csv)
        launches_per_step = 3 if world == 1 else 6
    else:
        exchange = os.environ.get("RLMD_B200_EXCHANGE", "p2p") if world > 1 else None
        # sweep + 4 x (pass, resolve); across GPUs over peer memory 4 x (pass, push, owner) + 3 waits + collect
        launches_per_step = 1 + 8 + (0 if world == 1 else 8)

    # ---- end to end through the reference's entry point
    e2e = None if args.no_e2e else measure_e2e(args, torch, dist, engine, lev_exp, np, dev, world, group, outcomes,
                                              packed, table, top_total)

    secondary = None if args.no_secondary else run_secondary(torch, dist, engine, lev_exp, np, dev, rank, world,
                                                             hbm_peak)
    cpu = None
    if rank == 0 and not args.no_cpu_baseline:
        cpu = measure_cpu_baseline(args, torch)
    if world > 1:
        dist.barrier()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    # algorithmic bytes: one read of this GPU's outcome array per launch (1/4 B per investor-step packed, 1 B as uint8)
    kernel = ("log_discrete_packed_kernel" if packed else "log_discrete_stream_kernel")
    achieved = n * row_bytes / sweep_s / 1e9
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(tpath) and n == N_INVESTORS:
        try:
            tj = json.load(open(tpath))
            traffic = (tj.get(kernel + ("_tally" if args.stats == "tally" else "")) or tj.get(kernel, {})
                       ).get("dram_bytes_per_launch")
        except Exception:
            traffic = None
    roofline = {
        "bound": "hbm", "kernel": kernel + ("<3, tally sink>" if args.stats == "tally" else "<3>"),
        "achieved": achieved, "peak": hbm_peak,
        "unit": "GB/s", "frac": achieved / hbm_peak, "traffic": traffic,
        "peak_source": f"MEASURED_PEAKS.json hbm_gbs ({peak_kind})",
        "algorithmic_bytes_per_launch": n * row_bytes, "bytes_per_investor_step": row_bytes / h,
        "avg_launch_ms": sweep_s * 1e3,
        "alone": {"avg_launch_ms": alone_s * 1e3, "achieved": n * row_bytes / alone_s / 1e9,
                  "frac": n * row_bytes / alone_s / 1e9 / hbm_peak,
                  "note": "the same launch, 20 times after the timed region"},
    }
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": warm_done, "ms_per_step": 1e3 * elapsed / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None,
        "dtype": ("2-bit codes" if packed else "u8 codes") + ", int32 counts, f64 log-wealth, f32 wealth",
        "data": "synthetic (on-device Philox4x32-10 die rolls, seed 420)",
        "config": {
            "workload": WORKLOAD, "investors_per_gpu": n, "horizon": h, "leverages": g, "top": top_total,
            "mode": {"tally": "log-domain count sweep -> tally of count tuples -> weighted exact statistics",
                     "rows": "log-domain final sweep -> data_T -> 4-pass row statistics"}[args.stats],
            "sharding": f"investors x{world}",
            "pipeline": ("depth 2: the statistics (and their cross-GPU exchange) of step i run beside the sweep of "
                         "step i+1 on a second stream" if depth == 2 else
                         "depth 1: each sweep waits for the previous step's statistics") +
                        (" (engine default: 2 across GPUs, 1 on one GPU)" if not (args.pipeline or args.no_pipeline)
                         else " (forced by flag)"),
            "statistics_exchange": "none (one GPU)" if world == 1 else
                                   ("one exchange per step: the ranks' distinct-tuple lists over NVLink peer memory"
                                    if args.stats == "tally" else "four per step (radix histograms), peer memory"),
            "outcome_format": "packed 2-bit codes (2.5 GB per GPU)" if packed else "uint8 codes (10 GB per GPU)",
            "l2": f"inputs ({n * row_bytes / 1e9:.1f} GB per GPU) exceed the 126 MB L2; no explicit flush",
        },
        "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e,
        "gpu_launches": launches_per_step * args.steps, "clocks": clocks,
        "path_steps_per_s": value * g, "other_depth": extra_rates.get("other_depth"),
        "other_stats_path": extra_rates.get("other_stats_path"), "secondary": secondary,
        "check": {"median_wealth_lev0": float(stats[0, 9]), "mean_wealth_lev0": float(stats[0, 0]),
                  "tally_vs_rows": agree},
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


def measure_e2e(args, torch, dist, engine, lev_exp, np, dev, world, group, outcomes, packed, table, top_total):
    """
    End to end through the reference's entry point: lev_exp.dice_fixed_final_lev(device, outcomes, top,
    value_0, up_r, down_r, mid_r, lev_low, lev_high, lev_incr) exactly as lev/dice_roll.py:147-150 calls
    it, `outcomes` an int64 [N,H] tensor in pinned HOST memory, stdout captured.  Inside the timed
    region: H2D of the int64 rows (two staging buffers), ingest + count, statistics, D2H of the
    statistics, formatting.  The engine-format host arrays (uint8, 2-bit) go through
    engine.lev_final_stats, the function the entry point itself calls.
    """
    import contextlib
    import io

    h = HORIZON
    n = outcomes.shape[0]
    codes = outcomes.unpack() if packed else outcomes            # uint8 [n, h] on the device

    def pinned(shape, dtype, rows):
        while True:   # halve the sample if the host refuses to pin that much
            try:
                return torch.empty((rows,) + shape, dtype=dtype, pin_memory=True), rows
            except RuntimeError:
                rows //= 2
                if rows < 1000:
                    raise

    def same_rows(rows):
        if world > 1:   # every rank must run the same sample size (the statistics are collective)
            t = torch.tensor([rows], dtype=torch.int64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            rows = int(t[0])
        return rows

    def timed(fn, steps):
        fn()      # warm-up (allocates the staging buffers / the tally)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(steps):
            fn()
        b.record()
        torch.cuda.synchronize()
        dt, = _max_over_ranks(torch, dist, dev, world, [a.elapsed_time(b) * 1e-3])
        return dt

    steps = max(1, min(args.steps, args.e2e_steps))
    out = {}
    if world > 1:
        lev_exp.set_process_group(group)
    try:
        # --- the reference's dtype: int64
        rows = min(n, args.e2e_investors)
        host, rows = pinned((h,), torch.int64, rows)
        rows = same_rows(rows)
        host = host[:rows]
        for r0 in range(0, rows, 65536):          # widen on the device in pieces, copy down
            r1 = min(rows, r0 + 65536)
            host[r0:r1].copy_(codes[r0:r1].to(torch.int64))
        torch.cuda.synchronize()
        top = TOP * world if rows == n else max(1, int(rows * world * 1e-4))
        text = io.StringIO()

        def call():
            with contextlib.redirect_stdout(text):
                lev_exp.dice_fixed_final_lev(dev, host, top, torch.tensor(V0), *RETURNS, *GRID)

        dt = timed(call, steps)
        lines = text.getvalue().splitlines()
        out = {
            "value": rows * world * h * steps / dt, "unit": UNIT, "h2d_bytes_per_step": rows * h * 8,
            "d2h_bytes_per_step": 20 * 12 * 8 + 8 * 8, "investors_per_gpu": rows, "steps": steps,
            "host_format": "int64 [N,H] (torch.distributions.Categorical.sample, lev/dice_roll.py:147-148), pinned",
            "call": "rlmd_b200.lev_exp.dice_fixed_final_lev(device, outcomes, top, value_0, up_r, down_r, mid_r, "
                    "lev_low, lev_high, lev_incr) - the reference's own signature (lev/lev_exp.py:508), stdout captured",
            "h2d_gbs_per_gpu": rows * h * 8 / (dt / steps) / 1e9,
            "printed_lines_per_call": len(lines) // (steps + 1),
            "note": "PCIe-bound: 8 bytes cross the bus per die roll in the reference's format",
        }
        # --- the platform's ceiling for this feed: the same pinned buffer copied H2D by every rank at once,
        #     nothing else running (a bare cudaMemcpyAsync loop): what the PCIe links + host memory deliver
        gib = min(host.numel() * 8, 4 << 30)
        src_b = host.view(torch.uint8).reshape(-1)[:gib]
        dst_b = torch.empty(gib, dtype=torch.uint8, device=dev)
        dtc = timed(lambda: dst_b.copy_(src_b, non_blocking=True), 4)
        out["h2d_ceiling"] = {"gbs_per_gpu": gib * 4 / dtc / 1e9, "gbs_all_gpus": world * gib * 4 / dtc / 1e9,
                              "note": f"{gib >> 20} MiB pinned -> device, {world} rank(s) at the same time, 4 copies; "
                                      "the e2e call above reaches h2d_gbs_per_gpu of it"}
        del host, src_b, dst_b
        # --- the engine's host formats through the same statistics path
        for name, width, dtype in (("uint8_host_codes", h, torch.uint8),
                                   ("packed2_host_codes", -(-((h + 3) // 4) // 16) * 16, torch.uint8)):
            hb, r2 = pinned((width,), dtype, n)
            r2 = same_rows(r2)
            hb = hb[:r2]
            if name.startswith("uint8"):
                hb.copy_(codes[:r2])
                src = hb
            else:
                pk = outcomes if packed else engine.pack_codes(codes)
                hb.copy_(pk.data[:r2, :width])
                src = engine.PackedCodes(hb, h)
            torch.cuda.synchronize()
            top2 = TOP * world if r2 == n else max(1, int(r2 * world * 1e-4))

            def call2():
                return engine.lev_final_stats(table, V0, top2, src, device=dev, group=group,
                                              n_total=r2 * world).cpu()

            dt2 = timed(call2, steps)
            out[name] = {"value": r2 * world * h * steps / dt2, "h2d_bytes_per_step": r2 * width,
                         "investors_per_gpu": r2, "h2d_gbs_per_gpu": r2 * width / (dt2 / steps) / 1e9,
                         "call": "rlmd_b200.engine.lev_final_stats(table, value_0, top, host_outcomes)"}
            del hb, src
    finally:
        if world > 1:
            lev_exp.set_process_group(None)
    return out


def run_gpu_gbm(args):
    """
    --workload gbm: lev/gbm.py's gbm_fixed_final_lev (lev/lev_exp.py:935-1005) at BASELINE's C4 size -
    1.25e7 investors x 1e4 steps per GPU (1e8 investors over 8 GPUs), outcomes drawn on the device
    (Philox4x32-10 + Box-Muller; 4 TB of fp32 returns can be resident nowhere).  One step = sweep ->
    data_T / log-wealth [10, N] -> the reference's 12 statistics per leverage over ALL shards
    (b200_rowstats, peer-memory exchange) + growth-rate summaries (valid runs, mean, median, 5th
    percentile; b200_growth_summary).
    """
    import numpy as np
    import torch
    import torch.distributed as dist

    from rlmd_b200 import engine, lev_exp

    world, rank, local_rank, dev, group = init_dist(torch, dist)
    peaks, peak_kind = load_peaks()
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    n, h = args.gbm_investors, HORIZON
    lev = np.asarray(lev_exp.param_range(*GBM_GRID), dtype=np.float32)
    g = len(lev)
    n_total, top_total = n * world, max(1, int(n * world * 1e-4))
    depth = 2 if args.pipeline else 1 if args.no_pipeline else None       # None: the engine's default (2 for GBM)
    pipe = engine.FinalSweepPipeline("gbm", lev, V0, top_total, device=dev, group=group, n_total=n_total, depth=depth)
    pipe.timing = True
    depth = pipe.depth
    holder = {}
    ev = [None] * args.steps
    cur = torch.cuda.current_stream()

    def step(i):
        holder["stats"], holder["growth"] = pipe.submit_philox(n, h, seed=420, investor_offset=rank * n,
                                                               log_mean=GBM_MEAN, sigma=GBM_SIGMA)
        if i is not None:
            ev[i] = pipe.last_sweep

    def after():
        cur.wait_stream(pipe.sweep_stream)
        cur.wait_stream(pipe.stats_stream)

    elapsed, clocks, warm_done = timed_steps(torch, dist, world, local_rank, args, step, after)
    pipe.synchronize()
    sweep_s = sum(a.elapsed_time(b) for a, b in ev) * 1e-3 / args.steps
    elapsed, sweep_s = _max_over_ranks(torch, dist, dev, world, [elapsed, sweep_s])
    value = n_total * h * args.steps / elapsed
    stats = holder["stats"].cpu().numpy()
    growth = holder["growth"].cpu().numpy()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, stats=stats, growth=growth)

    # e2e: the entry point with Philox-drawn outcomes has no host input; the host-facing call is the on-disk
    # script contract (lev_scripts.gbm): statistics and growth summaries read back to the host every step
    def e2e_call():
        step(None)
        after()
        return holder["stats"].cpu(), holder["growth"].cpu()

    e2e_call()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    e_steps = max(1, min(args.steps, args.e2e_steps))
    for _ in range(e_steps):
        s_host, g_host = e2e_call()
    b.record()
    torch.cuda.synchronize()
    dte, = _max_over_ranks(torch, dist, dev, world, [a.elapsed_time(b) * 1e-3])
    e2e = {"value": n_total * h * e_steps / dte, "unit": UNIT, "h2d_bytes_per_step": 0,
           "d2h_bytes_per_step": int(s_host.numel() * 8 + g_host.numel() * 8), "steps": e_steps,
           "note": "outcomes are drawn on the device (the reference's 4 TB fp32 array cannot exist): nothing to "
                   "copy in; the statistics and growth summaries are read back to the host every step"}
    cpu = None
    if rank == 0 and not args.no_cpu_baseline:
        cpu = measure_cpu_baseline(args, torch)
    if world > 1:
        dist.barrier()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0
    roof = gbm_roofline(n * h / sweep_s, sweep_s * 1e3)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": warm_done,
        "ms_per_step": 1e3 * elapsed / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32 draws, f32 partial sums folded into f64, f32 wealth",
        "data": "synthetic (on-device Philox4x32-10 + Box-Muller, seed 420)",
        "config": {"workload": GBM_WORKLOAD, "investors_per_gpu": n, "horizon": h, "leverages": g, "top": top_total,
                   "mu_sigma": [0.05, GBM_SIGMA], "sharding": f"investors x{world}",
                   "pipeline": f"depth {depth}: " + ("the statistics of step i (HBM-bound) run beside the sweep of step "
                               "i+1 (issue-bound) on a second stream" if depth == 2 else "sweep, then its statistics"),
                   "statistics": "12 reference statistics per leverage (radix select over all shards) + growth-rate "
                                 "summaries (valid runs, mean, 5th percentile, median)",
                   "l2": "no resident input (outcomes are generated in registers); data_T + the state [3,N] "
                         f"({(g * 4 + 24) * n / 1e9:.1f} GB per GPU) exceed the 126 MB L2"},
        "roofline": roof, "cpu_baseline": cpu, "e2e": e2e,
        "gpu_launches": args.steps * (1 + 9 + 14 + (0 if world == 1 else 8)), "clocks": clocks,
        "path_steps_per_s": value * g,
        "sweep_share_of_step": sweep_s / (elapsed / args.steps),
        "check": {"valid_runs": [int(v) for v in growth[:, 0]], "median_wealth": [float(v) for v in stats[:, 9]],
                  "growth_mean": [float(v) for v in growth[:, 1]], "growth_p05": [float(v) for v in growth[:, 6]]},
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default 2000; 10 for --workload gbm)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="dice", choices=["dice", "gbm"],
                    help="dice: BASELINE configs[1] (the headline); gbm: configs[3], 1.25e7 investors per GPU, Philox")
    ap.add_argument("--investors", type=int, default=N_INVESTORS, help="investors per GPU (dice)")
    ap.add_argument("--gbm-investors", type=int, default=12_500_000, help="investors per GPU (gbm)")
    ap.add_argument("--format", default="packed2", choices=["packed2", "u8"],
                    help="resident outcome format: 2-bit packed codes (default) or one uint8 per roll")
    ap.add_argument("--stats", default="tally", choices=["tally", "rows"],
                    help="statistics path: tally of count tuples (default) or data_T + row statistics")
    ap.add_argument("--pipeline", action="store_true",
                    help="force depth 2: the statistics of step i beside the sweep of step i+1 (two streams)")
    ap.add_argument("--no-pipeline", action="store_true",
                    help="force depth 1: steps strictly one after the other (default: the engine's choice - depth 2 "
                         "across GPUs, depth 1 on one GPU; the other depth's rate is reported as `other_depth`)")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--e2e-investors", type=int, default=250_000,
                    help="investors per GPU of the int64 end-to-end call (20 GB of pinned host memory per GPU)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the GBM-Philox / replay / collector side numbers")
    ap.add_argument("--cpu-sample", type=int, default=60_000, help="investors in the cpu_baseline sample")
    ap.add_argument("--ref-sample", type=int, default=4_000, help="investors per step of --impl reference")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 10 if args.workload == "gbm" else 2000          # a GBM step is ~100 ms
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        # the reference arm sizes its sample from a timing probe: its inputs differ from run to run
        ap.error("--dump-outputs needs --impl b200")
    if args.impl == "reference":
        return run_reference(args)
    return run_gpu(args)


if __name__ == "__main__":
    sys.exit(main())

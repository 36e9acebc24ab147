"""
Torch restatement of the per-step series contracts (*_smart_lev and
*_big_brain_lev), written op for op after oracle/lev_oracle.py so that it runs
on the CPU (pinned there against the NumPy oracle by tests/test_series_ref.py)
and on the GPU at the sizes the engine's chunked series are built for
(tests/test_series_shapes_gpu.py), where the NumPy oracle cannot go.

  smart_lev      discrete chain: w <- w * f[:, code_t] in fp32, one multiply per
                 step (bit-exact by construction: the library is built with
                 -fmad=false).
  gbm_smart_lev  GBM wealth the way the engine forms it (GbmAcc in lev_sweep.cu):
                 fp32 partial sums of x folded into an fp64 sum after every step t
                 with (t & 31) == 31, then fl32(exp(log V0 + l S_t)).  Saturation
                 follows the reference's fp32 chain: it is sticky per (leverage,
                 investor) in time order - the first of "log wealth above ln FLT_MAX"
                 (inf for good) and "below ln 2^-150" (0 for good) decides.
  big_brain      lev_oracle.big_brain over the whole grid as one [P, N] tensor per
                 step: fp32 for coin; fp64 wealth for dice, with fp64 or fp32
                 leverage as the retention branch dictates.

Statistics are taken one step at a time (`step_stats`): torch.sort, lower medians,
fp64 mean / MAD / std with lev_oracle.group_stats' non-finite rules, then
engine.stats_to_reference_dtype.  Nothing larger than one step's [rows, N] is ever
held in fp64.
"""
from __future__ import annotations

import math

import numpy as np
import torch

LOG_FLT_MAX = 88.72283905206835      # ln(FLT_MAX)
LOG_FLT_ZERO = -103.97207708399179   # ln(2^-150): below it fp32 rounds to 0


def _group_moments(v64: torch.Tensor):
    """(mean, mad, std) of every row of a finite fp64 [R, n] block, population std."""
    mean = v64.mean(dim=1)
    dev = v64 - mean[:, None]
    return mean, dev.abs().mean(dim=1), dev.square().mean(dim=1).sqrt()


def step_stats(v: torch.Tensor, top: int) -> torch.Tensor:
    """
    The 12 statistics (lev_oracle.STAT_ROWS order) of every row of v [R, N] (fp32 or
    fp64) as float64 [R, 12], before the cast to the reference's dtype.
    Groups: all, the `top` largest, the rest.  A group holding a non-finite value
    has mean nan (its element when it has only one), MAD and std nan; a group
    holding a nan has median nan (lev_oracle.group_stats).
    """
    r, n = v.shape
    a = torch.sort(v, dim=1).values           # ascending; nan sorts last, i.e. into the top group
    out = torch.empty((r, 12), dtype=torch.float64, device=v.device)
    nan = float("nan")
    groups = ((0, n), (n - top, n), (0, n - top))
    for j, (lo, hi) in enumerate(groups):
        g = a[:, lo:hi]
        size = hi - lo
        finite = torch.isfinite(g).all(dim=1)
        has_nan = torch.isnan(g).any(dim=1)
        g64 = g.to(torch.float64)
        mean, mad, std = _group_moments(torch.where(finite[:, None], g64, torch.zeros_like(g64)))
        bad_mean = g64[:, 0] if size == 1 else torch.full_like(mean, nan)
        out[:, 0 + j] = torch.where(finite, mean, bad_mean)
        out[:, 3 + j] = torch.where(finite, mad, torch.full_like(mad, nan))
        out[:, 6 + j] = torch.where(finite, std, torch.full_like(std, nan))
        med = g64[:, (size - 1) // 2]
        out[:, 9 + j] = torch.where(has_nan, torch.full_like(med, nan), med)
    return out


def reference_stats(v: torch.Tensor, top: int) -> torch.Tensor:
    """step_stats cast to the reference's dtype (fp32, with its fp32 MAD overflow)."""
    from rlmd_b200 import engine
    return engine.stats_to_reference_dtype(step_stats(v, top), v.shape[1], top)


# -------------------------------------------------------------------- discrete
def discrete_chain(codes: torch.Tensor, factors, value_0: float):
    """
    Yields (t, w) for t = 0..H-1: the fp32 wealth [G, N] after step t of the
    sequential chain ((V0 m_0) m_1) ... on codes' device (codes: uint8 [N, H]).
    """
    dev = codes.device
    f = torch.as_tensor(np.ascontiguousarray(factors, dtype=np.float32), device=dev)
    g = f.shape[0]
    n, h = codes.shape
    w = torch.full((g, n), float(np.float32(value_0)), dtype=torch.float32, device=dev)
    for t in range(h):
        w = w * f[:, codes[:, t].long()]
        yield t, w


def smart_lev(codes: torch.Tensor, factors, lev_row, top: int, value_0: float):
    """Discrete *_smart_lev: data [G,13,H-1] fp32 and data_T [G,N] fp32 on codes' device."""
    return _series(discrete_chain(codes, factors, value_0), codes.shape[1], lev_row, top, codes.device)


# ------------------------------------------------------------------------- GBM
def gbm_wealth(x: torch.Tensor, lev, value_0: float):
    """
    Yields (t, w) for t = 0..H-1: the engine's GBM wealth [G, N] fp32 after step t
    (x: fp32 [N, H] log-returns), with the reference's sticky saturation.
    """
    dev = x.device
    n, h = x.shape
    l64 = torch.as_tensor(np.asarray(lev, dtype=np.float32).astype(np.float64), device=dev)[:, None]
    log_v0 = math.log(float(np.float32(value_0)))
    base = torch.zeros(n, dtype=torch.float64, device=dev)     # folded fp64 sum
    p = torch.zeros(n, dtype=torch.float32, device=dev)        # fp32 partial sum since the last fold
    over = torch.zeros((l64.shape[0], n), dtype=torch.bool, device=dev)
    under = torch.zeros_like(over)
    inf = torch.tensor(float("inf"), dtype=torch.float32, device=dev)
    zero = torch.tensor(0.0, dtype=torch.float32, device=dev)
    for t in range(h):
        p = p + x[:, t]
        s = base + p.to(torch.float64)
        lw = l64 * s[None, :] + log_v0
        free = ~(over | under)
        over |= free & (lw > LOG_FLT_MAX)
        under |= free & (lw < LOG_FLT_ZERO)
        w = torch.where(over, inf, torch.where(under, zero, torch.exp(lw).to(torch.float32)))
        if (t & 31) == 31:
            base, p = s, torch.zeros_like(p)
        yield t, w


def gbm_smart_lev(x: torch.Tensor, lev, top: int, value_0: float):
    """GBM *_smart_lev: data [G,13,H-1] fp32 and data_T [G,N] fp32 on x's device."""
    return _series(gbm_wealth(x, lev, value_0), x.shape[1], lev, top, x.device)


def _series(steps, h: int, lev_row, top: int, dev):
    lev_row = torch.as_tensor(np.asarray(lev_row, dtype=np.float32), device=dev)
    data = torch.zeros((lev_row.shape[0], 13, max(h - 1, 0)), dtype=torch.float32, device=dev)
    data[:, 12, :] = lev_row[:, None]
    w = None
    for t, w in steps:
        if t >= 1:
            data[:, :12, t - 1] = reference_stats(w, top)
    return data, w


# ------------------------------------------------------------------ big brain
def _opt_lev_f32(v, v0, vmin, eta32, roll):
    """lev_oracle._opt_lev_f32 over [P, N] fp32 with per-point vmin / roll [P, 1] (fp32)."""
    lev0 = eta32 * (1.0 - vmin / v)
    floor_ = torch.where(v <= v0, vmin, v0 + roll * (v - v0))
    return torch.where(roll == 0, lev0, eta32 * (1.0 - floor_ / v))


def big_brain(kind: str, codes: torch.Tensor, top: int, value_0: float, returns, lev_factor: float, stop_grid,
              roll_grid):
    """
    lev_oracle.big_brain on codes' device: data [R,S,26,H-1] fp32 and the final
    wealth [R,S,N] (fp32 for coin, fp64 for dice).  returns = (up, down) for coin
    (code 1 up, 0 down), (up, down, mid) for dice (codes 0, 1, 2).
    """
    dev = codes.device
    n, h = codes.shape
    f32, f64 = torch.float32, torch.float64
    stop = np.asarray(stop_grid, dtype=np.float32)
    roll = np.asarray(roll_grid, dtype=np.float32)
    R, S = len(roll), len(stop)
    v0 = np.float32(value_0)
    eta64, eta32 = float(lev_factor), np.float32(lev_factor)
    # point p = j * S + i (retention outer, stop-loss inner)
    vmin_np = np.tile((stop * v0).astype(np.float32), R)
    roll_np = np.repeat(roll, S).astype(np.float32)
    lev0_np = np.array([float(eta64) * float(np.float32(np.float32(1) - np.float32(vm / v0))) for vm in vmin_np])
    vmin = torch.as_tensor(vmin_np, device=dev)[:, None]
    rollp = torch.as_tensor(roll_np, device=dev)[:, None]
    v0_t = torch.tensor(float(v0), dtype=f32, device=dev)
    eta32_t = torch.tensor(float(eta32), dtype=f32, device=dev)
    coin = kind == "coin"
    if coin:
        rv = torch.tensor([np.float32(returns[1]), np.float32(returns[0])], dtype=f32, device=dev)   # by code
    else:
        rv = torch.tensor([float(r) for r in returns[:3]], dtype=f64, device=dev)
    zero_roll = rollp == 0

    def opt(v):
        if coin:
            return _opt_lev_f32(v, v0_t, vmin, eta32_t, rollp)
        l64 = eta64 * (1.0 - vmin.to(f64) / v)
        l32 = _opt_lev_f32(v.to(f32), v0_t, vmin, eta32_t, rollp).to(f64)
        return torch.where(zero_roll, l64, l32)

    P = R * S
    data = torch.zeros((P, 26, max(h - 1, 0)), dtype=f32, device=dev)
    data[:, 24, :] = torch.as_tensor(np.tile(stop, R), device=dev)[:, None]
    data[:, 25, :] = rollp
    g = rv[codes[:, 0].long()][None, :]
    if coin:
        lev0 = torch.as_tensor(lev0_np.astype(np.float32), device=dev)[:, None]
        v = v0_t * (1.0 + lev0 * g)
    else:
        lev0 = torch.as_tensor(lev0_np, device=dev)[:, None]
        v = float(v0) * (1.0 + lev0 * g)
    lev = opt(v)
    for t in range(h - 1):
        data[:, 12:24, t] = reference_stats(lev, top)
        g = rv[codes[:, t + 1].long()][None, :]
        v = v * (1.0 + lev * g)
        lev = opt(v)
        data[:, 0:12, t] = reference_stats(v, top)
    return data.view(R, S, 26, max(h - 1, 0)), v.view(R, S, n)

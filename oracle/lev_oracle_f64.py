"""
TEST INFRASTRUCTURE ONLY - NumPy restatement of the reference's coin and GBM
leverage sweeps when it runs under torch.set_default_dtype(torch.float64)
(SURVEY.md section 8c, App. C "all-fp64 run").  Only tests/ may import this file;
the product (rlmd_b200/) never does.

For the coin and GBM every value is then float64: the grid T.tensor(param_range(...)),
the factors 1 + lev*r / exp(lev*x), the sequential chain value = value_0 * m[:,0];
value = value * m[:,t] (lev/lev_exp.py:160-212, :1042-1093) and the statistics.  One
IEEE fp64 rounding per operation, as torch-CPU performs it.  The fp32 restatements
and the statistic block live in oracle/lev_oracle.py.
"""
from __future__ import annotations

import numpy as np

from oracle.lev_oracle import group_stats, param_range, summary_stats


def lev_grid_f64(low: float, high: float, incr: float, up_r=None, down_r=None) -> np.ndarray:
    """float64 grid; negated iff -down_r > up_r (never for GBM: pass None)."""
    g = np.asarray(param_range(low, high, incr), dtype=np.float64)
    if up_r is not None and -down_r > up_r:
        g = -g
    return g


def coin_factors_f64(lev: np.ndarray, up_r: float, down_r: float) -> np.ndarray:
    """[G,2] float64, column = outcome value (0 -> down, 1 -> up)."""
    lev = np.asarray(lev, dtype=np.float64)
    return np.stack([1.0 + lev * down_r, 1.0 + lev * up_r], axis=1)


def chain_discrete_f64(outcomes: np.ndarray, factors: np.ndarray, value_0: float, keep_steps=False):
    """
    Sequential fp64 product per (grid point, investor).  keep_steps: False, True (every
    t = 1..H-1) or a collection of steps t to keep; returns data_T [G,N] and, when asked,
    a dict {t: [G,N] wealth after step t}.
    """
    oc = np.asarray(outcomes).astype(np.int64)
    n, h = oc.shape
    f = np.asarray(factors, dtype=np.float64)
    w = np.full((f.shape[0], n), float(value_0))
    steps = {}
    for t in range(h):
        w = w * f[:, oc[:, t]]
        if _keep(keep_steps, t):
            steps[t] = w.copy()
    return (w, steps) if keep_steps is not False else w


def chain_gbm_f64(x: np.ndarray, lev: np.ndarray, value_0: float, keep_steps=False):
    """GBM: factor = exp(l * x) in fp64; then the same sequential fp64 chain (keep_steps as above)."""
    x = np.asarray(x, dtype=np.float64)
    n, h = x.shape
    lev = np.asarray(lev, dtype=np.float64)
    w = np.full((lev.shape[0], n), float(value_0))
    steps = {}
    with np.errstate(over="ignore", invalid="ignore"):
        for t in range(h):
            w = w * np.exp(lev[:, None] * x[None, :, t])
            if _keep(keep_steps, t):
                steps[t] = w.copy()
    return (w, steps) if keep_steps is not False else w


def _keep(keep_steps, t: int) -> bool:
    if keep_steps is False:
        return False
    if keep_steps is True:
        return t >= 1
    return t in keep_steps


def summary_stats_f64(v: np.ndarray, top: int) -> np.ndarray:
    """summary_stats, with torch's answer for an empty adj group (top == n): nan mean / MAD / std / median."""
    v = np.asarray(v, dtype=np.float64)
    if top < v.shape[0]:
        return summary_stats(v, top)
    out = np.full(12, np.nan)
    mean, mad, std, med = group_stats(v)
    for gi in range(2):
        out[0 + gi], out[3 + gi], out[6 + gi], out[9 + gi] = mean, mad, std, med
    return out


def smart_lev_f64(outcomes, factors_or_lev, lev, top, value_0, gbm=False, steps=True):
    """
    Restates *_smart_lev under a float64 default: data [G,13,H-1] float64 (columns of the
    steps not in `steps` stay nan when `steps` is a subset of 1..H-1), data_T [G,N] float64.
    """
    chain = chain_gbm_f64 if gbm else chain_discrete_f64
    data_T, kept = chain(outcomes, factors_or_lev, value_0, keep_steps=steps)
    g, h = data_T.shape[0], np.asarray(outcomes).shape[1]
    data = np.full((g, 13, max(h - 1, 0)), np.nan)
    with np.errstate(over="ignore", invalid="ignore"):
        for t, w in kept.items():
            for gi in range(g):
                data[gi, :12, t - 1] = summary_stats_f64(w[gi], top)
    if h > 1:
        data[:, 12, :] = np.asarray(lev, dtype=np.float64)[:, None]
    return data, data_T


def fixed_final_lev_f64(outcomes, factors_or_lev, top, value_0, gbm=False) -> np.ndarray:
    """Restates *_fixed_final_lev under a float64 default (sequential product): [G,12] statistics."""
    w = chain_gbm_f64(outcomes, factors_or_lev, value_0) if gbm else \
        chain_discrete_f64(outcomes, factors_or_lev, value_0)
    with np.errstate(over="ignore", invalid="ignore"):
        return np.stack([summary_stats_f64(w[gi], top) for gi in range(w.shape[0])])

"""
TEST INFRASTRUCTURE ONLY (never imported by rlmd_b200/): a NumPy restatement of the
running log-return sum route the GPU takes for gbm_smart_lev(..., method="sum")
(rlmd_b200/csrc/gbm_sum.cu), pinned on the CPU against the reference's GBM fixtures
(tests/golden/lev_gbm_*.npz) and the per-investor statistics of oracle/lev_oracle.py.

  S_t    : an investor's running sum of log-returns after step t.  float32 x: 32 steps
           summed in fp32 on top of an fp64 base, S_t = base + (double)p, folded into the
           base after every step t with (t & 31) == 31 (GbmAcc, csrc/lev_kernels.cuh);
           float64 x: the sequential fp64 sum
  wealth : exp(log V0 + l S_t) in fp64, rounded to fp32 in fp32 mode (log V0 of the fp32
           V0, l the fp32 leverage there) - the series chain's wealth when it does not saturate
  route  : fp32, the chain saturates (inf above ln FLT_MAX, 0 below ln 2^-150) exactly when
           log V0 + l max S > ln FLT_MAX or log V0 + l min S < ln 2^-150 (swapped for l < 0),
           the extremes over every investor and step including the start value 0; fp64, both
           extreme paths strictly inside (DBL_MIN, DBL_MAX) with a margin of 1e-3 in log space
  stats  : lev_oracle.summary_stats of the closed-form wealth
"""
import math

import numpy as np

from . import lev_oracle as lo
from .lev_oracle_f64 import summary_stats_f64

F32 = np.float32
LOG_FLT_MAX = 88.72283905206835
LOG_FLT_ZERO = -103.97207708399179
ROUTE_MARGIN = 1e-3


def running_sum(x: np.ndarray) -> np.ndarray:
    """S float64 [H, N]: the S after every step (float32 x: with the fp32 partial sums and 32-step folds)."""
    x = np.asarray(x)
    n, h = x.shape
    if x.dtype == np.float64:
        return np.cumsum(x, axis=1).T.copy()
    x = x.astype(F32)
    out = np.empty((h, n))
    base = np.zeros(n)
    p = np.zeros(n, dtype=F32)
    for t in range(h):
        p = (p + x[:, t]).astype(F32)
        out[t] = base + p.astype(np.float64)
        if (t & 31) == 31:
            base = base + p.astype(np.float64)
            p = np.zeros(n, dtype=F32)
    return out


def log_v0(value_0: float, f32: bool) -> float:
    return math.log(float(F32(value_0)) if f32 else float(value_0))


def route_ok(S: np.ndarray, lev, value_0: float, f32: bool) -> np.ndarray:
    """bool [G]: which leverages take the running-sum statistics, from the S rows of every step."""
    lev = np.asarray(lev, dtype=F32 if f32 else np.float64).astype(np.float64)
    if not np.isfinite(S).all():
        return np.zeros(lev.shape[0], dtype=bool)
    smax, smin = max(float(S.max()), 0.0), min(float(S.min()), 0.0)
    lv0 = log_v0(value_0, f32)
    out = np.zeros(lev.shape[0], dtype=bool)
    for i, l in enumerate(lev):
        hi = lv0 + (l * smax if l >= 0 else l * smin)
        lo_ = lv0 + (l * smin if l >= 0 else l * smax)
        if f32:
            out[i] = not (hi > LOG_FLT_MAX) and not (lo_ < LOG_FLT_ZERO)
        else:
            out[i] = lo_ > math.log(np.finfo(np.float64).tiny) + ROUTE_MARGIN and \
                hi < math.log(np.finfo(np.float64).max) - ROUTE_MARGIN
    return out


def wealth(S_t: np.ndarray, l: float, value_0: float, f32: bool, exp=np.exp) -> np.ndarray:
    """The closed-form wealth of one leverage at one step; `exp` evaluates exp on fp64 arrays."""
    l = float(F32(l)) if f32 else float(l)
    with np.errstate(over="ignore"):
        e = exp(log_v0(value_0, f32) + l * np.asarray(S_t, dtype=np.float64))
    return e.astype(F32) if f32 else e


def sum_stats(S_t: np.ndarray, lev, value_0: float, top: int, f32: bool = True, exp=np.exp) -> np.ndarray:
    """float64 [G, 12]: the 12 statistics of every leverage's wealth at one step."""
    stats = summary_stats_f64 if not f32 else lo.summary_stats
    with np.errstate(over="ignore", invalid="ignore"):
        return np.stack([stats(wealth(S_t, l, value_0, f32, exp), top) for l in np.asarray(lev).reshape(-1)])

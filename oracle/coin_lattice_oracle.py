"""
TEST INFRASTRUCTURE ONLY (never imported by rlmd_b200/): a NumPy restatement of the
up-move count lattice the GPU takes for coin_smart_lev(..., method="counts")
(rlmd_b200/csrc/coin_lattice.cu), pinned on the CPU against the reference's fixtures
(tests/golden/lev_coin_*.npz) and the per-investor statistics of oracle/lev_oracle.py.

  k_t       : an investor's up-moves in steps 0..t (inclusive); wealth after step t is
              V0 u^k d^(t+1-k) at every leverage, monotone in k
  hist      : hist[t][k] = investors with k_t = k; kmin[t] / kmax[t] the occupied band
  value     : exp(log V0 + k log u + (t+1-k) log d) in fp64, rounded to fp32 in fp32
              mode (log V0 of the fp32 V0 there); the same expression, evaluated left to
              right, as the kernel's
  route     : a leverage takes the lattice only if its factors are > 0 and both extreme
              paths (kmin[t], kmax[t]) stay strictly inside (MIN, MAX) of the dtype's normal
              range with a margin of 1e-3 in log space at EVERY step: the fp32 / fp64 chain
              saturates path by path (inf and 0 absorb), the closed form does not
  statistics: lev_oracle.summary_stats of the per-investor lattice values
"""
import math

import numpy as np

from . import lev_oracle as lo
from .lev_oracle_f64 import summary_stats_f64

F32 = np.float32
ROUTE_MARGIN = 1e-3
_RANGE = {True: (float(np.finfo(np.float32).tiny), float(np.finfo(np.float32).max)),
          False: (float(np.finfo(np.float64).tiny), float(np.finfo(np.float64).max))}


def up_counts(codes: np.ndarray) -> np.ndarray:
    """[N,H] int64: k_t per investor and step (code 1 = up, codes taken modulo 2)."""
    return np.cumsum(np.asarray(codes).astype(np.int64) & 1, axis=1)


def lattice_hist(codes: np.ndarray, t_begin: int = 0, t_end=None):
    """(hist int64 [T, H+1], kmin [T], kmax [T], k_end [N]) of steps [t_begin, t_end);
    k_end is every investor's k after step t_end - 1 (0 when the range is empty)."""
    k = up_counts(codes)
    n, h = k.shape
    t_end = h if t_end is None else int(t_end)
    rows = range(int(t_begin), t_end)
    hist = np.zeros((len(rows), h + 1), dtype=np.int64)
    for i, t in enumerate(rows):
        hist[i] = np.bincount(k[:, t], minlength=h + 1)
    kmin = np.array([k[:, t].min() for t in rows], dtype=np.int64)
    kmax = np.array([k[:, t].max() for t in rows], dtype=np.int64)
    k_end = k[:, t_end - 1] if t_end > 0 else np.zeros(n, dtype=np.int64)
    return hist, kmin, kmax, k_end


def lattice_logs(factors: np.ndarray, value_0: float, f32: bool):
    """(log V0, log u [G], log d [G]) in fp64; factors [G,2] = (down, up) as the sweep holds them.  The C
    library's log (math.log), as the engine takes it; nan for a factor <= 0."""
    f = np.asarray(factors, dtype=np.float32 if f32 else np.float64).astype(np.float64)
    v0 = float(F32(value_0)) if f32 else float(value_0)
    logs = np.array([[math.log(x) if x > 0 else math.nan for x in row] for row in f]).reshape(-1, 2)
    return math.log(v0), logs[:, 1], logs[:, 0]


def lattice_values(lv0: float, lu: float, ld: float, t: int, k: np.ndarray, f32: bool, exp=np.exp) -> np.ndarray:
    """fp64 wealth of the investors with k up-moves after step t.  `exp` maps an fp64 array to its
    exponentials: the GPU tests pass the device's, whose last ulp can differ from NumPy's."""
    k = np.asarray(k, dtype=np.float64)
    x = lv0 + k * lu + (t + 1 - k) * ld
    v = np.asarray(exp(x), dtype=np.float64)
    if f32:
        with np.errstate(over="ignore"):
            v = v.astype(np.float32).astype(np.float64)
    return v


def route_ok(factors: np.ndarray, value_0: float, kmin: np.ndarray, kmax: np.ndarray, t_begin: int,
             f32: bool) -> np.ndarray:
    """bool [G]: the leverages that may take the lattice over the steps t_begin + i of kmin / kmax."""
    lv0, lu, ld = lattice_logs(factors, value_0, f32)
    lo_, hi_ = _RANGE[f32]
    lo_, hi_ = math.log(lo_) + ROUTE_MARGIN, math.log(hi_) - ROUTE_MARGIN
    f = np.asarray(factors, dtype=np.float64)
    ok = (f > 0).all(axis=1)
    t = np.arange(int(t_begin), int(t_begin) + len(kmin))
    for g in range(f.shape[0]):
        if not ok[g]:
            continue
        ends = [lv0 + kk * lu[g] + (t + 1 - kk) * ld[g] for kk in (np.asarray(kmin), np.asarray(kmax))]
        ok[g] = bool(np.all(np.minimum(*ends) > lo_) and np.all(np.maximum(*ends) < hi_))
    return ok


def lattice_stats(hist: np.ndarray, t_begin: int, factors: np.ndarray, value_0: float, top: int, f32: bool,
                  exp=np.exp) -> np.ndarray:
    """float64 [G, T, 12]: summary_stats of the per-investor lattice values of every leverage and step."""
    lv0, lu, ld = lattice_logs(factors, value_0, f32)
    g_n, t_n = len(lu), hist.shape[0]
    out = np.empty((g_n, t_n, 12))
    k_all = np.arange(hist.shape[1])
    with np.errstate(over="ignore", invalid="ignore"):
        for i in range(t_n):
            occ = hist[i] > 0
            k, c = k_all[occ], hist[i][occ]
            for g in range(g_n):
                v = np.repeat(lattice_values(lv0, lu[g], ld[g], int(t_begin) + i, k, f32, exp), c)
                out[g, i] = lo.summary_stats(v, top) if top < v.shape[0] else summary_stats_f64(v, top)
    return out

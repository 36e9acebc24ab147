"""
TEST INFRASTRUCTURE ONLY (never imported by rlmd_b200/): a NumPy restatement of the
count-tuple lattice the GPU takes for dice_smart_lev / dice_sh_smart_lev(..., method="tuples")
(rlmd_b200/csrc/dice_lattice.cu), pinned on the CPU against the reference's fixtures
(tests/golden/lev_dice*.npz) and the per-investor statistics of oracle/lev_oracle.py.

  (a_t, b_t) : an investor's up-moves (code 0) and down-moves (code 1) in steps 0..t
               (inclusive); c_t = t+1-a-b mid-moves (code 2); wealth after step t is
               V0 u^a d^b m^c at every leverage
  cells      : the (a, b) occupied at step t with their investor counts; the bounds
               amin/amax/bmin/bmax of step t are those of its occupied cells, and its box
               [amax-amin+1][bmax-bmin+1] is the histogram the kernels fill (row-major, a major)
  x          : log V0 + a log u + b log d + c log m in fp64, left to right (logs of the fp32 V0
               and factors); the cell's wealth is fl32(exp(x)), monotone in x
  route      : a leverage takes the lattice only if its three factors are > 0 and, at EVERY
               step, the min and the max of x over the occupied cells lie strictly inside
               (ln FLT_MIN, ln FLT_MAX) with a margin of 1e-3: the fp32 chain saturates path
               by path (inf and 0 absorb), the closed form does not
  statistics : lev_oracle.summary_stats of the per-investor cell values
"""
import math

import numpy as np

from . import lev_oracle as lo
from .lev_oracle_f64 import summary_stats_f64

F32 = np.float32
ROUTE_MARGIN = 1e-3
LW_LO = math.log(float(np.finfo(np.float32).tiny)) + ROUTE_MARGIN
LW_HI = math.log(float(np.finfo(np.float32).max)) - ROUTE_MARGIN


def tuple_counts(codes: np.ndarray):
    """([N,H], [N,H]) int64: a_t and b_t per investor and step."""
    c = np.asarray(codes)
    return np.cumsum(c == 0, axis=1, dtype=np.int64), np.cumsum(c == 1, axis=1, dtype=np.int64)


def lattice_bounds(codes: np.ndarray, t_begin: int = 0, t_end=None):
    """(bounds int64 [4, T] = amin, amax, bmin, bmax of steps [t_begin, t_end), ab_end int64 [2, N]):
    ab_end is every investor's (a, b) after step t_end - 1."""
    a, b = tuple_counts(codes)
    t_end = a.shape[1] if t_end is None else int(t_end)
    sl = slice(int(t_begin), t_end)
    bounds = np.stack([a[:, sl].min(0), a[:, sl].max(0), b[:, sl].min(0), b[:, sl].max(0)])
    return bounds, np.stack([a[:, t_end - 1], b[:, t_end - 1]])


def step_box(codes_ab, t: int) -> np.ndarray:
    """int64 [amax-amin+1, bmax-bmin+1]: investors per (a, b) at step t; codes_ab = tuple_counts(codes)."""
    a, b = codes_ab[0][:, t], codes_ab[1][:, t]
    wb = b.max() - b.min() + 1
    flat = np.bincount((a - a.min()) * wb + (b - b.min()), minlength=(a.max() - a.min() + 1) * wb)
    return flat.reshape(-1, wb)


def cells(codes_ab, t: int):
    """(a, b, count) of the cells occupied at step t."""
    box = step_box(codes_ab, t)
    ia, ib = np.nonzero(box)
    return ia + codes_ab[0][:, t].min(), ib + codes_ab[1][:, t].min(), box[ia, ib]


def lattice_logs(factors: np.ndarray, value_0: float):
    """(log V0, log u [G], log d [G], log m [G]) in fp64 of the fp32 factors [G,3] (columns = codes 0 up, 1 down,
    2 mid) and the fp32 V0; the C library's log (math.log), as the engine takes it; nan for a factor <= 0."""
    f = np.asarray(factors, dtype=np.float32).astype(np.float64)
    logs = np.array([[math.log(x) if x > 0 else math.nan for x in row] for row in f]).reshape(-1, 3)
    return math.log(float(F32(value_0))), logs[:, 0], logs[:, 1], logs[:, 2]


def cell_x(lv0: float, lu: float, ld: float, lm: float, t: int, a, b) -> np.ndarray:
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return lv0 + a * lu + b * ld + (t + 1 - a - b) * lm


def cell_values(x, exp=np.exp) -> np.ndarray:
    """fl32(exp(x)) as fp64.  `exp` maps an fp64 array to its exponentials: the GPU tests pass the device's,
    whose last ulp can differ from NumPy's."""
    with np.errstate(over="ignore"):
        return np.asarray(exp(np.asarray(x, dtype=np.float64)), dtype=np.float64).astype(np.float32).astype(np.float64)


def route_ok(factors: np.ndarray, value_0: float, codes: np.ndarray) -> np.ndarray:
    """bool [G]: the leverages that may take the lattice over every step of the codes."""
    lv0, lu, ld, lm = lattice_logs(factors, value_0)
    ok = (np.asarray(factors, dtype=np.float64) > 0).all(axis=1)
    ab = tuple_counts(codes)
    for t in range(ab[0].shape[1]):
        a, b, _ = cells(ab, t)
        for g in np.flatnonzero(ok):
            x = cell_x(lv0, lu[g], ld[g], lm[g], t, a, b)
            ok[g] = x.min() > LW_LO and x.max() < LW_HI
    return ok


def lattice_stats(codes: np.ndarray, steps, factors: np.ndarray, value_0: float, top: int,
                  exp=np.exp) -> np.ndarray:
    """float64 [G, len(steps), 12]: summary_stats of the per-investor cell values of every leverage and step."""
    lv0, lu, ld, lm = lattice_logs(factors, value_0)
    ab = tuple_counts(codes)
    steps = list(steps)
    out = np.empty((len(lu), len(steps), 12))
    with np.errstate(over="ignore", invalid="ignore"):
        for i, t in enumerate(steps):
            a, b, c = cells(ab, t)
            for g in range(len(lu)):
                v = np.repeat(cell_values(cell_x(lv0, lu[g], ld[g], lm[g], t, a, b), exp), c)
                out[g, i] = lo.summary_stats(v, top) if top < v.shape[0] else summary_stats_f64(v, top)
    return out

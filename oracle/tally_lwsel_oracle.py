"""
TEST INFRASTRUCTURE ONLY (never imported by rlmd_b200/): a NumPy restatement of the
log-wealth route of tally_select_kernel (rlmd_b200/csrc/tally.cu), pinned against the
sort-based order statistics of oracle/tally_oracle.py.

  log wealth  : the kernel's fp64 expression per bin (n_k = 0 terms skipped); it is linear
                in the count tuple, so over the (n_1, n_2) box of the bin list it lies
                between the values at the box's corners (K <= 3, finite log factors)
  bins        : NBINS equal bins of log wealth over that range - ordered by wealth, since
                fl32(exp(.)) is monotone
  selection   : the weighted histogram of the bins gives each target rank's bin and the rank
                left inside it; the bin's tuples sorted by (fp32 key, count) give the value
  checks      : no key below a target's bin above the target and none above it below; at most
                CAND tuples in a target's bin.  For thr (ascending rank n - K) strictly, since the
                sums beside its bin are taken as > thr / < thr - unless thr is 0 or +inf, whose
                copies beside its bin are counted as its ties.  A failed check means the
                radix route (None here)
"""
import math

import numpy as np

NBINS = 2048
CAND = 512
KEY_ZERO, KEY_INF = 0x80000000, 0xFF800000     # float_key(0.0), float_key(inf)


def float_key(w: np.ndarray) -> np.ndarray:
    """common.cuh float_key: the order-preserving map fp32 -> uint32 (NaN greatest)."""
    b = np.ascontiguousarray(w, dtype=np.float32).view(np.uint32).astype(np.uint64)
    k = np.where(b & 0x80000000, ~b & 0xFFFFFFFF, b | 0x80000000)
    k = np.where((b & 0x7FFFFFFF) > 0x7F800000, 0xFFFFFFFF, k)
    return k.astype(np.uint64)


def log_wealth(tuples: np.ndarray, lm: np.ndarray, value_0: float) -> np.ndarray:
    """[B] fp64: log V0 + sum_k n_k log m_k, added in k order, n_k = 0 terms skipped."""
    lw = np.full(tuples.shape[0], math.log(float(np.float32(value_0))))
    for k in range(tuples.shape[1]):
        nk = tuples[:, k].astype(np.float64)
        with np.errstate(invalid="ignore"):
            lw = lw + np.where(nk > 0, nk * lm[k], 0.0)
    return lw


def lw_range(tuples: np.ndarray, lm: np.ndarray, value_0: float):
    """(lo, hi) of the linear log wealth over the (n_1, n_2) box of the list, or None: the radix route."""
    k = tuples.shape[1]
    if k > 3 or len(tuples) == 0 or not np.isfinite(lm).all():
        return None
    h = float(tuples[0].sum())
    a = (int(tuples[:, 1].min()), int(tuples[:, 1].max()))
    b = (int(tuples[:, 2].min()), int(tuples[:, 2].max())) if k == 3 else (0, 0)
    logv0 = math.log(float(np.float32(value_0)))
    vals = []
    for n2 in b:
        for n1 in a:
            v = logv0 + (h - n1 - n2) * lm[0] + n1 * lm[1]
            if k == 3:
                v += n2 * lm[2]
            vals.append(v)
    lo, hi = min(vals), max(vals)
    return (lo, hi) if hi > lo and math.isfinite(hi - lo) else None


def select(lw: np.ndarray, wealth: np.ndarray, counts: np.ndarray, rng, top: int, cand: int = CAND):
    """The fp32 values at ascending ranks (n-1)//2, n-K, n-K+(K-1)//2, (n-K-1)//2 and the number of
    investors above thr, from the log-wealth bins over `rng`; None where a check fails."""
    n, k = int(counts.sum()), int(top)
    lo, hi = rng
    t = (lw - lo) * (NBINS / (hi - lo))
    b = np.where(t >= NBINS - 1, NBINS - 1, np.where(t > 0, np.floor(np.where(t > 0, t, 0)), 0)).astype(np.int64)
    pre = np.cumsum(np.bincount(b, weights=counts, minlength=NBINS).astype(np.int64))
    keys = float_key(wealth)
    out = []
    for j, rk in enumerate(((n - 1) // 2, n - k, n - k + (k - 1) // 2, (n - k - 1) // 2)):
        bq = int(np.searchsorted(pre, rk, side="right"))
        rem = rk - (int(pre[bq - 1]) if bq > 0 else 0)
        inb, below, above = b == bq, b < bq, b > bq
        if int(inb.sum()) > cand:
            return None
        ck, cc = keys[inb], counts[inb]
        order = np.lexsort((cc, ck))
        ck, cc = ck[order], cc[order]
        v = int(ck[np.searchsorted(np.cumsum(cc), rem, side="right")])
        lo_max = int(keys[below].max()) if below.any() else 0
        hi_min = int(keys[above].min()) if above.any() else 0xFFFFFFFF
        apart = v in (KEY_ZERO, KEY_INF) or lo_max < v < hi_min
        if not lo_max <= v <= hi_min or (j == 1 and not apart):
            return None
        out.append(v)
        if j == 1:
            b1 = bq
    # investors above thr as the kernel counts them: the bins above thr's, where +inf / 0 are ties if thr is
    # +inf / 0, and the tuples of thr's bin above it
    thr, above = out[1], b > b1
    sat = (keys == KEY_INF) | (keys == KEY_ZERO)
    n_gt = int(counts[above & ~sat].sum()) + int(counts[(b == b1) & (keys > thr)].sum())
    for key in (KEY_INF, KEY_ZERO):
        if thr != key:
            n_gt += int(counts[above & (keys == key)].sum())
    vals = np.array(out, dtype=np.uint64)
    return key_float(vals), n_gt


def key_float(k: np.ndarray) -> np.ndarray:
    """common.cuh key_float: the inverse of float_key."""
    k = np.asarray(k, dtype=np.uint64)
    b = np.where(k & 0x80000000, k & 0x7FFFFFFF, ~k & 0xFFFFFFFF)
    b = np.where(k == 0xFFFFFFFF, 0x7FC00000, b)
    return b.astype(np.uint32).view(np.float32)

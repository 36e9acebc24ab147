"""
The log-wealth route of the tally statistics on the CPU (oracle/tally_lwsel_oracle.py): where its
checks pass, the four target values and the top / rest split are those of a full sort of the bins;
where they fail (non-finite log factors, a flat grid point, wealth out of order with the log-wealth
bins, an overfull bin) the grid point is sent to the radix route.
"""
import numpy as np
import pytest

import golden_io
from oracle import tally_lwsel_oracle as lws
from oracle import tally_oracle as to
from test_oracle_tally import DISCRETE, factors_of


def by_sort(wealth, counts, top):
    """(values at the four target ranks, investors above thr) from a full sort."""
    n, k = int(counts.sum()), int(top)
    keys = lws.float_key(wealth)
    o = np.argsort(keys, kind="stable")
    cum = np.cumsum(counts[o])
    at = [int(keys[o][np.searchsorted(cum, r, side="right")])
          for r in ((n - 1) // 2, n - k, n - k + (k - 1) // 2, (n - k - 1) // 2)]
    return lws.key_float(np.array(at, dtype=np.uint64)), int(counts[keys > at[1]].sum())


def route(tuples, counts, lm, v0, top, wealth=None, cand=lws.CAND):
    rng = lws.lw_range(tuples, lm, v0)
    if rng is None:
        return None
    lw = lws.log_wealth(tuples, lm, v0)
    if wealth is None:
        with np.errstate(over="ignore"):
            wealth = np.exp(lw).astype(np.float32)
    return lws.select(lw, wealth, counts, rng, top, cand)


def check_grid(tuples, counts, f, v0, top):
    """Every grid point: the route's answer (where it applies) against the sort; returns how many took it."""
    with np.errstate(divide="ignore"):
        lm = np.log(f.astype(np.float64))
    w = to.bin_wealth(tuples, f, v0)
    taken = 0
    for g in range(f.shape[0]):
        got = route(tuples, counts, lm[g], v0, top)
        if got is None:
            continue
        taken += 1
        want = by_sort(w[g], counts, top)
        assert np.array_equal(got[0].view(np.uint32), want[0].view(np.uint32)) and got[1] == want[1], (g, got, want)
        st = to.stats_from_bins(w[g], counts, top)
        assert np.array_equal(got[0][[0, 2, 3]].astype(np.float64), st[9:12])
    return taken


@pytest.mark.parametrize("case", DISCRETE, ids=lambda c: c["name"])
def test_route_equals_the_sort_on_every_fixture(case):
    oc = golden_io.draw_outcomes(case)
    f = factors_of(case)
    tuples, counts = to.bins_of(oc, f.shape[1])
    taken = check_grid(tuples, counts, f, case["v0"], case["top"])
    with np.errstate(divide="ignore"):
        finite = np.isfinite(np.log(f.astype(np.float64))).all(axis=1).sum()
    assert taken >= finite // 2, (taken, finite)


@pytest.mark.parametrize("top", [1, 2, 7, 39, 40, 41, 199])
def test_ties_zero_and_inf_rows(top):
    """test_oracle_tally's tie / inf / zero rows: factor 0 (log -inf) and a flat row take the radix route."""
    rs = np.random.RandomState(top)
    oc = rs.choice(3, size=(200, 12), p=[0.2, 0.2, 0.6]).astype(np.uint8)
    oc[:40] = oc[0]
    f = np.float32([[1.5, 0.5, 1.05], [3.0e30, 0.0, 1.0], [1.0, 1.0, 1.0], [2.0, 0.0, 1.0], [3.0e30, 0.5, 1.0]])
    tuples, counts = to.bins_of(oc, 3)
    check_grid(tuples, counts, f, 100.0, top)
    with np.errstate(divide="ignore"):
        lm = np.log(f.astype(np.float64))
    for g in (1, 2, 3):
        assert route(tuples, counts, lm[g], 100.0, top) is None


@pytest.mark.parametrize("seed", range(6))
def test_random_tuple_sets_and_the_fall_back(seed):
    """Non-iid tuple sets with random counts and factors (K = 2 and 3, wealth over- and underflowing fp32);
    wealth shuffled against the log wealth or an overfull bin must be refused, never answered wrongly."""
    rs = np.random.RandomState(seed)
    k = 2 if seed % 3 == 0 else 3
    h = int(rs.randint(20, 3000))
    m = int(rs.randint(50, 4000))
    n1 = rs.randint(0, h // 2, size=m)
    n2 = rs.randint(0, h // 2, size=m) if k == 3 else np.zeros(m, np.int64)
    tup = np.stack([h - n1 - n2, n1] + ([n2] if k == 3 else []), axis=1)
    tuples, first = np.unique(tup, axis=0, return_index=True)
    tuples = tuples[np.argsort(first)]
    counts = rs.randint(1, 50, size=len(tuples)).astype(np.int64)
    counts[rs.randint(len(tuples))] = 5000                       # one heavy tuple: ties at the targets
    f = np.exp(rs.uniform(-0.3, 0.3, size=(12, k)) * rs.choice([0.01, 0.3, 3.0], size=(12, 1))).astype(np.float32)
    n = int(counts.sum())
    for top in (1, int(rs.randint(2, n - 1)), n - 1):
        check_grid(tuples, counts, f, 100.0, top)
    lm = np.log(f[0].astype(np.float64))
    refused = 0
    for _ in range(5):
        lw = lws.log_wealth(tuples, lm, 100.0)
        with np.errstate(over="ignore"):
            w = np.exp(lw).astype(np.float32)
        rs.shuffle(w)                                            # wealth no longer follows the log wealth
        got = lws.select(lw, w, counts, lws.lw_range(tuples, lm, 100.0), 3)
        if got is None:
            refused += 1
            continue
        want = by_sort(w, counts, 3)
        assert np.array_equal(got[0].view(np.uint32), want[0].view(np.uint32)) and got[1] == want[1]
    assert refused > 0
    assert route(tuples, counts, lm, 100.0, 3, cand=0) is None   # a target's bin holds more tuples than fit


def test_flagship_shape_takes_the_route_at_every_leverage():
    """1e6 investors x 1e4 die rolls, the bench's 20 leverages and top 100: above leverage 0.1 the best
    investors' wealth overflows fp32 (thr = +inf with copies in many bins) - still the log-wealth route."""
    from rlmd_b200 import lev_exp
    rs = np.random.RandomState(0)
    tuples, counts = np.unique(rs.multinomial(10_000, [1 / 6, 1 / 6, 2 / 3], size=1_000_000), axis=0,
                               return_counts=True)
    lev = np.asarray(lev_exp.param_range(0.05, 1.0, 0.05), np.float32)
    f = lev_exp.dice_factor_table(lev, 0.5, -0.5, 0.05)
    assert check_grid(tuples, counts.astype(np.int64), f, 100.0, 100) == len(lev)

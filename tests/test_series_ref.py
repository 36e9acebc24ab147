"""
Pins the torch restatement of the per-step series (tests/series_ref.py) on the
CPU against the NumPy oracle (oracle/lev_oracle.py) on the fixtures' inputs, so
that tests/test_series_shapes_gpu.py can use it as the reference at sizes the
oracle cannot reach.  CPU only.
"""
import numpy as np
import pytest
import torch

import golden_io
import series_ref
from oracle import lev_oracle as lo
from test_oracle_bigbrain import assert_bigbrain_close
from test_oracle_lev import assert_stats_close, oracle_inputs

def u32(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def stat_columns(case):
    """Every step of the small cases; the fixture's kept columns of the long ones."""
    if case["n"] * case["h"] <= 1_000_000:
        return list(range(case["h"] - 1))
    return golden_io.kept_columns(case)


def oracle_stats(steps, cols, top):
    """lev_oracle.summary_stats of steps[t] ([G,N]) at the columns t-1 in cols -> [G,12,len(cols)] fp32."""
    from rlmd_b200 import engine
    g, n = steps[-1].shape
    out = np.zeros((g, 12, len(cols)), dtype=np.float32)
    with np.errstate(all="ignore"):
        for j, c in enumerate(cols):
            st = np.stack([lo.summary_stats(steps[c + 1][gi], top) for gi in range(g)])
            out[:, :, j] = engine.stats_to_reference_dtype(st, n, top)
    return out


DISCRETE = [c for c in golden_io.LEV_CASES if c["kind"] != "gbm"]
GBM = [c for c in golden_io.LEV_CASES if c["kind"] == "gbm"]


@pytest.mark.parametrize("case", DISCRETE, ids=lambda c: c["name"])
def test_discrete_series_matches_oracle(case):
    oc, f, lev, _ = oracle_inputs(case)
    want_T, steps = lo.chain_discrete(oc, f, case["v0"], keep_steps=True)
    steps = [None] + steps                       # steps[t]: the wealth after step t (t >= 1)
    codes = torch.as_tensor(oc)
    got = [w.clone() for _, w in series_ref.discrete_chain(codes, f, case["v0"])]
    for t in range(1, case["h"]):
        assert np.array_equal(u32(got[t].numpy()), u32(steps[t])), t
    data, data_T = series_ref.smart_lev(codes, f, lev, case["top"], case["v0"])
    assert np.array_equal(u32(data_T.numpy()), u32(want_T))
    cols = stat_columns(case)
    want = oracle_stats(steps, cols, case["top"])
    data = data.numpy()
    assert np.array_equal(data[:, 12], np.broadcast_to(lev[:, None], data[:, 12].shape))
    sel = data[:, :12, cols]
    assert np.array_equal(u32(sel[:, 9:12]), u32(want[:, 9:12])), "order statistics must be bit-exact"
    assert_stats_close(sel[:, :9], want[:, :9], rtol=3e-7, noise=1e-12)


TINY = 1e-30


def assert_gbm_wealth_close(got, want, h):
    """
    got / want: the wealth after steps 1..H-1 ([G,N] each).  The same inf pattern at
    every step; relative 1e-5 max(1, H/500) while the fp32 chain has stayed above
    1e-30; below it both must be below 2e-30 (0 included).  The chain is no
    yardstick among denormals: a factor above 1/2 rounds 2^-149 back to 2^-149, so
    the chain can hold the smallest denormal for good where log wealth has long
    passed ln 2^-150, and a chain that climbs back out has lost its digits there
    (both seen in gbm_overflow at l = 2, and under exp(-0.5) per step).
    """
    been_low = np.zeros(want[0].shape, dtype=bool)
    for t, (a, b) in enumerate(zip(got, want)):
        assert np.array_equal(np.isinf(a), np.isinf(b)), t
        assert not np.isnan(a).any()
        low = b < TINY
        been_low |= low
        ok = np.isfinite(b) & ~been_low
        if ok.any():
            rel = np.abs(a[ok].astype(np.float64) - b[ok]) / b[ok]
            assert rel.max() <= 1e-5 * max(1.0, h / 500), (t, rel.max())
        assert (a[low] < 2 * TINY).all(), t


@pytest.mark.parametrize("case", GBM, ids=lambda c: c["name"])
def test_gbm_series_matches_oracle_chain(case):
    oc, _, lev, _ = oracle_inputs(case)
    want_T, steps = lo.chain_gbm(oc, lev, case["v0"], keep_steps=True)
    steps = [None] + steps
    got = [w.clone().numpy() for _, w in series_ref.gbm_wealth(torch.as_tensor(oc), lev, case["v0"])]
    assert_gbm_wealth_close(got[1:], steps[1:], case["h"])
    data, data_T = series_ref.gbm_smart_lev(torch.as_tensor(oc), lev, case["top"], case["v0"])
    assert np.array_equal(u32(data_T.numpy()), u32(got[-1]))
    # the statistics of the restated wealth: order statistics bit-exact, moments close
    cols = stat_columns(case)
    want = oracle_stats(got, cols, case["top"])
    sel = data.numpy()[:, :12, cols]
    assert np.array_equal(u32(sel[:, 9:12]), u32(want[:, 9:12]))
    assert_stats_close(sel[:, :9], want[:, :9], rtol=3e-7, noise=1e-12)


def sticky_paths(h=600):
    """
    Deterministic +-1 log-return paths.  Row 0 falls for 150 steps, then climbs for
    450: at l = 1, V0 = 100 the fp32 chain underflows to 0 at step 108 and stays
    there, although log wealth passes ln FLT_MAX again from step 384 on.  Row 1 is
    its mirror image (inf from step 84 for good), rows 2-3 only fall / climb,
    row 4 stays flat, rows 5-7 are small seeded draws.
    """
    x = np.zeros((8, h), dtype=np.float32)
    x[0, :150], x[0, 150:] = -1, 1
    x[1, :150], x[1, 150:] = 1, -1
    x[2], x[3] = -1, 1
    rs = np.random.RandomState(17)
    x[5:] = (-0.05 + 0.447 * rs.standard_normal((3, h))).astype(np.float32)
    return x


STICKY_LEV = np.float32([-1.0, -0.5, 0.5, 1.0])


def test_gbm_saturation_is_sticky_in_time_order():
    x = sticky_paths()
    h = x.shape[1]
    want_T, steps = lo.chain_gbm(x, STICKY_LEV, 100.0, keep_steps=True)
    steps = [None] + steps
    got = [w.clone().numpy() for _, w in series_ref.gbm_wealth(torch.as_tensor(x), STICKY_LEV, 100.0)]
    assert_gbm_wealth_close(got[1:], steps[1:], h)
    for t in range(1, h):
        # at l = +-1 every factor is e^-1 < 1/2 on the way down: the chain reaches 0 exactly where the rule does
        assert np.array_equal(got[t][[0, 3]] == 0, steps[t][[0, 3]] == 0), t
    g1 = 3                                                 # l = 1
    w0 = np.stack([w[g1, 0] for w in got])
    assert (w0[:108] > 0).all() and (w0[108:] == 0).all()   # 0 from step 108 to the end
    w1 = np.stack([w[g1, 1] for w in got])
    assert np.isfinite(w1[:84]).all() and np.isinf(w1[84:]).all()
    # l = -1 sees the mirror images
    assert np.array_equal(np.stack([w[0, 1] for w in got]) == 0, w0 == 0)


@pytest.mark.parametrize("case", golden_io.BIGBRAIN_CASES, ids=lambda c: c["name"])
def test_big_brain_matches_oracle(case):
    oc = golden_io.draw_outcomes(case)
    returns = (case["up_r"], case["down_r"]) + ((case["mid_r"],) if case["kind"] == "dice" else ())
    stop, roll = lo.param_range(*case["stop"]), lo.param_range(*case["roll"])
    eta = golden_io.bigbrain_lev_factor(case)
    want, want_w = lo.big_brain(case["kind"], oc, case["top"], case["v0"], returns, eta, stop, roll,
                                want_wealth=True)
    data, w = series_ref.big_brain(case["kind"], torch.as_tensor(oc), case["top"], case["v0"], returns, eta, stop,
                                   roll)
    w = w.numpy()
    if case["kind"] == "coin":
        assert w.dtype == np.float32 and np.array_equal(u32(w), u32(want_w.astype(np.float32)))
    else:
        assert w.dtype == np.float64 and np.array_equal(w.view(np.uint64), want_w.view(np.uint64))
    data = data.numpy()
    assert_bigbrain_close(data, want)
    for base in (0, 12):
        assert_stats_close(data[:, :, base:base + 9], want[:, :, base:base + 9], rtol=3e-7, noise=1e-12)


def test_step_stats_non_finite_rules():
    """inf / nan / 0 rows follow lev_oracle.group_stats, one-element top groups included."""
    inf, nan = np.inf, np.nan
    rows = np.float32([
        [1, 2, 3, 4, 5, 6],
        [inf, 2, 3, 4, 5, 6],
        [inf, inf, inf, inf, inf, inf],
        [0, 0, 0, 0, 0, 7],
        [0, 0, 0, 0, 0, 0],
        [nan, 1, 2, 3, inf, 0],
        [2, 1, 2, 1, 2, 1],
    ])
    from rlmd_b200 import engine
    for top in (1, 2, 5):
        got = series_ref.reference_stats(torch.as_tensor(rows), top).numpy()
        with np.errstate(all="ignore"):
            want = engine.stats_to_reference_dtype(np.stack([lo.summary_stats(r, top) for r in rows]), 6, top)
        assert np.array_equal(np.isnan(got), np.isnan(want))
        fin = ~np.isnan(want)
        np.testing.assert_allclose(got[fin], want[fin], rtol=1e-7, atol=0)

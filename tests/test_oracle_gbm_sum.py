"""
Pins oracle/gbm_sum_oracle.py - the running log-return sum behind gbm_smart_lev(..., method="sum") -
against the reference's GBM fixtures, at the drop-in tolerances of tests/test_lev_dropin_gpu.py.  CPU only.
"""
import numpy as np
import pytest

import golden_io
from oracle import gbm_sum_oracle as gs
from oracle import lev_oracle as lo
from test_oracle_lev import assert_stats_close

GBM_CASES = [c for c in golden_io.LEV_CASES if c["kind"] == "gbm"]
# leverages whose fp32 chain underflows to 0 for some investor: they keep the chain
CHAIN_LEVERAGES = {"gbm_overflow": [0.8, 1.4, 2.0]}


def test_running_sum_folds_every_32_steps():
    rs = np.random.RandomState(5)
    x = (rs.standard_normal((7, 97)) * 0.3).astype(np.float32)
    S = gs.running_sum(x)
    for t in (0, 30, 31, 32, 63, 64, 96):
        base = x[:, :(t + 1) // 32 * 32].astype(np.float64)
        want = np.zeros(7)
        for b in range(0, base.shape[1], 32):     # fold per tile: fp32 partial sum, then fp64 add
            p = np.zeros(7, dtype=np.float32)
            for j in range(b, b + 32):
                p = (p + x[:, j]).astype(np.float32)
            want = want + p.astype(np.float64)
        p = np.zeros(7, dtype=np.float32)
        for j in range((t + 1) // 32 * 32, t + 1):
            p = (p + x[:, j]).astype(np.float32)
        want = want + p.astype(np.float64)
        assert np.array_equal(S[t], want)
    x64 = x.astype(np.float64)
    assert np.array_equal(gs.running_sum(x64)[-1], np.cumsum(x64, axis=1)[:, -1])


@pytest.mark.parametrize("case", GBM_CASES, ids=lambda c: c["name"])
def test_route_decisions(case):
    x = golden_io.draw_outcomes(case)
    lev = lo.lev_grid(*case["grid"])
    ok = gs.route_ok(gs.running_sum(x), lev, case["v0"], True)
    assert [round(float(v), 6) for v in lev[~ok]] == CHAIN_LEVERAGES.get(case["name"], [])
    # the rule is exact: a routed leverage's fp32 chain never saturates, an unrouted one does
    _, steps = lo.chain_gbm(x, lev, case["v0"], keep_steps=True)
    for g in range(lev.shape[0]):
        sat = any(((w[g] == 0) | np.isinf(w[g])).any() for w in steps)
        assert sat == (not ok[g])


@pytest.mark.parametrize("case", GBM_CASES, ids=lambda c: c["name"])
def test_routed_statistics_meet_the_reference(case):
    x = golden_io.draw_outcomes(case)
    gold = golden_io.load("lev_" + case["name"], x)
    lev = lo.lev_grid(*case["grid"])
    S = gs.running_sum(x)
    ok = gs.route_ok(S, lev, case["v0"], True)
    steps = np.asarray(gold["cols"]) + 1           # column c of data holds step c + 1
    got = np.stack([gs.sum_stats(S[t], lev[ok], case["v0"], case["top"]) for t in steps], 2)   # [G, 12, cols]
    want = gold["data"][ok, :12]
    got = got.astype(np.float32)
    if case["name"] != "gbm_overflow":
        assert_stats_close(got, want, rtol=2e-5 * max(1.0, case["h"] / 500))
    else:
        normal = np.abs(want) > 1e-30
        assert_stats_close(np.where(normal, got, 0), np.where(normal, want, 0), rtol=2e-4)
    assert np.array_equal(lev[ok], gold["data"][ok, 12, 0])


def test_float64_route_keeps_far_leverages_on_the_chain():
    """Under a float64 default the range is wide: GBM at H = 4000 stays inside it up to l = 2.0."""
    case = golden_io.lev_case("gbm_overflow")
    x = golden_io.draw_outcomes(case).astype(np.float64)
    lev = np.asarray(lo.lev_grid(*case["grid"]), dtype=np.float64)
    assert gs.route_ok(gs.running_sum(x), lev, case["v0"], False).all()
    big = np.array([2.0, 5.0])
    assert gs.route_ok(gs.running_sum(x), big, case["v0"], False).tolist() == [True, False]

"""
Pins oracle/dice_lattice_oracle.py - the count-tuple lattice behind dice_smart_lev /
dice_sh_smart_lev(..., method="tuples") - against the reference's dice fixtures.  CPU only.
"""
import numpy as np
import pytest

import golden_io
from oracle import dice_lattice_oracle as dl
from oracle import lev_oracle as lo
from test_oracle_coin_lattice import assert_lattice_close, lattice_tol

DICE_CASES = [c for c in golden_io.LEV_CASES if c["kind"] in ("dice", "dice_sh")]
# leverages whose occupied cells leave fp32's normal range at some step: they keep the chain
CHAIN_LEVERAGES = {"dicesh_testscale": [0.5]}


def case_factors(case):
    lev = lo.lev_grid(*case["grid"], case["up_r"], case["down_r"])
    if case["kind"] == "dice":
        return lev, lo.dice_factors(lev, case["up_r"], case["down_r"], case["mid_r"])
    return lev, lo.dice_sh_factors(lev, case["up_r"], case["down_r"], case["mid_r"], *case["sh"])


def test_bounds_and_boxes_equal_cumsum_counts():
    rs = np.random.RandomState(5)
    for n, h in ((1, 1), (5, 2), (77, 33), (300, 97)):
        oc = rs.choice(3, size=(n, h), p=[0.2, 0.3, 0.5]).astype(np.uint8)
        a = np.cumsum(oc == 0, axis=1)
        b = np.cumsum(oc == 1, axis=1)
        ab = dl.tuple_counts(oc)
        for t0, t1 in ((0, h), (h // 3, h), (0, max(1, h // 2))):
            bounds, ab_end = dl.lattice_bounds(oc, t0, t1)
            assert bounds.shape == (4, t1 - t0)
            assert np.array_equal(ab_end, np.stack([a[:, t1 - 1], b[:, t1 - 1]]))
            for i, t in enumerate(range(t0, t1)):
                assert list(bounds[:, i]) == [a[:, t].min(), a[:, t].max(), b[:, t].min(), b[:, t].max()]
                box = dl.step_box(ab, t)
                assert box.shape == (bounds[1, i] - bounds[0, i] + 1, bounds[3, i] - bounds[2, i] + 1)
                assert box.sum() == n
                for j in range(n):
                    assert box[a[j, t] - bounds[0, i], b[j, t] - bounds[2, i]] > 0
                ca, cb, cc = dl.cells(ab, t)
                assert cc.sum() == n and (cc > 0).all()
                pairs = {(x, y) for x, y in zip(a[:, t], b[:, t])}
                assert pairs == set(zip(ca.tolist(), cb.tolist()))


@pytest.mark.parametrize("case", DICE_CASES, ids=lambda c: c["name"])
def test_route_decisions(case):
    oc = golden_io.draw_outcomes(case)
    lev, f = case_factors(case)
    ok = dl.route_ok(f, case["v0"], oc)
    assert [round(float(x), 6) for x in lev[~ok]] == CHAIN_LEVERAGES.get(case["name"], [])


@pytest.mark.parametrize("case", DICE_CASES, ids=lambda c: c["name"])
def test_routed_statistics_meet_the_reference(case):
    oc = golden_io.draw_outcomes(case)
    gold = golden_io.load("lev_" + case["name"], oc)
    lev, f = case_factors(case)
    ok = dl.route_ok(f, case["v0"], oc)
    steps = np.asarray(gold["cols"]) + 1           # column c of data holds step c + 1
    got = dl.lattice_stats(oc, steps, f[ok], case["v0"], case["top"])
    want = np.moveaxis(gold["data"][ok, :12], 1, 2)    # [G_routed, cols, 12]
    assert_lattice_close(got.astype(np.float32), want, lattice_tol(case["h"]))
    assert np.array_equal(lev[ok], gold["data"][ok, 12, 0])


def test_zero_factor_and_underflow_keep_the_chain():
    """A factor of 0 (down_r = -1 at l = 1) and a long horizon whose high leverages underflow."""
    rs = np.random.RandomState(8)
    oc = rs.choice(3, size=(200, 40), p=[1 / 6, 1 / 6, 2 / 3]).astype(np.uint8)
    lev = np.asarray([0.5, 1.0], dtype=np.float32)
    f = lo.dice_factors(lev, 0.5, -1.0, 0.05)
    assert list(dl.route_ok(f, 100.0, oc)) == [True, False]
    oc = rs.choice(3, size=(50, 3000), p=[0.1, 0.6, 0.3]).astype(np.uint8)
    lev = np.asarray([0.1, 0.5, 1.0], dtype=np.float32)
    f = lo.dice_factors(lev, 0.5, -0.5, 0.05)
    assert list(dl.route_ok(f, 100.0, oc)) == [True, False, False]

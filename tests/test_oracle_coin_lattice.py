"""
Pins oracle/coin_lattice_oracle.py - the up-move count lattice behind
coin_smart_lev(..., method="counts") - against the reference's coin fixtures.  CPU only.
"""
import math

import numpy as np
import pytest

import golden_io
from oracle import coin_lattice_oracle as cl
from oracle import lev_oracle as lo

COIN_CASES = [c for c in golden_io.LEV_CASES if c["kind"] == "coin"]
# leverages whose extreme paths leave fp32's normal range: they keep the chain
CHAIN_LEVERAGES = {"coin_long": [0.8, 1.0], "coin_overflow": [0.6, 1.0]}


def lattice_tol(h: int) -> float:
    """The LOG-mode tolerance of the suite (tests/test_lev_gpu.py) with a factor 1.5."""
    return 1e-5 * max(1.0, math.sqrt(h / 300)) * 1.5


def assert_lattice_close(got, want, tol):
    """[..., 12] statistics: nan/inf patterns equal; means and medians within tol relative; MAD and std
    within tol times the larger of their own and their group's mean magnitude (equal-k investors share ONE
    lattice value, so a small group's spread can be 0 where the fp32 chain reports a few ulps of its mean)."""
    got = np.asarray(got, dtype=np.float64)
    want = np.asarray(want, dtype=np.float64)
    assert np.array_equal(np.isnan(got), np.isnan(want))
    inf = np.isinf(want)
    assert np.array_equal(got[inf], want[inf])
    fin = np.isfinite(want)
    scale = np.abs(want).copy()
    for j in range(3, 9):
        m = want[..., j % 3]
        scale[..., j] = np.maximum(scale[..., j], np.abs(np.where(np.isfinite(m), m, 0.0)))
    with np.errstate(invalid="ignore"):
        bad = fin & (np.abs(got - want) > tol * scale)
    assert not bad.any(), (np.argwhere(bad)[:5], got[bad][:5], want[bad][:5])


def test_hist_equals_cumsum_counts():
    rs = np.random.RandomState(3)
    for n, h in ((1, 1), (5, 2), (77, 33), (300, 97)):
        oc = (rs.random_sample((n, h)) < 0.4).astype(np.uint8)
        k = np.cumsum(oc.astype(np.int64), axis=1)
        for t0, t1 in ((0, h), (h // 3, h), (0, max(1, h // 2))):
            hist, kmin, kmax, k_end = cl.lattice_hist(oc, t0, t1)
            assert hist.shape == (t1 - t0, h + 1)
            for i, t in enumerate(range(t0, t1)):
                assert np.array_equal(hist[i], np.bincount(k[:, t], minlength=h + 1))
                assert kmin[i] == k[:, t].min() and kmax[i] == k[:, t].max()
                assert hist[i].sum() == n and hist[i, :kmin[i]].sum() == 0 and hist[i, kmax[i] + 1:].sum() == 0
            assert np.array_equal(k_end, k[:, t1 - 1])


@pytest.mark.parametrize("case", COIN_CASES, ids=lambda c: c["name"])
def test_route_decisions(case):
    oc = golden_io.draw_outcomes(case)
    lev = lo.lev_grid(*case["grid"], case["up_r"], case["down_r"])
    f = lo.coin_factors(lev, case["up_r"], case["down_r"])
    _, kmin, kmax, _ = cl.lattice_hist(oc)
    ok = cl.route_ok(f, case["v0"], kmin, kmax, 0, True)
    chain = [round(abs(float(x)), 6) for x in lev[~ok]]
    assert chain == CHAIN_LEVERAGES.get(case["name"], [])
    # under the float64 default every leverage of these fixtures stays in range
    f64 = np.stack([1.0 + lev.astype(np.float64) * case["down_r"], 1.0 + lev.astype(np.float64) * case["up_r"]], 1)
    assert cl.route_ok(f64, case["v0"], kmin, kmax, 0, False).all()


@pytest.mark.parametrize("case", COIN_CASES, ids=lambda c: c["name"])
def test_routed_statistics_meet_the_reference(case):
    oc = golden_io.draw_outcomes(case)
    gold = golden_io.load("lev_" + case["name"], oc)
    lev = lo.lev_grid(*case["grid"], case["up_r"], case["down_r"])
    f = lo.coin_factors(lev, case["up_r"], case["down_r"])
    hist, kmin, kmax, _ = cl.lattice_hist(oc)
    ok = cl.route_ok(f, case["v0"], kmin, kmax, 0, True)
    steps = np.asarray(gold["cols"]) + 1           # column c of data holds step c + 1
    got = np.stack([cl.lattice_stats(hist[t:t + 1], t, f[ok], case["v0"], case["top"], True)[:, 0] for t in steps], 1)
    want = np.moveaxis(gold["data"][ok, :12], 1, 2)    # [G_routed, cols, 12]
    assert_lattice_close(got.astype(np.float32), want, lattice_tol(case["h"]))
    assert np.array_equal(lev[ok], gold["data"][ok, 12, 0])

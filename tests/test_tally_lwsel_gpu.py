"""
The two routes of the tally statistics kernel (tally.cu, tally_select_kernel) on the same finalized
bins: the log-wealth route (the default for K <= 3) against the radix route forced with
B200_LEV_FLAG_RADIX_SELECT - order statistics bit for bit, moments to 1e-12 - and the info word that
counts the grid points on the radix route, for the inputs that must take it (K = 4, a zero factor, a
flat grid point, a log-wealth bin with more tuples than the leader holds).
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import torch as T

import golden_io
from oracle import lev_oracle as lo

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def assert_routes_agree(lat, rad, rtol=1e-12):
    lat, rad = np.asarray(lat, np.float64), np.asarray(rad, np.float64)
    assert np.array_equal(np.isnan(lat), np.isnan(rad)), (lat, rad)
    assert np.array_equal(lat[:, 9:12].view(np.uint64), rad[:, 9:12].view(np.uint64)), (lat[:, 9:12], rad[:, 9:12])
    fin = np.isfinite(rad)
    assert np.array_equal(lat[~fin & ~np.isnan(rad)], rad[~fin & ~np.isnan(rad)])
    scale = np.where(np.isfinite(rad[:, 0:1]), np.abs(rad[:, 0:1]), 0.0) + 1e-300
    err = np.abs(np.where(fin, lat - rad, 0.0))
    ok = (err <= rtol * np.maximum(np.abs(rad), scale)) | ~fin
    assert ok.all(), (np.argwhere(~ok)[:5], lat[~ok][:5], rad[~ok][:5])


def both_routes(t, f, v0, h, n, top):
    """(log-wealth route stats, radix stats, grid points the first call sent to the radix route)."""
    before = t.info()["radix_route"]
    lat = t.stats(f, v0, h, n_total=n, top=top).cpu().numpy()
    mid = t.info()["radix_route"]
    rad = t.stats(f, v0, h, n_total=n, top=top, radix_select=True).cpu().numpy()
    assert t.info()["radix_route"] - mid == f.shape[0]
    return lat, rad, mid - before


def tally_of(codes, k):
    from rlmd_b200 import tally
    t = tally.FinalTally(codes.shape[0])
    t.add(codes, k)
    t.finalize()
    return t


def test_flag_matches_the_header(tmp_path):
    from rlmd_b200 import _lib
    src = tmp_path / "f.c"
    src.write_text(f'#include <stdio.h>\n#include "{os.path.join(ROOT, "include", "rlmd_b200.h")}"\n'
                   'int main(void){printf("%d\\n", B200_LEV_FLAG_RADIX_SELECT); return 0;}\n')
    subprocess.check_call(["gcc", "-std=c99", "-o", str(tmp_path / "f"), str(src)])
    assert int(subprocess.check_output([str(tmp_path / "f")])) == _lib.LEV_FLAG_RADIX_SELECT


def test_c2_dice_takes_the_log_wealth_route():
    """The flagship shape: 1e6 investors x 1e4 die rolls, 20 leverages - every grid point on the new route."""
    from rlmd_b200 import engine, lev_exp
    n, h = 1_000_000, 10_000
    lev = np.asarray(lev_exp.param_range(0.05, 1.0, 0.05), np.float32)
    f = lev_exp.dice_factor_table(lev, 0.5, -0.5, 0.05)
    oc = engine.lev_draw("discrete", n, h, seed=420, probs=(1 / 6, 1 / 6, 2 / 3), packed=True)
    t = tally_of(oc, 3)
    lat, rad, radix = both_routes(t, f, 100.0, h, n, 100)
    assert radix == 0
    assert_routes_agree(lat, rad)
    again = t.stats(f, 100.0, h, n_total=n, top=100).cpu().numpy()
    assert np.array_equal(again.view(np.uint64), lat.view(np.uint64)), "not repeatable"


@pytest.mark.parametrize("name", ["coin_testscale", "dice_testscale", "dicesh_testscale", "coin_top7", "dice_top5",
                                  "dicesh_top3", "dice_tiny"])
def test_fixtures(name):
    from rlmd_b200 import engine
    case = golden_io.lev_case(name)
    oc = golden_io.draw_outcomes(case)
    lev = lo.lev_grid(*case["grid"], case["up_r"], case["down_r"])
    if case["kind"] == "coin":
        f, k = lo.coin_factors(lev, case["up_r"], case["down_r"]), 2
    elif case["kind"] == "dice":
        f, k = lo.dice_factors(lev, case["up_r"], case["down_r"], case["mid_r"]), 3
    else:
        f, k = lo.dice_sh_factors(lev, case["up_r"], case["down_r"], case["mid_r"], *case["sh"]), 3
    t = tally_of(engine.encode_codes(oc), k)
    lat, rad, _ = both_routes(t, f, case["v0"], oc.shape[1], oc.shape[0], case["top"])
    assert_routes_agree(lat, rad)


def test_coin_ties_infinities_zeros_and_flat_rows():
    """K = 2; every investor equal / half at +inf; a zero factor (log -inf) and a flat row go to the radix route."""
    from rlmd_b200 import engine
    n, h = 515, 40
    f = np.array([[1.5, 0.6], [2.0, 0.0], [1e30, 1.0], [1.0, 1.0]], dtype=np.float32)
    same = np.ones((n, h), dtype=np.uint8)
    same[:, ::2] = 0
    half = same.copy()
    half[: n // 2] = 1
    rs = np.random.RandomState(3)
    coin = (rs.uniform(size=(20000, 3000)) < 0.5).astype(np.uint8)
    for oc in (same, half, coin):
        t = tally_of(engine.encode_codes(oc), 2)
        lat, rad, radix = both_routes(t, f, 1.0, oc.shape[1], oc.shape[0], 3)
        assert_routes_agree(lat, rad)
        assert radix >= 2      # the zero factor and the flat row
    lat, rad, radix = both_routes(t, f[:1], 1.0, 3000, 20000, 3)
    assert radix == 0


def test_grid_of_130_and_four_outcomes():
    """A grid wider than one statistics tile (K = 3), and K = 4, which always takes the radix route."""
    from rlmd_b200 import engine
    rs = np.random.RandomState(5)
    for k in (3, 4):
        oc = rs.randint(0, k, size=(3001, 77)).astype(np.uint8)
        f = (1 + rs.uniform(-0.3, 0.5, size=(130, k))).astype(np.float32)
        t = tally_of(engine.encode_codes(oc), k)
        lat, rad, radix = both_routes(t, f, 10.0, 77, 3001, 9)
        assert_routes_agree(lat, rad)
        assert radix == (130 if k == 4 else 0)


def test_overfull_bin_takes_the_radix_route():
    """Three investors at the corners of the simplex widen the (n_1, n_2) box so far that the dense middle of
    the population falls into a few log-wealth bins of thousands of tuples each."""
    from rlmd_b200 import engine, lev_exp, tally
    n, h = 200_000, 20_000
    lev = np.asarray(lev_exp.param_range(0.1, 1.0, 0.3), np.float32)
    f = lev_exp.dice_factor_table(lev, 0.5, -0.5, 0.05)
    t = tally.FinalTally(n + 3)
    t.add(engine.lev_draw("discrete", n, h, seed=7, probs=(1 / 3, 1 / 3, 1 / 3), packed=True), 3)
    t.add(engine.encode_codes(np.repeat(np.arange(3, dtype=np.uint8)[:, None], h, axis=1)), 3)
    t.finalize()
    lat, rad, radix = both_routes(t, f, 100.0, h, n + 3, 50)
    assert radix == f.shape[0]
    assert_routes_agree(lat, rad)


@pytest.mark.parametrize("world", [2, 8])
def test_merged_rank_tallies_on_one_gpu(world):
    """The cross-GPU merge played on one GPU (as test_tally_gpu.test_merge_of_rank_tallies_on_one_gpu): the box
    of the merged list comes from the unique kernel; every rank takes the log-wealth route with identical
    results, and they agree with the radix route."""
    from rlmd_b200 import _lib, engine, tally
    from rlmd_b200._lib import check, lib, ptr, stream_ptr
    case = golden_io.lev_case("dice_top5")
    oc = golden_io.draw_outcomes(case)
    lev = lo.lev_grid(*case["grid"], case["up_r"], case["down_r"])
    f = lo.dice_factors(lev, case["up_r"], case["down_r"], case["mid_r"])
    n, h = oc.shape
    cuts = np.linspace(0, n, world + 1).astype(int)
    ranks = []
    for r in range(world):
        t = tally.FinalTally.__new__(tally.FinalTally)
        t.dev, t.group, t._staging, t.rows, t.horizon = T.device("cuda", 0), None, None, 0, None
        t.plan = _lib.TallyPlan()
        t.plan.rows_cap, t.plan.bins_cap, t.plan.grid_cap, t.plan.world = n, n, 64, world
        t.ws = T.empty((lib.b200_tally_workspace_bytes(C.byref(t.plan)) // 8,), dtype=T.int64, device="cuda")
        t.exchange = None
        t.ex_buf = T.zeros((lib.b200_tally_exchange_bytes(C.byref(t.plan)) // 8 + 1,), dtype=T.int64, device="cuda")
        check(lib.b200_tally_reset(C.byref(t.plan), ptr(t.ws), stream_ptr()))
        t.add(engine.encode_codes(oc[cuts[r]:cuts[r + 1]]), 3)
        ranks.append(t)
    peers = []
    for r in range(world):
        p = _lib.TallyPeers()
        p.world, p.rank, p.epoch = world, r, 1
        for q in range(world):
            p.exchange[q] = ranks[q].ex_buf.data_ptr()
        peers.append(p)
    for phase in (0, 1):
        for r, t in enumerate(ranks):
            check(lib.b200_tally_finalize(C.byref(t.plan), ptr(t.ws), C.byref(peers[r]), phase, stream_ptr()))
    single = tally_of(engine.encode_codes(oc), 3).stats(f, case["v0"], h, n_total=n, top=case["top"]).cpu().numpy()
    got = []
    for t in ranks:
        lat, rad, radix = both_routes(t, f, case["v0"], h, n, case["top"])
        assert radix < f.shape[0]
        assert_routes_agree(lat, rad)
        got.append(lat)
    for r in range(1, world):
        assert np.array_equal(got[r].view(np.uint64), got[0].view(np.uint64)), f"rank {r} differs from rank 0"
    assert_routes_agree(got[0], single, rtol=1e-13)

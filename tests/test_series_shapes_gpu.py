"""
The per-step series (engine.lev_series, engine.bigbrain_series) at the chunk
shapes they are planned for at production sizes, against the torch restatement
of the reference (tests/series_ref.py, pinned to the NumPy oracle on the CPU by
tests/test_series_ref.py) run on the same GPU.

engine.rowstats is wrapped so that each test records the rows of every call and
asserts the planned chunk shape was actually reached:

  dice, streamed / Philox   G = 10, N = 1e6, H = 700   192-step chunks (1920 rows), last 124
  dice with l = 2.0         G = 8,  N = 1e6, H = 300   256-step chunks; the down factor is 0
  coin p = 0.7, +0.5/-0.4   G = 3,  N = 1e6, H = 1000  672-step chunks (2016 rows); l = 1 ends nearly all inf
  dice, two chain tiles     G = 40, N = 2e5, H = 300   32-step chunks (1280 rows), last 12
  GBM, streamed / Philox    G = 10, N = 1e6, H = 700   192-step chunks
  GBM, +-1 paths            saturation sticky in time order across chunks
  big brain, coin / dice    P = 63, N = 1e6, H = 128   point tile 16, 16-step chunks from s = 1, last tile 15
  big brain, coin           P = 63, N = 2e5, H = 128   point tile 32, 32-step chunks (the 16-byte loads)
"""
import numpy as np
import pytest
import torch

import golden_io
import series_ref
from oracle import lev_oracle as lo
from test_oracle_lev import assert_stats_close
from test_series_ref import STICKY_LEV, sticky_paths

pytestmark = pytest.mark.gpu

N, TOP, V0 = 1_000_000, 100, 100.0
DICE = (1 / 6, 1 / 6, 2 / 3)
PEAK_BYTES = 60e9


@pytest.fixture(autouse=True)
def peak_memory():
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    yield
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated()
    print(f"peak device memory {peak / 1e9:.2f} GB")
    assert peak <= PEAK_BYTES


@pytest.fixture
def calls(monkeypatch):
    """Rows of every engine.rowstats call; `keep` also keeps copies of the dumps (small cases only)."""
    from rlmd_b200 import engine
    real = engine.rowstats
    rec = {"rows": [], "dumps": [], "keep": False}

    def wrapped(values, top, **kw):
        rec["rows"].append(values.shape[0])
        if rec["keep"]:
            rec["dumps"].append(values.clone())
        return real(values, top, **kw)

    monkeypatch.setattr(engine, "rowstats", wrapped)
    return rec


def assert_series_equal(got, want, *, ulp=0, rtol=3e-7, noise=1e-12):
    """data [G,13,H-1]: leverage row equal, order statistics within `ulp` fp32 ulps (same nan / inf), moments close."""
    g, w = got.cpu().numpy(), want.cpu().numpy()
    assert g.shape == w.shape
    assert np.array_equal(g[:, 12], w[:, 12])
    assert_order_stats(g[:, 9:12], w[:, 9:12], ulp)
    assert_stats_close(g[:, :9], w[:, :9], rtol=rtol, noise=noise)


def assert_order_stats(g, w, ulp):
    assert np.array_equal(np.isnan(g), np.isnan(w))
    assert np.array_equal(np.isinf(g), np.isinf(w)) and np.array_equal(g[np.isinf(g)], w[np.isinf(w)])
    gi, wi = g.view(np.uint32).astype(np.int64), w.view(np.uint32).astype(np.int64)
    fin = np.isfinite(w)
    diff = np.abs(gi - wi)[fin]
    assert diff.size == 0 or diff.max() <= ulp, (np.argwhere(np.abs(gi - wi) * fin > ulp)[:5], diff.max())


def assert_data_T(got, want, ulp=0):
    assert got.shape == want.shape and got.dtype == want.dtype
    assert_order_stats(got.cpu().numpy(), want.cpu().numpy(), ulp)


def chunk_rows(g, h, tc):
    """The rows of every rowstats call of lev_series at chunk length tc."""
    return [g * (min(h, t0 + tc) - t0) for t0 in range(0, h, tc)]


# ----------------------------------------------------------------- discrete
@pytest.fixture(scope="module")
def dice10():
    from rlmd_b200 import engine, lev_exp
    h = 700
    lev = lo.lev_grid(0.1, 1.0, 0.1)
    f = lev_exp.dice_factor_table(lev, 0.5, -0.5, 0.05)
    codes = engine.lev_draw("discrete", N, h, seed=701, probs=DICE)
    data, data_T = series_ref.smart_lev(codes, f, lev, TOP, V0)
    yield dict(h=h, lev=lev, f=f, codes=codes, data=data, data_T=data_T)
    del codes, data, data_T
    torch.cuda.empty_cache()


def test_dice_streamed_at_192_step_chunks(dice10, calls):
    from rlmd_b200 import engine
    d = dice10
    data, data_T = engine.lev_series("discrete", d["f"], d["lev"], V0, TOP, outcomes=d["codes"])
    assert calls["rows"] == [1920, 1920, 1920, 1240] == chunk_rows(10, 700, 192)
    assert_data_T(data_T, d["data_T"])
    assert_series_equal(data, d["data"])


def test_dice_philox_at_192_step_chunks(dice10, calls):
    from rlmd_b200 import engine
    d = dice10
    data, data_T = engine.lev_series("discrete", d["f"], d["lev"], V0, TOP, n_investors=N, horizon=d["h"], seed=701,
                                     probs=DICE)
    assert calls["rows"] == [1920, 1920, 1920, 1240]
    assert_data_T(data_T, d["data_T"])
    assert_series_equal(data, d["data"])


def run_discrete(calls, lev, f, n, h, probs, seed, rows):
    from rlmd_b200 import engine
    codes = engine.lev_draw("discrete", n, h, seed=seed, probs=probs)
    want, want_T = series_ref.smart_lev(codes, f, lev, TOP, V0)
    data, data_T = engine.lev_series("discrete", f, lev, V0, TOP, outcomes=codes)
    assert calls["rows"] == rows
    assert_data_T(data_T, want_T)
    assert_series_equal(data, want)
    return data, data_T


def test_dice_with_a_zero_down_factor(calls):
    """l = 2.0: 1 + 2 (-0.5) = 0, so nearly every row of that grid point is tied at exactly 0."""
    from rlmd_b200 import lev_exp
    lev = lo.lev_grid(0.25, 2.0, 0.25)
    f = lev_exp.dice_factor_table(lev, 0.5, -0.5, 0.05)
    assert f[-1, 1] == 0
    data, data_T = run_discrete(calls, lev, f, N, 300, DICE, 702, [2048, 352])
    assert float((data_T[-1] == 0).double().mean()) > 0.99
    assert float(data[-1, 9, -1]) == 0.0                       # the median of the last step is 0


def test_coin_overflow_gamble_at_672_step_chunks(calls):
    """p = 0.7, +0.5 / -0.4: at l = 1 nearly every investor's wealth passes FLT_MAX (inf medians, nan moments)."""
    from rlmd_b200 import lev_exp
    c = golden_io.lev_case("coin_overflow")
    lev = lo.lev_grid(*c["grid"], c["up_r"], c["down_r"])
    f = lev_exp.coin_factor_table(lev, c["up_r"], c["down_r"])
    data, data_T = run_discrete(calls, lev, f, N, 1000, (0.3, 0.7), 703, [2016, 984])
    assert float(torch.isinf(data_T[-1]).double().mean()) > 0.999
    assert bool(torch.isnan(data[-1, 0, -1])) and bool(torch.isinf(data[-1, 9, -1]))


def test_dice_grid_of_two_chain_tiles(calls):
    """G = 40 > 32: run_chain_discrete runs two tiles, the second dumped at g0 * tc * ldT."""
    from rlmd_b200 import lev_exp
    lev = lo.lev_grid(0.025, 1.0, 0.025)
    assert lev.shape == (40,)
    f = lev_exp.dice_factor_table(lev, 0.5, -0.5, 0.05)
    run_discrete(calls, lev, f, 200_000, 300, DICE, 704, [1280] * 9 + [480])


# ---------------------------------------------------------------------- GBM
@pytest.fixture(scope="module")
def gbm10():
    from rlmd_b200 import engine
    h = 700
    lev = lo.lev_grid(-1.0, 1.0, 0.2)
    x = engine.lev_draw("gbm", N, h, seed=705, log_mean=-0.05, sigma=0.447)
    data, data_T = series_ref.gbm_smart_lev(x, lev, TOP, V0)
    yield dict(h=h, lev=lev, x=x, data=data, data_T=data_T)
    del x, data, data_T
    torch.cuda.empty_cache()


@pytest.mark.parametrize("source", ["streamed", "philox"])
def test_gbm_at_192_step_chunks(gbm10, calls, source):
    """exp is not bit-pinned: order statistics and data_T within one fp32 ulp."""
    from rlmd_b200 import engine
    d = gbm10
    if source == "streamed":
        kw = dict(outcomes=d["x"])
    else:
        kw = dict(n_investors=N, horizon=d["h"], seed=705, log_mean=-0.05, sigma=0.447)
    data, data_T = engine.lev_series("gbm", d["lev"], d["lev"], V0, TOP, **kw)
    assert calls["rows"] == [1920, 1920, 1920, 1240]
    assert_data_T(data_T, d["data_T"], ulp=1)
    assert_series_equal(data, d["data"], ulp=1, rtol=1e-6)


def test_gbm_saturation_is_sticky_across_chunks(calls):
    """
    The +-1 paths of test_series_ref: a path that underflows first stays 0 after it
    climbs past ln FLT_MAX (and the mirror image stays inf), in 64-step chunks so the
    state carries the saturation from chunk to chunk.  Every dumped wealth is compared.
    """
    from rlmd_b200 import engine
    x = torch.as_tensor(sticky_paths(), device="cuda")
    n, h = x.shape
    calls["keep"] = True
    data, data_T = engine.lev_series("gbm", STICKY_LEV, STICKY_LEV, V0, 1, outcomes=x, chunk_steps=64)
    assert calls["rows"] == chunk_rows(4, h, 64)
    want = [w.clone() for _, w in series_ref.gbm_wealth(x, STICKY_LEV, V0)]
    t0 = 0
    for dump in calls["dumps"]:
        tc = dump.shape[0] // 4
        got = dump.view(4, tc, n)
        for k in range(tc):
            assert_order_stats(got[:, k].cpu().numpy(), want[t0 + k].cpu().numpy(), 1)
        t0 += tc
    assert t0 == h
    assert float(data_T[3, 0]) == 0.0 and float(data_T[0, 1]) == 0.0      # underflowed first (l = 1, and its mirror)
    assert bool(torch.isinf(data_T[3, 1])) and bool(torch.isinf(data_T[0, 0]))
    rs, rs_T = series_ref.gbm_smart_lev(x, STICKY_LEV, 1, V0)
    assert_data_T(data_T, rs_T, ulp=1)
    assert_series_equal(data, rs, ulp=1, rtol=1e-6)


def test_gbm_final_time_sweep_keeps_its_documented_rule():
    """
    The saturating final-time sweep (lev_sweep, mode "log") decides saturation from
    the running extremes of S alone: inf if log wealth ever passed ln FLT_MAX, else 0
    if it ever fell below ln 2^-150.  A path that underflowed and later climbed past
    ln FLT_MAX therefore ends at inf there, where the series (and the reference's
    chain) end at 0.
    """
    from rlmd_b200 import engine
    x = torch.as_tensor(sticky_paths(), device="cuda")
    fin = engine.lev_sweep("gbm", STICKY_LEV, V0, outcomes=x, mode="log")["data_T"].cpu().numpy()
    assert np.isinf(fin[3, 0]) and np.isinf(fin[0, 1])             # went both ways: inf wins
    assert fin[3, 2] == 0 and np.isinf(fin[3, 3])                  # one way only: as the chain


# ---------------------------------------------------------------- big brain
BB_STOP = np.float32([0.1, 0.2, 0.3, 0.4, 0.5, 0.6, 0.7, 0.8, 0.9])
BB_ROLL = np.float32([0.0, 0.1, 0.2, 0.3, 0.4, 0.5, 0.6])     # retention 0 and > 0 in one grid


def bb_rows(P, ptile, tc, h):
    """The rows of every rowstats call of bigbrain_series: point tiles outer, chunks from s = 1 inner."""
    rows = []
    for p0 in range(0, P, ptile):
        pc = min(ptile, P - p0)
        s = 1
        while s < h:
            e = min(h, s + tc)
            rows.append(pc * (e - s) * 2)
            s = e
    return rows


def run_big_brain(calls, kind, n, rows, seed):
    from rlmd_b200 import engine
    h = 128
    if kind == "coin":
        probs, returns, by_code = (0.5, 0.5), (0.5, -0.4), (-0.4, 0.5)
        eta = golden_io.bigbrain_lev_factor(dict(up_r=0.5, down_r=-0.4))
    else:
        probs, returns = DICE, (0.5, -0.5, 0.05)
        by_code = returns
        eta = golden_io.bigbrain_lev_factor(dict(up_r=0.5, down_r=-0.5))
    codes = engine.lev_draw("discrete", n, h, seed=seed, probs=probs)
    data, w = engine.bigbrain_series(kind, codes, TOP, V0, by_code, eta, BB_STOP, BB_ROLL)
    assert calls["rows"] == rows
    want, want_w = series_ref.big_brain(kind, codes, TOP, V0, returns, eta, BB_STOP, BB_ROLL)
    assert w.dtype == want_w.dtype
    if kind == "coin":
        assert torch.equal(w.view(torch.int32), want_w.view(torch.int32))
    else:
        assert torch.equal(w.view(torch.int64), want_w.view(torch.int64))
    g, r = data.cpu().numpy(), want.cpu().numpy()
    assert g.shape == r.shape == (7, 9, 26, h - 1)
    assert np.array_equal(g[:, :, 24:26], r[:, :, 24:26])
    # dice: the engine takes the moments of the fp32-rounded dump, the reference those of the fp64 values
    tol = dict(rtol=3e-7, noise=1e-12) if kind == "coin" else dict(rtol=1e-6, noise=2e-6)
    for base in (0, 12):
        assert_order_stats(g[:, :, base + 9:base + 12], r[:, :, base + 9:base + 12], 0)
        assert_stats_close(g[:, :, base:base + 9], r[:, :, base:base + 9], **tol)


@pytest.mark.parametrize("kind", ["coin", "dice"])
def test_big_brain_at_16_point_tiles(calls, kind):
    """N = 1e6: the 2 GB dump halves the point tile to 16; chunks start at s = 1 mod 16 (the byte-wise loads)."""
    rows = bb_rows(63, 16, 16, 128)
    assert rows[:8] == [512] * 7 + [480] and rows[-1] == 450
    run_big_brain(calls, kind, N, rows, 706 if kind == "coin" else 707)


def test_big_brain_coin_at_32_point_tiles(calls):
    """N = 2e5: point tile 32, 32-step chunks; codes rows are 16-byte aligned, so the 16-outcome loads are taken."""
    rows = bb_rows(63, 32, 32, 128)
    assert rows[0] == 2048
    run_big_brain(calls, "coin", 200_000, rows, 708)

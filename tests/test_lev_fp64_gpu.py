"""
The float64 leverage path on the GPU (the reference run under
torch.set_default_dtype(torch.float64)): b200_rowstats_f64 against oracle.summary_stats,
the fp64 chain (b200_lev_chunk_f64) against the fp64 oracle, and the coin / GBM shims and
scripts under a float64 default.
"""
import contextlib
import io
import os

import numpy as np
import pytest
import torch as T

from oracle import lev_oracle as lo
from oracle import lev_oracle_f64 as lo64

pytestmark = pytest.mark.gpu

SNP_LOG_MEAN = 0.0540025395205692 - 0.1897916175617430 ** 2 / 2
SNP_SIGMA = 0.1897916175617430


@pytest.fixture
def fp64_default():
    old = T.get_default_dtype()
    T.set_default_dtype(T.float64)
    try:
        yield
    finally:
        T.set_default_dtype(old)


def assert_stats(got, want, rtol=1e-12, median_rtol=None):
    """Medians bit-exact (NaN where the oracle has NaN; -0 == +0) unless median_rtol; moments: the same
    non-finite entries, finite ones within rtol."""
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    assert got.shape == want.shape
    cols = slice(0, 12) if median_rtol is not None else slice(0, 9)
    if median_rtol is None:
        np.testing.assert_array_equal(got[..., 9:12], want[..., 9:12])
    g, w = got[..., cols], want[..., cols]
    assert np.array_equal(np.isnan(g), np.isnan(w))
    assert np.array_equal(np.isposinf(g), np.isposinf(w)) and np.array_equal(np.isneginf(g), np.isneginf(w))
    fin = np.isfinite(w)
    scale = np.max(np.abs(w[fin])) if fin.any() else 1.0
    np.testing.assert_allclose(g[fin], w[fin], rtol=max(rtol, median_rtol or 0.0), atol=1e-14 * scale)


def assert_wealth(got, want, rtol):
    got, want = np.asarray(got), np.asarray(want)
    assert np.array_equal(np.isinf(got), np.isinf(want)) and not np.isnan(got).any()
    fin = np.isfinite(want)
    np.testing.assert_allclose(got[fin], want[fin], rtol=rtol, atol=0)


# ---------------------------------------------------------------- rowstats
def _rows_1e6():
    rs = np.random.RandomState(11)
    n = 1_000_000
    a = np.round(rs.lognormal(3.0, 1.0, n), 1)                   # positive, heavy ties
    b = rs.randn(n) + 3.0                                        # negative values, +-0, ties
    b[rs.choice(n, 5000, replace=False)] = 0.0
    b[rs.choice(n, 5000, replace=False)] = -0.0
    b[rs.choice(n, 20000, replace=False)] = 2.5
    c = rs.lognormal(0.0, 2.0, n)
    c[rs.choice(n, 3, replace=False)] = np.inf                   # +inf in the top group
    d = rs.randn(n) * 10
    d[rs.choice(n, 7, replace=False)] = np.nan
    e = rs.lognormal(0.0, 1.0, n)
    e[rs.choice(n, 11, replace=False)] = -np.inf
    return np.stack([a, b, c, d, e])


@pytest.mark.parametrize("which", ["top1", "top_n_minus_1"])
def test_rowstats_f64_1e6(which):
    from rlmd_b200 import engine

    v = _rows_1e6()
    n = v.shape[1]
    top = 1 if which == "top1" else n - 1
    got = engine.rowstats(T.as_tensor(v, device="cuda"), top).cpu().numpy()
    want = np.stack([lo64.summary_stats_f64(r, top) for r in v])
    assert_stats(got, want)


def test_rowstats_f64_tiny_rows():
    from rlmd_b200 import engine

    two = np.array([[1.0, 2.0], [-0.0, 0.0], [np.inf, 1.0], [np.nan, 3.0], [-np.inf, -5.0], [7.0, 7.0]])
    got = engine.rowstats(T.as_tensor(two, device="cuda"), 1).cpu().numpy()
    assert_stats(got, np.stack([lo64.summary_stats_f64(r, 1) for r in two]))
    one = np.array([[5.0], [-np.inf], [np.nan], [-0.0]])
    got = engine.rowstats(T.as_tensor(one, device="cuda"), 1).cpu().numpy()
    assert_stats(got, np.stack([lo64.summary_stats_f64(r, 1) for r in one]))
    # strided rows (a view with ld > n)
    v = _rows_1e6()[:3, :1000]
    buf = T.zeros((3, 1024), dtype=T.float64, device="cuda")
    buf[:, :1000] = T.as_tensor(v, device="cuda")
    got = engine.rowstats(buf[:, :1000], 10).cpu().numpy()
    assert_stats(got, np.stack([lo64.summary_stats_f64(r, 10) for r in v]))


def test_rowstats_f64_with_group_raises_before_launch():
    from rlmd_b200 import engine

    v = T.ones((2, 8), dtype=T.float64, device="cuda")
    with pytest.raises(ValueError, match="single-GPU"):
        engine.rowstats(v, 1, group=object())
    with pytest.raises(ValueError, match="single-GPU"):
        engine.lev_series("gbm", np.ones(1), np.ones(1), 100.0, 1, outcomes=v, group=object(), dtype=T.float64)


# ------------------------------------------------------------- fp64 chain
def _coin_codes(n, h, seed):
    from rlmd_b200 import engine

    return engine.lev_draw("discrete", n, h, seed=seed, probs=(0.5, 0.5))


def test_coin_series_f64_testscale():
    from rlmd_b200 import engine

    n, h, top = 10_000, 300, 1
    codes = _coin_codes(n, h, 7)
    oc = codes.cpu().numpy()
    lev = lo64.lev_grid_f64(0.1, 1.0, 0.1, 0.5, -0.4)
    f = lo64.coin_factors_f64(lev, 0.5, -0.4)
    want, want_T = lo64.smart_lev_f64(oc, f, lev, top, 100.0)
    for chunk_steps in (None, 37):
        data, data_T = engine.lev_series("discrete", f, lev, 100.0, top, outcomes=codes, dtype=T.float64,
                                         chunk_steps=chunk_steps)
        assert data.dtype == T.float64 and data_T.dtype == T.float64
        data, data_T = data.cpu().numpy(), data_T.cpu().numpy()
        assert np.array_equal(data_T.view(np.uint64), want_T.view(np.uint64))
        assert np.array_equal(data[:, 12], want[:, 12])
        assert_stats(data[:, :12].transpose(0, 2, 1), want[:, :12].transpose(0, 2, 1))
    stats, fin_T = engine.lev_final_f64("discrete", f, 100.0, top, codes)
    assert np.array_equal(fin_T.cpu().numpy(), want_T)
    assert_stats(stats.cpu().numpy(), lo64.fixed_final_lev_f64(oc, f, top, 100.0))


def test_coin_series_f64_c1_smart_size():
    """C1's smart size (1e6 x 3e3, G = 10): data_T bit-exact against the NumPy oracle on a sample of investors
    and against a torch fp64 restatement of the chain (IEEE multiplies on the GPU) on all of them; the
    statistics of three steps against oracle.summary_stats of the restated wealth."""
    from rlmd_b200 import engine

    n, h, top = 1_000_000, 3000, 100
    codes = _coin_codes(n, h, 8)
    lev = lo64.lev_grid_f64(0.1, 1.0, 0.1, 0.5, -0.4)
    f = lo64.coin_factors_f64(lev, 0.5, -0.4)
    data, data_T = engine.lev_series("discrete", f, lev, 100.0, top, outcomes=codes, dtype=T.float64)
    keep = (1, 1500, h - 1)
    tab = T.as_tensor(f, device="cuda")
    w = T.full((len(lev), n), 100.0, dtype=T.float64, device="cuda")
    kept = {}
    for t in range(h):
        w = w * tab[:, codes[:, t].long()]
        if t in keep:
            kept[t] = w.cpu().numpy()
    assert T.equal(data_T, w)
    sample = np.random.RandomState(0).choice(n, 2000, replace=False)
    want_T = lo64.chain_discrete_f64(codes.cpu().numpy()[sample], f, 100.0)
    assert np.array_equal(data_T.cpu().numpy()[:, sample], want_T)
    got = data.cpu().numpy()
    assert np.array_equal(got[:, 12], np.broadcast_to(lev[:, None], got[:, 12].shape))
    for t in keep:
        want = np.stack([lo64.summary_stats_f64(kept[t][g], top) for g in range(len(lev))])
        assert_stats(got[:, :12, t - 1], want)


def _gbm_x(n, h, seed):
    g = T.Generator(device="cuda").manual_seed(seed)
    return SNP_LOG_MEAN + SNP_SIGMA * T.randn((n, h), generator=g, dtype=T.float64, device="cuda")


def test_gbm_series_f64_h1e4():
    """H = 1e4 with l = 0.4 (finite in fp64, inf in the reference's fp32) and l = 2.0 (overflows in fp64 too)."""
    from rlmd_b200 import engine

    n, h, top = 2000, 10_000, 2
    x = _gbm_x(n, h, 9)
    xc = x.cpu().numpy()
    lev = np.array([-0.4, 0.2, 0.4, 2.0])
    keep = {1, 4321, h - 1}
    want, want_T = lo64.smart_lev_f64(xc, lev, lev, top, 100.0, gbm=True, steps=keep)
    data, data_T = engine.lev_series("gbm", lev, lev, 100.0, top, outcomes=x, dtype=T.float64)
    data, data_T = data.cpu().numpy(), data_T.cpu().numpy()
    rtol = 1e-15 * h
    assert_wealth(data_T, want_T, rtol)
    assert np.isfinite(data_T[2]).all() and np.isinf(data_T[3]).any()
    for t in keep:
        assert_stats(data[:, :12, t - 1], want[:, :12, t - 1], rtol=rtol, median_rtol=rtol)
    stats, fin_T = engine.lev_final_f64("gbm", lev, 100.0, top, x)
    assert np.array_equal(fin_T.cpu().numpy(), data_T)
    assert_stats(stats.cpu().numpy(), want[:, :12, -1], rtol=rtol, median_rtol=rtol)


# ------------------------------------------------------------------ shims
def _run(fn, *args):
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        r = fn(*args)
    return r, buf.getvalue()


def _coin_text(lev, stats, smart):
    s = np.array(stats, dtype=np.float64)
    if smart:
        s[:, 11] = s[:, 10]          # coin_smart_lev prints med_top in the adj line
    return lo.format_final(lev, s) + "\n"


def test_coin_shims_fp64(fp64_default):
    from rlmd_b200 import lev_exp

    n, h, top = 10_000, 300, 1
    oc = (np.random.RandomState(12).rand(n, h) < 0.5).astype(np.float64)
    outcomes = T.as_tensor(oc)          # the reference's Bernoulli draw under a float64 default
    assert outcomes.dtype == T.float64
    dev = T.device("cuda:0")
    lev = lo64.lev_grid_f64(0.1, 1.0, 0.1, 0.5, -0.4)
    f = lo64.coin_factors_f64(lev, 0.5, -0.4)
    want, want_T = lo64.smart_lev_f64(oc.astype(np.uint8), f, lev, top, 100.0)
    (data, data_T), text = _run(lev_exp.coin_smart_lev, dev, outcomes, n, h, top, 100.0, 0.5, -0.4, 0.1, 1.0, 0.1)
    assert data.dtype == T.float64 and data_T.dtype == T.float64 and data.is_cuda and data_T.is_cuda
    assert np.array_equal(data_T.cpu().numpy(), want_T)
    d = data.cpu().numpy()
    assert np.array_equal(d[:, 12], want[:, 12])
    assert_stats(d[:, :12].transpose(0, 2, 1), want[:, :12].transpose(0, 2, 1))
    assert text == _coin_text(lev, want[:, :12, -1], smart=True)
    # the sign flip of the grid (-down_r > up_r)
    lev_neg = lo64.lev_grid_f64(0.1, 0.5, 0.1, 0.3, -0.6)
    assert (lev_neg < 0).all()
    _, text = _run(lev_exp.coin_fixed_final_lev, dev, outcomes, top, 100.0, 0.3, -0.6, 0.1, 0.5, 0.1)
    fin = lo64.fixed_final_lev_f64(oc.astype(np.uint8), lo64.coin_factors_f64(lev_neg, 0.3, -0.6), top, 100.0)
    assert text == _coin_text(lev_neg, fin, smart=False)


def test_gbm_shims_fp64(fp64_default):
    from rlmd_b200 import lev_exp

    n, h, top = 2000, 500, 1
    x = _gbm_x(n, h, 13).cpu()           # host float64, as Normal(...).sample holds it
    dev = T.device("cuda:0")
    lev = lo64.lev_grid_f64(0.2, 2.0, 0.2)
    want, want_T = lo64.smart_lev_f64(x.numpy(), lev, lev, top, 100.0, gbm=True, steps={h - 1})
    (data, data_T), text = _run(lev_exp.gbm_smart_lev, dev, x, n, h, top, 100.0, 0.2, 2.0, 0.2)
    assert data.dtype == T.float64 and data_T.dtype == T.float64
    rtol = 1e-15 * h
    assert_wealth(data_T.cpu().numpy(), want_T, rtol)
    assert_stats(data[:, :12, -1].cpu().numpy(), want[:, :12, -1], rtol=rtol, median_rtol=rtol)
    assert text == lo.format_final(lev, data[:, :12, -1].cpu().numpy()) + "\n"
    assert text.count("lev ") == len(lev)
    _, text = _run(lev_exp.gbm_fixed_final_lev, dev, x, top, 100.0, 0.2, 2.0, 0.2)
    assert text == lo.format_final(lev, want[:, :12, -1]) + "\n"


def _other_paths():
    """dice (smart and final) and GBM with float32 outcomes: outputs and printed text."""
    from rlmd_b200 import lev_exp

    dev = T.device("cuda:0")
    rs = np.random.RandomState(14)
    oc = T.as_tensor(rs.choice(3, size=(3000, 200), p=[1 / 6, 1 / 6, 2 / 3]).astype(np.int64))
    x = T.as_tensor((SNP_LOG_MEAN + SNP_SIGMA * rs.randn(3000, 200)).astype(np.float32))
    out = []
    out.append(_run(lev_exp.dice_smart_lev, dev, oc, 3000, 200, 2, 100.0, 0.5, -0.5, 0.05, 0.1, 1.0, 0.1))
    out.append(_run(lev_exp.dice_fixed_final_lev, dev, oc, 2, 100.0, 0.5, -0.5, 0.05, 0.1, 1.0, 0.1))
    out.append(_run(lev_exp.gbm_smart_lev, dev, x, 3000, 200, 2, 100.0, 0.2, 2.0, 0.2))
    out.append(_run(lev_exp.gbm_fixed_final_lev, dev, x, 2, 100.0, 0.2, 2.0, 0.2))
    return out


def test_other_paths_unchanged_under_fp64_default():
    base = _other_paths()
    old = T.get_default_dtype()
    T.set_default_dtype(T.float64)
    try:
        f64 = _other_paths()
    finally:
        T.set_default_dtype(old)
    for (r0, t0), (r1, t1) in zip(base, f64):
        assert t0 == t1
        if r0 is not None:
            for a, b in zip(r0, r1):
                assert a.dtype == T.float32 and T.equal(a, b)


def test_float32_default_unchanged():
    from rlmd_b200 import lev_exp

    assert T.get_default_dtype() == T.float32
    oc = T.as_tensor((np.random.RandomState(15).rand(2000, 100) < 0.5).astype(np.float64))
    (data, data_T), _ = _run(lev_exp.coin_smart_lev, T.device("cuda:0"), oc, 2000, 100, 1, 100.0, 0.5, -0.4,
                             0.1, 1.0, 0.1)
    assert data.dtype == T.float32 and data_T.dtype == T.float32
    lev = lo.lev_grid(0.1, 1.0, 0.1, 0.5, -0.4)
    want_T = lo.chain_discrete(oc.numpy().astype(np.uint8), lo.coin_factors(lev, 0.5, -0.4), 100.0)
    assert np.array_equal(data_T.cpu().numpy().view(np.uint32), want_T.view(np.uint32))


def test_fp64_path_refuses_a_process_group(fp64_default):
    from rlmd_b200 import lev_exp

    oc = T.zeros((16, 8))
    lev_exp.set_process_group(object())
    try:
        with pytest.raises(ValueError, match="one GPU"):
            _run(lev_exp.coin_smart_lev, T.device("cuda:0"), oc, 16, 8, 1, 100.0, 0.5, -0.4, 0.1, 1.0, 0.1)
        with pytest.raises(ValueError, match="one GPU"):
            _run(lev_exp.gbm_fixed_final_lev, T.device("cuda:0"), oc, 1, 100.0, 0.2, 1.0, 0.2)
    finally:
        lev_exp.set_process_group(None)


# ---------------------------------------------------------------- scripts
def test_scripts_write_float64_files(fp64_default, tmp_path):
    from rlmd_b200 import lev_exp, lev_scripts

    dev = T.device("cuda:0")
    n, h = 4000, 120
    oc = T.as_tensor((np.random.RandomState(16).rand(n, h) < 0.5).astype(np.float64))
    small = dict(s3=(0.5, 0.5, 0.1), r3=(0.7, 0.7, 0.05))
    with contextlib.redirect_stdout(io.StringIO()):
        lev_scripts.coin_flip(str(tmp_path), outcomes=oc, galaxy=False, investors=n, horizon=h, **small)
        d, dT = lev_exp.coin_smart_lev(dev, oc, n, h, 1, 1e2, 0.5, -0.4, 0.1, 1.0, 0.1)
    for name, t in (("coin_inv1_val", d), ("coin_inv1_val_T", dT)):
        a = np.load(os.path.join(tmp_path, name + ".npy"))
        assert a.dtype == np.float64 and np.array_equal(a, t.cpu().numpy(), equal_nan=True)

    xs = [_gbm_x(n, h, 17).cpu(), _gbm_x(n, h, 18).cpu()]
    with contextlib.redirect_stdout(io.StringIO()):
        lev_scripts.gbm(str(tmp_path), outcomes=xs, investors=n, horizon=h)
        d, dT = lev_exp.gbm_smart_lev(dev, xs[1], n, h, 1, 1e2, 0.2, 2.0, 0.2)
    for name, t in (("gbm_snp_inv1_val", d), ("gbm_snp_inv1_val_T", dT)):
        a = np.load(os.path.join(tmp_path, name + ".npy"))
        assert a.dtype == np.float64 and np.array_equal(a, t.cpu().numpy(), equal_nan=True)
    assert np.load(os.path.join(tmp_path, "gbm_op_inv1_val.npy")).dtype == np.float64

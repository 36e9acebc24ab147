"""
gbm_smart_lev(..., method="sum"): the running log-return sum (csrc/gbm_sum.cu) against a torch restatement of
S, the row statistics of the chain route's own wealth dumps, the reference's fixtures and the default route.
"""
import contextlib
import ctypes as C
import io
import math

import numpy as np
import pytest
import torch

import golden_io
from oracle import lev_oracle as lo
from test_coin_lattice_gpu import assert_same_series
from test_oracle_gbm_sum import CHAIN_LEVERAGES
from test_oracle_lev import assert_stats_close
from test_series_ref import STICKY_LEV, sticky_paths

pytestmark = pytest.mark.gpu

GBM_CASES = [c for c in golden_io.LEV_CASES if c["kind"] == "gbm"]
U = 2.0 ** -53


def _x32(n, h, seed, mean=-0.05, sigma=0.447):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return (mean + sigma * torch.randn((n, h), generator=g, device="cuda")).to(torch.float32)


def _ties(n, h, seed):
    """x from {-0.1, 0, 0.1}: heavy ties of S."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    vals = torch.tensor([-0.1, 0.0, 0.1], dtype=torch.float32, device="cuda")
    return vals[torch.randint(0, 3, (n, h), generator=g, device="cuda")]


def torch_S(x):
    """S after every step, [H, N] float64: base + p.to(float64) as tests/series_ref.py (pure IEEE adds)."""
    n, h = x.shape
    out = torch.empty((h, n), dtype=torch.float64, device=x.device)
    if x.dtype == torch.float64:
        s = torch.zeros(n, dtype=torch.float64, device=x.device)
        for t in range(h):
            s = s + x[:, t]
            out[t] = s
        return out
    base = torch.zeros(n, dtype=torch.float64, device=x.device)
    p = torch.zeros(n, dtype=torch.float32, device=x.device)
    for t in range(h):
        p = p + x[:, t]
        out[t] = base + p.to(torch.float64)
        if (t & 31) == 31:
            base, p = out[t].clone(), torch.zeros_like(p)
    return out


def chain_dumps(x, lev, v0):
    """The series chain's own fp32 wealth after every step, [G, H, N] (b200_lev_chunk with a dump)."""
    from rlmd_b200 import _lib, engine
    f = np.ascontiguousarray(lev, dtype=np.float32)
    d, g, _, n, h, dev = engine._fill_desc("gbm", f, v0, x, None, None, "log", 0, 0, None, 0.0, 0.0, 0, None)
    state = torch.empty((5, n), dtype=torch.float64, device=dev)
    dump = torch.empty((g, h, n), dtype=torch.float32, device=dev)
    engine.check(_lib.lib.b200_lev_chunk(C.byref(d), engine.ptr(x), f.ctypes.data_as(C.POINTER(C.c_float)), 0, h,
                                         engine.ptr(state), engine.ptr(dump), engine.stream_ptr()))
    return dump, state


# --------------------------------------------------------------------------------------- S rows
@pytest.mark.parametrize("chunk", [32, 64, 96])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_S_rows_bit_identical(chunk, dtype):
    from rlmd_b200 import engine
    n, h = 1000, 97
    x = _x32(n, h, 3).to(dtype)
    want = torch_S(x)
    state = torch.empty((3, n), dtype=torch.float64, device="cuda")
    for t0 in range(0, h, chunk):
        t1 = min(h, t0 + chunk)
        rows = engine.gbm_sum_chunk(x, t0, t1, state)
        assert torch.equal(rows, want[t0:t1])
    assert torch.equal(state[0], want[-1])
    ext = torch.cat([torch.zeros((1, n), dtype=torch.float64, device="cuda"), want])
    assert torch.equal(state[1], ext.max(0).values) and torch.equal(state[2], ext.min(0).values)
    if dtype == torch.float32:       # the state the series chain and the LOG sweep carry
        _, st5 = chain_dumps(x, [1.0], 100.0)
        assert torch.equal(st5[:3], state)
        st3 = engine.lev_sweep("gbm", np.float32([1.0]), 100.0, outcomes=x, mode="log", want_state=True)["state"]
        assert torch.equal(st3, state)


# ----------------------------------------------------------------------- kernel against rowstats
GRIDS = {"pos": np.float32([0.2, 0.6, 1.0]), "neg": np.float32([-1.0, -0.4]),
         "mixed": np.float32([-1.0, -0.5, 0.0, 0.5, 1.0])}


@pytest.mark.parametrize("grid", sorted(GRIDS))
@pytest.mark.parametrize("n,h,tops,ties", [(2, 5, (1,), False), (3, 40, (1, 2), True), (4099, 40, (1, 7), False),
                                            (4099, 40, (1, 7), True), (1_000_000, 6, (1, 100), False)])
def test_stats_kernel_matches_rowstats_fp32(grid, n, h, tops, ties):
    from rlmd_b200 import engine
    lev = GRIDS[grid]
    x = _ties(n, h, n + h) if ties else _x32(n, h, n + h)
    dump, _ = chain_dumps(x, lev, 100.0)
    state = torch.empty((3, n), dtype=torch.float64, device="cuda")
    S = engine.gbm_sum_chunk(x, 0, h, state)
    for top in tops:
        got = engine.gbm_sum_stats(S, lev, 100.0, top).cpu().numpy()
        want = engine.rowstats(dump.view(-1, n), top).view(len(lev), h, 12).cpu().numpy()
        assert np.array_equal(got[..., 9:12], want[..., 9:12])
        np.testing.assert_allclose(got[..., :9], want[..., :9], rtol=1e-12, atol=0)


@pytest.mark.parametrize("grid", sorted(GRIDS))
@pytest.mark.parametrize("n,h,tops,ties", [(1, 5, (1,), False), (2, 5, (1, 2), False), (3, 40, (1, 3), True),
                                            (4099, 40, (1, 7, 4099), True), (1_000_000, 4, (1, 100), False)])
def test_stats_kernel_matches_rowstats_fp64(grid, n, h, tops, ties):
    """fp64 wealth exp(log V0 + l S) restated in torch, then b200_rowstats_f64; top == n: adj is NaN."""
    from rlmd_b200 import engine
    lev = GRIDS[grid].astype(np.float64)
    x = (_ties(n, h, n + h) if ties else _x32(n, h, n + h)).to(torch.float64)
    state = torch.empty((3, n), dtype=torch.float64, device="cuda")
    S = engine.gbm_sum_chunk(x, 0, h, state)
    l64 = torch.as_tensor(lev, device="cuda")[:, None, None]
    w = torch.exp(math.log(100.0) + l64 * S[None])
    for top in tops:
        got = engine.gbm_sum_stats(S, lev, 100.0, top, dtype=torch.float64).cpu().numpy()
        want = engine.rowstats(w.view(-1, n), top).view(len(lev), h, 12).cpu().numpy()
        assert np.array_equal(np.isnan(got), np.isnan(want))
        np.testing.assert_allclose(got[..., 9:12], want[..., 9:12], rtol=4 * U, atol=0)
        np.testing.assert_allclose(got[..., :9], want[..., :9], rtol=1e-12, atol=0)


# ------------------------------------------------------------------------------- end to end
def run_smart(case, x, method, dtype=torch.float32):
    from rlmd_b200 import lev_exp
    n, h, top, v0 = case["n"], case["h"], case["top"], case["v0"]
    buf = io.StringIO()
    old = torch.get_default_dtype()
    torch.set_default_dtype(dtype)
    try:
        with contextlib.redirect_stdout(buf):
            data, data_T = lev_exp.gbm_smart_lev(torch.device("cuda:0"), torch.as_tensor(x),
                                                 torch.tensor(n, dtype=torch.int32), torch.tensor(h, dtype=torch.int32),
                                                 top, torch.tensor(v0), *case["grid"], method=method)
    finally:
        torch.set_default_dtype(old)
    return data.cpu().numpy(), data_T.cpu().numpy(), buf.getvalue()


def assert_sum_matches_chain(s, c, routed):
    """Routed leverages: order statistics bit for bit, moments within rtol 1e-6 (fp64 summation order);
    the others, and every last column, as the chain's (moments up to the atomics' summation order)."""
    s, c = np.asarray(s), np.asarray(c)
    assert np.array_equal(s[:, 9:13].view(np.uint32), c[:, 9:13].view(np.uint32))
    np.testing.assert_allclose(s[routed, :9], c[routed, :9], rtol=1e-6, atol=0)
    assert_same_series(s[~routed], c[~routed])


@pytest.mark.parametrize("case", GBM_CASES, ids=lambda c: c["name"])
def test_smart_lev_sum_meets_the_reference_and_the_chain(case):
    x = golden_io.draw_outcomes(case)
    gold = golden_io.load("lev_" + case["name"], x)
    data, data_T, text = run_smart(case, x, "sum")
    chain, chain_T, chain_text = run_smart(case, x, "chain")
    assert np.array_equal(data_T.view(np.uint32), chain_T.view(np.uint32))
    assert text == chain_text
    lev = lo.lev_grid(*case["grid"])
    routed = np.array([round(float(v), 6) not in CHAIN_LEVERAGES.get(case["name"], []) for v in lev])
    assert_sum_matches_chain(data, chain, routed)
    got, want = data[:, :, gold["cols"]], gold["data"]
    assert np.array_equal(got[:, 12], want[:, 12])
    if case["name"] != "gbm_overflow":
        assert_stats_close(got[:, :12], want[:, :12], rtol=2e-5 * max(1.0, case["h"] / 500))
    else:
        normal = np.abs(want[:, :12]) > 1e-30
        assert_stats_close(np.where(normal, got[:, :12], 0), np.where(normal, want[:, :12], 0), rtol=2e-4)


def _sum_vs_chain(x, lev, top, v0, chunk_steps=None):
    from rlmd_b200 import engine
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    data, data_T, routed = engine.gbm_series_sum(lev, lev, v0, top, x, chunk_steps=chunk_steps)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    chain, chain_T = engine.lev_series("gbm", lev, lev, v0, top, outcomes=x)
    assert torch.equal(data_T.view(torch.int32), chain_T.view(torch.int32))      # NaN-aware, bit for bit
    assert_sum_matches_chain(data.cpu().numpy(), chain.cpu().numpy(), routed)
    return routed, peak


@pytest.mark.parametrize("grid", [(-1.0, 1.0, 0.2, 0.05, math.sqrt(0.2)), (0.2, 2.0, 0.2, 0.0540025395205692,
                                                                          0.1897916175617430)],
                         ids=["gbm_op", "gbm_snp"])
def test_production_shape_1e6_x_500(grid):
    """The GBM script's size: every leverage routed; besides data / data_T the route holds one chunk of S
    (256 MB) and the LOG sweep's state, never [G, steps, N] wealth."""
    from rlmd_b200 import lev_exp
    lo_, hi_, inc, mu, sigma = grid
    n, h, top = 1_000_000, 500, 100
    x = _x32(n, h, 11, mean=mu - sigma ** 2 / 2, sigma=sigma)
    lev = np.asarray(lev_exp.param_range(lo_, hi_, inc), dtype=np.float32)
    routed, peak = _sum_vs_chain(x, lev, top, 100.0)
    assert routed.all()
    g = len(lev)
    out = g * 13 * (h - 1) * 4 + g * n * 4
    assert peak <= out + (256 << 20) + 3 * 8 * n + (128 << 20), peak


def test_production_shape_gbm10():
    """tests/test_series_shapes_gpu.py's gbm10: 1e6 x 700, l = -1..1.  At l = -1 the chain of the investor with
    the lowest S passes ln FLT_MAX (inf for good): that leverage keeps the chain, the other ten are routed."""
    from rlmd_b200 import engine
    lev = lo.lev_grid(-1.0, 1.0, 0.2)
    x = engine.lev_draw("gbm", 1_000_000, 700, seed=705, log_mean=-0.05, sigma=0.447)
    routed, _ = _sum_vs_chain(x, lev, 100, 100.0)
    assert routed.tolist() == [False] + [True] * (len(lev) - 1)
    _, chain_T = engine.lev_series("gbm", lev[:1], lev[:1], 100.0, 100, outcomes=x)
    assert torch.isinf(chain_T).any()


def test_sticky_paths_fall_back():
    x = torch.as_tensor(sticky_paths(), device="cuda")
    routed, _ = _sum_vs_chain(x, STICKY_LEV, 2, 100.0)
    assert not routed.any()
    # a grid of small leverages stays in range on the same paths
    routed, _ = _sum_vs_chain(x, np.float32([-0.1, 0.05, 0.1]), 2, 100.0)
    assert routed.all()


@pytest.mark.parametrize("bad", [float("nan"), float("inf"), -float("inf")])
def test_non_finite_returns_send_the_grid_to_the_chain(bad):
    x = _x32(3000, 70, 21)
    x[17, 40] = bad
    routed, _ = _sum_vs_chain(x, np.float32([-0.5, 0.0, 0.5]), 3, 100.0)
    assert not routed.any()


@pytest.mark.parametrize("chunk", [32, 64, 96])
def test_chunk_steps_invariance(chunk):
    from rlmd_b200 import engine
    x = _x32(5000, 230, 23)
    lev = lo.lev_grid(-1.0, 1.0, 0.2)
    a = engine.gbm_series_sum(lev, lev, 100.0, 3, x)
    b = engine.gbm_series_sum(lev, lev, 100.0, 3, x, chunk_steps=chunk)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    x64 = x.double()
    a = engine.gbm_series_sum(lev, lev, 100.0, 3, x64, dtype=torch.float64)
    b = engine.gbm_series_sum(lev, lev, 100.0, 3, x64, dtype=torch.float64, chunk_steps=chunk)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


# ------------------------------------------------------------------------------------- float64
def f64_bound(x: torch.Tensor, lev, v0: float) -> float:
    """
    Worst-case relative difference between the fp64 chain's wealth V0 prod fl(exp(fl(l x_t))) and the
    closed form fl(exp(fl(log V0 + fl(l S)))), S the sequential fp64 sum, u = 2^-53, exp within 1 ulp (2u):
    per step the chain's log wealth errs by at most u |l x_t| (product l x) + 2u (exp) + u (product), and the
    closed form by |l| (H + 1) max|S| u (the H additions of S and the product l S) + u |log V0 + l S| + 2u.
    Order statistics move by at most that (a rank is monotone in every member); means add the two fp64
    summations (n u each); MAD and std are compared against their group's mean at twice the bound.
    """
    h = x.shape[1]
    sum_abs = float(x.abs().sum(1).max())
    smax = float(torch_S_abs_max(x))
    lv0 = abs(math.log(v0))
    d = max(U * (3 * h + abs(l) * sum_abs + abs(l) * (h + 2) * smax + lv0 + 2) for l in np.asarray(lev))
    return 2 * (math.expm1(d) + 2 * x.shape[0] * U)


def torch_S_abs_max(x):
    s = torch.zeros(x.shape[0], dtype=torch.float64, device=x.device)
    m = torch.zeros_like(s)
    for t in range(x.shape[1]):
        s = s + x[:, t]
        m = torch.maximum(m, s.abs())
    return m.max()


def assert_f64_close(got, want, tol):
    got, want = np.asarray(got), np.asarray(want)
    assert np.array_equal(np.isnan(got), np.isnan(want))
    assert np.array_equal(np.isinf(got), np.isinf(want)) and np.array_equal(got[np.isinf(got)], want[np.isinf(want)])
    scale = np.abs(want).copy()
    for j in range(3, 9):
        m = want[:, j % 3]
        scale[:, j] = np.maximum(scale[:, j], np.abs(np.where(np.isfinite(m), m, 0.0)))
    fin = np.isfinite(want)
    bad = fin & (np.abs(got - want) > tol * scale)
    assert not bad.any(), (np.argwhere(bad)[:5], got[bad][:5], want[bad][:5], tol)


def _f64_against_chain(x, lev, top, v0):
    from rlmd_b200 import engine
    data, data_T, routed = engine.gbm_series_sum(lev, lev, v0, top, x, dtype=torch.float64)
    want, want_T = engine.lev_series("gbm", lev, lev, v0, top, outcomes=x, dtype=torch.float64)
    assert torch.equal(data_T, want_T)
    data, want = data.cpu().numpy(), want.cpu().numpy()
    tol = f64_bound(x, lev[routed], v0) if routed.any() else 0.0
    for g in range(len(lev)):
        if routed[g]:
            for c in range(data.shape[2]):
                assert_f64_close(data[g:g + 1, :12, c], want[g:g + 1, :12, c], tol)
        else:
            assert np.array_equal(data[g, 9:], want[g, 9:], equal_nan=True)
            np.testing.assert_allclose(data[g, :9], want[g, :9], rtol=1e-12, atol=0)
    return routed


def test_f64_1e6_x_500():
    x = _x32(1_000_000, 500, 31, mean=0.0540025395205692 - 0.1897916175617430 ** 2 / 2,
             sigma=0.1897916175617430).double()
    assert _f64_against_chain(x, np.arange(1, 11) * 0.2, 100, 100.0).all()


def test_f64_h1e4():
    """test_lev_fp64_gpu's H = 1e4 inputs: l = 2.0 overflows fp64 and keeps the chain."""
    from test_lev_fp64_gpu import _gbm_x
    x = _gbm_x(2000, 10_000, 9)
    routed = _f64_against_chain(x, np.array([-0.4, 0.2, 0.4, 2.0]), 2, 100.0)
    assert routed.tolist() == [True, True, True, False]


def test_f64_sums_overflow():
    """Wealth just inside DBL_MAX: the fp64 sums overflow - inf / NaN where lev_series_f64 has them."""
    g = torch.Generator(device="cuda").manual_seed(41)
    n, h = 1000, 64
    x = 0.5 + 0.01 * torch.randn((n, h), generator=g, dtype=torch.float64, device="cuda")
    x[:, h // 2:] = 0.0          # S (and every investor's wealth) stays near its maximum for the second half
    smax = float(torch_S(x).max())
    l_over = (709.0 - math.log(100.0)) / smax
    lev = np.array([0.1, l_over])
    routed = _f64_against_chain(x, lev, 3, 100.0)
    assert routed.all()
    from rlmd_b200 import engine
    data, _, _ = engine.gbm_series_sum(lev, lev, 100.0, 3, x, dtype=torch.float64)
    assert np.isinf(data[1, 0, -2].item())                     # the mean of all overflows


# ------------------------------------------------------------------------------------------- API
def test_method_validation_and_process_group():
    from rlmd_b200 import engine, lev_exp
    case = golden_io.lev_case("gbm_snp_top4")
    x = golden_io.draw_outcomes(case)
    with pytest.raises(ValueError):
        run_smart(case, x, "counts")
    with pytest.raises(ValueError):
        run_smart(case, x, "lattice")
    lev = lo.lev_grid(*case["grid"])
    xt = torch.as_tensor(x, device="cuda")
    with pytest.raises(ValueError):
        engine.lev_series("gbm", lev, lev, 100.0, 2, outcomes=xt, method="counts")
    with pytest.raises(ValueError):
        engine.lev_series("gbm", lev, lev, 100.0, 2, outcomes=xt, method="sum", n_total=2 * x.shape[0])
    with pytest.raises(ValueError):
        engine.lev_series("gbm", lev, lev, 100.0, 2, outcomes=xt, method="sum", group=object())
    lev_exp.set_process_group(object())
    try:
        with pytest.raises(ValueError):
            run_smart(case, x, "sum")
        with lev_exp.series_method("sum"), pytest.raises(ValueError):
            run_smart(case, x, None)
    finally:
        lev_exp.set_process_group(None)


def test_series_method_nesting():
    from rlmd_b200 import lev_exp
    case = golden_io.lev_case("gbm_testscale")
    x = golden_io.draw_outcomes(case)
    chain, _, _ = run_smart(case, x, "chain")
    summ, _, _ = run_smart(case, x, "sum")
    with lev_exp.series_method("sum"):
        inside, _, _ = run_smart(case, x, None)
        with lev_exp.series_method("counts"):
            nested, _, _ = run_smart(case, x, None)          # "counts" is the coin's: GBM takes the chain
        with lev_exp.series_method("chain"):
            nested2, _, _ = run_smart(case, x, None)
    after, _, _ = run_smart(case, x, None)
    routed = np.ones(chain.shape[0], dtype=bool)
    np.testing.assert_array_equal(inside[:, :, :-1], summ[:, :, :-1])
    assert_same_series(nested, chain)
    assert_same_series(nested2, chain)
    assert_same_series(after, chain)
    assert_sum_matches_chain(inside, chain, routed)
    with pytest.raises(ValueError):
        lev_exp.series_method("lattice")


def test_lev_scripts_gbm_series_sum():
    from rlmd_b200 import lev_scripts
    with contextlib.redirect_stdout(io.StringIO()):
        a = lev_scripts.gbm(None, series="sum", seed=5, investors=5000, horizon=60)
        b = lev_scripts.gbm(None, series="chain", seed=5, investors=5000, horizon=60)
    for name in ("gbm_op", "gbm_snp"):
        assert np.array_equal(a[name + "_inv1_val_T"], b[name + "_inv1_val_T"])
        routed = np.ones(a[name + "_inv1_val"].shape[0], dtype=bool)
        assert_sum_matches_chain(a[name + "_inv1_val"], b[name + "_inv1_val"], routed)


def test_few_investors_long_horizon():
    """N = 300, H = 7e4: chunks of at most 2048 steps (the statistics take at most 65535 rows per call), the
    same columns as the chain."""
    x = _x32(300, 70_000, 51, mean=0.0, sigma=0.01)
    routed, peak = _sum_vs_chain(x, np.float32([-1.0, 0.5, 1.0]), 2, 100.0)
    assert routed.all()
    assert peak <= 400 << 20, peak


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("h", [1, 2])
def test_short_horizons_route_nothing(h, dtype):
    """H <= 2: no column comes from the running sum (column H-2 is the chain's), so nothing is routed."""
    from rlmd_b200 import engine
    x = _x32(500, h, 53).to(dtype)
    lev = np.array([-0.5, 0.5])
    data, data_T, routed = engine.gbm_series_sum(lev, lev, 100.0, 3, x, dtype=dtype)
    chain, chain_T = engine.lev_series("gbm", lev, lev, 100.0, 3, outcomes=x, dtype=dtype)
    assert not routed.any()
    assert torch.equal(data_T, chain_T)
    assert data.shape == chain.shape
    if h == 2:
        assert torch.equal(data[:, 9:13], chain[:, 9:13])

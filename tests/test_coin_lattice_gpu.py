"""
coin_smart_lev(..., method="counts"): the up-move count lattice (csrc/coin_lattice.cu) against the NumPy
restatement (oracle/coin_lattice_oracle.py), the reference's coin fixtures and the default chain route.
"""
import contextlib
import io
import math

import numpy as np
import pytest
import torch

import golden_io
from oracle import coin_lattice_oracle as cl
from oracle import lev_oracle as lo
from oracle import lev_oracle_f64 as lo64
from test_oracle_coin_lattice import CHAIN_LEVERAGES, assert_lattice_close, lattice_tol

pytestmark = pytest.mark.gpu

COIN_CASES = [c for c in golden_io.LEV_CASES if c["kind"] == "coin"]


def device_exp(x):
    """The device's fp64 exp (the kernel's): NumPy's can differ in the last ulp."""
    return torch.exp(torch.as_tensor(np.asarray(x, dtype=np.float64), device="cuda")).cpu().numpy()


def codes_of(oc: np.ndarray, layout: str):
    from rlmd_b200 import engine
    if layout == "u8":          # engine.encode_codes: rows padded to 16 bytes (vector loads)
        return engine.encode_codes(torch.as_tensor(oc), n_outcomes=2)
    if layout == "u8_tight":    # row stride H: unaligned rows (byte loads)
        return torch.as_tensor(oc, device="cuda")
    return engine.pack_codes(engine.encode_codes(torch.as_tensor(oc), n_outcomes=2), bits=1)


def walk_counts(codes, h, chunk):
    """(hist, kmin, kmax) of every step and the final k state, walked in chunks of `chunk` steps."""
    from rlmd_b200 import engine
    n = codes.shape[0]
    k = torch.full((n,), -7, dtype=torch.int32, device="cuda")      # ignored at t_begin = 0
    rows = []
    for t0 in range(0, h, chunk):
        hs, lo_, hi_ = engine.coin_lattice_count(codes, t0, min(h, t0 + chunk), k)
        rows.append((hs.cpu().numpy(), lo_.cpu().numpy(), hi_.cpu().numpy()))
    return (np.concatenate([r[0] for r in rows]), np.concatenate([r[1] for r in rows]),
            np.concatenate([r[2] for r in rows]), k.cpu().numpy())


COUNT_SHAPES = [
    # (n, h, p_up, chunk steps)
    (1, 2, 0.5, (1, 2)),
    (5, 2, 0.5, (1,)),
    (77, 33, 0.4, (1, 7, 33)),
    (1000, 97, 0.5, (32, 40, 97)),
    (4099, 301, 0.6, (64, 301)),
    (200000, 37, 0.5, (37,)),            # several blocks, two investors per thread
    (700000, 45, 0.5, (45,)),            # eight investors per thread
]


@pytest.mark.parametrize("layout", ["u8", "u8_tight", "bits1"])
@pytest.mark.parametrize("shape", COUNT_SHAPES, ids=lambda s: f"n{s[0]}_h{s[1]}")
def test_count_matches_oracle(shape, layout):
    n, h, p, chunks = shape
    rs = np.random.RandomState(n + h)
    oc = (rs.random_sample((n, h)) < p).astype(np.uint8)
    want = cl.lattice_hist(oc)
    codes = codes_of(oc, layout)
    for chunk in chunks:
        got = walk_counts(codes, h, chunk)
        for a, b in zip(got, want):
            assert np.array_equal(a, b), (chunk, layout)


def test_count_wide_band_and_long_horizon():
    """Investors that drift apart (half nearly always up, half nearly always down: a block's band outgrows its
    shared-memory window), and H = 1e4 walked in chunks."""
    rs = np.random.RandomState(11)
    n, h = 3000, 10000
    p = np.where(np.arange(n) % 2 == 0, 0.97, 0.03)[:, None]
    oc = (rs.random_sample((n, h)) < p).astype(np.uint8)
    want = cl.lattice_hist(oc)
    for layout, chunk in (("u8", 4096), ("bits1", 3000)):
        got = walk_counts(codes_of(oc, layout), h, chunk)
        for a, b in zip(got, want):
            assert np.array_equal(a, b), layout


STATS_CASES = [
    # (name, n, h, p_up, up_r, down_r, lev, top)
    ("top1", 1001, 64, 0.5, 0.5, -0.4, (0.2, 0.5, 1.0), 1),
    ("top7_ties", 300, 40, 0.5, 0.5, -0.4, (0.3, 0.9), 7),       # few k values: the threshold's bin is split
    ("negated", 777, 33, 0.6, 0.3, -0.5, (-0.2, -0.6), 2),      # -down_r > up_r: wealth falls with k
    ("one_investor", 1, 20, 0.5, 0.5, -0.4, (0.5,), 1),
]


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64], ids=["fp32", "fp64"])
@pytest.mark.parametrize("case", STATS_CASES, ids=lambda c: c[0])
def test_stats_match_oracle(case, dtype):
    from rlmd_b200 import engine, lev_exp
    _, n, h, p, up_r, down_r, lev, top = case
    rs = np.random.RandomState(n)
    oc = (rs.random_sample((n, h)) < p).astype(np.uint8)
    f32 = dtype == torch.float32
    lev = np.asarray(lev, dtype=np.float32 if f32 else np.float64)
    f = lev_exp.coin_factor_table(lev, up_r, down_r) if f32 else lev_exp.coin_factor_table64(lev, up_r, down_r)
    tops = (top,) if f32 or n == 1 else (top, n)        # top == n: the adj group is empty (nan)
    codes = codes_of(oc, "u8")
    k = torch.zeros(n, dtype=torch.int32, device="cuda")
    hs, kmin, kmax = engine.coin_lattice_count(codes, 0, h, k)
    hist_np = hs.cpu().numpy()
    for tp in tops:
        got, fails = engine.coin_lattice_stats(hs, kmin, kmax, 0, f, 100.0, tp, n, dtype=dtype)
        got = got.cpu().numpy()
        want = cl.lattice_stats(hist_np, 0, f, 100.0, tp, f32, exp=device_exp)
        assert np.array_equal(got[..., 9:12], want[..., 9:12], equal_nan=True), "order statistics must be exact"
        assert np.array_equal(np.isnan(got), np.isnan(want))
        scale = np.abs(want[..., :9]).copy()
        for j in range(3, 9):
            scale[..., j] = np.maximum(scale[..., j], np.abs(want[..., j % 3]))
        fin = np.isfinite(want[..., :9])
        assert (np.abs(got[..., :9] - want[..., :9])[fin] <= 1e-12 * scale[fin]).all()
        ok = cl.route_ok(f, 100.0, kmin.cpu().numpy(), kmax.cpu().numpy(), 0, f32)
        assert np.array_equal(fails.cpu().numpy() == 0, ok)


def assert_same_series(a, b):
    """Two runs of the series: medians and the leverage row bit for bit; the moments up to summation order
    (the row statistics of the chain's columns add fp64 partial sums with atomics)."""
    a, b = np.asarray(a), np.asarray(b)
    assert np.array_equal(a[:, 9:13].view(np.uint32 if a.dtype == np.float32 else np.uint64),
                          b[:, 9:13].view(np.uint32 if b.dtype == np.float32 else np.uint64))
    np.testing.assert_allclose(a[:, :9], b[:, :9], rtol=1e-6, atol=0)


def run_smart(case, oc, method, dtype=torch.float32):
    from rlmd_b200 import lev_exp
    n, h, top, v0 = case["n"], case["h"], case["top"], case["v0"]
    buf = io.StringIO()
    old = torch.get_default_dtype()
    torch.set_default_dtype(dtype)
    try:
        with contextlib.redirect_stdout(buf):
            data, data_T = lev_exp.coin_smart_lev(torch.device("cuda:0"), torch.tensor(oc.astype(np.float32)),
                                                  torch.tensor(n, dtype=torch.int32), torch.tensor(h, dtype=torch.int32),
                                                  top, torch.tensor(v0), case["up_r"], case["down_r"], *case["grid"],
                                                  method=method)
    finally:
        torch.set_default_dtype(old)
    return data.cpu().numpy(), data_T.cpu().numpy(), buf.getvalue()


@pytest.mark.parametrize("case", COIN_CASES, ids=lambda c: c["name"])
def test_smart_lev_counts_meets_the_reference(case):
    from rlmd_b200 import engine, lev_exp
    oc = golden_io.draw_outcomes(case)
    gold = golden_io.load("lev_" + case["name"], oc)
    data, data_T, text = run_smart(case, oc, "counts")
    ref, ref_T, ref_text = run_smart(case, oc, "chain")
    assert data.dtype == np.float32 and data.shape == ref.shape
    # data_T: the chain's, bit for bit; the printed report is the default route's
    assert np.array_equal(data_T.view(np.uint32), gold["data_T"].view(np.uint32))
    assert text == ref_text
    # the last column: row statistics of the same data_T (medians exact; moments up to summation order)
    assert np.array_equal(data[:, 9:13, -1].view(np.uint32), ref[:, 9:13, -1].view(np.uint32))
    np.testing.assert_allclose(data[:, :9, -1], ref[:, :9, -1], rtol=1e-6, atol=0)
    cols = gold["cols"]
    got, want = data[:, :, cols], gold["data"]
    assert np.array_equal(got[:, 12], want[:, 12])
    assert np.array_equal(got[:, 9:12, -1].view(np.uint32), want[:, 9:12, -1].view(np.uint32))
    assert_lattice_close(np.moveaxis(got[:, :12], 1, 2), np.moveaxis(want[:, :12], 1, 2), lattice_tol(case["h"]))
    # the route: these leverages keep the chain, and their columns are the default route's statistics
    lev = lo.lev_grid(*case["grid"], case["up_r"], case["down_r"])
    f = lev_exp.coin_factor_table(lev, case["up_r"], case["down_r"])
    _, _, routed = engine.coin_series_counts(f, lev, case["v0"], case["top"], engine.encode_codes(oc, n_outcomes=2))
    assert [round(abs(float(x)), 6) for x in lev[~routed]] == CHAIN_LEVERAGES.get(case["name"], [])
    assert_same_series(data[~routed], ref[~routed])


@pytest.mark.parametrize("chunk", [1, 7, 64])
def test_counts_is_chunk_invariant(chunk):
    from rlmd_b200 import engine, lev_exp
    case = golden_io.lev_case("coin_top7")
    oc = golden_io.draw_outcomes(case)
    lev = lo.lev_grid(*case["grid"], case["up_r"], case["down_r"])
    f = lev_exp.coin_factor_table(lev, case["up_r"], case["down_r"])
    codes = engine.encode_codes(oc, n_outcomes=2)
    a = engine.coin_series_counts(f, lev, 100.0, 7, codes)
    b = engine.coin_series_counts(f, lev, 100.0, 7, codes, chunk_steps=chunk)
    assert a[2].all() and np.array_equal(a[2], b[2]) and torch.equal(a[1], b[1])
    assert torch.equal(a[0][:, :, :-1], b[0][:, :, :-1])         # the lattice's columns: bit for bit
    assert_same_series(a[0].cpu().numpy(), b[0].cpu().numpy())


def f64_inputs(n, h, seed, p=0.5, grid=(0.1, 1.0, 0.1)):
    from rlmd_b200 import engine, lev_exp
    lev = lev_exp._grid64(*grid, 0.5, -0.4)
    f = lev_exp.coin_factor_table64(lev, 0.5, -0.4)
    codes = engine.lev_draw("discrete", n, h, seed=seed, probs=(1 - p, p))
    return lev, f, codes


@pytest.mark.parametrize("shape", [(10000, 300, 1), (1_000_000, 3000, 1)], ids=["testscale", "C1_smart"])
def test_f64_counts_against_the_fp64_chain(shape):
    """Under a float64 default: every leverage routed, within 1e-12 * max(1, H/3000) of lev_series_f64."""
    from rlmd_b200 import engine
    n, h, top = shape
    lev, f, codes = f64_inputs(n, h, seed=h)
    data, data_T, routed = engine.coin_series_counts(f, lev, 100.0, top, codes, dtype=torch.float64)
    assert routed.all() and data.dtype == torch.float64
    ref, ref_T = engine.lev_series_f64("discrete", f, lev, 100.0, top, codes)
    assert torch.equal(data_T, ref_T)
    assert torch.equal(data[:, 9:13], ref[:, 9:13]) or _close(data[:, 9:13], ref[:, 9:13], 1e-12 * max(1.0, h / 3000))
    assert _close(data[:, :9], ref[:, :9], 1e-12 * max(1.0, h / 3000), mean_scaled=True)
    assert torch.equal(data[:, :, -1][:, 9:], ref[:, :, -1][:, 9:])


def _close(a, b, rtol, mean_scaled=False):
    a, b = a.double(), b.double()
    if not torch.equal(torch.isnan(a), torch.isnan(b)):
        return False
    scale = b.abs().clone()
    if mean_scaled:
        for j in range(3, 9):
            scale[:, j] = torch.maximum(scale[:, j], b[:, j % 3].abs())
    fin = torch.isfinite(b)
    return bool(((a - b).abs()[fin] <= rtol * scale[fin]).all())


def test_f64_counts_meets_the_oracle_at_testscale():
    """coin_testscale under a float64 default through coin_smart_lev: the all-fp64 restatement of the reference."""
    case = golden_io.lev_case("coin_testscale")
    oc = golden_io.draw_outcomes(case)
    data, data_T, text = run_smart(case, oc, "counts", torch.float64)
    ref, ref_T, ref_text = run_smart(case, oc, "chain", torch.float64)
    assert data.dtype == np.float64 and np.array_equal(data_T, ref_T) and text == ref_text
    lev = lo64.lev_grid_f64(*case["grid"], case["up_r"], case["down_r"])
    steps = set(golden_io.kept_columns(case))
    want, want_T = lo64.smart_lev_f64(oc, lo64.coin_factors_f64(lev, case["up_r"], case["down_r"]), lev,
                                      case["top"], case["v0"], steps={c + 1 for c in steps})
    assert np.array_equal(data_T, want_T)
    cols = sorted(steps)
    assert _close(torch.as_tensor(data[:, :12, cols]), torch.as_tensor(want[:, :12, cols]), 1e-12, mean_scaled=True)


def test_series_method_context_and_default():
    from rlmd_b200 import lev_exp
    case = golden_io.lev_case("coin_long")
    oc = golden_io.draw_outcomes(case)
    default, _, _ = run_smart(case, oc, None)
    chain, _, _ = run_smart(case, oc, "chain")
    counts, _, _ = run_smart(case, oc, "counts")
    routed = np.array([abs(float(x)) not in CHAIN_LEVERAGES["coin_long"] for x in default[:, 12, 0]])
    assert_same_series(default, chain)                              # the default is the chain
    assert not np.array_equal(default[routed, 9:12], counts[routed, 9:12])
    with lev_exp.series_method("counts"):
        inside, _, _ = run_smart(case, oc, None)
        with lev_exp.series_method("chain"):
            nested, _, _ = run_smart(case, oc, None)
    after, _, _ = run_smart(case, oc, None)
    assert np.array_equal(inside[routed, :, :-1], counts[routed, :, :-1], equal_nan=True)
    assert_same_series(inside, counts)
    assert_same_series(nested, chain)
    assert_same_series(after, chain)
    with pytest.raises(ValueError):
        lev_exp.series_method("lattice")


def test_counts_refuses_a_process_group():
    from rlmd_b200 import lev_exp
    case = golden_io.lev_case("coin_top7")
    oc = golden_io.draw_outcomes(case)
    lev_exp.set_process_group(object())
    try:
        with pytest.raises(ValueError):
            run_smart(case, oc, "counts")
        with lev_exp.series_method("counts"), pytest.raises(ValueError):
            run_smart(case, oc, None)
    finally:
        lev_exp.set_process_group(None)


def test_lev_series_method_counts():
    from rlmd_b200 import engine, lev_exp
    case = golden_io.lev_case("coin_flip_sign")
    oc = golden_io.draw_outcomes(case)
    lev = lo.lev_grid(*case["grid"], case["up_r"], case["down_r"])
    f = lev_exp.coin_factor_table(lev, case["up_r"], case["down_r"])
    codes = engine.encode_codes(oc, n_outcomes=2)
    a = engine.lev_series("discrete", f, lev, 100.0, 2, outcomes=codes, method="counts")
    b = engine.coin_series_counts(f, lev, 100.0, 2, codes)
    assert torch.equal(a[0][:, :, :-1], b[0][:, :, :-1]) and torch.equal(a[1], b[1])
    assert_same_series(a[0].cpu().numpy(), b[0].cpu().numpy())
    dice = lev_exp.dice_factor_table(lev, 0.5, -0.5, 0.05)
    with pytest.raises(ValueError):
        engine.lev_series("discrete", dice, lev, 100.0, 2, outcomes=codes, method="counts")
    with pytest.raises(ValueError):
        engine.lev_series("gbm", lev, lev, 100.0, 2, n_investors=10, horizon=10, method="counts")
    with pytest.raises(ValueError):
        engine.lev_series("discrete", f, lev, 100.0, 2, outcomes=codes, method="tally")


def test_lattice_refuses_bad_arguments():
    from rlmd_b200 import engine
    from rlmd_b200._lib import B200Error
    codes = engine.encode_codes(np.zeros((10, 40), dtype=np.uint8), n_outcomes=2)
    k = torch.zeros(10, dtype=torch.int32, device="cuda")
    with pytest.raises(B200Error):
        engine.coin_lattice_count(codes, 5, 5, k)
    with pytest.raises(B200Error):
        engine.coin_lattice_count(codes, 0, 41, k)
    with pytest.raises(ValueError):
        engine.coin_lattice_count(engine.pack_codes(codes, bits=2), 0, 40, k)
    hs, lo_, hi_ = engine.coin_lattice_count(codes, 0, 40, k)
    with pytest.raises(B200Error):
        engine.coin_lattice_stats(hs, lo_, hi_, 0, np.array([[0.6, 1.5]]), 100.0, 11, 10)
    assert math.isfinite(float(engine.coin_lattice_stats(hs, lo_, hi_, 0, np.array([[0.6, 1.5]]), 100.0, 10,
                                                        10)[0][0, -1, 0]))

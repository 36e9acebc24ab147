"""
dice_smart_lev / dice_sh_smart_lev(..., method="tuples"): the count-tuple lattice (csrc/dice_lattice.cu) against
the NumPy restatement (oracle/dice_lattice_oracle.py), the reference's dice fixtures and the default chain route.
"""
import contextlib
import io
import os

import numpy as np
import pytest
import torch

import golden_io
from oracle import dice_lattice_oracle as dl
from oracle import lev_oracle as lo
from test_oracle_coin_lattice import assert_lattice_close, lattice_tol
from test_oracle_dice_lattice import CHAIN_LEVERAGES, DICE_CASES, case_factors

pytestmark = pytest.mark.gpu

DICE_P = (1 / 6, 1 / 6, 2 / 3)


def device_exp(x):
    """The device's fp64 exp (the kernel's): NumPy's can differ in the last ulp."""
    return torch.exp(torch.as_tensor(np.asarray(x, dtype=np.float64), device="cuda")).cpu().numpy()


def draw(n, h, p, seed):
    return np.random.RandomState(seed).choice(3, size=(n, h), p=p).astype(np.uint8)


def codes_of(oc: np.ndarray, layout: str):
    from rlmd_b200 import engine
    if layout == "u8":          # engine.encode_codes: rows padded to 16 bytes (vector loads)
        return engine.encode_codes(torch.as_tensor(oc), n_outcomes=3)
    return torch.as_tensor(oc, device="cuda")      # row stride H: unaligned rows (byte loads)


def step_offsets(bounds: np.ndarray) -> np.ndarray:
    area = (bounds[1] - bounds[0] + 1) * (bounds[3] - bounds[2] + 1)
    return np.concatenate([[0], np.cumsum(area)]).astype(np.int64)


def walk(codes, h, chunk):
    """(bounds [4,H], per-step boxes, bounds state, count state) walked in chunks of `chunk` steps."""
    from rlmd_b200 import engine
    n = codes.shape[0]
    ab = torch.full((2, n), -7, dtype=torch.int32, device="cuda")      # ignored at t_begin = 0
    cols = []
    for t0 in range(0, h, chunk):
        cols.append(engine.dice_lattice_bounds(codes, t0, min(h, t0 + chunk), ab).cpu().numpy())
    bounds = np.concatenate(cols, axis=1)
    abc = torch.full((2, n), -7, dtype=torch.int32, device="cuda")
    boxes = []
    for t0 in range(0, h, chunk):
        t1 = min(h, t0 + chunk)
        b = bounds[:, t0:t1]
        off = step_offsets(b)
        hs = engine.dice_lattice_count(codes, t0, t1, abc, torch.as_tensor(b, device="cuda").contiguous(),
                                       torch.as_tensor(off[:-1], device="cuda"), int(off[-1])).cpu().numpy()
        for i in range(t1 - t0):
            boxes.append(hs[off[i]:off[i + 1]].reshape(b[1, i] - b[0, i] + 1, -1))
    return bounds, boxes, ab.cpu().numpy(), abc.cpu().numpy()


COUNT_SHAPES = [
    # (n, h, probabilities of up / down / mid, chunk steps)
    (1, 2, DICE_P, (1, 2)),
    (5, 2, DICE_P, (1,)),
    (77, 33, (0.3, 0.3, 0.4), (1, 7, 33)),
    (1000, 97, DICE_P, (32, 40, 97)),
    (4099, 301, (0.05, 0.8, 0.15), (64, 301)),          # skewed
    (200000, 37, DICE_P, (37,)),                       # several blocks, two investors per thread
    (700000, 45, (0.45, 0.1, 0.45), (13, 45)),         # four investors per thread
]


@pytest.mark.parametrize("layout", ["u8", "u8_tight"])
@pytest.mark.parametrize("shape", COUNT_SHAPES, ids=lambda s: f"n{s[0]}_h{s[1]}")
def test_bounds_counts_and_state_match_oracle(shape, layout):
    n, h, p, chunks = shape
    oc = draw(n, h, p, n + h)
    want_bounds, want_ab = dl.lattice_bounds(oc)
    ab = dl.tuple_counts(oc)
    want_boxes = [dl.step_box(ab, t) for t in range(h)]
    codes = codes_of(oc, layout)
    for chunk in chunks:
        bounds, boxes, st_bounds, st_count = walk(codes, h, chunk)
        assert np.array_equal(bounds, want_bounds), (chunk, layout)
        assert np.array_equal(st_bounds, want_ab) and np.array_equal(st_count, want_ab), (chunk, layout)
        for t in range(h):
            assert np.array_equal(boxes[t], want_boxes[t]), (chunk, layout, t)


def test_counts_at_production_shape():
    """1e6 x 700 against a torch restatement: cumulative counts per row, then bincount per step."""
    from rlmd_b200 import engine
    n, h = 1_000_000, 700
    codes = engine.lev_draw("discrete", n, h, seed=17, probs=DICE_P)
    ab = torch.empty((2, n), dtype=torch.int32, device="cuda")
    bounds = engine.dice_lattice_bounds(codes, 0, h, ab)
    a = torch.cumsum(codes[:, :h] == 0, dim=1, dtype=torch.int32)
    b = torch.cumsum(codes[:, :h] == 1, dim=1, dtype=torch.int32)
    want = torch.stack([a.amin(0), a.amax(0), b.amin(0), b.amax(0)])
    assert torch.equal(bounds, want)
    assert torch.equal(ab, torch.stack([a[:, -1], b[:, -1]]))
    offsets, chunks = engine.dice_lattice_plan(bounds.cpu().numpy(), 2 << 20)
    assert len(chunks) > 1
    off_dev = torch.as_tensor(offsets, device="cuda")
    abc = torch.empty_like(ab)
    bn = bounds.cpu().numpy()
    for t0, t1, cells in chunks:
        hs = engine.dice_lattice_count(codes, t0, t1, abc, bounds[:, t0:t1], off_dev[t0:t1], cells)
        for t in range(t0, t1):
            wb = int(bn[3, t] - bn[2, t] + 1)
            area = int(bn[1, t] - bn[0, t] + 1) * wb
            idx = (a[:, t] - int(bn[0, t])).long() * wb + (b[:, t] - int(bn[2, t])).long()
            ref = torch.bincount(idx, minlength=area).to(torch.int32)
            got = hs[int(offsets[t]):int(offsets[t]) + area]
            assert torch.equal(got, ref), t
    assert torch.equal(abc, ab)


STATS_CASES = [
    # (name, n, h, probabilities, factor kind, lev, top)
    ("top1", 1001, 64, DICE_P, "dice", (0.2, 0.5, 1.0), 1),
    ("top7_ties", 300, 6, DICE_P, "dice", (0.3, 0.9), 7),         # few cells: the threshold's cell is split
    ("insured", 777, 50, DICE_P, "dice_sh", (0.73, 0.85, 1.0), 3),
    ("skewed", 5000, 300, (0.05, 0.8, 0.15), "dice", (0.1, 0.6), 4),
    ("one_investor", 1, 20, DICE_P, "dice", (0.5,), 1),
    ("wide", 20000, 400, DICE_P, "dice", (0.05, 0.5, 1.0), 10),
]


def factors_of(kind, lev):
    lev = np.asarray(lev, dtype=np.float32)
    if kind == "dice":
        return lo.dice_factors(lev, 0.5, -0.5, 0.05)
    return lo.dice_sh_factors(lev, 0.5, -0.5, 0.05, *golden_io.SH)


@pytest.mark.parametrize("case", STATS_CASES, ids=lambda c: c[0])
def test_stats_match_oracle(case):
    from rlmd_b200 import engine
    _, n, h, p, kind, lev, top = case
    oc = draw(n, h, p, n + 1)
    f = factors_of(kind, lev)
    codes = codes_of(oc, "u8")
    ab = torch.empty((2, n), dtype=torch.int32, device="cuda")
    bounds = engine.dice_lattice_bounds(codes, 0, h, ab)
    offsets, chunks = engine.dice_lattice_plan(bounds.cpu().numpy(), 256 << 20)
    assert len(chunks) == 1
    off = torch.as_tensor(offsets, device="cuda")
    hs = engine.dice_lattice_count(codes, 0, h, torch.empty_like(ab), bounds, off, chunks[0][2])
    for tp in sorted({top, n}):          # top == n: the adj group is empty (nan)
        got, fails = engine.dice_lattice_stats(hs, bounds, off, 0, f, 100.0, tp, n)
        got = got.cpu().numpy()
        want = dl.lattice_stats(oc, range(h), f, 100.0, tp, exp=device_exp)
        assert np.array_equal(got[..., 9:12], want[..., 9:12], equal_nan=True), "order statistics must be exact"
        assert np.array_equal(np.isnan(got), np.isnan(want))
        scale = np.abs(want[..., :9]).copy()
        for j in range(3, 9):
            scale[..., j] = np.maximum(scale[..., j], np.abs(want[..., j % 3]))
        fin = np.isfinite(want[..., :9])
        assert (np.abs(got[..., :9] - want[..., :9])[fin] <= 1e-12 * scale[fin]).all()
        assert np.array_equal(fails.cpu().numpy() == 0, dl.route_ok(f, 100.0, oc))


def assert_same_series(a, b):
    """Two runs of the series: medians and the leverage row bit for bit; the moments up to summation order
    (the row statistics of the chain's columns add fp64 partial sums with atomics)."""
    a, b = np.asarray(a), np.asarray(b)
    assert np.array_equal(a[:, 9:13].view(np.uint32), b[:, 9:13].view(np.uint32))
    np.testing.assert_allclose(a[:, :9], b[:, :9], rtol=1e-6, atol=0)


def run_smart(case, oc, method):
    """dice_smart_lev / dice_sh_smart_lev as the reference's scripts call them -> (data, data_T, printed text)."""
    from rlmd_b200 import lev_exp
    n, h = oc.shape
    buf = io.StringIO()
    args = (torch.device("cuda:0"), torch.tensor(oc.astype(np.float32)), torch.tensor(n, dtype=torch.int32),
            torch.tensor(h, dtype=torch.int32), case["top"], torch.tensor(case["v0"]), case["up_r"], case["down_r"],
            case["mid_r"])
    with contextlib.redirect_stdout(buf):
        if case["kind"] == "dice":
            data, data_T = lev_exp.dice_smart_lev(*args, *case["grid"], method=method)
        else:
            data, data_T = lev_exp.dice_sh_smart_lev(*args, *case["sh"], *case["grid"], method=method)
    return data.cpu().numpy(), data_T.cpu().numpy(), buf.getvalue()


def check_against_chain(data, data_T, text, ref, ref_T, ref_text, routed, h):
    assert data.dtype == np.float32 and data.shape == ref.shape
    assert np.array_equal(data_T.view(np.uint32), ref_T.view(np.uint32))
    assert text == ref_text
    if data.shape[2] == 0:
        return
    assert np.array_equal(data[:, 9:13, -1].view(np.uint32), ref[:, 9:13, -1].view(np.uint32))
    np.testing.assert_allclose(data[:, :9, -1], ref[:, :9, -1], rtol=1e-6, atol=0)
    assert np.array_equal(data[:, 12], ref[:, 12])
    assert_lattice_close(np.moveaxis(data[routed, :12], 1, 2), np.moveaxis(ref[routed, :12], 1, 2), lattice_tol(h))
    assert_same_series(data[~routed], ref[~routed])


@pytest.mark.parametrize("case", DICE_CASES, ids=lambda c: c["name"])
def test_smart_lev_tuples_meets_the_reference_and_the_chain(case):
    from rlmd_b200 import engine
    oc = golden_io.draw_outcomes(case)
    gold = golden_io.load("lev_" + case["name"], oc)
    data, data_T, text = run_smart(case, oc, "tuples")
    ref, ref_T, ref_text = run_smart(case, oc, "chain")
    assert np.array_equal(data_T.view(np.uint32), gold["data_T"].view(np.uint32))
    lev, f = case_factors(case)
    _, _, routed = engine.dice_series_tuples(f, lev, case["v0"], case["top"], engine.encode_codes(oc, n_outcomes=3))
    want_chain = CHAIN_LEVERAGES.get(case["name"], []) if case["h"] > 2 else [round(float(x), 6) for x in lev]
    assert [round(float(x), 6) for x in lev[~routed]] == want_chain
    check_against_chain(data, data_T, text, ref, ref_T, ref_text, routed, case["h"])
    cols = gold["cols"]
    got, want = data[:, :, cols], gold["data"]
    assert np.array_equal(got[:, 12], want[:, 12])
    assert np.array_equal(got[:, 9:12, -1].view(np.uint32), want[:, 9:12, -1].view(np.uint32))
    assert_lattice_close(np.moveaxis(got[:, :12], 1, 2), np.moveaxis(want[:, :12], 1, 2), lattice_tol(case["h"]))


SCRIPT = dict(kind="dice", top=100, v0=100.0, up_r=0.5, down_r=-0.5, mid_r=0.05, grid=(0.1, 1.0, 0.1))
SCRIPT_SH = dict(kind="dice_sh", top=100, v0=100.0, up_r=0.5, down_r=-0.5, mid_r=0.05, sh=golden_io.SH,
                 grid=(0.73, 1.0, 0.03))


@pytest.mark.parametrize("shape", [("dice", 1_000_000, 700), ("dice_sh", 1_000_000, 700), ("dice", 1_000_000, 5000)],
                         ids=["dice_1e6x700", "dicesh_1e6x700", "dice_script_1e6x5e3"])
def test_production_shapes_against_the_chain(shape):
    """The dice script's grid (l1 = 0.1..1.0, G = 10, top 100) and dice_sh's (0.73..1.0) at 1e6 investors."""
    from rlmd_b200 import engine
    kind, n, h = shape
    case = SCRIPT if kind == "dice" else SCRIPT_SH
    codes = engine.lev_draw("discrete", n, h, seed=h + len(kind), probs=DICE_P)
    lev, f = case_factors(case)
    data, data_T, routed = engine.dice_series_tuples(f, lev, 100.0, 100, codes)
    ref, ref_T = engine.lev_series("discrete", f, lev, 100.0, 100, outcomes=codes)
    # at H = 5e3 the lowest cells of l = 0.8, 0.9 and 1.0 pass below FLT_MIN: those keep the chain
    assert [round(float(x), 6) for x in lev[~routed]] == ([0.8, 0.9, 1.0] if h == 5000 else [])
    check_against_chain(data.cpu().numpy(), data_T.cpu().numpy(), "", ref.cpu().numpy(), ref_T.cpu().numpy(), "",
                        routed, h)


def test_results_do_not_depend_on_chunking():
    from rlmd_b200 import engine
    case = golden_io.lev_case("dice_testscale")
    oc = golden_io.draw_outcomes(case)
    lev, f = case_factors(case)
    codes = engine.encode_codes(oc, n_outcomes=3)
    a = engine.dice_series_tuples(f, lev, 100.0, 1, codes)
    bounds = engine.dice_lattice_bounds(codes, 0, oc.shape[1], torch.empty((2, oc.shape[0]), dtype=torch.int32,
                                                                           device="cuda")).cpu().numpy()
    small = 4 * int(((bounds[1] - bounds[0] + 1) * (bounds[3] - bounds[2] + 1)).max())
    assert len(engine.dice_lattice_plan(bounds, small)[1]) > 20
    b = engine.dice_series_tuples(f, lev, 100.0, 1, codes, chunk_bytes=small)
    assert a[2].all() and np.array_equal(a[2], b[2]) and torch.equal(a[1], b[1])
    assert torch.equal(a[0][:, :, :-1], b[0][:, :, :-1])         # the lattice's columns: bit for bit
    assert_same_series(a[0].cpu().numpy(), b[0].cpu().numpy())


def route_case(oc, f, lev, chunk_bytes=256 << 20):
    from rlmd_b200 import engine
    codes = engine.encode_codes(oc, n_outcomes=3)
    data, data_T, routed = engine.dice_series_tuples(f, lev, 100.0, 2, codes, chunk_bytes=chunk_bytes)
    ref, ref_T = engine.lev_series("discrete", f, lev, 100.0, 2, outcomes=codes)
    assert torch.equal(data_T, ref_T)
    check_against_chain(data.cpu().numpy(), data_T.cpu().numpy(), "", ref.cpu().numpy(), ref_T.cpu().numpy(), "",
                        routed, oc.shape[1])
    return routed


def test_route_edges():
    from rlmd_b200 import engine
    # a zero factor: down_r = -1 at l = 1
    oc = draw(2000, 40, DICE_P, 8)
    lev = np.asarray([0.5, 1.0], dtype=np.float32)
    assert list(route_case(oc, lo.dice_factors(lev, 0.5, -1.0, 0.05), lev)) == [True, False]
    # a long horizon whose high leverages underflow
    oc = draw(500, 3000, (0.1, 0.6, 0.3), 9)
    lev = np.asarray([0.1, 0.5, 1.0], dtype=np.float32)
    f = lo.dice_factors(lev, 0.5, -0.5, 0.05)
    routed = route_case(oc, f, lev)
    assert list(routed) == [True, False, False] and np.array_equal(routed, dl.route_ok(f, 100.0, oc))
    # a spread too wide for the budget: rows of all-up and all-down codes; the whole grid keeps the chain
    oc = np.zeros((64, 3000), dtype=np.uint8)
    oc[1::2] = 1
    oc[::4, ::3] = 2
    lev = np.asarray([0.05, 0.1], dtype=np.float32)
    f = lo.dice_factors(lev, 0.5, -0.5, 0.05)
    assert list(route_case(oc, f, lev)) == [True, False]          # (l = 0.1: the all-down rows underflow)
    bounds, _ = dl.lattice_bounds(oc)
    assert engine.dice_lattice_plan(bounds, 1 << 20) is None
    assert not route_case(oc, f, lev, chunk_bytes=1 << 20).any()
    # H <= 2: no column comes from the route
    for h in (1, 2):
        assert not route_case(draw(300, h, DICE_P, h), lo.dice_factors(lev, 0.5, -0.5, 0.05), lev).any()


def test_series_method_blocks_and_errors():
    from rlmd_b200 import engine, lev_exp
    case = golden_io.lev_case("dice_top5")
    oc = golden_io.draw_outcomes(case)
    chain, _, _ = run_smart(case, oc, "chain")
    tuples, _, _ = run_smart(case, oc, "tuples")
    assert not np.array_equal(chain[:, 9:12, :-1], tuples[:, 9:12, :-1])
    assert_same_series(run_smart(case, oc, None)[0], chain)            # the default is the chain
    for own_of_others in ("counts", "sum"):
        with lev_exp.series_method(own_of_others):
            assert_same_series(run_smart(case, oc, None)[0], chain)
    with lev_exp.series_method("tuples"):
        assert np.array_equal(run_smart(case, oc, None)[0], tuples)
        with lev_exp.series_method("counts"):
            assert_same_series(run_smart(case, oc, None)[0], chain)
        with lev_exp.series_method("chain"):
            assert_same_series(run_smart(case, oc, None)[0], chain)
        with pytest.raises(ValueError):
            run_smart(case, oc, "counts")
        # the coin ignores "tuples"
        coin = golden_io.lev_case("coin_top7")
        coc = golden_io.draw_outcomes(coin)
        lev = lo.lev_grid(*coin["grid"], coin["up_r"], coin["down_r"])
        with contextlib.redirect_stdout(io.StringIO()):
            d, _ = lev_exp.coin_smart_lev(torch.device("cuda:0"), torch.tensor(coc.astype(np.float32)), None, None,
                                          coin["top"], coin["v0"], coin["up_r"], coin["down_r"], *coin["grid"])
        ref, _ = engine.lev_series("discrete", lev_exp.coin_factor_table(lev, coin["up_r"], coin["down_r"]), lev,
                                   100.0, coin["top"], outcomes=engine.encode_codes(coc, n_outcomes=2))
        assert_same_series(d.cpu().numpy(), ref.cpu().numpy())
    assert np.array_equal(run_smart(case, oc, None)[0], chain)
    lev_exp.set_process_group(object())
    try:
        with pytest.raises(ValueError):
            run_smart(case, oc, "tuples")
        with lev_exp.series_method("tuples"), pytest.raises(ValueError):
            run_smart(case, oc, None)
    finally:
        lev_exp.set_process_group(None)
    lev, f = case_factors(case)
    codes = engine.encode_codes(oc, n_outcomes=3)
    a = engine.lev_series("discrete", f, lev, 100.0, 5, outcomes=codes, method="tuples")
    b = engine.dice_series_tuples(f, lev, 100.0, 5, codes)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    with pytest.raises(ValueError):
        engine.lev_series("discrete", f, lev, 100.0, 5, outcomes=codes, method="tuples", group=object())
    with pytest.raises(ValueError):
        engine.lev_series("discrete", lev_exp.coin_factor_table(lev, 0.5, -0.4), lev, 100.0, 5, outcomes=codes,
                          method="tuples")
    with pytest.raises(ValueError):
        engine.lev_series("gbm", lev, lev, 100.0, 2, outcomes=torch.zeros((10, 10), device="cuda"), method="tuples")
    for bad in ("lattice", "tally"):
        with pytest.raises(ValueError):
            lev_exp.series_method(bad)


def test_scripts_write_the_same_files(tmp_path):
    from rlmd_b200 import lev_scripts
    for fn, name in ((lev_scripts.dice_roll, "dice"), (lev_scripts.dice_roll_sh, "dice_sh")):
        kw = dict(seed=5, investors=5000, horizon=60)
        if name == "dice":
            kw.update(s3=(0.5, 0.5, 0.1), r3=(0.45, 0.55, 0.05))
        with contextlib.redirect_stdout(io.StringIO()):
            a = fn(str(tmp_path / "t") + "/", series="tuples", **kw)
            b = fn(str(tmp_path / "c") + "/", series="chain", **kw)
        assert sorted(os.listdir(tmp_path / "t")) == sorted(os.listdir(tmp_path / "c"))
        assert sorted(a) == sorted(b)
        for k in a:
            if k.endswith("_inv1_val"):
                assert_lattice_close(np.moveaxis(a[k][:, :12], 1, 2), np.moveaxis(b[k][:, :12], 1, 2), lattice_tol(60))
                assert np.array_equal(a[k][:, :, -1], b[k][:, :, -1]) or \
                    np.allclose(a[k][:, :, -1], b[k][:, :, -1], rtol=1e-6, atol=0)
            else:
                assert np.array_equal(a[k], b[k]), k

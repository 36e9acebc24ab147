"""
The tally path (count tuples -> weighted exact statistics; tally.cu, lev_ingest.cu)
against the CPU oracle and against the general path (LOG sweep -> data_T ->
b200_rowstats), and the reference-format ingest.  All calls go through the C ABI.
"""
import contextlib
import io
import json
import os

import numpy as np
import pytest
import torch as T

import golden_io
import tally_sets
from oracle import lev_oracle as lo

pytestmark = pytest.mark.gpu

DISCRETE = [c for c in golden_io.LEV_CASES if c["kind"] != "gbm"]


def factors_of(case):
    lev = lo.lev_grid(*case["grid"], case["up_r"], case["down_r"])
    if case["kind"] == "coin":
        return lev, lo.coin_factors(lev, case["up_r"], case["down_r"])
    if case["kind"] == "dice":
        return lev, lo.dice_factors(lev, case["up_r"], case["down_r"], case["mid_r"])
    return lev, lo.dice_sh_factors(lev, case["up_r"], case["down_r"], case["mid_r"], *case["sh"])


def oracle_stats(oc, f, top, v0):
    """The 12 statistics of fl32(exp(log-wealth)) per leverage: what the LOG sweep's data_T holds."""
    lw = lo.log_wealth_discrete(oc, f, v0)
    with np.errstate(over="ignore", invalid="ignore"):
        w = np.exp(lw).astype(np.float32)
        return np.stack([lo.summary_stats(w[g], top) for g in range(w.shape[0])]), w


def assert_same_stats(got, want, rtol=1e-11):
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    assert np.array_equal(np.isnan(got), np.isnan(want)), (got, want)
    # order statistics: the same fp32 value, bit for bit
    assert np.array_equal(got[:, 9:12][~np.isnan(got[:, 9:12])], want[:, 9:12][~np.isnan(want[:, 9:12])])
    fin = np.isfinite(want)
    assert np.array_equal(got[~fin & ~np.isnan(want)], want[~fin & ~np.isnan(want)])
    # mad / std of (nearly) equal groups: relative to the mean
    scale = np.where(np.isfinite(want[:, 0:1]), np.abs(want[:, 0:1]), 0.0) + 1e-300
    with np.errstate(invalid="ignore"):
        err = np.abs(got - want)
    ok = (err <= rtol * np.maximum(np.abs(want), scale)) | ~fin
    assert ok.all(), (np.argwhere(~ok)[:5], got[~ok][:5], want[~ok][:5])


@pytest.mark.parametrize("case", DISCRETE, ids=lambda c: c["name"])
def test_tally_stats_match_general_path_and_oracle(case):
    from rlmd_b200 import engine
    oc = golden_io.draw_outcomes(case)
    lev, f = factors_of(case)
    top, v0 = case["top"], case["v0"]
    codes = engine.encode_codes(oc)
    got = engine.lev_final_stats(f, v0, top, codes).cpu().numpy()
    res = engine.lev_sweep("discrete", f, v0, outcomes=codes, mode="log")
    general = engine.rowstats(res["data_T"], top).cpu().numpy()
    assert_same_stats(got, general)
    want, w = oracle_stats(oc, f, top, v0)
    # the oracle's exp / log may differ from CUDA's in the last fp64 bit: an fp32 wealth can
    # move by one ulp, so compare with the fp32 data_T the GPU produced
    dT = res["data_T"].cpu().numpy()
    fin = np.isfinite(w) & np.isfinite(dT)
    assert np.array_equal(np.isinf(dT) | (fin & False), np.isinf(w)) or (np.isinf(dT) != np.isinf(w)).mean() < 0.01
    assert (np.abs(dT[fin].astype(np.float64) - w[fin]) <= 2.4e-7 * np.abs(w[fin])).all()
    ref = np.stack([lo.summary_stats(res["data_T"][g].cpu().numpy(), top) for g in range(f.shape[0])])
    assert_same_stats(got, ref, rtol=1e-10)


FORMATS = [("int64", T.int64), ("int32", T.int32), ("float32", T.float32), ("float64", T.float64),
           ("uint8", T.uint8), ("bool", T.bool)]


@pytest.mark.parametrize("name,dtype", FORMATS)
@pytest.mark.parametrize("where", ["cuda", "host", "pinned"])
def test_ingest_every_reference_format(name, dtype, where):
    """The same outcomes in every accepted dtype / location give the same counts, codes and statistics."""
    from rlmd_b200 import engine, tally
    kind = "coin" if dtype == T.bool else "dice"
    case = golden_io.lev_case("coin_top7" if kind == "coin" else "dice_top5")
    oc = golden_io.draw_outcomes(case)
    lev, f = factors_of(case)
    k = f.shape[1]
    src = T.tensor(oc).to(dtype)
    if where == "cuda":
        src = src.cuda()
    elif where == "pinned":
        src = src.pin_memory()
    want = engine.lev_final_stats(f, case["v0"], case["top"], engine.encode_codes(oc)).cpu().numpy()
    info = {}
    got = engine.lev_final_stats(f, case["v0"], case["top"], src, info=info).cpu().numpy()
    # the same tuples, listed in whatever order the compaction found them: fp64 sums agree to rounding
    assert_same_stats(got, want, rtol=1e-13)
    assert info["bad_outcomes"] == 0 and not info["overflow"]
    assert info["h2d_bytes"] == (0 if where == "cuda" else src.numel() * src.element_size())
    # codes + counts sinks
    codes = engine.encode_codes(src, n_outcomes=k)
    assert np.array_equal(codes.cpu().numpy(), oc)
    if where == "cuda":
        t = tally.FinalTally(oc.shape[0])
        counts = T.empty((oc.shape[0], k), dtype=T.int32, device="cuda")
        t.add(src, k, counts=counts)
        t.finalize()
        assert np.array_equal(counts.cpu().numpy(), lo.counts_discrete(oc, k))
        assert t.check()["bins"] == len({tuple(r) for r in lo.counts_discrete(oc, k)})


def test_host_chunks_and_row_blocks_do_not_change_the_result():
    from rlmd_b200 import engine, tally
    case = golden_io.lev_case("dice_top5")
    oc = golden_io.draw_outcomes(case)
    lev, f = factors_of(case)
    n, h = oc.shape
    want = engine.lev_final_stats(f, case["v0"], case["top"], engine.encode_codes(oc)).cpu().numpy()
    host = T.tensor(oc.astype(np.int64))
    t = tally.FinalTally(n)
    t.add_host(host, 3, chunk_bytes=h * 8 * 37)        # 37-row chunks: many staging round trips
    t.finalize()
    got = t.stats(f, case["v0"], h, n_total=n, top=case["top"]).cpu().numpy()
    t.check()
    # same tuples, possibly listed in another order: fp64 sums agree to rounding
    assert_same_stats(got, want, rtol=1e-13)
    # two row blocks on the device, one of them packed
    codes = engine.encode_codes(oc)
    t.add(codes[:700], 3)
    t.add(engine.pack_codes(codes[700:].contiguous()), 3)
    t.finalize()
    got = t.stats(f, case["v0"], h, n_total=n, top=case["top"]).cpu().numpy()
    t.check()
    assert_same_stats(got, want, rtol=1e-13)
    # unaligned rows (odd horizon, sliced): the scalar path of the ingest kernel
    odd = T.tensor(oc.astype(np.float32))[:, 1:].cuda()
    sub = engine.lev_final_stats(f, case["v0"], case["top"], odd).cpu().numpy()
    ref = engine.lev_final_stats(f, case["v0"], case["top"], engine.encode_codes(oc[:, 1:])).cpu().numpy()
    assert_same_stats(sub, ref, rtol=1e-13)


def test_bad_outcomes_and_overflow_are_reported():
    from rlmd_b200 import engine, lev_exp, tally
    case = golden_io.lev_case("dice_top5")
    oc = golden_io.draw_outcomes(case).astype(np.int64)
    lev, f = factors_of(case)
    bad = oc.copy()
    bad[3, 5] = 7
    bad[9, 0] = -1
    with pytest.raises(ValueError, match="2 outcomes outside"):
        engine.lev_final_stats(f, case["v0"], case["top"], T.tensor(bad).cuda())
    # a plan too small for the distinct tuples of this input -> overflow, and the statistics are NaN
    n, h = oc.shape
    small = tally.FinalTally(n, bins_cap=16)
    small.add(T.tensor(oc).cuda(), 3)
    small.finalize()
    st = small.stats(f, case["v0"], h, n_total=n, top=case["top"])
    assert T.isnan(st).all()
    with pytest.raises(tally.TallyOverflow):
        small.check()
    # after the reset that check() did, the same object works again when the input fits
    few = np.zeros((n, h), dtype=np.int64)
    few[: n // 2, 0] = 1
    small.add(T.tensor(few).cuda(), 3)
    small.finalize()
    st = small.stats(f, case["v0"], h, n_total=n, top=case["top"]).cpu().numpy()
    assert small.check()["bins"] == 2
    ref = np.stack([lo.summary_stats(w, case["top"]) for w in
                    np.exp(lo.log_wealth_discrete(few, f, case["v0"])).astype(np.float32)])
    assert_same_stats(st, ref, rtol=1e-10)
    # the drop-in function falls back to the general path on overflow (same printed text)
    buf_a, buf_b = io.StringIO(), io.StringIO()
    with contextlib.redirect_stdout(buf_a):
        lev_exp.dice_fixed_final_lev(T.device("cuda:0"), T.tensor(oc), case["top"], T.tensor(1e2), 0.5, -0.5, 0.05,
                                     *case["grid"])
    engine._tally_cache.clear()
    old = tally.DEFAULT_BINS_CAP
    tally.DEFAULT_BINS_CAP = 16
    try:
        engine._tally_cache.clear()
        with contextlib.redirect_stdout(buf_b):
            lev_exp.dice_fixed_final_lev(T.device("cuda:0"), T.tensor(oc), case["top"], T.tensor(1e2), 0.5, -0.5,
                                         0.05, *case["grid"])
    finally:
        tally.DEFAULT_BINS_CAP = old
        engine._tally_cache.clear()
    assert buf_a.getvalue() == buf_b.getvalue() and buf_a.getvalue().count("lev ") == f.shape[0]


def test_ties_infinities_and_zeros():
    """Degenerate inputs: every investor equal; half the investors at +inf; all wealth zero."""
    from rlmd_b200 import engine
    n, h = 515, 40
    f = np.array([[1.5, 0.6], [2.0, 0.0], [1e30, 1.0]], dtype=np.float32)
    same = np.ones((n, h), dtype=np.uint8)
    same[:, ::2] = 0
    half = same.copy()
    half[: n // 2] = 1     # all up: overflows to inf at the third grid point, rest stay finite
    for oc in (same, half):
        codes = engine.encode_codes(oc)
        got = engine.lev_final_stats(f, 1.0, 3, codes).cpu().numpy()
        res = engine.lev_sweep("discrete", f, 1.0, outcomes=codes, mode="log")
        want = engine.rowstats(res["data_T"], 3).cpu().numpy()
        assert_same_stats(got, want, rtol=1e-12)
        ref = np.stack([lo.summary_stats(res["data_T"][g].cpu().numpy(), 3) for g in range(3)])
        assert_same_stats(got, ref, rtol=1e-10)


def test_four_outcomes_and_coin_and_large_grid():
    """K = 4 (engine-only) and a grid wider than one statistics tile."""
    from rlmd_b200 import engine
    rs = np.random.RandomState(5)
    oc = rs.randint(0, 4, size=(3001, 77)).astype(np.uint8)
    f = (1 + rs.uniform(-0.3, 0.5, size=(130, 4))).astype(np.float32)
    codes = engine.encode_codes(oc)
    got = engine.lev_final_stats(f, 10.0, 9, codes).cpu().numpy()
    parts = []
    for g0 in range(0, 130, 64):
        res = engine.lev_sweep("discrete", f[g0:g0 + 64], 10.0, outcomes=codes, mode="log")
        parts.append(engine.rowstats(res["data_T"], 9).cpu().numpy())
    assert_same_stats(got, np.concatenate(parts))


FINAL_TEXT = os.path.join(golden_io.GOLDEN_DIR, "final_text.json")


@pytest.mark.parametrize("name", ["coin_testscale", "dice_testscale", "dicesh_testscale", "gbm_testscale", "coin_top7",
                                  "dice_top5", "dicesh_top3", "gbm_snp_top4", "coin_flip_sign", "dice_tiny"])
@pytest.mark.parametrize("where", ["host", "cuda"])
def test_fixed_final_prints_the_reference_text(name, where):
    """
    {coin,dice,dice_sh,gbm}_fixed_final_lev called as the reference scripts call them
    (reference dtypes, host or device tensors): the printed text equals, line for line,
    what the unmodified reference printed on the same outcomes
    (tests/golden/final_text.json, written by tests/golden/gen_golden_final_text.py).
    """
    from rlmd_b200 import lev_exp
    case = golden_io.lev_case(name)
    oc = golden_io.draw_outcomes(case)
    want = json.load(open(FINAL_TEXT))[name]
    dev, v0, top, grid = T.device("cuda:0"), T.tensor(case["v0"]), case["top"], case["grid"]
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        if case["kind"] == "coin":
            t = T.tensor(oc.astype(np.float32))
            lev_exp.coin_fixed_final_lev(dev, t.cuda() if where == "cuda" else t, top, v0, case["up_r"],
                                         case["down_r"], *grid)
        elif case["kind"] == "dice":
            t = T.tensor(oc.astype(np.int64))
            lev_exp.dice_fixed_final_lev(dev, t.cuda() if where == "cuda" else t, top, v0, case["up_r"],
                                         case["down_r"], case["mid_r"], *grid)
        elif case["kind"] == "dice_sh":
            t = T.tensor(oc.astype(np.int64))
            lev_exp.dice_sh_fixed_final_lev(dev, t.cuda() if where == "cuda" else t, top, v0, case["up_r"],
                                            case["down_r"], case["mid_r"], *case["sh"], *grid)
        else:
            t = T.tensor(oc)
            lev_exp.gbm_fixed_final_lev(dev, t.cuda() if where == "cuda" else t, top, v0, *grid)
    got = buf.getvalue().rstrip("\n").splitlines()
    want = want.splitlines()
    assert len(got) == len(want)
    for a, b in zip(got, want):
        assert a == b, (a, b)


@pytest.mark.parametrize("world", [2, 3, 8])
def test_merge_of_rank_tallies_on_one_gpu(world):
    """
    The cross-GPU merge (publish -> wait -> merge in rank order, first occurrence wins) played
    on ONE GPU: every rank has its own workspace and exchange buffer in this process, all
    ranks publish (phase 0) before any rank merges (phase 1) - so no kernel waits for a kernel
    queued behind it.  Every rank must end with the identical bin list (bit-identical
    statistics) and with the statistics of the undivided population.
    """
    from rlmd_b200 import engine

    case = golden_io.lev_case("dice_top5")
    oc = golden_io.draw_outcomes(case)
    lev, f = factors_of(case)
    n, h = oc.shape
    codes = engine.encode_codes(oc)
    want = engine.lev_final_stats(f, case["v0"], case["top"], codes).cpu().numpy()
    # uneven shards, one of them empty when there are enough ranks
    cuts = tally_sets.shard_cuts(n, world)
    ranks = tally_sets.one_gpu_ranks(world, n, n)
    for epoch in (1, 2, 3):      # successive sweeps alternate between the two published lists
        sl = slice(None) if epoch != 2 else slice(0, h - 3)      # another horizon in between
        ref = want if epoch != 2 else engine.lev_final_stats(f, case["v0"], case["top"],
                                                             engine.encode_codes(oc[:, sl])).cpu().numpy()
        hh = oc[:, sl].shape[1]
        for r, t in enumerate(ranks):
            t.rows = 0
            if cuts[r + 1] > cuts[r]:
                t.add(engine.encode_codes(oc[cuts[r]:cuts[r + 1], sl]), 3)
        tally_sets.merge_on_one_gpu(ranks, epoch)
        got = [t.stats(f, case["v0"], hh, n_total=n, top=case["top"]).cpu().numpy() for t in ranks]
        for r, t in enumerate(ranks):
            i = t.info()
            assert not (i["overflow"] or i["timed_out"] or i["count_mismatch"] or i["bad_outcomes"]), (r, i)
            assert np.array_equal(got[r], got[0]), f"rank {r} differs from rank 0"
        assert_same_stats(got[0], ref, rtol=1e-13)
    distinct = len({tuple(c) for c in lo.counts_discrete(oc, 3)})
    assert ranks[0].info()["bins"] == distinct


@pytest.mark.parametrize("world", [2, 3, 8])
def test_merge_of_long_rank_lists_on_one_gpu(world):
    """
    The same merge on the 150 000 distinct tuples of tally_sets' wide K = 3 set, shuffled over uneven shards
    (one empty): every rank's list is tens of thousands of bins long and shares tuples with the others, so
    the mark / unique kernels walk many chunks of MERGE_CHUNK positions, each placed after the first
    occurrences of all earlier chunks, and rebuild the (n_1, n_2) box.  The merged list (about 150 k bins,
    spilling in both select shapes) gives every rank bit-identical statistics, equal to the reference and to
    the undivided tally, with the six-CTA and the two-CTA (beside_sweep: 8-GPU depth 2) select.
    """
    s = tally_sets.get("wide3")
    want = tally_sets.set_reference("wide3")
    codes = tally_sets.rows(s)
    single = tally_sets.tally_in_blocks(codes, 3)
    whole = single.stats(s["f"], s["v0"], s["h"], n_total=s["n"], top=s["top"]).cpu().numpy()
    del single
    cuts = tally_sets.shard_cuts(s["n"], world)
    ranks = tally_sets.one_gpu_ranks(world, int(np.diff(cuts).max()), len(s["tuples"]))
    for r, t in enumerate(ranks):
        if cuts[r + 1] > cuts[r]:
            t.add(codes[cuts[r]:cuts[r + 1]], 3)
    tally_sets.merge_on_one_gpu(ranks, 1)
    box = tally_sets.box_of(s["tuples"])
    for beside in (False, True):
        got = [t.stats(s["f"], s["v0"], s["h"], n_total=s["n"], top=s["top"], beside_sweep=beside).cpu().numpy()
               for t in ranks]
        for r, t in enumerate(ranks):
            i = t.info()
            assert not (i["overflow"] or i["timed_out"] or i["count_mismatch"] or i["bad_outcomes"]), (r, i)
            assert i["bins"] == len(s["tuples"]), (r, i)
            assert tally_sets.box_words(t) == box, r
            assert np.array_equal(got[r].view(np.uint64), got[0].view(np.uint64)), f"rank {r} differs from rank 0"
        assert_same_stats(got[0], want, rtol=1e-12)
        assert_same_stats(got[0], whole, rtol=1e-13)


def test_pipeline_depths_agree():
    """Statistics beside the next sweep (depth 2: two tallies, two streams, the select kernel in its two-CTA
    shape, B200_LEV_FLAG_BESIDE_SWEEP) equal the strictly sequential pipeline and the one-shot call."""
    from rlmd_b200 import engine
    rs = np.random.RandomState(12)
    n, h, top = 60_000, 500, 6
    f = np.float32([[1.25, 0.75, 1.025], [1.5, 0.5, 1.05], [1.9, 0.1, 1.09]])
    arrays = [engine.pack_codes(engine.encode_codes(rs.choice(3, size=(n, h), p=[1 / 6, 1 / 6, 2 / 3]).astype(np.uint8)))
              for _ in range(5)]
    want = [engine.lev_final_stats(f, 100.0, top, a) for a in arrays]
    for depth in (1, 2):
        pipe = engine.FinalSweepPipeline("discrete", f, 100.0, top, depth=depth)
        got = [pipe.submit(a) for a in arrays]
        pipe.synchronize()
        for g_, w_ in zip(got, want):
            assert T.equal(g_[:, 9:12], w_[:, 9:12]) and T.allclose(g_, w_, rtol=1e-12, atol=0), depth

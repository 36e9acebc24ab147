"""
The tally chain launched early (programmatic dependent launch): at pipeline depth 1 the count kernel of step i+1
streams its rows while step i's select kernel runs and waits for it only before its first tally insertion; the
compaction and the select start under the kernel before them and wait before they read the table.  Every step
must give what the same outcome array gives alone.  B200_PDL is read once per process, so the runs with and
without early launches are made in interpreters of their own.
"""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch as T

from test_tally_gpu import assert_same_stats

pytestmark = pytest.mark.gpu

TESTS = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(TESTS)
V0, TOP = 100.0, 100


def _inputs():
    """(outcomes, factor table) of three sweeps that differ in K, format and distinct-tuple count: the flagship
    dice draw (K = 3, 1e6 x 1e4, 45 561 tuples), a skewed K = 3 draw over 3000 steps (fewer tuples) and the
    one-bit coin (K = 2)."""
    from rlmd_b200 import engine, lev_exp
    lev = np.asarray(lev_exp.param_range(0.05, 1.0, 0.05), np.float32)
    dice = lev_exp.dice_factor_table(lev, 0.5, -0.5, 0.05)
    coin = lev_exp.coin_factor_table(lev, 0.5, -0.4)
    n = 1_000_000
    return [
        (engine.lev_draw("discrete", n, 10_000, seed=420, probs=(1 / 6, 1 / 6, 2 / 3), packed=True), dice),
        (engine.lev_draw("discrete", n, 3_000, seed=7, probs=(0.3, 0.1, 0.6), packed=True), dice),
        (engine.lev_draw("discrete", n, 3_000, seed=11, probs=(0.5, 0.5), packed=True, bits=1), coin),
    ]


def _child(mode: str, out_dir: str) -> None:
    """mode "chain": 12 back-to-back pipeline steps cycling through the inputs (timing on, as in bench.py);
    mode "alone": every input once through lev_final_stats, each after a device synchronise."""
    from rlmd_b200 import engine
    ins = _inputs()
    if mode == "chain":
        pipe = engine.FinalSweepPipeline("discrete", ins[0][1], V0, TOP, depth=1)
        pipe.timing = True
        out = [pipe.submit(oc, factors=f) for _ in range(4) for oc, f in ins]
        pipe.synchronize()        # raises on overflow, a count mismatch or bad outcomes
        info = pipe.tallies[0].info()
        assert not (info["overflow"] or info["count_mismatch"] or info["bad_outcomes"]), info
    else:
        out = []
        for oc, f in ins:
            T.cuda.synchronize()
            out.append(engine.lev_final_stats(f, V0, TOP, oc))
    for i, s in enumerate(out):
        np.save(os.path.join(out_dir, f"{mode}_{i}.npy"), s.cpu().numpy())


def _run_child(mode: str, pdl: str, out_dir) -> None:
    env = dict(os.environ, B200_PDL=pdl)
    code = ("import sys; sys.path.insert(0, sys.argv[3]); import test_final_step_overlap_gpu as m; "
            "m._child(sys.argv[1], sys.argv[2])")
    p = subprocess.run([sys.executable, "-c", code, mode, str(out_dir), TESTS], env=env, cwd=ROOT,
                       capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stderr[-4000:]


def test_back_to_back_steps_equal_isolated_steps(tmp_path):
    """Twelve depth-1 steps with early launches against each input alone without them: order statistics
    bit-identical, moments to 1e-14 (the compaction's append order varies from run to run)."""
    _run_child("chain", "1", tmp_path)
    _run_child("alone", "0", tmp_path)
    alone = [np.load(tmp_path / f"alone_{j}.npy") for j in range(3)]
    for i in range(12):
        got = np.load(tmp_path / f"chain_{i}.npy")
        want = alone[i % 3]
        assert np.array_equal(got[:, 9:12].view(np.uint64), want[:, 9:12].view(np.uint64)), i
        assert_same_stats(got, want, rtol=1e-14)


@pytest.mark.parametrize("early", [False, True], ids=["plain", "early_start"])
def test_repeated_adds_multiply_every_count(early):
    """add() four times without a finalize (each count kernel, launched early or not, waits for the one before it
    only before it inserts), then one finalize: the tally holds every tuple four times, so the statistics at
    4 n rows and top 4 K are those of one add()."""
    from rlmd_b200 import tally
    oc, f = _inputs()[1]
    n, h = oc.shape
    one = tally.FinalTally(n)
    one.add(oc, 3)
    one.finalize()
    want = one.stats(f, V0, h, n_total=n, top=TOP).cpu().numpy()
    bins = one.check()["bins"]
    rep = tally.FinalTally(4 * n)
    for _ in range(4):
        rep.add(oc, 3, early_start=early)
    rep.finalize()
    got = rep.stats(f, V0, h, n_total=4 * n, top=4 * TOP).cpu().numpy()
    info = rep.check()
    assert info["bins"] == bins and not info["count_mismatch"], info
    assert np.array_equal(got[:, 9:12].view(np.uint64), want[:, 9:12].view(np.uint64))
    assert_same_stats(got, want, rtol=1e-12)


def test_k4_radix_route_and_overflow_under_early_launches():
    """K = 4 on the forced radix route, steps launched early back to back, equals each step alone; then an
    overflowing step (a plan of 1024 bins against 45 561 tuples) gives NaN statistics and TallyOverflow, and the
    next step, launched early behind it, recovers after the reset."""
    from rlmd_b200 import engine, lev_exp, tally
    lev = np.asarray(lev_exp.param_range(0.05, 1.0, 0.05), np.float32)
    f4 = np.stack([1 + lev * r for r in (0.6, -0.5, 0.05, 0.2)], axis=1).astype(np.float32)
    n, h = 400_000, 2_000
    arrays = [engine.lev_draw("discrete", n, h, seed=s, probs=(0.2, 0.2, 0.3, 0.3), packed=True) for s in (1, 2)]

    def step(t, oc, early):
        t.add(oc, 4, early_start=early)
        t.finalize()
        return t.stats(f4, V0, h, n_total=n, top=TOP, radix_select=True)

    alone = []
    for oc in arrays:
        T.cuda.synchronize()
        alone.append(step(tally.FinalTally(n), oc, False).cpu().numpy())
    t = tally.FinalTally(n)
    got = [step(t, arrays[i % 2], True) for i in range(6)]
    info = t.check()
    assert info["radix_route"] == f4.shape[0] and not info["count_mismatch"], info   # (counted since the last finalize)
    for i, s in enumerate(got):
        s = s.cpu().numpy()
        assert np.array_equal(s[:, 9:12].view(np.uint64), alone[i % 2][:, 9:12].view(np.uint64)), i
        assert_same_stats(s, alone[i % 2], rtol=1e-14)

    ins = _inputs()
    (dice, fd), (small, fs) = ins[0], ins[2]
    t = tally.FinalTally(dice.shape[0], bins_cap=1024)
    bad = step_k(t, dice, fd, 3)
    with pytest.raises(tally.TallyOverflow):
        t.check()
    assert np.isnan(bad.cpu().numpy()).all()
    good = step_k(t, small, fs, 2).cpu().numpy()
    assert not t.check()["overflow"]
    want = engine.lev_final_stats(fs, V0, TOP, small).cpu().numpy()
    assert np.array_equal(good[:, 9:12].view(np.uint64), want[:, 9:12].view(np.uint64))
    assert_same_stats(good, want, rtol=1e-14)


def step_k(t, oc, f, k):
    t.add(oc, k, early_start=True)
    t.finalize()
    return t.stats(f, V0, oc.shape[1], n_total=oc.shape[0], top=TOP)

"""
The tally statistics (tally.cu) at production list sizes and in every launch shape of tally_select_kernel,
against the weighted order statistics of oracle/tally_oracle.py on the GPU's own bin wealth: bin lists whose
slices exceed the shared-memory cache of a CTA (the spilled bins are written to and read back from the global
wbuf; on the log-wealth route a spilled bin's log-wealth bin is recomputed from its key), the two-CTA shape
(beside_sweep, pipeline depth 2), every cluster size 1..16 and a cache of 0 or 7 bins (B200_SELECT_CLUSTER /
B200_SELECT_CACHE, read once per process: each setting runs in its own interpreter), and the (n_1, n_2) box
header words of the list.  The inputs are tuple sets chosen in tests/tally_sets.py; the merges of rank lists
longer than one chunk are in test_tally_gpu.py.
"""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch as T

import tally_sets as ts
from oracle import tally_oracle as to
from test_tally_gpu import assert_same_stats

pytestmark = pytest.mark.gpu

RADIX_ONLY = {"wide3": 3, "coin2": 4, "quad4": None}   # rows that may leave the log-wealth route (None: all of them)


@pytest.mark.parametrize("name", ["wide3", "coin2", "quad4"])
def test_spilled_bins_in_both_shapes_and_both_routes(name):
    """Default (six CTAs), beside_sweep (two), radix_select and both: every call equals the reference; the forced
    calls add G to the radix count, K = 4 always takes the radix route, the others mostly the log-wealth route."""
    s = ts.get(name)
    want = ts.set_reference(name)
    g = s["f"].shape[0]
    t = ts.tally_in_blocks(ts.rows(s), s["k"])
    info = t.info()
    assert info["bins"] == len(s["tuples"]) and not (info["overflow"] or info["bad_outcomes"]), info
    assert ts.box_words(t) == ts.box_of(s["tuples"])
    for beside, radix in ts.FLAGS:
        before = t.info()["radix_route"]
        got = t.stats(s["f"], s["v0"], s["h"], n_total=s["n"], top=s["top"], beside_sweep=beside,
                      radix_select=radix).cpu().numpy()
        took = t.info()["radix_route"] - before
        assert_same_stats(got, want, rtol=1e-12)
        if radix or RADIX_ONLY[name] is None:
            assert took == g, (beside, radix, took)
        else:
            assert took <= RADIX_ONLY[name], (beside, took)
    assert not t.info()["count_mismatch"]


def test_wide_set_matches_the_general_path():
    """The same rows through the LOG sweep (data_T) and b200_rowstats: no oracle in between."""
    from rlmd_b200 import engine
    s = ts.get("wide3")
    codes = ts.rows(s)
    t = ts.tally_in_blocks(codes, 3)
    got = t.stats(s["f"], s["v0"], s["h"], n_total=s["n"], top=s["top"]).cpu().numpy()
    general = engine.rowstats(engine.lev_sweep("discrete", s["f"], s["v0"], outcomes=codes, mode="log")["data_T"],
                              s["top"]).cpu().numpy()
    assert_same_stats(got, general, rtol=1e-12)


@pytest.mark.parametrize("source", ["wide3", "c2"])
def test_pipeline_depths_at_production_size(source):
    """FinalSweepPipeline at depth 2 (the select kernel beside the next sweep, two CTAs: both lists spill) and depth
    1 (six CTAs): order statistics bit-equal, moments to 1e-12; the wide set also against the reference.  C2 is
    the flagship draw (1e6 investors x 1e4 die rolls, 45 561 bins: it spills only in the two-CTA shape)."""
    from rlmd_b200 import engine, lev_exp
    if source == "wide3":
        s = ts.get("wide3")
        arrays = [ts.rows(s)]
        f, v0, top, want = s["f"], s["v0"], s["top"], ts.set_reference("wide3")
    else:
        f = lev_exp.dice_factor_table(np.asarray(lev_exp.param_range(0.05, 1.0, 0.05), np.float32), 0.5, -0.5, 0.05)
        arrays = [engine.lev_draw("discrete", 1_000_000, 10_000, seed=420, probs=(1 / 6, 1 / 6, 2 / 3), packed=True)]
        v0, top, want = 100.0, 100, None
        bins = ts.tally_in_blocks(arrays[0], 3, blocks=1).info()["bins"]
        assert ts.spills(bins, 2) and not ts.spills(bins, 6), bins
    arrays = arrays * 3      # successive submissions alternate between the two tallies at depth 2
    res = {}
    for depth in (1, 2):
        pipe = engine.FinalSweepPipeline("discrete", f, v0, top, depth=depth)
        res[depth] = [pipe.submit(a) for a in arrays]
        pipe.synchronize()
        res[depth] = [x.cpu().numpy() for x in res[depth]]
    for one, two in zip(res[1], res[2]):
        assert np.array_equal(one[:, 9:12].view(np.uint64), two[:, 9:12].view(np.uint64))
        assert_same_stats(two, one, rtol=1e-12)
        if want is not None:
            assert_same_stats(one, want, rtol=1e-12)
            assert_same_stats(two, want, rtol=1e-12)


SHAPES = [(1, 0), (2, 0), (3, 0), (6, 0), (8, 0), (16, 0), (3, 7)]


@pytest.mark.parametrize("cluster,cache", SHAPES, ids=[f"cluster{c}-cache{k}" for c, k in SHAPES])
def test_every_cluster_and_cache_size(cluster, cache, tmp_path):
    """B200_SELECT_CLUSTER x B200_SELECT_CACHE in a child interpreter (cache 0: every bin spills, even for the small
    fixtures; 7: the cache ends inside a warp).  The child saves the four calls of every input; each must equal
    the reference, and the forced calls send every grid point to the radix route."""
    env = dict(os.environ, B200_SELECT_CLUSTER=str(cluster), B200_SELECT_CACHE=str(cache))
    code = "import sys; sys.path.insert(0, sys.argv[2]); import tally_sets; tally_sets.run_child(sys.argv[1])"
    p = subprocess.run([sys.executable, "-c", code, str(tmp_path), ts.TESTS], env=env, cwd=ts.ROOT,
                       capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stderr[-4000:]
    inputs = {name: (to.bins_of(oc, k), oc.shape[1], f, v0, top)
              for name, (oc, k, f, v0, top) in ts.small_inputs().items()}
    s = ts.get("wide3")
    for name, ((tuples, mult), h, f, v0, top) in inputs.items():
        want = ts.reference(tuples, mult, h, f, v0, top)
        for i in range(len(ts.FLAGS)):
            assert_same_stats(np.load(tmp_path / f"{name}_{i}.npy"), want, rtol=1e-12)
        radix = np.load(tmp_path / f"{name}_radix.npy")
        assert radix[2] == radix[3] == f.shape[0], (name, radix)
    want = ts.set_reference("wide3")
    for i in range(len(ts.FLAGS)):
        assert_same_stats(np.load(tmp_path / f"wide3_{i}.npy"), want, rtol=1e-12)
    radix = np.load(tmp_path / "wide3_radix.npy")
    assert radix[2] == radix[3] == s["f"].shape[0], radix
    # every target's log-wealth bin holds at most 256 tuples (test_tally_shapes.py): even one CTA takes the route
    assert radix[0] <= RADIX_ONLY["wide3"] and radix[1] <= RADIX_ONLY["wide3"], radix

"""
The chosen-tuple inputs of test_tally_shapes_gpu.py (tests/tally_sets.py) on the CPU: the expanded rows give back
the chosen tuples and multiplicities, and the large sets have the properties the GPU tests rely on - bin lists
above the select kernel's spill thresholds, per-rank lists longer than one merge chunk that share tuples, a
threshold tuple whose copies are split between the top group and the rest, and log-wealth bins small enough for
the log-wealth route.
"""
import numpy as np
import pytest
import torch as T

import tally_sets as ts
from oracle import lev_oracle as lo
from oracle import tally_lwsel_oracle as lw
from oracle import tally_oracle as to


@pytest.mark.parametrize("k,h", [(2, 1), (2, 9), (3, 7), (3, 64), (4, 33)])
def test_rows_give_back_the_chosen_tuples(k, h):
    rs = np.random.RandomState(k * 100 + h)
    cuts = np.sort(rs.randint(0, h + 1, size=(40, k - 1)), axis=1)
    tuples = np.diff(np.concatenate([np.zeros((40, 1), int), cuts, np.full((40, 1), h)], axis=1), axis=1)
    tuples = np.unique(tuples, axis=0)
    mult = rs.randint(1, 5, size=len(tuples))
    perm = rs.permutation(np.repeat(np.arange(len(tuples)), mult))
    codes = ts.expand(T.as_tensor(tuples[perm]), h, block=7).numpy()
    assert codes.shape == (mult.sum(), h) and codes.max() < k
    got, cnt = np.unique(lo.counts_discrete(codes, k), axis=0, return_counts=True)
    assert np.array_equal(got, tuples) and np.array_equal(cnt, mult)
    # the rows of one tuple are spread over the shuffled order
    assert not np.array_equal(perm, np.sort(perm))


def test_large_sets_cross_every_threshold():
    wide, coin, quad = ts.get("wide3"), ts.get("coin2"), ts.get("quad4")
    for s in (wide, coin, quad):
        assert len(np.unique(s["tuples"], axis=0)) == len(s["tuples"]) and (s["mult"] >= 1).all()
        assert (s["tuples"] >= 0).all() and (s["tuples"].sum(axis=1) == s["h"]).all()
        assert s["n"] == len(s["perm"]) and np.array_equal(np.bincount(s["perm"]), s["mult"])
    # bins per CTA above the shared-memory cache: the six-CTA default and the two-CTA shape beside a sweep
    for s in (wide, quad):
        assert ts.spills(len(s["tuples"]), 6) and ts.spills(len(s["tuples"]), 2)
    assert not ts.spills(len(coin["tuples"]), 6) and ts.spills(len(coin["tuples"]), 2)
    assert len(coin["tuples"]) == coin["h"] + 1        # every n1 in 0..H


@pytest.mark.parametrize("name", ["wide3", "coin2", "quad4"])
def test_threshold_tuple_is_split(name):
    """At the grid point `top` was chosen for, thr's copies go to both groups: 0 < ties in the top < ties."""
    s = ts.get(name)
    g = {"wide3": 9, "coin2": 9, "quad4": 3}[name]
    w = to.bin_wealth(s["tuples"], s["f"][g:g + 1], s["v0"])[0].astype(np.float64)
    order = np.argsort(-w, kind="stable")
    cum = np.cumsum(s["mult"][order])
    j = int(np.searchsorted(cum, s["top"] - 1, side="right"))
    above = int(cum[j - 1]) if j > 0 else 0
    assert s["mult"][order[j]] > 1 and above < s["top"] < above + s["mult"][order[j]]
    assert (w == w[order[j]]).sum() == 1


@pytest.mark.parametrize("world", [2, 3, 8])
def test_merge_shards_are_longer_than_one_chunk_and_overlap(world):
    s = ts.get("wide3")
    cuts = ts.shard_cuts(s["n"], world)
    lists = [np.unique(s["perm"][a:b]) for a, b in zip(cuts[:-1], cuts[1:])]
    sizes = [len(x) for x in lists]
    assert (0 in sizes) == (world >= 3)
    assert all(m == 0 or m > 8 * ts.MERGE_CHUNK for m in sizes)
    assert sum(sizes) > 60 * ts.MERGE_CHUNK
    seen = np.concatenate(lists)
    assert len(np.unique(seen)) == len(s["tuples"]) < len(seen)        # every tuple, many on several ranks


@pytest.mark.parametrize("name", ["wide3", "coin2"])
def test_log_wealth_bins_fit_the_candidate_lists(name):
    """On the dice / small-leverage rows the target ranks' log-wealth bins hold at most 256 tuples (the per-CTA
    limit, so even one CTA could hold a whole bin) and every check of the route passes: the kernel is expected
    to take the log-wealth route there with spilled bins.  The flat row and the zero factor are refused."""
    s = ts.get(name)
    g_route = 20
    with np.errstate(divide="ignore"):
        lm = np.log(s["f"].astype(np.float64))
    wealth = to.bin_wealth(s["tuples"], s["f"], s["v0"])
    for g in range(g_route):
        rng = lw.lw_range(s["tuples"], lm[g], s["v0"])
        assert rng is not None
        lwg = lw.log_wealth(s["tuples"], lm[g], s["v0"])
        assert lw.select(lwg, wealth[g], s["mult"], rng, s["top"], cand=256) is not None, g
    flat = s["f"].shape[0] - 1
    zero = s["f"].shape[0] - (3 if name == "wide3" else 2)
    assert lw.lw_range(s["tuples"], lm[flat], s["v0"]) is None and lw.lw_range(s["tuples"], lm[zero], s["v0"]) is None

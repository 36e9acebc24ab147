"""
Inputs of the tally statistics (rlmd_b200/csrc/tally.cu) whose count tuples are CHOSEN, not drawn: distinct
tuples [B,K] and their multiplicities [B] are picked on the CPU with a seeded RNG, and the outcome rows are
expanded from them (code[i, t] = (t >= n0_i) + (t >= n0_i + n1_i) + ...; only the counts matter) in a
shuffled investor order.  So the bin list has a known length, which puts it above the select kernel's
shared-memory cache (SEL_CACHE bins per CTA; the rest spill to the global wbuf) and the merges above one
chunk of MERGE_CHUNK concatenation positions.

The reference is oracle/tally_oracle.stats_from_bins fed with the GPU's own fp32 wealth of every bin: the
LOG sweep's data_T of ONE representative row per tuple (a bin's wealth is bit-identical to the data_T of its
investors, DESIGN.md 4.1; NumPy's exp may differ by one ulp).

Used by test_tally_shapes.py (CPU), test_tally_shapes_gpu.py and test_tally_gpu.py, and by the child
interpreters of test_tally_shapes_gpu.py (run_child), which read the select kernel's environment once.
"""
import os
import re
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TESTS = os.path.join(ROOT, "tests")
for _p in (ROOT, TESTS):
    if _p not in sys.path:
        sys.path.insert(0, _p)

from oracle import lev_oracle as lo  # noqa: E402
from oracle import tally_oracle as to  # noqa: E402


def _header_constant(name: str) -> int:
    src = open(os.path.join(ROOT, "rlmd_b200", "csrc", "tally.cuh")).read()
    return int(re.search(r"\b" + name + r"\s*=\s*(\d+)", src).group(1))


TH_BOX = _header_constant("TH_BOX")
TH_WORDS = _header_constant("TH_WORDS")
TALLY_COUNT_BITS = _header_constant("TALLY_COUNT_BITS")
TALLY_MAX_HORIZON = (1 << TALLY_COUNT_BITS) - 1
SEL_CACHE = 16384          # default bins per CTA kept in shared memory (select_shape, tally.cu)
MERGE_CHUNK = 2048         # concatenation positions per block of the mark / unique kernels (tally.cu)


def bins_per_cta(b: int, cluster: int) -> int:
    """The slice of the bin list one CTA of a `cluster`-CTA select cluster holds (tally_select_kernel)."""
    return ((b + cluster - 1) // cluster + 3) & ~3


def spills(b: int, cluster: int, cache: int = SEL_CACHE) -> bool:
    return bins_per_cta(b, cluster) > cache


# ------------------------------------------------------------------ the sets
DICE_LEV = np.asarray([0.05 * i for i in range(1, 21)], np.float32)   # the dice script's 20 leverages


def _wide3():
    """K = 3: 150 000 distinct (n1, n2) drawn uniformly from the triangle n1 + n2 <= 1200, multiplicities 1-4."""
    rs = np.random.RandomState(20261)
    h, b = 1200, 150_000
    tri = (h + 1) * (h + 2) // 2
    idx = np.sort(rs.choice(tri, size=b, replace=False))
    # row n1 of the triangle holds n2 = 0 .. h - n1: it starts at n1 (h + 1) - n1 (n1 - 1) / 2
    starts = np.array([n1 * (h + 1) - n1 * (n1 - 1) // 2 for n1 in range(h + 1)])
    n1 = np.searchsorted(starts, idx, side="right") - 1
    n2 = idx - starts[n1]
    tuples = np.stack([h - n1 - n2, n1, n2], axis=1)
    f = np.concatenate([lo.dice_factors(DICE_LEV, 0.5, -0.5, 0.05),
                        np.float32([[1.5, 0.0, 1.05],      # a zero factor: log -inf, the radix route
                                    [1e30, 1e-30, 1.0],    # saturates to +inf and to 0, thr included
                                    [1.0, 1.0, 1.0]])])    # flat
    return dict(tuples=tuples, mult=rs.randint(1, 5, size=b), h=h, f=f, v0=100.0, rs=rs, top_grid=9,
                top_at=0.02)


def _coin2():
    """K = 2, long horizon: every n1 in 0..40 000 (40 001 bins: above the two-CTA shape's spill threshold only)."""
    rs = np.random.RandomState(20262)
    h = 40_000
    n1 = np.arange(h + 1)
    tuples = np.stack([h - n1, n1], axis=1)
    lev = np.concatenate([[0.0005 * i for i in range(1, 21)], [0.05, 0.5]]).astype(np.float32)
    f = np.concatenate([lo.coin_factors(lev, 0.5, -0.4), np.float32([[0.0, 1.5], [1.0, 1.0]])])
    return dict(tuples=tuples, mult=rs.randint(1, 3, size=h + 1), h=h, f=f, v0=100.0, rs=rs, top_grid=9,
                top_at=0.1)


def _quad4():
    """K = 4 (the radix route only): 120 000 distinct (n1, n2, n3) with n1 + n2 + n3 <= 120, multiplicities 1-4."""
    rs = np.random.RandomState(20263)
    h, b = 120, 120_000
    a = np.arange(h + 1)
    n1, n2, n3 = [x.ravel() for x in np.meshgrid(a, a, a, indexing="ij")]
    ok = n1 + n2 + n3 <= h
    n1, n2, n3 = n1[ok], n2[ok], n3[ok]
    pick = np.sort(rs.choice(n1.size, size=b, replace=False))
    n1, n2, n3 = n1[pick], n2[pick], n3[pick]
    tuples = np.stack([h - n1 - n2 - n3, n1, n2, n3], axis=1)
    f = np.concatenate([(1 + rs.uniform(-0.3, 0.5, size=(20, 4))).astype(np.float32), np.ones((1, 4), np.float32)])
    return dict(tuples=tuples, mult=rs.randint(1, 5, size=b), h=h, f=f, v0=10.0, rs=rs, top_grid=3, top_at=0.05)


_SETS = {"wide3": _wide3, "coin2": _coin2, "quad4": _quad4}
_cache = {}


def split_top(tuples, mult, f_row, v0, at: float) -> int:
    """A `top` whose threshold tuple (at the grid point of `f_row`) has multiplicity > 1 and a wealth no other
    tuple shares: one copy goes to the top group, the others to the rest."""
    w = to.bin_wealth(tuples, f_row[None], v0)[0].astype(np.float64)
    order = np.argsort(-w, kind="stable")
    ws, ms = w[order], mult[order]
    cum = np.cumsum(ms)
    i = int(np.searchsorted(cum, at * cum[-1]))
    while not (ms[i] > 1 and np.isfinite(ws[i]) and ws[i - 1] > ws[i] > ws[i + 1]):
        i += 1
    return int(cum[i - 1]) + 1


def get(name: str) -> dict:
    """{tuples [B,K] int64, mult [B], h, k, f [G,K] fp32, v0, top, perm [N]: the tuple of every investor row}."""
    if name not in _cache:
        s = _SETS[name]()
        rs = s.pop("rs")
        s["tuples"] = s["tuples"].astype(np.int64)
        s["mult"] = s["mult"].astype(np.int64)
        s["k"] = s["tuples"].shape[1]
        s["n"] = int(s["mult"].sum())
        s["top"] = split_top(s["tuples"], s["mult"], s["f"][s.pop("top_grid")], s["v0"], s.pop("top_at"))
        s["perm"] = rs.permutation(np.repeat(np.arange(len(s["mult"])), s["mult"]))
        _cache[name] = s
    return _cache[name]


# ------------------------------------------------------------------ rows
def expand(tuples, h: int, block: int = 8192):
    """uint8 codes [N,h] (a torch tensor on the device of `tuples`, int64 [N,K]) whose counts are `tuples`."""
    import torch
    n, k = tuples.shape
    t = torch.arange(h, device=tuples.device)
    edge = torch.cumsum(tuples[:, :-1], dim=1)          # n0, n0 + n1, ...
    out = torch.empty((n, h), dtype=torch.uint8, device=tuples.device)
    for r0 in range(0, n, block):
        e = edge[r0:r0 + block]
        o = torch.zeros((e.shape[0], h), dtype=torch.uint8, device=tuples.device)
        for j in range(k - 1):
            o += (t[None, :] >= e[:, j:j + 1]).to(torch.uint8)
        out[r0:r0 + block] = o
    return out


def rows(s: dict, device="cuda"):
    """The set's investor rows (uint8 codes [N,h], shuffled) on `device`."""
    import torch
    return expand(torch.as_tensor(s["tuples"][s["perm"]], device=device), s["h"])


def tally_in_blocks(codes, k: int, blocks: int = 3):
    """A FinalTally of `codes` (uint8 codes, added in row blocks, or PackedCodes, added whole), finalized."""
    import torch
    from rlmd_b200 import tally
    t = tally.FinalTally(codes.shape[0])
    if not isinstance(codes, torch.Tensor):
        blocks = 1
    cuts = np.linspace(0, codes.shape[0], blocks + 1).astype(int)
    for a, b in zip(cuts[:-1], cuts[1:]):
        t.add(codes[a:b] if blocks > 1 else codes, k)
    t.finalize()
    return t


# ------------------------------------------------------------------ reference
def bin_wealth_gpu(tuples, h: int, f, v0):
    """[G,B] fp32: the LOG sweep's data_T of one representative row per tuple."""
    import torch
    from rlmd_b200 import engine
    reps = expand(torch.as_tensor(np.asarray(tuples, np.int64), device="cuda"), h)
    return engine.lev_sweep("discrete", f, v0, outcomes=reps, mode="log")["data_T"].cpu().numpy()


def reference(tuples, mult, h: int, f, v0, top: int):
    w = bin_wealth_gpu(tuples, h, f, v0)
    return np.stack([to.stats_from_bins(w[g], mult, top) for g in range(w.shape[0])])


_refs = {}


def set_reference(name: str):
    if name not in _refs:
        s = get(name)
        _refs[name] = reference(s["tuples"], s["mult"], s["h"], s["f"], s["v0"], s["top"])
    return _refs[name]


def box_of(tuples) -> list:
    """The four box header words of a bin list: (M - min n1, max n1, M - min n2, max n2), M = TALLY_MAX_HORIZON."""
    n1 = tuples[:, 1]
    n2 = tuples[:, 2] if tuples.shape[1] > 2 else np.zeros_like(n1)
    return [TALLY_MAX_HORIZON - int(n1.min()), int(n1.max()), TALLY_MAX_HORIZON - int(n2.min()), int(n2.max())]


def box_words(t) -> list:
    """The box words at the start of a tally's workspace."""
    return t.ws[:TH_WORDS].cpu().tolist()[TH_BOX:TH_BOX + 4]


def shard_cuts(n: int, world: int):
    """Uneven row shards; rank 1 is empty when there are three ranks or more."""
    cuts = np.linspace(0, n, world + 1).astype(int)
    cuts[1:-1] += np.arange(1, world) * 7 % 50
    if world >= 3:
        cuts[2] = cuts[1]
    return cuts


def one_gpu_ranks(world: int, rows_cap: int, bins_cap: int):
    """`world` FinalTally objects in THIS process, each with its own workspace and exchange buffer: the cross-GPU
    merge played on one GPU (every rank publishes with phase 0 before any rank merges with phase 1)."""
    import ctypes as C

    import torch as T
    from rlmd_b200 import _lib, tally
    from rlmd_b200._lib import check, lib, ptr, stream_ptr
    ranks = []
    for r in range(world):
        t = tally.FinalTally.__new__(tally.FinalTally)
        t.dev, t.group, t._staging, t.rows, t.horizon = T.device("cuda", 0), None, None, 0, None
        t.plan = _lib.TallyPlan()
        t.plan.rows_cap, t.plan.bins_cap, t.plan.grid_cap, t.plan.world = rows_cap, bins_cap, 64, world
        t.ws = T.empty((lib.b200_tally_workspace_bytes(C.byref(t.plan)) // 8,), dtype=T.int64, device="cuda")
        t.exchange = None
        t.ex_buf = T.zeros((lib.b200_tally_exchange_bytes(C.byref(t.plan)) // 8 + 1,), dtype=T.int64, device="cuda")
        check(lib.b200_tally_reset(C.byref(t.plan), ptr(t.ws), stream_ptr()))
        ranks.append(t)
    return ranks


def merge_on_one_gpu(ranks, epoch: int) -> None:
    import ctypes as C

    from rlmd_b200 import _lib
    from rlmd_b200._lib import check, lib, ptr, stream_ptr
    world = len(ranks)
    peers = []
    for r in range(world):
        p = _lib.TallyPeers()
        p.world, p.rank, p.epoch = world, r, epoch
        for q in range(world):
            p.exchange[q] = ranks[q].ex_buf.data_ptr()
        peers.append(p)
    for phase in (0, 1):
        for r, t in enumerate(ranks):
            check(lib.b200_tally_finalize(C.byref(t.plan), ptr(t.ws), C.byref(peers[r]), phase, stream_ptr()))


# ------------------------------------------------------------------ every cluster and cache size
TIES_F = np.array([[1.5, 0.6], [2.0, 0.0], [1e30, 1.0], [1.0, 1.0]], dtype=np.float32)
FLAGS = [(False, False), (True, False), (False, True), (True, True)]    # (beside_sweep, radix_select)


def small_inputs():
    """name -> (outcomes [N,H] uint8, K, factors, v0, top): three fixtures and the coin ties / +inf / zero rows of
    test_tally_lwsel_gpu.test_coin_ties_infinities_zeros_and_flat_rows."""
    import golden_io
    out = {}
    for name in ("coin_top7", "dice_top5", "dicesh_top3"):
        case = golden_io.lev_case(name)
        lev = lo.lev_grid(*case["grid"], case["up_r"], case["down_r"])
        if case["kind"] == "coin":
            f, k = lo.coin_factors(lev, case["up_r"], case["down_r"]), 2
        elif case["kind"] == "dice":
            f, k = lo.dice_factors(lev, case["up_r"], case["down_r"], case["mid_r"]), 3
        else:
            f, k = lo.dice_sh_factors(lev, case["up_r"], case["down_r"], case["mid_r"], *case["sh"]), 3
        out[name] = (golden_io.draw_outcomes(case).astype(np.uint8), k, f, case["v0"], case["top"])
    n, h = 515, 40
    same = np.ones((n, h), dtype=np.uint8)
    same[:, ::2] = 0
    half = same.copy()
    half[: n // 2] = 1
    coin = (np.random.RandomState(3).uniform(size=(20000, 3000)) < 0.5).astype(np.uint8)
    for name, oc in (("same", same), ("half", half), ("coin", coin)):
        out[name] = (oc, 2, TIES_F, 1.0, 3)
    return out


def run_child(out_dir: str) -> None:
    """The four statistics calls (FLAGS) on every small input and the wide set, saved as <name>_<i>.npy, and
    the grid points each call sent to the radix route as <name>_radix.npy.  Meant for a fresh interpreter whose
    environment sets B200_SELECT_CLUSTER / B200_SELECT_CACHE."""
    from rlmd_b200 import engine
    inputs = {name: (engine.encode_codes(oc), k, f, v0, top, oc.shape[0], oc.shape[1])
              for name, (oc, k, f, v0, top) in small_inputs().items()}
    s = get("wide3")
    inputs["wide3"] = (rows(s), 3, s["f"], s["v0"], s["top"], s["n"], s["h"])
    for name, (codes, k, f, v0, top, n, h) in inputs.items():
        t = tally_in_blocks(codes, k)
        radix = []
        for i, (beside, rad) in enumerate(FLAGS):
            before = t.info()["radix_route"]
            st = t.stats(f, v0, h, n_total=n, top=top, beside_sweep=beside, radix_select=rad).cpu().numpy()
            info = t.info()
            assert not (info["overflow"] or info["count_mismatch"]), (name, info)
            radix.append(info["radix_route"] - before)
            np.save(os.path.join(out_dir, f"{name}_{i}.npy"), st)
        np.save(os.path.join(out_dir, f"{name}_radix.npy"), np.asarray(radix))
        del t, codes

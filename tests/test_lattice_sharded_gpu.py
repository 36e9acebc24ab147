"""
coin_series_counts(..., group=) and dice_series_tuples(..., group=): the count-lattice series on investor shards
must return, on every rank, the one-GPU result on the concatenated codes - the lattice's columns and `routed` bit
for bit, the sharded chain's columns (unrouted leverages, the last column) with exact order statistics - and each
rank's slice of data_T.  On one GPU: 2 and 3 gloo ranks sharing cuda:0; on two GPUs: NCCL ranks at a larger shape.
"""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import golden_io
from oracle import lev_oracle as lo
from test_oracle_dice_lattice import case_factors

pytestmark = pytest.mark.gpu

DICE_P = (1 / 6, 1 / 6, 2 / 3)


def _free_port() -> int:
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _coin_inputs(case):
    from rlmd_b200 import lev_exp
    lev = lo.lev_grid(*case["grid"], case["up_r"], case["down_r"])
    return lev, lev_exp.coin_factor_table(lev, case["up_r"], case["down_r"])


def even_cuts(n, world):
    """The shard boundaries of sharding.shard_range: sizes differ by at most one."""
    from rlmd_b200 import sharding
    return [0] + [sum(sharding.shard_range(n, world, q)) for q in range(world)]


def _wide_rows(n, h):
    """Rows of all-up and all-down codes: together with any other rows their box spans (t+2)^2 cells at step t."""
    oc = np.zeros((n, h), dtype=np.uint8)
    oc[1::2] = 1
    return oc


def cases(world):
    """(name, kind, codes [N,H], lev, factors, v0, top, extra keyword arguments, shard cuts [world + 1])."""
    even = lambda n: even_cuts(n, world)
    out = []
    top7 = golden_io.lev_case("coin_top7")
    oc = golden_io.draw_outcomes(top7)
    lev, f = _coin_inputs(top7)
    unequal = [0, 500, 2001] if world == 2 else [0, 0, 1000, 2001]          # world 3: rank 0 holds no investor
    out.append(("coin_top7", "coin", oc, lev, f, 100.0, 7, {}, unequal))
    out.append(("coin_top7_chunks", "coin", oc, lev, f, 100.0, 7, {"chunk_steps": 7}, even(2001)))
    over = golden_io.lev_case("coin_overflow")
    lev, f = _coin_inputs(over)
    out.append(("coin_overflow", "coin", golden_io.draw_outcomes(over), lev, f, 100.0, 3, {}, even(400)))
    for h in (1, 2):
        lev, f = _coin_inputs(top7)
        oc = (np.random.RandomState(h).random_sample((301, h)) < 0.5).astype(np.uint8)
        out.append((f"coin_h{h}", "coin", oc, lev, f, 100.0, 2, {}, even(301)))

    dts = golden_io.lev_case("dice_testscale")
    oc = golden_io.draw_outcomes(dts)
    lev, f = case_factors(dts)
    unequal = [0, 3000, 10000] if world == 2 else [0, 4000, 4000, 10000]    # world 3: rank 1 holds no investor
    out.append(("dice_testscale", "dice", oc, lev, f, 100.0, 1, {}, unequal))
    out.append(("dice_chunks", "dice", oc, lev, f, 100.0, 3, {"chunk_bytes": 1 << 16}, even(10000)))
    dsh = golden_io.lev_case("dicesh_testscale")
    lev, f = case_factors(dsh)
    out.append(("dicesh_testscale", "dice", golden_io.draw_outcomes(dsh), lev, f, 100.0, 1, {}, even(10000)))
    lev = np.asarray([0.3, 0.6], dtype=np.float32)
    f = lo.dice_factors(lev, 0.5, -0.5, 0.05)
    for h in (1, 2):
        oc = np.random.RandomState(10 + h).choice(3, size=(301, h), p=DICE_P).astype(np.uint8)
        out.append((f"dice_h{h}", "dice", oc, lev, f, 100.0, 2, {}, even(301)))
    # the last rank's rows alone make the box too wide for the budget: nothing is routed on any rank
    lev = np.asarray([0.05, 0.1], dtype=np.float32)
    rest = np.random.RandomState(5).choice(3, size=(1000 * (world - 1), 200), p=DICE_P).astype(np.uint8)
    oc = np.concatenate([rest, _wide_rows(64, 200)])
    cuts = [1000 * r for r in range(world)] + [oc.shape[0]]
    out.append(("dice_budget", "dice", oc, lev, lo.dice_factors(lev, 0.5, -0.5, 0.05), 100.0, 2,
                {"chunk_bytes": 1 << 16}, cuts))
    return out


def run(kind, codes, lev, f, v0, top, kw, group=None):
    from rlmd_b200 import engine
    fn = engine.coin_series_counts if kind == "coin" else engine.dice_series_tuples
    return fn(f, lev, v0, top, codes, group=group, **kw)


def encode(oc, kind, device="cuda"):
    from rlmd_b200 import engine
    return engine.encode_codes(torch.as_tensor(oc), device=device, n_outcomes=2 if kind == "coin" else 3)


def _gloo_worker(rank, world, port, out_dir):
    from rlmd_b200 import engine

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RLMD_B200_EXCHANGE="nccl")
    torch.cuda.set_device(0)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    g = dist.group.WORLD
    try:
        for name, kind, oc, lev, f, v0, top, kw, cuts in cases(world):
            data, data_T, routed = run(kind, encode(oc[cuts[rank]:cuts[rank + 1]], kind), lev, f, v0, top, kw, g)
            np.savez(os.path.join(out_dir, f"{name}_{rank}.npz"), data=data.cpu().numpy(),
                     data_T=data_T.cpu().numpy(), routed=routed)
        # refusals: every rank raises ValueError, and the group is still usable afterwards
        refused = []
        top7 = golden_io.lev_case("coin_top7")
        lev, f = _coin_inputs(top7)
        oc = golden_io.draw_outcomes(top7)[rank::world]
        try:
            engine.coin_series_counts(f, lev, 100.0, 7, encode(oc, "coin"), dtype=torch.float64, group=g)
        except ValueError:
            refused.append("fp64")
        try:
            engine.coin_series_counts(f, lev, 100.0, 7, encode(oc[:, :30 + rank], "coin"), group=g)
        except ValueError:
            refused.append("coin_h")
        dts = golden_io.lev_case("dice_testscale")
        lev, f = case_factors(dts)
        oc = golden_io.draw_outcomes(dts)[rank::world]
        try:
            engine.dice_series_tuples(f, lev, 100.0, 1, encode(oc[:, :40 + rank], "dice"), group=g)
        except ValueError:
            refused.append("dice_h")
        try:           # one rank's codes are not a CUDA tensor: refused there, and the others raise with it
            codes = encode(oc[:, :40], "dice")
            engine.dice_series_tuples(f, lev, 100.0, 1, codes.cpu() if rank == world - 1 else codes, group=g)
        except ValueError:
            refused.append("dice_local")
        from rlmd_b200 import sharding
        assert sharding.global_count(1, g, "cuda") == world
        np.save(os.path.join(out_dir, f"refused_{rank}.npy"), np.array(refused))
    finally:
        dist.destroy_process_group()


def check_rank(got, want, cuts, rank):
    """One rank's (data, data_T, routed) against the one-GPU call on the concatenated codes."""
    data, data_T, routed = got["data"], got["data_T"], got["routed"]
    w_data, w_T, w_routed = want
    assert data.dtype == np.float32 and data.shape == w_data.shape
    assert np.array_equal(routed, w_routed)
    assert np.array_equal(data_T.view(np.uint32), w_T[:, cuts[rank]:cuts[rank + 1]].view(np.uint32))
    if data.shape[2] == 0:
        return
    # the lattice's columns (every column but the last) of routed leverages, and the leverage row: bit for bit
    assert np.array_equal(data[routed, :, :-1].view(np.uint32), w_data[routed, :, :-1].view(np.uint32))
    assert np.array_equal(data[:, 12].view(np.uint32), w_data[:, 12].view(np.uint32))
    # the sharded chain's columns: unrouted leverages and the last column.  Order statistics exact; the float64
    # moments sum in another order (agree to ~1e-12) and can round to fp32 one ulp apart
    for got_c, want_c in ((data[~routed, :12], w_data[~routed, :12]), (data[:, :12, -1:], w_data[:, :12, -1:])):
        assert np.array_equal(got_c[:, 9:12].view(np.uint32), want_c[:, 9:12].view(np.uint32))
        np.testing.assert_allclose(got_c[:, :9], want_c[:, :9], rtol=2.0 ** -23, atol=0)


@pytest.mark.parametrize("world", [2, 3])
def test_gloo_ranks_on_one_gpu_equal_one_call(tmp_path, world):
    from rlmd_b200 import engine

    mp.spawn(_gloo_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    seen_routed, seen_unrouted = set(), set()
    for name, kind, oc, lev, f, v0, top, kw, cuts in cases(world):
        d, t, r = run(kind, encode(oc, kind), lev, f, v0, top, kw)
        want = (d.cpu().numpy(), t.cpu().numpy(), r)
        (seen_routed if r.any() else seen_unrouted).add(name)
        for rank in range(world):
            check_rank(np.load(tmp_path / f"{name}_{rank}.npz"), want, cuts, rank)
        if name == "dice_budget":     # the first rank's rows alone fit the budget; the concatenation does not
            def plan(rows):
                b = engine.dice_lattice_bounds(encode(rows, "dice"), 0, rows.shape[1],
                                               torch.empty((2, rows.shape[0]), dtype=torch.int32, device="cuda"))
                return engine.dice_lattice_plan(b.cpu().numpy(), kw["chunk_bytes"])
            assert plan(oc[:cuts[1]]) is not None and plan(oc) is None and not r.any()
        if name == "dice_chunks":
            assert r.all()
    # both walks took the lattice, and the chain fallback under a group was exercised
    assert {"coin_top7", "coin_overflow", "dice_testscale", "dicesh_testscale"} <= seen_routed
    over = [c for c in cases(world) if c[0] == "coin_overflow"][0]
    assert not run("coin", encode(over[2], "coin"), *over[3:8])[2].all()
    for rank in range(world):
        assert sorted(np.load(tmp_path / f"refused_{rank}.npy").tolist()) == ["coin_h", "dice_h", "dice_local", "fp64"]


def _nccl_worker(rank, world, port, out_dir):
    from rlmd_b200 import engine, sharding

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    g = dist.group.WORLD
    try:
        for kind, n, h, seed in NCCL_SHAPES:
            off, cnt = sharding.shard_range(n, world, rank)
            probs = (0.5, 0.5) if kind == "coin" else DICE_P
            codes = engine.lev_draw("discrete", cnt, h, seed=seed, investor_offset=off, probs=probs)
            lev, f = nccl_grid(kind)
            data, data_T, routed = run(kind, codes, lev, f, 100.0, 100, {}, g)
            np.savez(os.path.join(out_dir, f"{kind}_{rank}.npz"), data=data.cpu().numpy(),
                     data_T=data_T.cpu().numpy(), routed=routed)
            del codes, data_T
            torch.cuda.empty_cache()
    finally:
        dist.destroy_process_group()


# production-like shapes: the coin at C1's smart size, the dice script's grid (1e6 investors in all)
NCCL_SHAPES = [("coin", 1_000_000, 3000, 31), ("dice", 1_000_000, 2000, 32)]


def nccl_grid(kind):
    from rlmd_b200 import lev_exp
    lev = np.asarray(lev_exp.param_range(0.1, 1.0, 0.1), dtype=np.float32)
    if kind == "coin":
        return lev, lev_exp.coin_factor_table(lev, 0.5, -0.4)
    return lev, lev_exp.dice_factor_table(lev, 0.5, -0.5, 0.05)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_gpus_equal_one():
    import tempfile

    from rlmd_b200 import engine

    world = 2
    with tempfile.TemporaryDirectory() as out_dir:
        mp.spawn(_nccl_worker, args=(world, _free_port(), out_dir), nprocs=world, join=True)
        for kind, n, h, seed in NCCL_SHAPES:
            probs = (0.5, 0.5) if kind == "coin" else DICE_P
            codes = engine.lev_draw("discrete", n, h, seed=seed, probs=probs)
            lev, f = nccl_grid(kind)
            d, t, r = run(kind, codes, lev, f, 100.0, 100, {})
            want = (d.cpu().numpy(), t.cpu().numpy(), r)
            del codes, t
            assert r.any()
            cuts = even_cuts(n, world)
            for rank in range(world):
                check_rank(np.load(os.path.join(out_dir, f"{kind}_{rank}.npz")), want, cuts, rank)

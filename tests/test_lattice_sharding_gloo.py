"""
The host-side helpers of the sharded count-lattice series on CPU (gloo ranks, host tensors):
sharding.agree raises on every rank at once, and sharding.gather_steps reassembles the per-rank step slices.
"""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp


def _free_port() -> int:
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, out_dir):
    from rlmd_b200 import sharding

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    g = dist.group.WORLD
    seen = []
    try:
        sharding.agree([300, 10, 2 ** 40 + 7, -1], g, "cpu")
        seen.append("same")
        for name, values, refused in (("mismatch", [300 + (rank == world - 1), 10], ""),
                                      ("refused", [300, 10], "bad codes" if rank == 0 else "")):
            try:
                sharding.agree(values, g, "cpu", refused)
            except ValueError as exc:
                seen.append(name + (":own" if "bad codes" in str(exc) else ""))
        for steps in (1, 2, 7, 12):
            off, cnt = sharding.shard_range(steps, world, rank)
            block = torch.arange(off, off + cnt, dtype=torch.float64).repeat(3, 1)[:, :, None] * torch.ones(1, 1, 12)
            got = sharding.gather_steps(block, steps, g)
            want = torch.arange(steps, dtype=torch.float64).repeat(3, 1)[:, :, None] * torch.ones(1, 1, 12)
            assert torch.equal(got, want), (steps, got)
        seen.append("gather")
        assert sharding.global_count(1, g, "cpu") == world        # the group is still in step
    finally:
        np.save(os.path.join(out_dir, f"seen{rank}.npy"), np.array(seen))
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_agree_and_gather_steps(tmp_path, world):
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    for rank in range(world):
        seen = np.load(tmp_path / f"seen{rank}.npy").tolist()
        assert seen == ["same", "mismatch", "refused:own" if rank == 0 else "refused", "gather"]

"""
Host-side logic of the multi-GPU path (SURVEY.md section 8e): the sweep shards
by INVESTOR - one process per GPU, every rank holds the whole leverage grid and a
contiguous block of investor rows, Philox counters carry the global investor id -
so there is no data-path collective.  The only exchange is inside the
cross-investor statistics: after each pass of b200_rowstats the per-row partial
sums and radix histograms named by b200_rowstats_exchange are summed over ranks
(and, for the count-lattice series, the integer histograms themselves: `agree`
and `gather_steps` are that walk's helpers - engine.coin_series_counts).

Nothing here launches a kernel, so the module is exercised on CPU with the gloo
backend (tests/test_sharding_gloo.py) as well as with NCCL on the GPUs.
"""
from __future__ import annotations

import ctypes as C
from typing import Callable, Tuple

import torch

from ._lib import check, lib

N_PHASES = 5


def shard_range(n_total: int, world: int, rank: int) -> Tuple[int, int]:
    """(offset, count) of the contiguous investor block of `rank`: sizes differ by at most one."""
    if not 0 <= rank < world:
        raise ValueError("rank outside the world")
    base, extra = divmod(int(n_total), int(world))
    count = base + (1 if rank < extra else 0)
    offset = rank * base + min(rank, extra)
    return offset, count


def exchange_words(phase: int, what: str = "rowstats") -> Tuple[int, int, int, int, int]:
    """(int_offset, int_count, double_offset, double_count, words_per_row) to sum after `phase`."""
    ex = (C.c_int64 * 5)()
    fn = lib.b200_rowstats_exchange if what == "rowstats" else lib.b200_growth_exchange
    check(fn(int(phase), ex))
    return tuple(int(v) for v in ex)


def global_count(n_local: int, group, device) -> int:
    """Sum of the ranks' local investor counts."""
    import torch.distributed as dist

    t = torch.tensor([int(n_local)], dtype=torch.int64, device=device)
    dist.all_reduce(t, group=group)
    return int(t.item())


def agree(values, group, device, refused: str = "") -> None:
    """
    Collective check that every rank of `group` called with the same `values` (integers: sizes, flags, checksums
    of the arguments).  `refused` is this rank's own ValueError message when its local inputs failed validation;
    it still takes part, so that every rank raises together instead of one waiting in a later collective.
    """
    import torch.distributed as dist

    v = torch.tensor([0 if refused else 1] + [int(x) for x in values], dtype=torch.int64, device=device)
    both = torch.cat([v, -v])            # one MAX all-reduce: the maxima, then minus the minima
    dist.all_reduce(both, op=dist.ReduceOp.MAX, group=group)
    hi, lo = both[:v.numel()].tolist(), (-both[v.numel():]).tolist()
    if refused:
        raise ValueError(refused)
    if lo[0] == 0:
        raise ValueError("rlmd_b200: another rank's inputs were refused (see that rank's error)")
    if hi != lo:
        raise ValueError("rlmd_b200: the ranks disagree on the call's shape or arguments (horizon, grid, top, "
                         "factors, chunking)")


def gather_steps(block: torch.Tensor, steps: int, group) -> torch.Tensor:
    """
    The all-gather of per-step results split by shard_range over the steps: `block` [G, count, ...] holds this
    rank's steps; returns [G, steps, ...] of every rank's blocks in rank order (identical on every rank).
    The blocks travel padded to the largest count.
    """
    import torch.distributed as dist

    world = dist.get_world_size(group)
    per = (steps + world - 1) // world
    pad = block.new_zeros((block.shape[0], per) + tuple(block.shape[2:]))
    pad[:, :block.shape[1]] = block
    parts = [torch.empty_like(pad) for _ in range(world)]
    dist.all_gather(parts, pad, group=group)
    return torch.cat([p[:, :shard_range(steps, world, r)[1]] for r, p in enumerate(parts)], dim=1)


class PeerWorkspace:
    """
    The statistics workspaces of all ranks of `group` (the GPUs of one node), each
    mapped into every process through torch's symmetric memory (CUDA IPC over
    NVLink), for b200_rowstats_p2p: two workspaces per rank (successive calls
    alternate: a peer may still be summing the previous call's histograms) and one
    flag block, plus two alternating staging areas.  Rows are owned round-robin: every rank
    pushes a row's partial sums into its owner's staging area, the owner sums and resolves
    the rows it owns and stores the resolved words into every workspace (rowstats.cu).  Construction and `peer_set` are collective: every rank must make
    the same calls in the same order, and the calls of one workspace must execute
    one after the other on the GPU - engine.rowstats chains them with an event
    (`last_call`), whatever streams they are issued on.
    """

    FLAG_WORDS = 64   # B200_PEER_FLAG_WORDS uint32 ([8 ranks][8 flags], error word, tickets) in 8-byte slots
    ERROR_WORD = 64   # B200_PEER_FLAG_ERROR_WORD

    def __init__(self, rows: int, group, device):
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm

        from ._lib import MAX_PEERS

        self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        if self.world > MAX_PEERS:
            raise ValueError(f"the peer-memory exchange spans at most {MAX_PEERS} GPUs of one node")
        self.rows = int(rows)
        self.row_words = int(lib.b200_rowstats_workspace_bytes(1)) // 8
        self.stage_rows = (self.rows + self.world - 1) // self.world       # owned rows per source rank
        self.stage_words = int(lib.b200_rowstats_stage_bytes(self.rows, self.world)) // 8
        # two alternating workspaces, the flags, two alternating staging areas
        words = 2 * self.rows * self.row_words + self.FLAG_WORDS + 2 * self.stage_words
        self.buf = symm.empty(words, dtype=torch.int64, device=device)
        self.buf.zero_()
        self.handle = symm.rendezvous(self.buf, group)
        self.ptrs = [int(p) for p in self.handle.buffer_ptrs]
        torch.cuda.synchronize(device)
        dist.barrier(group=group)          # every rank's flags are zero before anyone signals
        self.epoch = 0
        self.last_call = None     # event after the last b200_rowstats_p2p on this workspace (engine.rowstats)

    def peer_set(self):
        """The b200_peer_set of the next call (advances the epoch: collective)."""
        from ._lib import PeerSet

        self.epoch += 1
        parity = self.epoch & 1
        ps = PeerSet()
        ps.world, ps.rank, ps.epoch = self.world, self.rank, self.epoch
        for r in range(self.world):
            ps.workspace[r] = self.ptrs[r] + 8 * parity * self.rows * self.row_words
            ps.flags[r] = self.ptrs[r] + 8 * 2 * self.rows * self.row_words
            ps.stage[r] = self.ptrs[r] + 8 * (2 * self.rows * self.row_words + self.FLAG_WORDS + parity * self.stage_words)
        ps.stage_rows = self.stage_rows
        return ps

    def timed_out(self, clear: bool = False) -> bool:
        """True when a resolve kernel gave up waiting for a peer (its statistics are NaN)."""
        flags = self.buf[2 * self.rows * self.row_words:2 * self.rows * self.row_words + self.FLAG_WORDS].view(torch.int32)
        hit = bool(flags[self.ERROR_WORD].item())
        if hit and clear:
            flags[self.ERROR_WORD] = 0
        return hit


_peer_cache = {}
_peer_ok = {}


def _key(group, device):
    d = torch.device(device)
    index = d.index if d.index is not None else torch.cuda.current_device()
    return (id(group), index)


def raise_if_peers_timed_out(group, device) -> None:
    """
    After a synchronisation point: raises when a resolve step of the peer-memory exchange gave up
    waiting for a peer's flag (~60 s; the statistics of that call are NaN).  Costs one 4-byte
    device-to-host read; a no-op when the group does not use the peer-memory exchange.
    """
    pw = _peer_cache.get(_key(group, device))
    if pw is not None and pw.timed_out(clear=True):      # (the error word is cleared: later calls start clean)
        raise RuntimeError("rlmd_b200: a rank did not reach the statistics exchange within 60 s "
                           "(peer-memory flags); the statistics of that call are NaN")


def peer_memory_available(group, device) -> bool:
    """
    Whether the ranks of `group` can map each other's memory (torch symmetric
    memory: the GPUs of one node with peer access).  Decided once per group by ALL
    ranks together (a collective: a rank that cannot allocate vetoes for everyone),
    so that every rank takes the same exchange path afterwards.
    """
    import sys

    import torch.distributed as dist

    key = _key(group, device)
    if key not in _peer_ok:
        ok = 1
        try:
            _peer_cache[key] = PeerWorkspace(64, group, device)
        except Exception as exc:  # noqa: BLE001 - any failure means "use the all-reduce path"
            ok = 0
            print(f"rlmd_b200: peer-memory exchange unavailable ({exc}); using NCCL all-reduces", file=sys.stderr)
        t = torch.tensor([ok], dtype=torch.int32, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MIN, group=group)
        _peer_ok[key] = bool(t.item())
        if not _peer_ok[key]:
            _peer_cache.pop(key, None)
    return _peer_ok[key]


def peer_workspace(rows: int, group, device) -> PeerWorkspace:
    """Cached per (group, device); grown (collectively) when a call needs more rows."""
    key = _key(group, device)
    pw = _peer_cache.get(key)
    if pw is None or pw.rows < rows:
        if pw is not None:
            # peers may still be reading the old workspaces: every rank finishes its work, then all let go together
            import torch.distributed as dist

            torch.cuda.synchronize(device)
            dist.barrier(group=group)
        pw = PeerWorkspace(max(rows, 64), group, device)
        _peer_cache[key] = pw
    return pw


def exchange_phases(run_phase: Callable[[int], None], workspace: torch.Tensor, group, what: str = "rowstats",
                    n_phases: int = N_PHASES) -> None:
    """
    Drives the statistics passes of one rank: `run_phase(p)` launches phase p on
    the local rows (filling this rank's partials in `workspace` [rows, words],
    int64), after which the phase's exchange region is all-reduced (SUM) so that
    every rank resolves the same global histogram walk in phase p+1.
    """
    import torch.distributed as dist

    if workspace.is_cuda:
        # one packed fp64 all-reduce per phase (pack / unpack kernels of the C ABI)
        from ._lib import ptr, stream_ptr

        rows, words = workspace.shape
        with torch.cuda.device(workspace.device):
            for phase in range(n_phases):
                run_phase(phase)
                io, ic, do, dc, _ = exchange_words(phase, what)
                if ic + dc == 0:
                    continue
                staging = torch.empty((rows, ic + dc), dtype=torch.float64, device=workspace.device)
                check(lib.b200_exchange_pack(ptr(workspace), words, rows, io, ic, do, dc, ptr(staging), stream_ptr()))
                dist.all_reduce(staging, group=group)
                check(lib.b200_exchange_unpack(ptr(workspace), words, rows, io, ic, do, dc, ptr(staging),
                                               stream_ptr()))
        return

    # host tensors (gloo, the CPU tests of this module): the same exchange, region by region
    ws_f = workspace.view(torch.float64)
    for phase in range(n_phases):
        run_phase(phase)
        io, ic, do, dc, _ = exchange_words(phase, what)
        if ic:
            part = workspace[:, io:io + ic].contiguous()
            dist.all_reduce(part, group=group)
            workspace[:, io:io + ic] = part
        if dc:
            part = ws_f[:, do:do + dc].contiguous()
            dist.all_reduce(part, group=group)
            ws_f[:, do:do + dc] = part

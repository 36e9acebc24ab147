"""
Final-time statistics of the discrete sweeps from outcome-count tuples - the
route every `{coin,dice,dice_sh}_fixed_final_lev` call takes
(lev/lev_exp.py:56-125, :508-583, :1121-1206).

    outcomes (any format, device or host)
      -> count kernel / ingest kernel with the tally as its sink   (one read of the outcomes)
      -> finalize: distinct count tuples (across GPUs: one exchange of bin lists)
      -> statistics of any number of leverage grids                 (no [G,N] array anywhere)

Accepted outcome formats
  * the engine's: uint8 codes [N,H] on the GPU, or engine.PackedCodes (2-bit);
  * the reference's, exactly as its scripts hold them: fp32 {0,1}
    (Bernoulli.sample, lev/coin_flip.py:160), int64 {0,1,2} (Categorical.sample,
    lev/dice_roll.py:147), and int32 / fp64 / uint8 / bool - on the GPU, or in
    host memory (pinned or pageable), which is walked in row chunks through two
    device staging buffers so that the copy of chunk i+1 overlaps the ingest of
    chunk i and the device never holds more than two chunks of the source.

Thin ctypes calls into librlmd_b200.so (tally.cu, lev_ingest.cu, lev_sweep.cu);
torch is the allocator and the stream provider.  No CPU path.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import numpy as np
import torch

from . import _lib
from ._lib import LevDesc, TallyPeers, TallyPlan, check, lib, ptr, require_cuda, stream_ptr

_SRC_TYPES = {
    torch.uint8: _lib.DT_U8, torch.bool: _lib.DT_U8, torch.int32: _lib.DT_I32, torch.int64: _lib.DT_I64,
    torch.float32: _lib.DT_F32, torch.float64: _lib.DT_F64,
}

DEFAULT_BINS_CAP = 1 << 22


class TallyOverflow(RuntimeError):
    """More distinct count tuples than the plan's bins_cap: use lev_sweep + rowstats for this input."""


class TallyUnavailable(TallyOverflow):
    """The ranks of the group cannot map each other's memory (no peer access): the tally's exchange cannot be
    set up; callers take the general path (lev_sweep + rowstats with the NCCL exchange), like on overflow."""


class TallyExchange:
    """
    One rank's peer-mapped exchange buffer (torch symmetric memory: CUDA IPC over
    NVLink) for b200_tally_finalize: two alternating bin lists and the arrival flags.
    Every FinalTally owns its own - its epochs and flags are private to the
    sequence of finalize calls made on that object (calls of ONE FinalTally must
    be issued in the same order on every rank; different FinalTally objects are
    independent and may run on different streams).  Construction is collective.
    """

    def __init__(self, nbytes: int, group, device):
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm

        self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        self.buf = symm.empty((nbytes + 7) // 8, dtype=torch.int64, device=device)
        self.buf.zero_()
        self.handle = symm.rendezvous(self.buf, group)
        self.ptrs = [int(p) for p in self.handle.buffer_ptrs]
        torch.cuda.synchronize(device)
        dist.barrier(group=group)      # every rank's flags are zero before anyone signals
        self.epoch = 0

    def next_peers(self) -> TallyPeers:
        self.epoch += 1
        p = TallyPeers()
        p.world, p.rank, p.epoch = self.world, self.rank, self.epoch
        for r in range(self.world):
            p.exchange[r] = self.ptrs[r]
        return p


class FinalTally:
    """
    Plan + workspace of the tally path for up to `rows_cap` investor rows per sweep
    on this GPU.  `group`: a torch.distributed process group whose ranks each hold
    an investor shard (one node, peer access); the statistics are then global and
    bit-identical on every rank.

        t = FinalTally(n, device=dev)
        t.add(outcomes, n_outcomes=3)          # any accepted format; may be called per row block
        t.finalize()
        stats = t.stats(table, 100.0, horizon, n_total=n, top=100)   # float64 [G,12] on the GPU
        t.check()                              # host sync: raises on overflow / bad outcomes / time-out
    """

    def __init__(self, rows_cap: int, *, device="cuda", group=None, bins_cap: Optional[int] = None,
                 grid_cap: int = _lib.MAX_GRID, world_rows: Optional[int] = None):
        require_cuda()
        self.dev = torch.device(device)
        if self.dev.index is None:
            self.dev = torch.device("cuda", torch.cuda.current_device())
        self.group = group
        world = 1
        if group is not None:
            import torch.distributed as dist

            world = dist.get_world_size(group)
        rows_cap = max(int(rows_cap), 1)
        total = int(world_rows) if world_rows is not None else rows_cap * world
        self.plan = TallyPlan()
        self.plan.rows_cap = rows_cap
        self.plan.bins_cap = int(bins_cap) if bins_cap is not None else max(1024, min(total, DEFAULT_BINS_CAP))
        self.plan.grid_cap = int(grid_cap)
        self.plan.world = world
        nbytes = lib.b200_tally_workspace_bytes(C.byref(self.plan))
        if nbytes < 0:
            raise _lib.B200Error(_lib.B200_EINVAL, lib.b200_last_error().decode())
        with torch.cuda.device(self.dev):
            self.ws = torch.empty((nbytes // 8,), dtype=torch.int64, device=self.dev)
            self.exchange = None
            if world > 1:
                self.exchange = TallyExchange(lib.b200_tally_exchange_bytes(C.byref(self.plan)), group, self.dev)
            check(lib.b200_tally_reset(C.byref(self.plan), ptr(self.ws), stream_ptr()))
        self._staging = None
        self.rows = 0            # rows added since the last finalize (host bookkeeping)
        self.horizon = None

    # ------------------------------------------------------------------ filling
    def reset(self) -> None:
        with torch.cuda.device(self.dev):
            check(lib.b200_tally_reset(C.byref(self.plan), ptr(self.ws), stream_ptr()))
        self.rows = 0

    def _note(self, n: int, h: int) -> None:
        if self.horizon is not None and self.rows > 0 and self.horizon != h:
            raise ValueError("every row block of one sweep must have the same horizon")
        if self.rows + n > self.plan.rows_cap:
            raise ValueError(f"more than rows_cap = {self.plan.rows_cap} rows in one sweep")
        if h > _lib.TALLY_MAX_HORIZON:
            raise ValueError("the tally path needs horizon < 2^21")
        self.horizon = h
        self.rows += n

    def add(self, outcomes, n_outcomes: int, *, counts: Optional[torch.Tensor] = None,
            codes_out: Optional[torch.Tensor] = None, early_start: bool = False) -> None:
        """
        Tallies the rows of `outcomes` (a CUDA tensor [N,H] in any accepted format, or
        PackedCodes) on the current stream.  `counts` (int32 [N,K]) and `codes_out`
        (uint8 [N, >=H], reference formats only) are optional extra sinks.
        early_start: packed outcomes only - the count kernel may start while the stream's previous kernel
        runs (B200_LEV_FLAG_EARLY_START); only when that kernel does not write the outcomes.
        """
        from .engine import PackedCodes

        k = int(n_outcomes)
        with torch.cuda.device(self.dev):
            if isinstance(outcomes, PackedCodes) or (outcomes.dtype == torch.uint8 and codes_out is None):
                packed = isinstance(outcomes, PackedCodes)
                data = outcomes.data if packed else outcomes
                n, h = outcomes.shape
                if not data.is_cuda or data.dim() != 2 or (n > 1 and data.stride(1) != 1):
                    raise ValueError("outcomes must be a [N,H] CUDA tensor with unit inner stride")
                self._note(n, h)
                d = LevDesc()
                d.kind, d.mode, d.source = _lib.LEV_DISCRETE, _lib.MODE_LOG, _lib.SRC_STREAM
                d.n_investors, d.horizon, d.n_grid, d.n_outcomes = n, h, 1, k
                d.value_0 = 1.0
                d.outcome_bits = outcomes.bits if packed else 8
                d.ld_outcomes = data.stride(0) if n > 1 else data.shape[1]
                d.flags = _lib.LEV_FLAG_EARLY_START if early_start else 0
                check(lib.b200_lev_tally(C.byref(d), ptr(data), C.byref(self.plan), ptr(self.ws), ptr(counts),
                                         stream_ptr()))
                return
            t = outcomes
            if t.dtype not in _SRC_TYPES:
                raise TypeError(f"outcomes of dtype {t.dtype} are not an accepted format")
            if not t.is_cuda or t.dim() != 2 or (t.shape[0] > 1 and t.stride(1) != 1):
                raise ValueError("outcomes must be a [N,H] CUDA tensor with unit inner stride")
            n, h = t.shape
            self._note(n, h)
            ld = t.stride(0) if n > 1 else max(t.stride(0), h)
            ldc = 0
            if codes_out is not None:
                if codes_out.dtype != torch.uint8 or codes_out.shape[0] != n or codes_out.shape[1] < h:
                    raise ValueError("codes_out must be uint8 [N, >=H]")
                ldc = codes_out.stride(0) if n > 1 else codes_out.shape[1]
            check(lib.b200_lev_ingest(ptr(t), _SRC_TYPES[t.dtype], n, h, ld, k, ptr(codes_out), ldc, ptr(counts),
                                      C.byref(self.plan), ptr(self.ws), stream_ptr()))

    def add_host(self, host: torch.Tensor, n_outcomes: int, *, chunk_bytes: int = 256 << 20,
                 horizon: Optional[int] = None) -> int:
        """
        Tallies a HOST array (any accepted format, or PackedCodes over a host tensor):
        row chunks travel through two device staging buffers on a copy stream while the
        previous chunk is ingested.  Returns the bytes copied host -> device.
        """
        from .engine import PackedCodes, _copy_stream

        packed = isinstance(host, PackedCodes)
        src = host.data if packed else host
        if src.is_cuda or src.dim() != 2:
            raise ValueError("add_host takes a 2-D host tensor (or PackedCodes over one)")
        n = src.shape[0]
        h = host.horizon if packed else src.shape[1]
        if n == 0:
            return 0
        if src.stride(1) != 1:
            src = src.contiguous()
        if src.dtype == torch.bool:
            src = src.view(torch.uint8)
        width = src.shape[1]
        row_bytes = width * src.element_size()
        rows = int(max(1, min(n, chunk_bytes // max(row_bytes, 1))))
        with torch.cuda.device(self.dev):
            key = (src.dtype, rows, width)
            if self._staging is None or self._staging[0] != key:
                self._staging = (key, [torch.empty((rows, width), dtype=src.dtype, device=self.dev) for _ in range(2)],
                                 [torch.cuda.Event() for _ in range(2)], [torch.cuda.Event() for _ in range(2)])
            _, bufs, ready, done = self._staging
            comp = torch.cuda.current_stream()
            copy = _copy_stream(self.dev)
            copy.wait_stream(comp)
            for i, r0 in enumerate(range(0, n, rows)):
                m = min(rows, n - r0)
                b = bufs[i & 1]
                if i >= 2:
                    copy.wait_event(done[i & 1])
                with torch.cuda.stream(copy):
                    b[:m].copy_(src[r0:r0 + m], non_blocking=True)
                    ready[i & 1].record(copy)
                comp.wait_event(ready[i & 1])
                self.add(PackedCodes(b[:m], h, host.bits) if packed else b[:m], n_outcomes)
                done[i & 1].record(comp)
            copy.wait_event(done[0])
            copy.wait_event(done[1])
        return n * row_bytes

    # -------------------------------------------------------------- statistics
    def finalize(self) -> None:
        with torch.cuda.device(self.dev):
            peers = self.exchange.next_peers() if self.exchange is not None else None
            check(lib.b200_tally_finalize(C.byref(self.plan), ptr(self.ws), C.byref(peers) if peers else None, -1,
                                          stream_ptr()))
        self.rows = 0

    def stats(self, factors: np.ndarray, value_0: float, horizon: int, *, n_total: int, top: int,
              beside_sweep: bool = False, radix_select: bool = False) -> torch.Tensor:
        """The 12 statistics (engine.STAT_NAMES order) of every grid point: float64 [G,12] on the GPU.
        beside_sweep: the call runs beside another kernel (B200_LEV_FLAG_BESIDE_SWEEP: a smaller footprint).
        radix_select: every grid point takes the radix route (B200_LEV_FLAG_RADIX_SELECT), for comparisons."""
        f = np.ascontiguousarray(factors, dtype=np.float32)
        if f.ndim != 2:
            raise ValueError("factors must be [G,K]")
        g, k = f.shape
        out = torch.empty((g, 12), dtype=torch.float64, device=self.dev)
        d = LevDesc()
        d.kind, d.mode, d.source = _lib.LEV_DISCRETE, _lib.MODE_LOG, _lib.SRC_STREAM
        d.horizon, d.n_outcomes, d.value_0 = int(horizon), k, float(value_0)
        d.flags = (_lib.LEV_FLAG_BESIDE_SWEEP if beside_sweep else 0) | (_lib.LEV_FLAG_RADIX_SELECT if radix_select else 0)
        with torch.cuda.device(self.dev):
            for g0 in range(0, g, self.plan.grid_cap):
                tile = np.ascontiguousarray(f[g0:g0 + self.plan.grid_cap])
                d.n_grid = tile.shape[0]
                check(lib.b200_tally_stats(C.byref(self.plan), ptr(self.ws), C.byref(d),
                                           tile.ctypes.data_as(C.POINTER(C.c_float)), int(n_total), int(top),
                                           ptr(out[g0:]), stream_ptr()))
        return out

    def info(self) -> dict:
        """The info words (one small device-to-host read; synchronises the current stream).  With a group
        this is COLLECTIVE: the words are the maximum over the ranks."""
        w = self.ws[:_lib.TALLY_INFO_WORDS]
        if self.group is not None:     # every rank must see (and act on) the same verdict
            import torch.distributed as dist

            w = w.clone()
            dist.all_reduce(w, op=dist.ReduceOp.MAX, group=self.group)
        w = w.cpu().tolist()
        return {"bins": w[0], "overflow": bool(w[1]), "bad_outcomes": w[2], "timed_out": bool(w[3]),
                "count_mismatch": bool(w[4]), "radix_route": w[5]}

    def check(self) -> dict:
        """info() + raise on anything that invalidates the statistics (and reset the tally)."""
        i = self.info()
        if i["overflow"] or i["bad_outcomes"] or i["timed_out"] or i["count_mismatch"]:
            self.reset()
        if i["timed_out"]:
            raise RuntimeError("rlmd_b200: a rank's bins did not arrive within 30 s (peer-memory exchange)")
        if i["bad_outcomes"]:
            raise ValueError(f"{i['bad_outcomes']} outcomes outside 0..K-1: the reference would use such a value as "
                             "the factor itself (lev/lev_exp.py:541); not supported")
        if i["overflow"]:
            raise TallyOverflow(f"more than {self.plan.bins_cap} distinct outcome-count tuples")
        if i["count_mismatch"]:
            raise RuntimeError("rlmd_b200: the tallied rows do not add up to n_total")
        return i

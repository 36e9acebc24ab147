"""
Engine-level calls (thin ctypes wrappers; torch tensors are only buffers).

Every function here launches CUDA kernels through the C ABI on the current
torch stream and fails loudly without a GPU - there is no CPU path.
"""
from __future__ import annotations

import ctypes as C
import math
import os
from typing import Optional, Sequence

import numpy as np
import torch

from . import _lib
from ._lib import BigBrainDesc, LevDesc, check, lib, ptr, require_cuda, stream_ptr

STAT_NAMES = (
    "mean", "mean_top", "mean_adj", "mad", "mad_top", "mad_adj",
    "std", "std_top", "std_adj", "med", "med_top", "med_adj",
)


def _round_up(x: int, m: int) -> int:
    return (x + m - 1) // m * m


def device_info() -> dict:
    require_cuda()
    a, b, c = C.c_int32(), C.c_int32(), C.c_int32()
    check(lib.b200_device_info(C.byref(a), C.byref(b), C.byref(c)))
    return {"sm_count": a.value, "cc": (b.value, c.value)}


# ----------------------------------------------------------------- outcomes
def _cuda_device(device=None) -> torch.device:
    """The CUDA device a call runs on: `device` when it names one, else the current one
    (the reference scripts pass T.device("cpu") with VRAM = False, lev/coin_flip.py:67,137)."""
    if device is not None:
        d = torch.device(device)
        if d.type == "cuda":
            return d if d.index is not None else torch.device("cuda", torch.cuda.current_device())
    return torch.device("cuda", torch.cuda.current_device())


def encode_codes(outcomes, device=None, n_outcomes: int = 4, chunk_bytes: int = 256 << 20) -> torch.Tensor:
    """
    Reference-format outcomes ([N,H] fp32 {0,1} for the coin, int64 {0,1,2} for
    the dice; lev/coin_flip.py:160-161, lev/dice_roll.py:147-148; host or device,
    also int32 / fp64 / uint8 / bool / NumPy) -> the engine format: uint8 codes
    [N, ld] on the GPU with ld = H rounded up to 16 so that the TMA path applies.
    Returns a view [N,H] of the padded buffer.  The conversion is b200_lev_ingest;
    a host array is walked in row chunks through two staging buffers (the device
    never holds more than two chunks of the wide source format).
    n_outcomes = 2: code = (x == 1), the coin's rule (lev/lev_exp.py:85).
    """
    require_cuda()
    from . import tally as _tally

    t = torch.as_tensor(outcomes)
    if t.dtype == torch.bool:
        t = t.view(torch.uint8)
    if t.dtype not in _tally._SRC_TYPES:
        raise TypeError(f"outcomes of dtype {t.dtype} are not an accepted format")
    n, h = t.shape
    dev = t.device if t.is_cuda else _cuda_device(device)
    ld = _round_up(h, 16)
    if t.stride(1) != 1:
        t = t.contiguous()
    with torch.cuda.device(dev):
        buf = torch.zeros((n, ld), dtype=torch.uint8, device=dev)
        if n == 0:
            return buf[:, :h]

        def ingest(src, dst):
            m = src.shape[0]
            lds = src.stride(0) if m > 1 else max(src.stride(0), h)
            check(lib.b200_lev_ingest(ptr(src), _tally._SRC_TYPES[src.dtype], m, h, lds, int(n_outcomes), ptr(dst), ld,
                                      None, None, None, stream_ptr()))

        if t.is_cuda:
            ingest(t, buf)
            return buf[:, :h]
        rows = int(max(1, min(n, chunk_bytes // max(h * t.element_size(), 1))))
        stage = [torch.empty((rows, h), dtype=t.dtype, device=dev) for _ in range(2)]
        comp, copy = torch.cuda.current_stream(), _copy_stream(dev)
        ready = [torch.cuda.Event() for _ in range(2)]
        done = [torch.cuda.Event() for _ in range(2)]
        copy.wait_stream(comp)
        for i, r0 in enumerate(range(0, n, rows)):
            m = min(rows, n - r0)
            if i >= 2:
                copy.wait_event(done[i & 1])
            with torch.cuda.stream(copy):
                stage[i & 1][:m].copy_(t[r0:r0 + m], non_blocking=True)
                ready[i & 1].record(copy)
            comp.wait_event(ready[i & 1])
            ingest(stage[i & 1][:m], buf[r0:r0 + m])
            done[i & 1].record(comp)
        for b in stage:
            b.record_stream(copy)
    return buf[:, :h]


class PackedCodes:
    """
    Discrete outcomes at two bits each (`bits` = 2): `data` is uint8 [N, ld] (CUDA, or
    pinned host memory for the host paths), four codes per byte - step t of a row in byte
    t >> 2, bits 2*(t&3)..+1 - with ld = ceil(H/4) rounded up to 16 bytes and zero
    pad bits.  A die roll carries 1.25 bits: the LOG sweep, which is bound by the
    read of the outcome array, moves a quarter of the bytes (the CHAIN kernels,
    bound by instruction issue, take uint8 codes).
    `bits` = 1: the coin's format, ONE bit per flip (K = 2; step t in byte t >> 3, bit t & 7,
    ld = ceil(H/8) rounded up to 16): half the bytes again.
    """

    def __init__(self, data: torch.Tensor, horizon: int, bits: int = 2):
        if bits not in (1, 2):
            raise ValueError("bits must be 1 or 2")
        if data.dtype != torch.uint8 or data.dim() != 2 or (data.shape[0] > 1 and data.stride(1) != 1):
            raise ValueError("packed outcomes are a uint8 [N, ld] tensor with unit inner stride")
        if data.shape[1] * (8 // bits) < horizon:
            raise ValueError("packed outcomes: fewer than ceil(horizon * bits / 8) bytes per row")
        self.data, self.horizon, self.bits = data, int(horizon), int(bits)

    @property
    def shape(self):
        return (self.data.shape[0], self.horizon)

    def unpack(self) -> torch.Tensor:
        """uint8 codes [N,H] (torch ops; for tests and one-off conversions)."""
        d = self.data
        sh = torch.arange(0, 8, self.bits, device=d.device, dtype=torch.uint8)
        codes = (d.unsqueeze(-1) >> sh) & ((1 << self.bits) - 1)
        return codes.reshape(d.shape[0], -1)[:, : self.horizon].contiguous()


def pack_codes(codes: torch.Tensor, bits: int = 2) -> PackedCodes:
    """uint8 codes [N,H] on the GPU (encode_codes / lev_draw) -> PackedCodes (b200_lev_pack_bits)."""
    require_cuda()
    if not codes.is_cuda or codes.dtype != torch.uint8 or codes.dim() != 2 or codes.stride(1) != 1:
        raise ValueError("codes must be a [N,H] uint8 CUDA tensor with unit inner stride")
    n, h = codes.shape
    per = 8 // int(bits)
    ldb = _round_up((h + per - 1) // per, 16)
    out = torch.empty((n, ldb), dtype=torch.uint8, device=codes.device)
    ld = codes.stride(0) if n > 1 else max(codes.stride(0), h)
    with torch.cuda.device(codes.device):
        check(lib.b200_lev_pack_bits(ptr(codes), n, h, ld, ptr(out), ldb, int(bits), stream_ptr()))
    return PackedCodes(out, h, int(bits))


def encode_returns(x, device=None, chunk_bytes: int = 256 << 20) -> torch.Tensor:
    """GBM log-returns (host or device, fp32 or fp64) -> fp32 [N, ld] on the GPU, ld a multiple of 4 (16 bytes).
    A host array travels in row chunks (never a second whole copy of it on the device)."""
    require_cuda()
    t = torch.as_tensor(x)
    n, h = t.shape
    dev = t.device if t.is_cuda else _cuda_device(device)
    ld = _round_up(h, 4)
    with torch.cuda.device(dev):
        buf = torch.zeros((n, ld), dtype=torch.float32, device=dev)
        if t.is_cuda:
            buf[:, :h].copy_(t)
        else:
            rows = int(max(1, min(max(n, 1), chunk_bytes // max(h * t.element_size(), 1))))
            for r0 in range(0, n, rows):
                buf[r0:r0 + rows, :h].copy_(t[r0:r0 + rows], non_blocking=True)
    return buf[:, :h]


def philox_thresholds(probs: Sequence[float]) -> list:
    """Cumulative probabilities -> uint32 thresholds: code = #{k: u >= thr[k]}."""
    thr, acc = [], 0.0
    for p in probs[:-1]:
        acc += float(p)
        thr.append(min(int(math.floor(acc * 4294967296.0)), 0xFFFFFFFF))
    return thr


# -------------------------------------------------------------------- sweep
def lev_sweep(
    kind: str,
    factors: np.ndarray,
    value_0: float,
    *,
    outcomes: Optional[torch.Tensor] = None,
    n_investors: Optional[int] = None,
    horizon: Optional[int] = None,
    mode: str = "chain",
    want_data_T: bool = True,
    want_log_w: bool = False,
    want_counts: bool = False,
    seed: int = 0,
    investor_offset: int = 0,
    probs: Optional[Sequence[float]] = None,
    log_mean: float = 0.0,
    sigma: float = 0.0,
    variant: int = 0,
    out_data_T: Optional[torch.Tensor] = None,
    device=None,
    final_only: bool = False,
    want_state: bool = False,
) -> dict:
    """
    One launch over the whole leverage grid (b200_lev_sweep).

    kind      "discrete" (factors [G,K] fp32) or "gbm" (factors = lev[G] fp32)
    outcomes  CUDA tensor [N,H] uint8 (discrete) / float32 (gbm), row stride
              arbitrary (unit inner stride), or PackedCodes (discrete, LOG mode);
              None -> Philox draws on device
    mode      "chain" (exact fp32 product; discrete only) or "log"
    final_only  GBM: data_T without the running-extremes saturation, i.e. what gbm_fixed_final_lev's
              torch.prod holds (B200_LEV_FLAG_FINAL_ONLY); the default is gbm_smart_lev's chain, saturated
              from the running extremes of S: inf if log wealth ever passed ln FLT_MAX, else 0 if it ever
              fell below ln 2^-150 (the reference's chain keeps whichever came first; the two differ only
              on a path that did both - lev_series follows the reference; DESIGN.md section 4)
    want_state  GBM: also return "state" = float64 [3,N] (S, running max, running min of the summed
              log-returns): the leverage-independent state every row's log wealth log V0 + l S follows
              from (B200_LEV_FLAG_STATE_OUT; excludes want_log_w) - see gbm_growth_summary
    returns   {"data_T": [G,N] f32, "log_w": [G,N] f64, "counts": [N,K] i32}
    """
    require_cuda()
    f = np.ascontiguousarray(factors, dtype=np.float32)
    d, g, k, n, h, dev = _fill_desc(kind, f, value_0, outcomes, n_investors, horizon, mode, seed, investor_offset,
                                    probs, log_mean, sigma, variant, device)
    if final_only:
        d.flags |= _lib.LEV_FLAG_FINAL_ONLY
    if want_state:
        if kind != "gbm" or want_log_w:
            raise ValueError("want_state is a GBM output and replaces log_w")
        d.flags |= _lib.LEV_FLAG_STATE_OUT

    res = {}
    with torch.cuda.device(dev):
        data_T = log_w = counts = None
        if want_data_T:
            data_T = out_data_T if out_data_T is not None else torch.empty((g, n), dtype=torch.float32, device=dev)
            if tuple(data_T.shape) != (g, n) or data_T.dtype != torch.float32 or (n > 1 and data_T.stride(1) != 1):
                raise ValueError("out_data_T must be a float32 [G,N] tensor with unit inner stride")
            if g > 1 and n > 0:
                d.ld_out = data_T.stride(0)
            if want_log_w and d.ld_out not in (0, n):
                raise ValueError("log_w and a strided out_data_T cannot be combined")
        if want_log_w:
            log_w = torch.empty((g, n), dtype=torch.float64, device=dev)
        state = None
        if want_state:
            state = log_w = torch.empty((3, n), dtype=torch.float64, device=dev)
        if want_counts:
            counts = torch.empty((n, k), dtype=torch.int32, device=dev)
        oc = outcomes.data if isinstance(outcomes, PackedCodes) else outcomes
        check(lib.b200_lev_sweep(C.byref(d), ptr(oc), f.ctypes.data_as(C.POINTER(C.c_float)),
                                 ptr(data_T), ptr(log_w), ptr(counts), stream_ptr()))
    res["data_T"], res["log_w"], res["counts"] = data_T, None if want_state else log_w, counts
    if want_state:
        res["state"] = state
    return res


def lev_grid_sweep(factors: np.ndarray, value_0: float, outcomes, *, want_log_w: bool = False,
                   counts: Optional[torch.Tensor] = None) -> dict:
    """
    Final-time LOG sweep of a discrete gamble over a grid of ANY size (factors
    [G,K] fp32, G unbounded): the wealth depends on the outcomes only through
    their counts, so the outcome array (uint8 codes or PackedCodes) is read ONCE
    (b200_lev_sweep -> counts [N,K]) and every tile of 64 grid points is then one
    b200_lev_from_counts launch over the counts.  This is the engine's route to
    BASELINE's 2-D grid of lev/dice_roll_sh.py (leverage x insurance fraction,
    lev_exp.grid2d_factor_table: G = La * Lb).  Pass `counts` to reuse a previous
    call's counts (another grid over the same outcomes: no pass over the outcomes).
    Returns {"data_T": [G,N] f32, "log_w": [G,N] f64 or None, "counts": [N,K] i32};
    bit-identical to lev_sweep(mode="log") tile by tile.
    """
    require_cuda()
    f = np.ascontiguousarray(factors, dtype=np.float32)
    if f.ndim != 2:
        raise ValueError("factors must be [G,K]")
    g, k = f.shape
    n, h = outcomes.shape
    dev = outcomes.data.device if isinstance(outcomes, PackedCodes) else outcomes.device
    with torch.cuda.device(dev):
        if counts is None:
            counts = lev_sweep("discrete", f[:1], value_0, outcomes=outcomes, mode="log", want_data_T=False,
                               want_counts=True)["counts"]
        elif tuple(counts.shape) != (n, k) or counts.dtype != torch.int32 or not counts.is_contiguous():
            raise ValueError("counts must be a contiguous int32 [N,K] tensor")
        data_T = torch.empty((g, n), dtype=torch.float32, device=dev)
        log_w = torch.empty((g, n), dtype=torch.float64, device=dev) if want_log_w else None
        d = LevDesc()
        d.kind, d.mode, d.source = _lib.LEV_DISCRETE, _lib.MODE_LOG, _lib.SRC_STREAM
        d.n_investors, d.horizon, d.ld_outcomes, d.n_outcomes = n, max(h, 1), max(h, 1), k
        d.value_0 = float(value_0)
        for g0 in range(0, g, _lib.MAX_GRID):
            tile = np.ascontiguousarray(f[g0:g0 + _lib.MAX_GRID])
            d.n_grid = tile.shape[0]
            check(lib.b200_lev_from_counts(C.byref(d), ptr(counts), tile.ctypes.data_as(C.POINTER(C.c_float)),
                                           ptr(data_T[g0:]), ptr(log_w[g0:]) if want_log_w else None, stream_ptr()))
    return {"data_T": data_T, "log_w": log_w, "counts": counts}


def lev_draw(kind: str, n_investors: int, horizon: int, *, seed: int = 0, investor_offset: int = 0,
             probs=None, log_mean: float = 0.0, sigma: float = 0.0, device="cuda", packed: bool = False, bits: int = 2):
    """The outcome array a Philox sweep with the same arguments consumes (packed=True: PackedCodes of `bits`
    bits per outcome - 1 for a two-outcome gamble's one-bit format)."""
    require_cuda()
    d = LevDesc()
    d.n_investors, d.horizon = int(n_investors), int(horizon)
    d.n_grid, d.mode, d.source = 1, _lib.MODE_LOG, _lib.SRC_PHILOX
    d.seed, d.investor_offset = int(seed) & 0xFFFFFFFFFFFFFFFF, int(investor_offset)
    if kind == "discrete":
        d.kind, d.n_outcomes = _lib.LEV_DISCRETE, len(probs)
        for i, v in enumerate(philox_thresholds(probs)):
            d.thresholds[i] = v
        if packed:
            if bits == 1 and len(probs) != 2:
                raise ValueError("one bit per outcome needs a two-outcome gamble")
            per = 8 // int(bits)
            ld = _round_up((horizon + per - 1) // per, 16)
            d.outcome_bits = int(bits)
        else:
            ld = _round_up(horizon, 16)
        out = torch.zeros((n_investors, ld), dtype=torch.uint8, device=device)
    else:
        if packed:
            raise ValueError("packed outcomes are discrete codes")
        d.kind, d.log_mean, d.sigma = _lib.LEV_GBM, float(log_mean), float(sigma)
        ld = _round_up(horizon, 4)
        out = torch.zeros((n_investors, ld), dtype=torch.float32, device=device)
    d.ld_outcomes = ld
    with torch.cuda.device(out.device):
        check(lib.b200_lev_draw(C.byref(d), ptr(out), stream_ptr()))
    if packed:
        return PackedCodes(out, horizon, int(bits))
    return out[:, :horizon]


def _fill_desc(kind, f, value_0, outcomes, n_investors, horizon, mode, seed, investor_offset, probs, log_mean,
               sigma, variant, device):
    d = LevDesc()
    if kind == "discrete":
        d.kind = _lib.LEV_DISCRETE
        g, k = f.shape
        d.n_outcomes = k
    elif kind == "gbm":
        d.kind = _lib.LEV_GBM
        g, k = f.shape[0], 0
    else:
        raise ValueError("kind must be 'discrete' or 'gbm'")
    d.n_grid = g
    d.mode = {"chain": _lib.MODE_CHAIN, "log": _lib.MODE_LOG}[mode]
    d.value_0 = float(value_0)
    d.variant = int(variant)
    d.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    d.investor_offset = int(investor_offset)
    d.log_mean, d.sigma = float(log_mean), float(sigma)
    if isinstance(outcomes, PackedCodes):
        if kind != "discrete" or mode != "log":
            raise ValueError("packed outcomes feed the discrete LOG sweep (the CHAIN kernels take uint8 codes)")
        if not outcomes.data.is_cuda:
            raise ValueError("outcomes must live on the GPU")
        n, h = outcomes.shape
        d.source, d.outcome_bits = _lib.SRC_STREAM, outcomes.bits
        d.ld_outcomes = outcomes.data.stride(0) if n > 1 else outcomes.data.shape[1]
        dev = outcomes.data.device
    elif outcomes is not None:
        if not outcomes.is_cuda:
            raise ValueError("outcomes must live on the GPU (see encode_codes / encode_returns)")
        want = torch.uint8 if kind == "discrete" else torch.float32
        if outcomes.dtype != want or outcomes.dim() != 2 or outcomes.stride(1) != 1:
            raise ValueError(f"outcomes must be a [N,H] {want} tensor with unit inner stride")
        n, h = outcomes.shape
        d.source = _lib.SRC_STREAM
        d.ld_outcomes = outcomes.stride(0) if n > 1 else max(outcomes.stride(0), h)
        dev = outcomes.device
    else:
        if n_investors is None or horizon is None:
            raise ValueError("Philox mode needs n_investors and horizon")
        n, h = int(n_investors), int(horizon)
        d.source = _lib.SRC_PHILOX
        d.ld_outcomes = h
        dev = torch.device(device or "cuda")
        if kind == "discrete":
            for i, v in enumerate(philox_thresholds(probs)):
                d.thresholds[i] = v
    d.n_investors, d.horizon = n, h
    return d, g, k, n, h, dev


def lev_series(
    kind: str,
    factors: np.ndarray,
    lev_row: np.ndarray,
    value_0: float,
    top: int,
    *,
    outcomes: Optional[torch.Tensor] = None,
    n_investors: Optional[int] = None,
    horizon: Optional[int] = None,
    seed: int = 0,
    investor_offset: int = 0,
    probs: Optional[Sequence[float]] = None,
    log_mean: float = 0.0,
    sigma: float = 0.0,
    variant: int = 0,
    chunk_steps: Optional[int] = None,
    chunk_bytes: int = 8 << 30,
    n_total: Optional[int] = None,
    group=None,
    device=None,
    dtype: torch.dtype = torch.float32,
):
    """
    Per-step statistics of the whole grid (the *_smart_lev contract):
    returns data [G,13,H-1] fp32 (rows: the 12 statistics in the reference's
    order, then the leverage) and data_T [G,N] fp32 (wealth after step H-1).
    dtype=torch.float64: the reference run under a float64 default dtype - see
    lev_series_f64 (factors float64, data / data_T float64, one GPU).

    The horizon is walked in chunks: b200_lev_chunk dumps the wealth after every
    step of the chunk to a [G*steps, N] buffer, b200_rowstats reduces every row,
    and the statistics are scattered into `data` (step t -> column t-1).
    With `group`, the rows are investor shards and the statistics are global.
    A chunk is up to `chunk_bytes` (8 GB of the 180) and 2048 rows: the statistics'
    launch and cross-GPU latencies (4 exchange steps per chunk) are paid once per chunk.
    """
    if dtype == torch.float64:
        if group is not None:
            raise ValueError("float64 sweeps are single-GPU")
        if n_total is not None and outcomes is not None and int(n_total) != outcomes.shape[0]:
            raise ValueError("float64 sweeps are single-GPU: n_total must be the number of investors")
        return lev_series_f64(kind, factors, lev_row, value_0, top, outcomes, chunk_steps=chunk_steps,
                              chunk_bytes=chunk_bytes)
    if dtype != torch.float32:
        raise ValueError("dtype must be torch.float32 or torch.float64")
    require_cuda()
    f = np.ascontiguousarray(factors, dtype=np.float32)
    mode = "chain" if kind == "discrete" else "log"
    d, g, k, n, h, dev = _fill_desc(kind, f, value_0, outcomes, n_investors, horizon, mode, seed, investor_offset,
                                    probs, log_mean, sigma, variant, device)
    n_total = n if n_total is None else int(n_total)
    fptr = f.ctypes.data_as(C.POINTER(C.c_float))
    with torch.cuda.device(dev):
        data = torch.zeros((g, 13, max(h - 1, 0)), dtype=torch.float32, device=dev)
        if h > 1:
            data[:, 12, :] = torch.as_tensor(np.asarray(lev_row, dtype=np.float32), device=dev)[:, None]
        if kind == "discrete":
            state = torch.empty((g, n), dtype=torch.float32, device=dev)
        else:
            state = torch.empty((5, n), dtype=torch.float64, device=dev)   # S, max, min, overflow / underflow masks
        if chunk_steps is None:
            n_ref = max(n, 1)
            if group is not None:   # every rank must walk the same chunks (one exchange per chunk)
                import torch.distributed as dist

                t = torch.tensor([n_ref], dtype=torch.int64, device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
                n_ref = int(t.item())
            chunk_steps = max(32, min(h, chunk_bytes // max(4 * g * n_ref, 1), 2048 // g))
        tc_max = max(32, (int(chunk_steps) // 32) * 32)
        tc_max = min(tc_max, (h + 31) // 32 * 32)
        chunk = torch.empty((g * tc_max * max(n, 1),), dtype=torch.float32, device=dev)
        ws = rowstats_workspace(g * tc_max, dev)
        last = None
        for t0 in range(0, h, tc_max):
            t1 = min(h, t0 + tc_max)
            tc = t1 - t0
            dump = chunk[: g * tc * n].view(g * tc, n)
            check(lib.b200_lev_chunk(C.byref(d), ptr(outcomes), fptr, t0, t1, ptr(state), ptr(dump), stream_ptr()))
            if n > 0 or group is not None:      # a rank with an empty shard still takes part in the exchange
                st = rowstats(dump, top, n_total=n_total, group=group, workspace=ws[: g * tc]).view(g, tc, 12)
                lo = max(t0, 1)
                if t1 > lo:
                    data[:, :12, lo - 1:t1 - 1] = stats_to_reference_dtype(st[:, lo - t0:, :], n_total, top).permute(0, 2, 1)
            last = dump.view(g, tc, n)[:, tc - 1, :]
        data_T = state if kind == "discrete" else last.clone()
        if group is not None:
            from . import sharding

            torch.cuda.current_stream().synchronize()
            sharding.raise_if_peers_timed_out(group, dev)
    return data, data_T


def _desc_f64(kind: str, factors, outcomes):
    """The b200_lev_chunk_f64 descriptor and float64 factor table of a streamed sweep."""
    want = {"discrete": torch.uint8, "gbm": torch.float64}.get(kind)
    if want is None:
        raise ValueError("kind must be 'discrete' or 'gbm'")
    if not isinstance(outcomes, torch.Tensor) or not outcomes.is_cuda or outcomes.dtype != want \
            or outcomes.dim() != 2 or outcomes.stride(1) != 1:
        raise ValueError(f"float64 sweeps stream outcomes: a [N,H] {want} CUDA tensor with unit inner stride")
    f = np.ascontiguousarray(factors, dtype=np.float64)
    d = LevDesc()
    if kind == "discrete":
        if f.ndim != 2:
            raise ValueError("factors must be [G,K]")
        d.kind, d.n_outcomes = _lib.LEV_DISCRETE, f.shape[1]
    else:
        f = f.reshape(-1)
        d.kind = _lib.LEV_GBM
    g = f.shape[0]
    if not 1 <= g <= _lib.MAX_GRID:
        raise ValueError(f"float64 sweeps take 1..{_lib.MAX_GRID} grid points (got {g})")
    n, h = outcomes.shape
    d.n_grid, d.n_investors, d.horizon = g, n, h
    d.source, d.mode = _lib.SRC_STREAM, _lib.MODE_CHAIN
    d.ld_outcomes = outcomes.stride(0) if n > 1 else max(outcomes.stride(0), h)
    return d, f, g, n, h


def lev_series_f64(kind: str, factors, lev_row, value_0: float, top: int, outcomes: torch.Tensor, *,
                   chunk_steps: Optional[int] = None, chunk_bytes: int = 8 << 30):
    """
    lev_series for the reference run under torch.set_default_dtype(torch.float64), on one GPU:
    the exact fp64 chain value = value_0 * m_0, value = value * m_t (b200_lev_chunk_f64) and
    the statistics of float64 rows (b200_rowstats_f64).
    kind "discrete": outcomes uint8 codes [N,H], factors float64 [G,K];
    kind "gbm": outcomes float64 x [N,H], factors = float64 lev [G] (m = exp(l x)).
    Returns data [G,13,H-1] and data_T [G,N], float64 on the GPU.  A chunk is up to
    `chunk_bytes` of 8-byte wealth and 2048 rows.
    """
    require_cuda()
    d, f, g, n, h = _desc_f64(kind, factors, outcomes)
    fptr = f.ctypes.data_as(C.POINTER(C.c_double))
    dev = outcomes.device
    with torch.cuda.device(dev):
        data = torch.zeros((g, 13, max(h - 1, 0)), dtype=torch.float64, device=dev)
        if h > 1:
            data[:, 12, :] = torch.as_tensor(np.asarray(lev_row, dtype=np.float64), device=dev)[:, None]
        state = torch.full((g, n), float(value_0), dtype=torch.float64, device=dev)
        if chunk_steps is None:
            chunk_steps = min(h, chunk_bytes // max(8 * g * n, 1), 2048 // g)
        tc_max = max(1, min(int(chunk_steps), h))
        chunk = torch.empty((g * tc_max * max(n, 1),), dtype=torch.float64, device=dev)
        ws = rowstats_f64_workspace(g * tc_max, dev)
        for t0 in range(0, h, tc_max):
            t1 = min(h, t0 + tc_max)
            tc = t1 - t0
            dump = chunk[: g * tc * n].view(g * tc, n)
            check(lib.b200_lev_chunk_f64(C.byref(d), ptr(outcomes), fptr, t0, t1, ptr(state), ptr(dump), stream_ptr()))
            lo = max(t0, 1)
            if n > 0 and t1 > lo:
                st = rowstats(dump, top, workspace=ws[: g * tc]).view(g, tc, 12)
                data[:, :12, lo - 1:t1 - 1] = st[:, lo - t0:, :].permute(0, 2, 1)
    return data, state


def lev_final_f64(kind: str, factors, value_0: float, top: int, outcomes: torch.Tensor):
    """
    The *_fixed_final_lev counterpart of lev_series_f64 (same inputs): the fp64 chain over the whole
    horizon without a dump, then the statistics of the float64 rows.
    Returns (stats [G,12], data_T [G,N]), float64 on the GPU.
    """
    require_cuda()
    d, f, g, n, h = _desc_f64(kind, factors, outcomes)
    dev = outcomes.device
    with torch.cuda.device(dev):
        data_T = torch.full((g, n), float(value_0), dtype=torch.float64, device=dev)
        check(lib.b200_lev_chunk_f64(C.byref(d), ptr(outcomes), f.ctypes.data_as(C.POINTER(C.c_double)), 0, h,
                                     ptr(data_T), None, stream_ptr()))
        stats = rowstats(data_T, top) if n > 0 else torch.full((g, 12), float("nan"), dtype=torch.float64, device=dev)
    return stats, data_T


_copy_streams = {}


def _copy_stream(dev) -> "torch.cuda.Stream":
    """One H2D stream per device, kept: a fresh stream per call also means a fresh allocator pool per call."""
    key = str(dev)
    if key not in _copy_streams:
        with torch.cuda.device(dev):
            _copy_streams[key] = torch.cuda.Stream()
    return _copy_streams[key]


def lev_final_host(kind: str, factors: np.ndarray, value_0: float, top: int, outcomes_host, *,
                   mode: str = "log", chunk_rows: Optional[int] = None, variant: int = 0, device="cuda",
                   return_data_T: bool = False, group=None, n_total: Optional[int] = None, final_only: bool = False):
    """
    The *_fixed_final_lev hot path for outcomes that live in HOST memory
    (pinned for overlap): investor rows are independent, so the array is walked
    in row chunks through two device staging buffers - the H2D copy of chunk i+1
    overlaps the sweep of chunk i - and the statistics come back to the host.
    `outcomes_host`: uint8 codes / fp32 returns [N,H], or PackedCodes over a host
    tensor (a quarter of the bytes over PCIe).  Rows whose byte length is a multiple
    of 16 (every PackedCodes made by pack_codes / lev_draw; H a multiple of 16 / 4
    otherwise) travel as ONE contiguous copy per chunk; other widths make each
    chunk a pitched copy through a device temporary, which is much slower.
    Returns float64 [G,12] numpy (and data_T on the device when asked).
    """
    require_cuda()
    packed = isinstance(outcomes_host, PackedCodes)
    host = outcomes_host.data if packed else outcomes_host
    if host.is_cuda or host.dim() != 2:
        raise ValueError("outcomes_host must be a 2-D host tensor (or PackedCodes over one)")
    want = torch.uint8 if kind == "discrete" else torch.float32
    if host.dtype != want:
        raise ValueError(f"outcomes_host must be {want}")
    if packed and (kind != "discrete" or mode != "log"):
        raise ValueError("packed outcomes feed the discrete LOG sweep")
    f = np.ascontiguousarray(factors, dtype=np.float32)
    g = f.shape[0]
    n, h = outcomes_host.shape
    w = host.shape[1] if packed else h                      # row width in elements of `host`
    dev = torch.device(device)
    ld = _round_up(w, 16 if kind == "discrete" else 4)
    if chunk_rows is None:
        chunk_rows = max(1024, (256 << 20) // (ld * host.element_size()))
    chunk_rows = min(chunk_rows, max(n, 1))
    with torch.cuda.device(dev):
        data_T = torch.empty((g, n), dtype=torch.float32, device=dev)
        bufs = [torch.empty((chunk_rows, ld), dtype=want, device=dev) for _ in range(2)]
        comp = torch.cuda.current_stream()
        copy = _copy_stream(dev)
        ready = [torch.cuda.Event() for _ in range(2)]
        done = [torch.cuda.Event() for _ in range(2)]
        copy.wait_stream(comp)
        for i, r0 in enumerate(range(0, n, chunk_rows)):
            rows = min(chunk_rows, n - r0)
            b = bufs[i & 1]
            if i >= 2:
                copy.wait_event(done[i & 1])
            with torch.cuda.stream(copy):
                b[:rows, :w].copy_(host[r0:r0 + rows], non_blocking=True)
                ready[i & 1].record(copy)
            comp.wait_event(ready[i & 1])
            oc = PackedCodes(b[:rows], h, outcomes_host.bits) if packed else b[:rows, :h]
            lev_sweep(kind, f, value_0, outcomes=oc, mode=mode, variant=variant, out_data_T=data_T[:, r0:r0 + rows],
                      final_only=final_only)
            done[i & 1].record(comp)
        if n > 0 or group is not None:      # a rank with an empty shard still takes part in the exchange
            stats = rowstats(data_T, top, n_total=n_total, group=group).cpu().numpy()
        else:
            stats = np.zeros((g, 12))
        if group is not None:
            from . import sharding

            sharding.raise_if_peers_timed_out(group, dev)
    return (stats, data_T) if return_data_T else stats


_tally_cache = {}


def final_tally(rows: int, device, group=None):
    """
    The cached tally.FinalTally of (device, group) with room for `rows` investor rows
    (grown when a call needs more).  With `group` this is COLLECTIVE the first time
    and whenever it grows: every rank must call it with its own row count in the same
    order (the capacity is the largest row count of the group).
    """
    from . import tally as _tally

    dev = _cuda_device(device)
    key = (dev.index, id(group))
    t = _tally_cache.get(key)
    need = max(int(rows), 1)
    if group is not None:
        import torch.distributed as dist

        grow = torch.tensor([need if (t is None or t.plan.rows_cap < need) else 0], dtype=torch.int64, device=dev)
        dist.all_reduce(grow, op=dist.ReduceOp.MAX, group=group)
        need = int(grow.item())
        if need == 0:
            return t
    elif t is not None and t.plan.rows_cap >= need:
        return t
    if group is not None:
        from . import sharding

        if not sharding.peer_memory_available(group, dev):      # decided by all ranks together
            raise _tally.TallyUnavailable("no peer-mapped memory between the ranks of this group")
    if t is not None:
        torch.cuda.synchronize(dev)          # peers may still read the old exchange buffer
        if group is not None:
            import torch.distributed as dist

            dist.barrier(group=group)
    t = _tally.FinalTally(need, device=dev, group=group)
    _tally_cache[key] = t
    return t


def lev_final_stats(factors: np.ndarray, value_0: float, top: int, outcomes, *, device=None, group=None,
                    n_total: Optional[int] = None, check: bool = True, tally=None, info: Optional[dict] = None):
    """
    The *_fixed_final_lev hot path of the DISCRETE gambles (lev/lev_exp.py:56-125,
    :508-583, :1121-1206) for outcomes in ANY accepted format, on the GPU or in host
    memory: one read of the outcomes by a count / ingest kernel whose sink is the
    tally of count tuples, then the reference's 12 statistics of every leverage from
    the distinct tuples (tally.py; no data_T, no [G,N] pass).  factors [G,K] fp32.

    Returns float64 [G,12] on the GPU (engine.STAT_NAMES order).  With check=True the
    call ends with one small device-to-host read and raises ValueError (outcomes
    outside 0..K-1), tally.TallyOverflow (more distinct tuples than the plan holds:
    use lev_sweep + rowstats), or RuntimeError (a peer timed out).  `info`, when a
    dict, receives {"h2d_bytes": ...} and the tally's info words.
    With `group` the rows are this rank's investor shard; statistics are global.
    """
    require_cuda()
    f = np.ascontiguousarray(factors, dtype=np.float32)
    if f.ndim != 2:
        raise ValueError("factors must be [G,K]")
    k = f.shape[1]
    packed = isinstance(outcomes, PackedCodes)
    if not packed:
        outcomes = torch.as_tensor(outcomes)
    data = outcomes.data if packed else outcomes
    n, h = outcomes.shape
    dev = data.device if data.is_cuda else _cuda_device(device)
    if n_total is None:
        n_total = n
        if group is not None:
            from . import sharding

            n_total = sharding.global_count(n, group, dev)
    with torch.cuda.device(dev):
        t = tally if tally is not None else final_tally(n, dev, group)
        moved = 0
        if data.is_cuda:
            t.add(outcomes, k)
        else:
            moved = t.add_host(outcomes, k)
        t.finalize()
        stats = t.stats(f, float(value_0), h, n_total=int(n_total), top=int(top))
        if info is not None:
            info["h2d_bytes"] = moved
        if check:
            i = t.check()
            if info is not None:
                info.update(i)
    return stats


class FinalSweepPipeline:
    """
    A sequence of final-time sweeps (the *_fixed_final_lev hot path) on one GPU or
    one investor shard: float64 [G,12] statistics per submitted outcome array.

    statistics = "tally" (discrete gambles; the default for them): the count kernel's
    sink is the tally of count tuples and the statistics come from the distinct
    tuples (tally.py) - no data_T; across GPUs one exchange per sweep.
    statistics = "rows": LOG sweep -> data_T [G,N] -> b200_rowstats (GBM, and the
    checker of the tally path).
    depth = 2 runs the statistics of sweep i beside sweep i+1 (two streams, two
    tallies / data_T buffers); depth = 1 strictly one after the other.  Default: 2 with
    a `group` (the cross-GPU exchange's latency is hidden), 1 on a single GPU.

        pipe = FinalSweepPipeline("discrete", table, 100.0, top, device=dev)
        stats = [pipe.submit(oc) for oc in outcome_arrays]   # on the device
        pipe.synchronize()                                   # then read them (raises on overflow / time-out)
    """

    def __init__(self, kind: str, factors: np.ndarray, value_0: float, top: int, *, device="cuda", group=None,
                 n_total: Optional[int] = None, depth: Optional[int] = None, statistics: Optional[str] = None):
        require_cuda()
        self.kind, self.value_0, self.top = kind, float(value_0), int(top)
        self.factors = np.ascontiguousarray(factors, dtype=np.float32)
        self.group, self.n_total = group, n_total
        self.dev = _cuda_device(device)
        # default: across GPUs the statistics chain is mostly exchange latency (flags, peer reads) - it runs beside
        # the next sweep; on one GPU there is nothing to hide and the two kernels only take SMs from each other
        # (measured: 0.474 ms per step at depth 2 against 0.461 at depth 1)
        # (the GBM Philox sweep is bound by instruction issue, its statistics by HBM: they overlap well anywhere)
        self.depth = max(1, int(depth)) if depth is not None else (2 if (group is not None or kind == "gbm") else 1)
        self.statistics = statistics or ("tally" if kind == "discrete" else "rows")
        if self.statistics not in ("tally", "rows") or (self.statistics == "tally" and kind != "discrete"):
            raise ValueError("statistics must be 'tally' (discrete gambles) or 'rows'")
        if self.statistics == "tally" and group is not None:
            from . import sharding

            if not sharding.peer_memory_available(group, self.dev):     # collective; all ranks decide alike
                self.statistics = "rows"       # the general path, whose exchange can run over NCCL
        with torch.cuda.device(self.dev):
            # the statistics' short, dependent kernels go first whenever they are ready
            self.sweep_stream = torch.cuda.Stream()
            # depth 1 is strictly sequential: one stream (a cross-stream event wait per kernel costs microseconds)
            self.stats_stream = torch.cuda.Stream(priority=-1) if self.depth > 1 else self.sweep_stream
        self.data_T = [None] * self.depth
        self.ws = [None] * self.depth
        self.tallies = [None] * self.depth
        self.free = [None] * self.depth       # statistics that last read data_T[b] / tally[b]
        self.count = 0
        self.last_sweep = None                # (start, end) events of the last sweep, when timing is on
        self.timing = False
        self._timing_stream = None
        self._sweep_opens = None              # depth 1, timing on: the next sweep's start event

    def submit(self, outcomes, factors: Optional[np.ndarray] = None) -> torch.Tensor:
        f = self.factors if factors is None else np.ascontiguousarray(factors, dtype=np.float32)
        g = f.shape[0]
        n, h = outcomes.shape
        b = self.count % self.depth
        self.count += 1
        tally = self.statistics == "tally"
        # Depth 1 on the tally path: count kernel, compaction and select follow each other on one stream with
        # nothing between them but event waits and records without timing, so each kernel starts under the one before it
        # (programmatic dependent launch, B200_LEV_FLAG_EARLY_START): the sweep of this step streams its rows on
        # the SMs the previous step's select leaves free.  A record of a timing event would end that overlap,
        # so the sweep's timing events are taken on a stream of their own (_stamp).
        chain = tally and self.depth == 1
        if not (self.timing and chain):
            self._sweep_opens = None
        with torch.cuda.device(self.dev):
            cur = torch.cuda.current_stream()
            self.sweep_stream.wait_stream(cur)        # the caller produced `outcomes` on its stream
            data = outcomes.data if isinstance(outcomes, PackedCodes) else outcomes
            data.record_stream(self.sweep_stream)
            with torch.cuda.stream(self.sweep_stream):
                if self.free[b] is not None:
                    self.sweep_stream.wait_event(self.free[b])
                if tally and (self.tallies[b] is None or self.tallies[b].plan.rows_cap < n):
                    from . import tally as _tally

                    # on the sweep stream: the reset of its table runs before the count kernel fills it
                    self.tallies[b] = _tally.FinalTally(n, device=self.dev, group=self.group)   # collective with a group
                if not tally and (self.data_T[b] is None or tuple(self.data_T[b].shape) != (g, n)):
                    self.data_T[b] = torch.empty((g, n), dtype=torch.float32, device=self.dev)
                    self.ws[b] = rowstats_workspace(g, self.dev)
                if self.timing:
                    t0 = self._sweep_opens if chain and self._sweep_opens is not None else self._stamp()
                if tally:
                    self.tallies[b].add(outcomes, f.shape[1], early_start=chain)
                else:
                    lev_sweep(self.kind, f, self.value_0, outcomes=outcomes, mode="log", out_data_T=self.data_T[b])
                if self.timing:
                    self.last_sweep = (t0, self._stamp())
            n_total = self.n_total if self.n_total is not None else n
            with torch.cuda.stream(self.stats_stream):
                if self.depth > 1:
                    swept = torch.cuda.Event()
                    swept.record(self.sweep_stream)
                    self.stats_stream.wait_event(swept)
                if tally:
                    self.tallies[b].finalize()
                    if self.timing and chain:
                        # the next step's sweep starts under this step's select: its window opens here
                        self._sweep_opens = self._stamp()
                    stats = self.tallies[b].stats(f, self.value_0, h, n_total=n_total, top=self.top,
                                                  beside_sweep=self.depth > 1)
                else:
                    stats = rowstats(self.data_T[b], self.top, n_total=self.n_total, group=self.group,
                                     workspace=self.ws[b])
                if self.depth > 1:
                    done = torch.cuda.Event()
                    done.record(self.stats_stream)
                    self.free[b] = done
                stats.record_stream(cur)
        return stats

    def _stamp(self) -> torch.cuda.Event:
        """A timing event that completes with the work enqueued so far on the sweep stream: recorded on a
        stream of its own behind an event without timing, which leaves the sweep stream's kernels overlapping."""
        if self._timing_stream is None:
            self._timing_stream = torch.cuda.Stream(self.dev)
        mark = torch.cuda.Event()
        mark.record(self.sweep_stream)
        self._timing_stream.wait_event(mark)
        ev = torch.cuda.Event(enable_timing=True)
        ev.record(self._timing_stream)
        return ev

    def submit_philox(self, n_investors: int, horizon: int, *, seed: int, investor_offset: int = 0,
                      log_mean: float, sigma: float, growth_quantiles: Optional[Sequence[float]] = (0.05, 0.5)):
        """
        GBM with outcomes drawn on the device (lev/gbm.py at sizes whose fp32 outcome array cannot exist):
        Philox sweep -> data_T [G,N] + state [3,N] on the sweep stream; the 12 statistics per leverage and (when
        `growth_quantiles` is not None) the growth-rate summaries on the statistics stream, beside the next
        sweep.  Returns (stats [G,12], growth [G, 6 + len(q)] or None), float64 on the device.
        """
        if self.kind != "gbm":
            raise ValueError("submit_philox is the GBM path")
        lev = self.factors.reshape(-1)
        g, n = lev.shape[0], int(n_investors)
        b = self.count % self.depth
        self.count += 1
        with torch.cuda.device(self.dev):
            cur = torch.cuda.current_stream()
            self.sweep_stream.wait_stream(cur)
            with torch.cuda.stream(self.sweep_stream):
                if self.free[b] is not None:
                    self.sweep_stream.wait_event(self.free[b])
                if self.data_T[b] is None or tuple(self.data_T[b].shape) != (g, n):
                    self.data_T[b] = torch.empty((g, n), dtype=torch.float32, device=self.dev)
                    self.ws[b] = rowstats_workspace(g, self.dev)
                if self.timing:
                    t0 = torch.cuda.Event(enable_timing=True)
                    t0.record(self.sweep_stream)
                res = lev_sweep("gbm", lev, self.value_0, n_investors=n, horizon=int(horizon), seed=seed,
                                investor_offset=investor_offset, log_mean=log_mean, sigma=sigma, mode="log",
                                out_data_T=self.data_T[b], want_state=growth_quantiles is not None, device=self.dev)
                swept = torch.cuda.Event(enable_timing=self.timing)
                swept.record(self.sweep_stream)
                if self.timing:
                    self.last_sweep = (t0, swept)
            n_total = self.n_total if self.n_total is not None else n
            with torch.cuda.stream(self.stats_stream):
                self.stats_stream.wait_event(swept)
                stats = rowstats(self.data_T[b], self.top, n_total=n_total, group=self.group, workspace=self.ws[b])
                growth = None
                if growth_quantiles is not None:
                    res["state"].record_stream(self.stats_stream)
                    growth = gbm_growth_summary(res["state"], lev, int(horizon), self.value_0, data_T=self.data_T[b],
                                                quantiles=growth_quantiles, n_total=n_total, group=self.group)
                    growth.record_stream(cur)
                done = torch.cuda.Event()
                done.record(self.stats_stream)
                self.free[b] = done
                stats.record_stream(cur)
        return stats, growth

    def synchronize(self) -> None:
        self.sweep_stream.synchronize()
        self.stats_stream.synchronize()
        if self._timing_stream is not None:
            self._timing_stream.synchronize()
        for t in self.tallies:
            if t is not None:
                t.check()
        if self.group is not None and self.statistics == "rows":
            from . import sharding

            sharding.raise_if_peers_timed_out(self.group, self.dev)


# ----------------------------------------------------------------- rowstats
_FLT_MAX = 3.4028234663852886e38


def stats_to_reference_dtype(stats, n_total: int, top: int):
    """
    float64 [..., 12] statistics (torch tensor or NumPy) -> the reference's dtype, float32, with the one
    place where its fp32 ARITHMETIC shows: `mad = T.mean(T.abs(v - mean))` (lev/lev_exp.py:99, :102, :104)
    sums |v - mean| in fp32, so a group whose absolute deviations add up beyond FLT_MAX reports inf
    (seen in the reference harness's GBM sweep at leverage 4) - while std_mean's Welford update and the
    medians do not overflow.  Everything else is the plain cast.
    """
    sizes = (float(n_total), float(top), float(n_total - top))
    if isinstance(stats, torch.Tensor):
        out = stats.to(torch.float32)
        for j, m in enumerate(sizes):
            col = stats[..., 3 + j]
            out[..., 3 + j] = torch.where(col * m > _FLT_MAX, torch.full_like(out[..., 3 + j], float("inf")),
                                          out[..., 3 + j])
        return out
    st = np.asarray(stats, dtype=np.float64)
    with np.errstate(over="ignore"):
        out = st.astype(np.float32)
    for j, m in enumerate(sizes):
        with np.errstate(invalid="ignore", over="ignore"):
            out[..., 3 + j] = np.where(st[..., 3 + j] * m > _FLT_MAX, np.float32(np.inf), out[..., 3 + j])
    return out


def rowstats_workspace(rows: int, device) -> torch.Tensor:
    nbytes = lib.b200_rowstats_workspace_bytes(rows)
    return torch.empty((rows, nbytes // 8 // max(rows, 1)), dtype=torch.int64, device=device)


def rowstats_f64_workspace(rows: int, device) -> torch.Tensor:
    nbytes = lib.b200_rowstats_f64_workspace_bytes(rows)
    return torch.empty((rows, nbytes // 8 // max(rows, 1)), dtype=torch.int64, device=device)


def _rowstats_f64(values: torch.Tensor, top: int, n_total: Optional[int], workspace: Optional[torch.Tensor]):
    require_cuda()
    if values.dim() != 2 or not values.is_cuda or values.stride(1) != 1:
        raise ValueError("values must be a [rows,n] float64 CUDA tensor with unit inner stride")
    rows, n = values.shape
    if n_total is not None and int(n_total) != n:
        raise ValueError("float64 rows are single-GPU: n_total must equal the row length")
    ld = values.stride(0) if rows > 1 else max(values.stride(0), n)
    dev = values.device
    stats = torch.empty((rows, 12), dtype=torch.float64, device=dev)
    if rows == 0:
        return stats
    with torch.cuda.device(dev):
        ws = workspace if workspace is not None else rowstats_f64_workspace(rows, dev)
        check(lib.b200_rowstats_f64(ptr(values), rows, n, ld, int(top), ptr(ws), ptr(stats), stream_ptr()))
    return stats


def rowstats(values: torch.Tensor, top: int, *, n_total: Optional[int] = None, group=None,
             workspace: Optional[torch.Tensor] = None, exchange: Optional[str] = None) -> torch.Tensor:
    """
    The reference's 12 summary statistics for every row of `values` [rows, n]
    (fp32, CUDA, unit inner stride) -> float64 [rows, 12] (STAT_NAMES order).

    float64 rows (one GPU; `workspace` from rowstats_f64_workspace) take b200_rowstats_f64: the
    same statistics with exact fp64 order statistics, 1 <= top <= n (top == n: the adj group is
    empty and its statistics are NaN, as torch's).

    With `group` (a torch.distributed process group) the rows are investor
    shards of a global vector of n_total entries and every rank returns the global
    statistics.  exchange = "p2p" (default; RLMD_B200_EXCHANGE overrides): the
    resolve kernels sum the peers' partial histograms out of their memory over
    NVLink (b200_rowstats_p2p, GPUs of one node); "nccl": one packed all-reduce per
    pass between the kernels.
    """
    if values.dtype == torch.float64:
        if group is not None:
            raise ValueError("float64 rows are single-GPU")
        return _rowstats_f64(values, top, n_total, workspace)
    require_cuda()
    if values.dim() != 2 or values.dtype != torch.float32 or not values.is_cuda or values.stride(1) != 1:
        raise ValueError("values must be a [rows,n] float32 CUDA tensor with unit inner stride")
    rows, n = values.shape
    ld = values.stride(0) if rows > 1 else max(values.stride(0), n)
    n_total = n if n_total is None else int(n_total)
    dev = values.device
    stats = torch.empty((rows, 12), dtype=torch.float64, device=dev)
    if rows == 0:
        return stats
    with torch.cuda.device(dev):
        if group is None:
            ws = workspace if workspace is not None else rowstats_workspace(rows, dev)
            check(lib.b200_rowstats(ptr(values), rows, n, ld, n_total, int(top), ptr(ws), ptr(stats), -1, stream_ptr()))
            return stats
        from . import sharding

        how = exchange or os.environ.get("RLMD_B200_EXCHANGE", "p2p")
        if how not in ("p2p", "nccl"):
            raise ValueError("exchange must be 'p2p' or 'nccl'")
        if how == "p2p" and not sharding.peer_memory_available(group, dev):
            how = "nccl"     # no peer mapping between these GPUs: the all-reduce path (both run on the GPUs)
        if how == "p2p":
            # ONE workspace / flag block per (group, device): its calls must run one after the other on the GPU
            # (epochs and the alternating workspaces assume it).  Callers on different streams - two pipelines, a
            # pipeline and a direct call - are chained here with an event: call i+1 waits for call i.
            pw = sharding.peer_workspace(rows, group, dev)
            cur = torch.cuda.current_stream()
            if pw.last_call is not None:
                cur.wait_event(pw.last_call)
            ps = pw.peer_set()
            check(lib.b200_rowstats_p2p(ptr(values), rows, n, ld, n_total, int(top), C.byref(ps), ptr(stats),
                                        stream_ptr()))
            pw.last_call = torch.cuda.Event()
            pw.last_call.record(cur)
            return stats
        ws = workspace if workspace is not None else rowstats_workspace(rows, dev)

        def run_phase(phase):
            check(lib.b200_rowstats(ptr(values), rows, n, ld, n_total, int(top), ptr(ws), ptr(stats), phase,
                                    stream_ptr()))

        sharding.exchange_phases(run_phase, ws, group)
    return stats


# ------------------------------------------------------------ growth rates
GROWTH_NAMES = ("valid", "mean", "std", "mean_valid", "min", "max")


def growth_summary(log_w: torch.Tensor, horizon: int, value_0: float, *, data_T: Optional[torch.Tensor] = None,
                   quantiles: Sequence[float] = (0.05, 0.5), n_total: Optional[int] = None, group=None) -> torch.Tensor:
    """
    Time-average growth rates g = (log W_T - log V0) / H of every leverage row of
    `log_w` [G,N] (fp64, CUDA; the LOG sweep's output) reduced to
    float64 [G, 6 + len(quantiles)]: valid-run count (data_T finite and > 0), mean,
    population std, mean over the valid runs, min, max, then the quantiles
    (numpy's method="median_unbiased", the reference's percentile convention,
    tools/eval_episodes.py:276-315).  With `group` the rows are investor shards.
    """
    require_cuda()
    if log_w.dim() != 2 or log_w.dtype != torch.float64 or not log_w.is_cuda or log_w.stride(1) != 1:
        raise ValueError("log_w must be a [G,N] float64 CUDA tensor with unit inner stride")
    rows, n = log_w.shape
    q = [float(x) for x in quantiles]
    if len(q) > 3:
        raise ValueError("at most three quantiles per call")
    ld = log_w.stride(0) if rows > 1 else max(log_w.stride(0), n)
    ld_T = 0
    if data_T is not None:
        if tuple(data_T.shape) != (rows, n) or data_T.dtype != torch.float32 or data_T.stride(1) != 1:
            raise ValueError("data_T must be a float32 [G,N] tensor matching log_w")
        ld_T = data_T.stride(0) if rows > 1 else max(data_T.stride(0), n)
    n_total = n if n_total is None else int(n_total)
    dev = log_w.device
    out = torch.empty((rows, 6 + len(q)), dtype=torch.float64, device=dev)
    if rows == 0:
        return out
    qarr = (C.c_double * max(len(q), 1))(*q)
    with torch.cuda.device(dev):
        words = lib.b200_growth_workspace_bytes(1) // 8
        ws = torch.empty((rows, words), dtype=torch.int64, device=dev)

        def run_phase(phase):
            check(lib.b200_growth_summary(ptr(log_w), ptr(data_T), rows, n, ld, ld_T, n_total, math.log(float(value_0)),
                                          int(horizon), qarr, len(q), ptr(ws), ptr(out), phase, stream_ptr()))

        if group is None:
            run_phase(-1)
        else:
            from . import sharding

            sharding.exchange_phases(run_phase, ws, group, what="growth", n_phases=7)
    return out


def gbm_growth_summary(state: torch.Tensor, lev: np.ndarray, horizon: int, value_0: float, *,
                       data_T: Optional[torch.Tensor] = None, quantiles: Sequence[float] = (0.05, 0.5),
                       n_total: Optional[int] = None, group=None) -> torch.Tensor:
    """
    growth_summary for a GBM sweep from its leverage-independent state [3,N] (lev_sweep(..., want_state=True)):
    log wealth is log V0 + l S, so g = l S / H and every row's mean / std / min / max / quantiles follow from
    ONE set of statistics of S (the q-quantile of a row with l < 0 is l/H times S's (1-q)-quantile: type 8 is
    symmetric) - one selection over N doubles instead of G selections over G x N.  The valid-run counts (finite
    and positive fp32 wealth, per leverage) come from b200_gbm_valid: from the sweep's `data_T` when it is passed
    (one 4-byte read per run and leverage), else re-formed from the state.  Same layout as growth_summary:
    float64 [G, 6 + len(quantiles)].  With `group` the rows are investor shards.
    """
    require_cuda()
    if state.dim() != 2 or state.shape[0] != 3 or state.dtype != torch.float64 or not state.is_cuda \
            or not state.is_contiguous():
        raise ValueError("state must be the contiguous float64 [3,N] CUDA tensor of lev_sweep(want_state=True)")
    levf = np.ascontiguousarray(lev, dtype=np.float32).reshape(-1)
    g = levf.shape[0]
    n = state.shape[1]
    q = [float(x) for x in quantiles]
    need = sorted(set(q) | {1.0 - x for x in q})
    dev = state.device
    n_total = n if n_total is None else int(n_total)
    with torch.cuda.device(dev):
        valid = torch.empty((g, 2), dtype=torch.float64, device=dev)
        ld_T = 0
        if data_T is not None:
            if tuple(data_T.shape) != (g, n) or data_T.dtype != torch.float32 or (n > 1 and data_T.stride(1) != 1):
                raise ValueError("data_T must be the sweep's float32 [G,N] output")
            ld_T = data_T.stride(0) if g > 1 else max(data_T.stride(0), n)
        check(lib.b200_gbm_valid(ptr(state), ptr(data_T), n, ld_T, levf.ctypes.data_as(C.POINTER(C.c_float)), g,
                                 math.log(float(value_0)), ptr(valid), stream_ptr()))
        if group is not None:
            import torch.distributed as dist

            dist.all_reduce(valid, group=group)
        if len(need) > 3:
            raise ValueError("at most three distinct quantile levels of S per call (q and 1-q count)")
        base = growth_summary(state[0:1], 1, 1.0, quantiles=need, n_total=n_total, group=group)   # the row S itself
        key = (dev.index, tuple(q))
        if key not in _gbm_picks:
            _gbm_picks[key] = (torch.tensor([need.index(x) for x in q], dtype=torch.int32, device=dev),
                               torch.tensor([need.index(1.0 - x) for x in q], dtype=torch.int32, device=dev))
        pick_pos, pick_neg = _gbm_picks[key]
        out = torch.empty((g, 6 + len(q)), dtype=torch.float64, device=dev)
        check(lib.b200_gbm_growth_assemble(ptr(base), ptr(valid), levf.ctypes.data_as(C.POINTER(C.c_float)), g,
                                           int(horizon), len(q), ptr(pick_pos), ptr(pick_neg), ptr(out), stream_ptr()))
    return out


_gbm_picks = {}


# ---------------------------------------------------------------- big brain
def bigbrain_series(kind: str, outcomes: torch.Tensor, top: int, value_0: float, returns_by_code: Sequence[float],
                    lev_factor: float, stop_grid, roll_grid, *, chunk_bytes: int = 2 << 30, rows_cap: int = 2048,
                    chunk_steps: Optional[int] = None, n_total: Optional[int] = None, group=None):
    """
    State-dependent leverage over a retention x stop-loss grid (the *_big_brain_lev
    contract): data [R,S,26,H-1] fp32 on the GPU (rows 0..11 wealth statistics after
    each step, 12..23 leverage statistics before it, 24 stop-loss, 25 retention) and
    the final wealth [R,S,N] (fp32 for "coin", fp64 for "dice").

    outcomes: CUDA uint8 codes [N,H] (coin: 1 up / 0 down; dice: 0 up, 1 down, 2 mid);
    returns_by_code: the return of code 0,1,2; lev_factor: the float64 value of the
    scripts' LEV_FACTOR; grids: fp32 values as the reference's tensors hold them.
    The grid is walked in point tiles and the horizon in chunks: b200_bigbrain_chunk
    dumps leverage / wealth per step, b200_rowstats reduces every dumped row.
    """
    require_cuda()
    if not outcomes.is_cuda or outcomes.dtype != torch.uint8 or outcomes.dim() != 2 or outcomes.stride(1) != 1:
        raise ValueError("outcomes must be a [N,H] uint8 CUDA tensor with unit inner stride (engine.encode_codes)")
    n, h = outcomes.shape
    dev = outcomes.device
    stop = np.asarray(stop_grid, dtype=np.float32).reshape(-1)
    roll = np.asarray(roll_grid, dtype=np.float32).reshape(-1)
    R, S = len(roll), len(stop)
    P = R * S
    v0 = np.float32(value_0)
    eta64 = float(lev_factor)
    # point p = j * S + i  (retention j outer, stop-loss i inner; lev/lev_exp.py:314-318)
    vmin = np.tile((stop * v0).astype(np.float32), R)
    rollp = np.repeat(roll, S).astype(np.float32)
    inner = (np.float32(1) - (vmin / v0).astype(np.float32)).astype(np.float32)
    lev0 = eta64 * inner.astype(np.float64)          # 0-dim float64 arithmetic of step 0 (:327)
    d = BigBrainDesc()
    d.n_investors, d.horizon = n, h
    d.ld_outcomes = outcomes.stride(0) if n > 1 else max(outcomes.stride(0), h)
    d.kind = {"coin": _lib.BB_COIN, "dice": _lib.BB_DICE}[kind]
    d.value_0, d.lev_factor32, d.lev_factor64 = float(v0), float(np.float32(eta64)), eta64
    rb = list(returns_by_code) + [0.0] * (3 - len(returns_by_code))
    for k in range(3):
        d.returns[k] = float(rb[k])
    sdt = torch.float32 if kind == "coin" else torch.float64
    n_total = n if n_total is None else int(n_total)

    n_ref = max(n, 1)
    if group is not None:
        import torch.distributed as dist

        t = torch.tensor([n_ref], dtype=torch.int64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
        n_ref = int(t.item())
    ptile = min(P, 32, _lib.BB_MAX_POINTS)
    while True:
        tc = min(max(h - 1, 1), rows_cap // (2 * ptile), chunk_bytes // (8 * n_ref * ptile))
        if tc >= 16 or ptile == 1:
            break
        ptile = max(1, ptile // 2)
    tc = max(1, tc if chunk_steps is None else min(tc, int(chunk_steps)))

    with torch.cuda.device(dev):
        data = torch.zeros((P, 26, max(h - 1, 0)), dtype=torch.float32, device=dev)
        wealth = torch.empty((P, n), dtype=sdt, device=dev)
        if h > 1:
            data[:, 24, :] = torch.as_tensor(np.tile(stop, R), device=dev)[:, None]
            data[:, 25, :] = torch.as_tensor(rollp, device=dev)[:, None]
        dump_buf = torch.empty((ptile * tc * 2 * max(n, 1),), dtype=torch.float32, device=dev)
        ws = rowstats_workspace(ptile * tc * 2, dev)
        fptr = lambda a: a.ctypes.data_as(C.POINTER(C.c_float))
        for p0 in range(0, P, ptile):
            pc = min(ptile, P - p0)
            d.n_points = pc
            vm, rl, l0 = (np.ascontiguousarray(vmin[p0:p0 + pc]), np.ascontiguousarray(rollp[p0:p0 + pc]),
                          np.ascontiguousarray(lev0[p0:p0 + pc]))
            state = torch.empty((2, pc, max(n, 1)), dtype=sdt, device=dev)[:, :, :n].contiguous()
            s = 0
            while s < h:
                s_end = min(h, max(s, 1) + tc)
                s_lo = max(s, 1)
                steps = s_end - s_lo
                dump = dump_buf[: pc * steps * 2 * n].view(pc * steps * 2, n) if steps > 0 else None
                check(lib.b200_bigbrain_chunk(C.byref(d), ptr(outcomes), fptr(vm), fptr(rl),
                                              l0.ctypes.data_as(C.POINTER(C.c_double)), s, s_end, ptr(state),
                                              ptr(dump), stream_ptr()))
                if steps > 0 and (n > 0 or group is not None):
                    st = rowstats(dump, top, n_total=n_total, group=group, workspace=ws[: pc * steps * 2])
                    st = stats_to_reference_dtype(st, n_total, top).view(pc, steps, 2, 12)
                    data[p0:p0 + pc, 12:24, s_lo - 1:s_end - 1] = st[:, :, 0, :].permute(0, 2, 1)
                    data[p0:p0 + pc, 0:12, s_lo - 1:s_end - 1] = st[:, :, 1, :].permute(0, 2, 1)
                s = s_end
            wealth[p0:p0 + pc] = state[0]
        if group is not None:
            from . import sharding

            torch.cuda.current_stream().synchronize()
            sharding.raise_if_peers_timed_out(group, dev)
    return data.view(R, S, 26, max(h - 1, 0)), wealth.view(R, S, n)

"""
Drop-in for the reference's `lev/lev_exp.py`: the same function names,
positional signatures, return types, printed text and output layouts, with the
per-leverage / per-time-step Python loops replaced by CUDA launches
(rlmd_b200.engine -> librlmd_b200.so).

    sys.modules["lev.lev_exp"] = rlmd_b200.lev_exp      # INTEGRATION.md

Reference behaviour kept on the host, verbatim in meaning:
  * `param_range` - the grid with its truncation quirks (lev/lev_exp.py:29-53);
  * the grid becomes an fp32 tensor and is negated iff -down_r > up_r
    (:80-81 and siblings; never for GBM :961,1042);
  * factors are evaluated left to right in fp32 on 0-dim operands
    (`1 + lev * up_r`, `1 + lev * r + (1 - lev) * sh`; :85, :541-543, :1160-1166).
The `*_smart_lev` / `*_big_brain_lev` sweeps run in CHAIN mode (exact fp32
sequential product), so their `data_T` and medians are bit-identical to the
reference's.  The `*_fixed_final_lev` functions reduce with `torch.prod` in the
reference (order unspecified) and only print three significant digits: the
discrete ones run the log-domain count sweep whose sink is the tally of count
tuples (engine.lev_final_stats: one read of the outcomes in whatever format the
caller holds them, then weighted exact statistics of the distinct tuples), the
GBM one the log-domain sum.  `outcomes` may live on the GPU or in host memory,
in the reference's dtypes (fp32 {0,1}, int64 {0,1,2}, fp32 x) or the engine's
(uint8 codes, engine.PackedCodes); host arrays are streamed in row chunks.

Float64 default dtype (`torch.set_default_dtype(torch.float64)` before the reference's
outcomes are drawn and its functions called): the coin functions, and the GBM ones
when `outcomes` is float64 too, follow the reference's all-fp64 run - fp64 grid and
factors, the exact fp64 chain, statistics of the fp64 wealth, float64 tensors back
(engine.lev_series_f64 / lev_final_f64; one GPU).  Every other function and dtype
combination runs as under the float32 default.
"""
from __future__ import annotations

from typing import Tuple  # noqa: F401

import numpy as np
import torch as T

from . import engine

_F32 = np.float32


# ------------------------------------------------------------------- grid
def param_range(low: float, high: float, increment: float) -> list:
    """List of grid values from `low` to `high` in steps of `increment`.

    Python-double arithmetic with the reference's integer truncations
    (lev/lev_exp.py:29-53): int(low/incr) .. int(high/incr + 1), the fractional
    offset of `low` added back, an exact 0 dropped unless it is the only value.
    """
    k_lo = int(low / increment)
    k_hi = int(high / increment + 1)
    offset = low / increment - k_lo
    values = []
    for k in range(k_lo, k_hi):
        values.append((k + offset) * increment)
    if 0 in values and len(values) != 1:
        values.remove(0)
    return values


def _grid(lev_low, lev_high, lev_incr, up_r=None, down_r=None) -> np.ndarray:
    g = np.asarray(param_range(lev_low, lev_high, lev_incr), dtype=_F32)
    if up_r is not None and -down_r > up_r:
        g = -g
    return g


def _grid64(lev_low, lev_high, lev_incr, up_r=None, down_r=None) -> np.ndarray:
    """The grid of the float64 default: T.tensor(param_range(...)) holds the doubles, same negation rule."""
    g = np.asarray(param_range(lev_low, lev_high, lev_incr), dtype=np.float64)
    if up_r is not None and -down_r > up_r:
        g = -g
    return g


def coin_factor_table64(lev: np.ndarray, up_r: float, down_r: float) -> np.ndarray:
    """[G,2] float64: 1 + lev * r in double (lev/lev_exp.py:85 under a float64 default)."""
    lev = np.asarray(lev, dtype=np.float64)
    return np.stack([1.0 + lev * float(down_r), 1.0 + lev * float(up_r)], axis=1)


def _lin(lev: np.ndarray, r: float) -> np.ndarray:
    """fl32(1 + fl32(lev * fl32(r)))"""
    return (_F32(1) + lev * _F32(r)).astype(_F32)


def coin_factor_table(lev: np.ndarray, up_r: float, down_r: float) -> np.ndarray:
    """[G,2]: column = outcome value (0 = down, 1 = up), lev/lev_exp.py:85."""
    return np.stack([_lin(lev, down_r), _lin(lev, up_r)], axis=1)


def dice_factor_table(lev, up_r, down_r, mid_r) -> np.ndarray:
    """[G,3]: code 0 up, 1 down, 2 mid (lev/lev_exp.py:541-543)."""
    return np.stack([_lin(lev, up_r), _lin(lev, down_r), _lin(lev, mid_r)], axis=1)


def dice_sh_factor_table(lev, up_r, down_r, mid_r, sh_up_r, sh_down_r, sh_mid_r) -> np.ndarray:
    """[G,3]: (1 + l r) + (1 - l) sh in fp32 (lev/lev_exp.py:1160-1166)."""
    one_minus = (_F32(1) - lev).astype(_F32)
    cols = []
    for r, sh in ((up_r, sh_up_r), (down_r, sh_down_r), (mid_r, sh_mid_r)):
        cols.append((_lin(lev, r) + (one_minus * _F32(sh)).astype(_F32)).astype(_F32))
    return np.stack(cols, axis=1)


def grid2d_factor_table(a, b, returns, sh_returns) -> np.ndarray:
    """Engine-only 2-D grid (leverage x insurance fraction): m = (1 + a r) + b sh."""
    a = np.asarray(a, dtype=_F32)
    b = np.asarray(b, dtype=_F32)
    cols = [(_lin(a, r) + (b * _F32(s)).astype(_F32)).astype(_F32) for r, s in zip(returns, sh_returns)]
    return np.stack(cols, axis=1)


# -------------------------------------------------------------- plumbing
def dice_sh_grid2d(device, outcomes, top, value_0, up_r, down_r, mid_r, sh_up_r, sh_down_r, sh_mid_r, a_grid, b_grid,
                   want_data_T: bool = True):
    """
    Engine-only (BASELINE's 2-D grid of lev/dice_roll_sh.py): the final-time sweep of
    dice_sh_fixed_final_lev (lev/lev_exp.py:1121-1206) with the two coefficients of its factor
    `1 + l r_k + (1-l) sh_k` (:1160-1166) set free - m = (1 + a r_k) + b sh_k over a_grid x b_grid.
    One pass over the outcomes whatever the grid size (counts), then wealth and the reference's 12
    statistics per grid point.  Returns (stats [La,Lb,12] float64 CUDA, data_T [La,Lb,N] fp32 CUDA);
    the reference's 1-D grid is the line b = 1 - a.  want_data_T=False: the statistics come from the
    tally of count tuples (engine.lev_final_stats: no [G,N] array at all) and data_T is None.
    """
    a = np.asarray(a_grid, dtype=np.float32).reshape(-1)
    b = np.asarray(b_grid, dtype=np.float32).reshape(-1)
    # point (i, j) = (a_i, b_j), row-major
    table = grid2d_factor_table(np.repeat(a, len(b)), np.tile(b, len(a)), (up_r, down_r, mid_r),
                                (sh_up_r, sh_down_r, sh_mid_r))
    if not want_data_T:
        n = outcomes.shape[0]
        data = outcomes.data if isinstance(outcomes, engine.PackedCodes) else outcomes
        dev = data.device if isinstance(data, T.Tensor) and data.is_cuda else engine._cuda_device(device)
        stats = engine.lev_final_stats(table, _as_float(value_0), _as_int(top), outcomes, device=dev, group=_GROUP,
                                       n_total=_n_total(n, dev))
        return stats.view(len(a), len(b), 12), None
    codes = outcomes if isinstance(outcomes, engine.PackedCodes) else _codes(outcomes, 3, device)
    res = engine.lev_grid_sweep(table, _as_float(value_0), codes)
    data_T = res["data_T"]
    n = data_T.shape[1]
    stats = engine.rowstats(data_T, _as_int(top), n_total=_n_total(n, data_T.device), group=_GROUP)
    return stats.view(len(a), len(b), 12), data_T.view(len(a), len(b), n)


def _as_int(x) -> int:
    return int(x.item()) if isinstance(x, T.Tensor) else int(x)


def _as_float(x) -> float:
    return float(x.item()) if isinstance(x, T.Tensor) else float(x)


_codes_cache = {"on": False, "src": None, "version": None, "k": None, "codes": None}


def _codes(outcomes, n_outcomes: int, device=None) -> T.Tensor:
    """uint8 codes [N,H] on the GPU for the CHAIN kernels (engine.encode_codes: the ingest kernel; host
    arrays travel in row chunks)."""
    if isinstance(outcomes, T.Tensor) and outcomes.is_cuda and outcomes.dtype == T.uint8:
        return outcomes  # already in the engine format
    c = _codes_cache
    if c["on"] and isinstance(outcomes, T.Tensor) and c["src"] is outcomes and c["version"] == outcomes._version \
            and c["k"] == int(n_outcomes):
        return c["codes"]
    codes = engine.encode_codes(outcomes, device=device, n_outcomes=n_outcomes)
    if c["on"] and isinstance(outcomes, T.Tensor):
        c["src"], c["version"], c["k"], c["codes"] = outcomes, outcomes._version, int(n_outcomes), codes
    return codes


class reuse_codes:
    """
    `with lev_exp.reuse_codes():` - inside the block the conversion of an outcome tensor to the engine
    format is kept and reused while the SAME tensor object (same in-place version) is handed to the next
    sweep, as the scripts do (lev/coin_flip.py:163-227 passes one `outcomes` to five functions).  Off by
    default: a caller who rewrites the tensor's memory behind torch's back (a NumPy alias) would otherwise
    sweep stale codes.  Leaving the block frees the kept copy (10 GB for 1e6 x 1e4 outcomes).
    """

    def __enter__(self):
        _codes_cache["on"] = True
        return self

    def __exit__(self, *exc):
        _codes_cache.update(on=False, src=None, version=None, k=None, codes=None)
        return False


def _returns(outcomes, device=None) -> T.Tensor:
    if isinstance(outcomes, T.Tensor) and outcomes.is_cuda and outcomes.dtype == T.float32 \
            and outcomes.stride(1) == 1 and outcomes.stride(0) % 4 == 0:
        return outcomes
    return engine.encode_returns(outcomes, device=device)


_FINAL_FMT = """       lev {:1.0f}%:
                 avg mean/med/mad/std:  $ {:1.2e} / {:1.2e} / {:1.1e} / {:1.1e}
                 top mean/med/mad/std:  $ {:1.2e} / {:1.2e} / {:1.1e} / {:1.1e}
                 adj mean/med/mad/std:  $ {:1.2e} / {:1.2e} / {:1.1e} / {:1.1e}"""


def _print_final(lev: np.ndarray, stats: np.ndarray, smart: bool = False) -> None:
    """The reference's per-leverage report (lev/lev_exp.py:106-125).

    coin_smart_lev - and only it - prints med_top in the "adj" line (:227,231; the
    dice / dice_sh / gbm variants print med_adj, :691-695, :1108-1112, :1324-1328); kept (`smart`).
    """
    for l, s in zip(lev, stats):
        mean, mean_top, mean_adj, mad, mad_top, mad_adj, std, std_top, std_adj, med, med_top, med_adj = s
        print(_FINAL_FMT.format(float(l) * 100, mean, med, mad, std, mean_top, med_top, mad_top, std_top,
                                mean_adj, med_top if smart else med_adj, mad_adj, std_adj))


_GROUP = None


def set_process_group(group) -> None:
    """
    Multi-GPU use (one process per GPU, SURVEY.md section 8e): after this call the
    functions below treat `outcomes` as THIS RANK'S investor rows, `top` as the
    global top-K, and return global statistics on every rank (data_T stays the
    local shard).  `None` restores single-GPU behaviour.
    """
    global _GROUP
    _GROUP = group


def _n_total(n_local: int, device) -> int:
    from . import sharding
    return n_local if _GROUP is None else sharding.global_count(n_local, _GROUP, device)


def _fp64_coin() -> bool:
    """The coin follows the all-fp64 run under a float64 default (its values depend on the outcomes only
    through outcomes == 1, so their dtype does not matter)."""
    return T.get_default_dtype() == T.float64


def _fp64_gbm(outcomes) -> bool:
    """GBM follows the all-fp64 run under a float64 default with float64 outcomes."""
    if T.get_default_dtype() != T.float64:
        return False
    dt = getattr(outcomes, "dtype", None)
    if isinstance(dt, T.dtype):
        return dt == T.float64
    return dt is not None and np.dtype(dt) == np.float64


def _single_gpu_f64() -> None:
    if _GROUP is not None:
        raise ValueError("the float64 sweeps (float64 default dtype) run on one GPU: call set_process_group(None) "
                         "or run under the float32 default")


def _returns64(outcomes, device=None) -> T.Tensor:
    t = T.as_tensor(outcomes)
    dev = t.device if t.is_cuda else engine._cuda_device(device)
    return t.to(device=dev, dtype=T.float64).contiguous()


def _final_discrete(device, outcomes, table, top, value_0) -> np.ndarray:
    """Statistics [G,12] (in the reference's dtype) of a discrete final-time sweep: the tally path; inputs
    it cannot hold (more distinct count tuples than its plan, horizon >= 2^21) take the general path (LOG
    sweep -> data_T -> row statistics)."""
    from . import tally as _tally

    k = table.shape[1]
    n, h = outcomes.shape
    data = outcomes.data if isinstance(outcomes, engine.PackedCodes) else outcomes
    dev = data.device if isinstance(data, T.Tensor) and data.is_cuda else engine._cuda_device(device)
    n_total = _n_total(n, dev)
    stats = None
    if h <= _tally._lib.TALLY_MAX_HORIZON:
        try:
            stats = engine.lev_final_stats(table, _as_float(value_0), _as_int(top), outcomes, device=dev,
                                           group=_GROUP, n_total=n_total).cpu().numpy()
        except _tally.TallyOverflow:
            stats = None
    if stats is None:
        codes = outcomes if isinstance(outcomes, engine.PackedCodes) else _codes(outcomes, k, dev)
        res = engine.lev_sweep("discrete", table, _as_float(value_0), outcomes=codes, mode="log")
        stats = engine.rowstats(res["data_T"], _as_int(top), n_total=n_total, group=_GROUP).cpu().numpy()
    return engine.stats_to_reference_dtype(stats, n_total, _as_int(top))


# ----------------------------------------------------- fixed final leverage
def coin_fixed_final_lev(device, outcomes, top, value_0, up_r, down_r, lev_low, lev_high, lev_incr):
    """lev/lev_exp.py:56-125 - prints the final-time statistics per leverage."""
    if _fp64_coin():
        _single_gpu_f64()
        lev = _grid64(lev_low, lev_high, lev_incr, up_r, down_r)
        stats, _ = engine.lev_final_f64("discrete", coin_factor_table64(lev, up_r, down_r), _as_float(value_0),
                                        _as_int(top), _codes(outcomes, 2, device))
        _print_final(lev, stats.cpu().numpy())
        return
    lev = _grid(lev_low, lev_high, lev_incr, up_r, down_r)
    _print_final(lev, _final_discrete(device, outcomes, coin_factor_table(lev, up_r, down_r), top, value_0))


def dice_fixed_final_lev(device, outcomes, top, value_0, up_r, down_r, mid_r, lev_low, lev_high, lev_incr):
    """lev/lev_exp.py:508-583."""
    lev = _grid(lev_low, lev_high, lev_incr, up_r, down_r)
    _print_final(lev, _final_discrete(device, outcomes, dice_factor_table(lev, up_r, down_r, mid_r), top, value_0))


def dice_sh_fixed_final_lev(device, outcomes, top, value_0, up_r, down_r, mid_r, sh_up_r, sh_down_r, sh_mid_r,
                            lev_low, lev_high, lev_incr):
    """lev/lev_exp.py:1121-1206."""
    lev = _grid(lev_low, lev_high, lev_incr, up_r, down_r)
    table = dice_sh_factor_table(lev, up_r, down_r, mid_r, sh_up_r, sh_down_r, sh_mid_r)
    _print_final(lev, _final_discrete(device, outcomes, table, top, value_0))


def gbm_fixed_final_lev(device, outcomes, top, value_0, lev_low, lev_high, lev_incr):
    """lev/lev_exp.py:935-1005 (no sign flip of the grid).  Host outcomes are streamed in row chunks."""
    if _fp64_gbm(outcomes):
        _single_gpu_f64()
        lev = _grid64(lev_low, lev_high, lev_incr)
        stats, _ = engine.lev_final_f64("gbm", lev, _as_float(value_0), _as_int(top), _returns64(outcomes, device))
        _print_final(lev, stats.cpu().numpy())
        return
    lev = _grid(lev_low, lev_high, lev_incr)
    t = T.as_tensor(outcomes)
    dev = t.device if t.is_cuda else engine._cuda_device(device)
    n_total = _n_total(t.shape[0], dev)
    if not t.is_cuda:
        if t.dtype != T.float32:
            t = t.to(T.float32)
        stats = engine.lev_final_host("gbm", lev, _as_float(value_0), _as_int(top), t, mode="log", final_only=True,
                                      device=dev, group=_GROUP, n_total=n_total)
    else:
        x = _returns(t, device)
        res = engine.lev_sweep("gbm", lev, _as_float(value_0), outcomes=x, mode="log", final_only=True)
        stats = engine.rowstats(res["data_T"], _as_int(top), n_total=n_total, group=_GROUP).cpu().numpy()
    _print_final(lev, engine.stats_to_reference_dtype(stats, n_total, _as_int(top)))


# ------------------------------------------------------------ smart leverage
def _series(kind, outcomes, table, lev, investors, horizon, top, value_0, dtype=T.float32) -> Tuple[T.Tensor, T.Tensor]:
    n, h = outcomes.shape
    if (investors is not None and _as_int(investors) != n) or (horizon is not None and _as_int(horizon) != h):
        raise ValueError("investors/horizon do not match the shape of outcomes")
    return engine.lev_series(kind, table, lev, _as_float(value_0), int(top), outcomes=outcomes,
                             n_total=_n_total(n, outcomes.device), group=_GROUP, dtype=dtype)


def coin_smart_lev(device, outcomes, investors, horizon, top, value_0, up_r, down_r, lev_low, lev_high, lev_incr):
    """lev/lev_exp.py:128-237 -> (data [L,13,H-1], data_T [L,N]), fp32 on the GPU (float64 under a float64
    default dtype)."""
    if _fp64_coin():
        _single_gpu_f64()
        lev = _grid64(lev_low, lev_high, lev_incr, up_r, down_r)
        data, data_T = _series("discrete", _codes(outcomes, 2, device), coin_factor_table64(lev, up_r, down_r),
                               lev, investors, horizon, top, value_0, T.float64)
        _print_final(lev, data[:, :12, -1].cpu().numpy(), smart=True)
        return data, data_T
    lev = _grid(lev_low, lev_high, lev_incr, up_r, down_r)
    data, data_T = _series("discrete", _codes(outcomes, 2, device), coin_factor_table(lev, up_r, down_r), lev, investors,
                           horizon, top, value_0)
    _print_final(lev, data[:, :12, -1].double().cpu().numpy(), smart=True)
    return data, data_T


def dice_smart_lev(device, outcomes, investors, horizon, top, value_0, up_r, down_r, mid_r, lev_low, lev_high,
                   lev_incr):
    """lev/lev_exp.py:586-701."""
    lev = _grid(lev_low, lev_high, lev_incr, up_r, down_r)
    data, data_T = _series("discrete", _codes(outcomes, 3, device), dice_factor_table(lev, up_r, down_r, mid_r), lev, investors,
                           horizon, top, value_0)
    _print_final(lev, data[:, :12, -1].double().cpu().numpy())
    return data, data_T


def dice_sh_smart_lev(device, outcomes, investors, horizon, top, value_0, up_r, down_r, mid_r, sh_up_r, sh_down_r,
                      sh_mid_r, lev_low, lev_high, lev_incr):
    """lev/lev_exp.py:1209-1334."""
    lev = _grid(lev_low, lev_high, lev_incr, up_r, down_r)
    table = dice_sh_factor_table(lev, up_r, down_r, mid_r, sh_up_r, sh_down_r, sh_mid_r)
    data, data_T = _series("discrete", _codes(outcomes, 3, device), table, lev, investors, horizon, top, value_0)
    _print_final(lev, data[:, :12, -1].double().cpu().numpy())
    return data, data_T


def gbm_smart_lev(device, outcomes, investors, horizon, top, value_0, lev_low, lev_high, lev_incr):
    """lev/lev_exp.py:1008-1118 (float64 under a float64 default dtype with float64 outcomes)."""
    if _fp64_gbm(outcomes):
        _single_gpu_f64()
        lev = _grid64(lev_low, lev_high, lev_incr)
        data, data_T = _series("gbm", _returns64(outcomes, device), lev, lev, investors, horizon, top, value_0,
                               T.float64)
        _print_final(lev, data[:, :12, -1].cpu().numpy())
        return data, data_T
    lev = _grid(lev_low, lev_high, lev_incr)
    data, data_T = _series("gbm", _returns(outcomes, device), lev, lev, investors, horizon, top, value_0)
    _print_final(lev, data[:, :12, -1].double().cpu().numpy())
    return data, data_T


# ------------------------------------------------- state-dependent leverage
def coin_optimal_lev(value_t, value_0, value_min, lev_factor, roll):
    """lev/lev_exp.py:240-267 - element-wise helper, kept as the same torch expression
    (inside the sweeps the engine evaluates it in the CUDA chain, csrc/bigbrain.cu)."""
    if roll == 0:
        return lev_factor * (1 - T.maximum(value_min, value_min) / value_t)
    rolling_loss = T.where(value_t <= value_0, value_min, value_0 + roll * (value_t - value_0))
    return lev_factor * (1 - rolling_loss / value_t)


def dice_optimal_lev(device, value_t, value_0, value_min, lev_factor, roll):
    """lev/lev_exp.py:704-738 (the retention branch re-casts the wealth to fp32, :731)."""
    if roll == 0:
        return lev_factor * (1 - T.maximum(value_min, value_min) / value_t)
    value_t = T.as_tensor(value_t).to(dtype=T.float, device=device)
    rolling_loss = T.where(value_t <= value_0, value_min, value_0 + roll * (value_t - value_0))
    return lev_factor * (1 - rolling_loss / value_t)


_BB_FMT = """stop/roll {:1.0f}/{:1.0f}%:
                    avg mean/med/mad/std:  $ {:1.2e} / {:1.2e} / {:1.1e} / {:1.1e}  l {:1.2f} / {:1.2f} / {:1.1f} / {:1.1f}
                    top mean/med/mad/std:  $ {:1.2e} / {:1.2e} / {:1.1e} / {:1.1e}  l {:1.2f} / {:1.2f} / {:1.1f} / {:1.1f}
                    adj mean/med/mad/std:  $ {:1.2e} / {:1.2e} / {:1.1e} / {:1.1e}  l {:1.2f} / {:1.2f} / {:1.1f} / {:1.1f}"""


def _print_big_brain(data: T.Tensor) -> None:
    """The per-grid-point report of lev/lev_exp.py:417-449 (statistics of the last step)."""
    if data.shape[-1] == 0:
        return
    last = data[:, :, :, -1].cpu().numpy()
    for j in range(last.shape[0]):
        for i in range(last.shape[1]):
            v, l = last[j, i, 0:12], last[j, i, 12:24]
            args = [last[j, i, 24] * 100, last[j, i, 25] * 100]
            for g in range(3):      # all / top / adj: mean, med, mad, std of wealth then of leverage
                args += [v[0 + g], v[9 + g], v[3 + g], v[6 + g], l[0 + g], l[9 + g], l[3 + g], l[6 + g]]
            print(_BB_FMT.format(*args))


def _lev_factor64(lev_factor) -> float:
    return float(lev_factor.item()) if isinstance(lev_factor, T.Tensor) else float(lev_factor)


def _big_brain(device, kind, outcomes, investors, horizon, top, value_0, returns_by_code, lev_factor, stop, roll):
    codes = _codes(outcomes, len(returns_by_code), device)
    n, h = codes.shape
    if (investors is not None and _as_int(investors) != n) or (horizon is not None and _as_int(horizon) != h):
        raise ValueError("investors/horizon do not match the shape of outcomes")
    stop_grid = np.asarray(param_range(*stop), dtype=_F32)
    roll_grid = np.asarray(param_range(*roll), dtype=_F32)
    data, _ = engine.bigbrain_series(kind, codes, int(top), _as_float(value_0), returns_by_code,
                                     _lev_factor64(lev_factor), stop_grid, roll_grid,
                                     n_total=_n_total(n, codes.device), group=_GROUP)
    _print_big_brain(data)
    return data


def coin_big_brain_lev(device, outcomes, investors, horizon, top, value_0, up_r, down_r, lev_factor, stop_min,
                       stop_max, stop_incr, roll_min, roll_max, roll_incr):
    """lev/lev_exp.py:270-452 -> data [R,S,26,H-1] fp32 on the GPU."""
    return _big_brain(device, "coin", outcomes, investors, horizon, top, value_0, (down_r, up_r), lev_factor,
                      (stop_min, stop_max, stop_incr), (roll_min, roll_max, roll_incr))


def dice_big_brain_lev(device, outcomes, investors, horizon, top, value_0, up_r, down_r, mid_r, lev_factor, stop_min,
                       stop_max, stop_incr, roll_min, roll_max, roll_incr):
    """lev/lev_exp.py:741-932 -> data [R,S,26,H-1] fp32 on the GPU."""
    return _big_brain(device, "dice", outcomes, investors, horizon, top, value_0, (up_r, down_r, mid_r), lev_factor,
                      (stop_min, stop_max, stop_incr), (roll_min, roll_max, roll_incr))


def coin_galaxy_brain_lev(device, ru_min, ru_max, ru_incr, rd_min, rd_max, rd_incr, pu_min, pu_max, pu_incr):
    """
    lev/lev_exp.py:455-505 - Kelly table [len(pu), len(ru), len(ru), 4] fp32 of
    (pu, ru, rd, pu/rd - (1-pu)/ru).  Closed form on the host in Python-double
    arithmetic like the reference's triple loop (no kernel: 1e6 divisions); the
    table is allocated with len(ru) twice, as the reference does (:486).
    """
    ru = np.asarray(param_range(ru_min, ru_max, ru_incr), dtype=np.float64)
    rd = np.asarray(param_range(rd_min, rd_max, rd_incr), dtype=np.float64)
    pu = np.asarray(param_range(pu_min, pu_max, pu_incr), dtype=np.float64)
    if len(rd) > len(ru):
        raise IndexError("the reference's table holds len(ru_range) down-returns (lev/lev_exp.py:486)")
    table = np.zeros((len(pu), len(ru), len(ru), 4), dtype=np.float32)
    k = len(rd)
    table[:, :, :k, 0] = pu[:, None, None]
    table[:, :, :k, 1] = ru[None, :, None]
    table[:, :, :k, 2] = rd[None, None, :]
    table[:, :, :k, 3] = pu[:, None, None] / rd[None, None, :] - (1 - pu[:, None, None]) / ru[None, :, None]
    return T.as_tensor(table, device=device)

"""
The experiment section of the reference's `lev/*.py` scripts as callable
functions: same defaults, same sequence of `lev_exp` calls, and the same
on-disk contract - `<name>_inv1_val.npy`, `<name>_inv1_val_T.npy`,
`<name>_inv{2,3}_val.npy`, `coin_inv4_lev.npy` with identical shapes and the
dtype of the tensors saved (fp32; the inv1 arrays of the float64 paths of
`lev_exp` are float64) - so that the reference's plotting stage (`plotting/plots_multiverse.py`,
`lev/coin_flip.py:244-283`) runs on the engine's output unchanged.

Reference: lev/coin_flip.py:54-241, lev/dice_roll.py:54-218,
lev/dice_roll_sh.py:54-161, lev/gbm.py:54-157.

Outcomes are drawn on the GPU by the engine's Philox4x32-10 stream (seed 420 by
default, the scripts' `T.manual_seed(420)`; the torch CPU generator's stream is
not reproduced - pass `outcomes=` to inject a reference-drawn array).
`inv1_plot_inputs` is the arithmetic `plot_inv1` applies to the two inv1
arrays before drawing (log10 series, mean +/- MAD/std bands, 5th percentile).
"""
from __future__ import annotations

import os
import time
from typing import Dict, Optional

import numpy as np
import torch as T

from . import engine, lev_exp

# ---- defaults of the four scripts (lev/coin_flip.py:54-83 etc.) -------------
COIN = dict(investors=1e6, horizon=3e3, value_0=1e2, up_prob=0.5, up_r=0.5, down_r=-0.4, asym_lim=1e-12,
            l0=(0.05, 1.00, 0.05), l1=(0.10, 1.00, 0.10),
            s2=(0.10, 0.10, 0.10), r2=(0.00, 0.00, 0.10),
            s3=(0.05, 0.95, 0.05), r3=(0.70, 0.95, 0.05),
            ru=(0.20, 0.80, 0.001), rd=(0.20, 0.80, 0.001), pu=(0.25, 0.75, 0.25))
DICE = dict(investors=1e6, horizon=5e3, value_0=1e2, up_prob=1 / 6, down_prob=1 / 6, up_r=0.5, down_r=-0.5,
            mid_r=0.05, asym_lim=1e-12,
            l0=(0.05, 1.00, 0.05), l1=(0.10, 1.00, 0.10),
            s2=(0.10, 0.10, 0.10), r2=(0.00, 0.00, 0.10),
            s3=(0.05, 0.95, 0.05), r3=(0.45, 0.95, 0.05))
DICE_SH = dict(investors=1e6, horizon=2e3, value_0=1e2, up_prob=1 / 6, down_prob=1 / 6, up_r=0.5, down_r=-0.5,
               mid_r=0.05, sh_up_r=-1, sh_down_r=5, sh_mid_r=-1,
               l0=(0.73, 1.00, 0.03), l1=(0.73, 1.00, 0.03))
GBM = dict(investors=1e6, horizon=5e2, value_0=1e2,
           drift=[0.05, 0.0540025395205692], vol=[float(np.sqrt(0.2)), 0.1897916175617430],
           name=["gbm_op", "gbm_snp"],
           l0_l=[-1.0, 0.4], l0_h=[1.0, 4.0], l0_i=[0.2, 0.4],
           l1_l=[-1.0, 0.2], l1_h=[1.0, 2.0], l1_i=[0.2, 0.2])


def _reusing_codes(fn):
    """An injected reference-format `outcomes` tensor is converted to the engine format once per script."""
    import functools

    @functools.wraps(fn)
    def run(*a, **kw):
        with lev_exp.reuse_codes():
            return fn(*a, **kw)
    return run


def _cfg(defaults: dict, overrides: dict) -> dict:
    unknown = set(overrides) - set(defaults)
    if unknown:
        raise TypeError(f"unknown parameters: {sorted(unknown)}")
    c = dict(defaults)
    c.update(overrides)
    c["investors"], c["horizon"] = int(c["investors"]), int(c["horizon"])
    top = c["investors"] * 1e-4                      # TOP = INVESTORS * 1e-4 ...
    c["top"] = int(top) if top > 1 else 1            # ... minimum 1 (lev/coin_flip.py:142)
    return c


def _save(path_results: Optional[str], name: str, t: T.Tensor, out: Dict[str, np.ndarray]) -> None:
    a = t.cpu().numpy()
    out[name] = a
    if path_results is not None:
        os.makedirs(path_results, exist_ok=True)
        np.save(os.path.join(path_results, name + ".npy"), a)


def _lev_factor(up_r: float, down_r: float, asym_lim: float) -> float:
    """LEV_FACTOR of the scripts (lev/coin_flip.py:146-152): fp32 tensor arithmetic, returned as a double."""
    bigger = np.abs(down_r) if np.abs(up_r) >= np.abs(down_r) else -np.abs(up_r)
    f = T.tensor(1 / bigger)
    f = f - T.tensor(asym_lim) if np.abs(up_r) > np.abs(down_r) else f + T.tensor(asym_lim)
    return f


def _report(t0: float) -> None:
    total = time.perf_counter() - t0
    print("TOTAL TIME: {:1.0f}s = {:1.1f}m = {:1.2f}h".format(total, total / 60, total / 3600))


@_reusing_codes
def coin_flip(path_results: Optional[str] = "./results/multiverse/", *, seed: int = 420, outcomes=None,
              galaxy: bool = True, **overrides) -> Dict[str, np.ndarray]:
    """lev/coin_flip.py:154-241 -> coin_inv1_val[_T], coin_inv2_val, coin_inv3_val, coin_inv4_lev.

    Under a float64 default dtype coin_inv1_val[_T] are float64, as the reference's np.save of its fp64
    tensors (lev_exp's all-fp64 coin path); the big-brain and Kelly arrays stay fp32."""
    c = _cfg(COIN, overrides)
    dev = T.device("cuda")
    t0 = time.perf_counter()
    n, h = c["investors"], c["horizon"]
    if outcomes is None:
        outcomes = engine.lev_draw("discrete", n, h, seed=seed, probs=(1 - c["up_prob"], c["up_prob"]))
    out: Dict[str, np.ndarray] = {}
    lf = _lev_factor(c["up_r"], c["down_r"], c["asym_lim"])
    lev_exp.coin_fixed_final_lev(dev, outcomes, c["top"], c["value_0"], c["up_r"], c["down_r"], *c["l0"])
    d, dT = lev_exp.coin_smart_lev(dev, outcomes, n, h, c["top"], c["value_0"], c["up_r"], c["down_r"], *c["l1"])
    _save(path_results, "coin_inv1_val", d, out)
    _save(path_results, "coin_inv1_val_T", dT, out)
    for tag, s, r in (("coin_inv2_val", c["s2"], c["r2"]), ("coin_inv3_val", c["s3"], c["r3"])):
        bb = lev_exp.coin_big_brain_lev(dev, outcomes, n, h, c["top"], c["value_0"], c["up_r"], c["down_r"], lf,
                                        s[0], s[1], s[2], r[0], r[1], r[2])
        _save(path_results, tag, bb, out)
    if galaxy:
        g = lev_exp.coin_galaxy_brain_lev(dev, *c["ru"], *c["rd"], *c["pu"])
        _save(path_results, "coin_inv4_lev", g, out)
    _report(t0)
    return out


@_reusing_codes
def dice_roll(path_results: Optional[str] = "./results/multiverse/", *, seed: int = 420, outcomes=None,
              **overrides) -> Dict[str, np.ndarray]:
    """lev/dice_roll.py:143-218 -> dice_inv1_val[_T], dice_inv2_val, dice_inv3_val."""
    c = _cfg(DICE, overrides)
    dev = T.device("cuda")
    t0 = time.perf_counter()
    n, h = c["investors"], c["horizon"]
    if outcomes is None:
        probs = (c["up_prob"], c["down_prob"], 1 - c["up_prob"] - c["down_prob"])
        outcomes = engine.lev_draw("discrete", n, h, seed=seed, probs=probs)
    out: Dict[str, np.ndarray] = {}
    lf = _lev_factor(c["up_r"], c["down_r"], c["asym_lim"])
    rets = (c["up_r"], c["down_r"], c["mid_r"])
    lev_exp.dice_fixed_final_lev(dev, outcomes, c["top"], c["value_0"], *rets, *c["l0"])
    d, dT = lev_exp.dice_smart_lev(dev, outcomes, n, h, c["top"], c["value_0"], *rets, *c["l1"])
    _save(path_results, "dice_inv1_val", d, out)
    _save(path_results, "dice_inv1_val_T", dT, out)
    for tag, s, r in (("dice_inv2_val", c["s2"], c["r2"]), ("dice_inv3_val", c["s3"], c["r3"])):
        bb = lev_exp.dice_big_brain_lev(dev, outcomes, n, h, c["top"], c["value_0"], *rets, lf,
                                        s[0], s[1], s[2], r[0], r[1], r[2])
        _save(path_results, tag, bb, out)
    _report(t0)
    return out


@_reusing_codes
def dice_roll_sh(path_results: Optional[str] = "./results/multiverse/", *, seed: int = 420, outcomes=None,
                 **overrides) -> Dict[str, np.ndarray]:
    """lev/dice_roll_sh.py:122-161 -> dice_sh_inv1_val[_T]."""
    c = _cfg(DICE_SH, overrides)
    dev = T.device("cuda")
    t0 = time.perf_counter()
    n, h = c["investors"], c["horizon"]
    if outcomes is None:
        probs = (c["up_prob"], c["down_prob"], 1 - c["up_prob"] - c["down_prob"])
        outcomes = engine.lev_draw("discrete", n, h, seed=seed, probs=probs)
    out: Dict[str, np.ndarray] = {}
    rets = (c["up_r"], c["down_r"], c["mid_r"], c["sh_up_r"], c["sh_down_r"], c["sh_mid_r"])
    lev_exp.dice_sh_fixed_final_lev(dev, outcomes, c["top"], c["value_0"], *rets, *c["l0"])
    d, dT = lev_exp.dice_sh_smart_lev(dev, outcomes, n, h, c["top"], c["value_0"], *rets, *c["l1"])
    _save(path_results, "dice_sh_inv1_val", d, out)
    _save(path_results, "dice_sh_inv1_val_T", dT, out)
    _report(t0)
    return out


def gbm(path_results: Optional[str] = "./results/multiverse/", *, seed: int = 420, outcomes=None,
        **overrides) -> Dict[str, np.ndarray]:
    """lev/gbm.py:112-157 -> {gbm_op,gbm_snp}_inv1_val[_T]; `outcomes` = one array per environment.

    The engine's own draws (engine.lev_draw) are float32, so without `outcomes` the sweeps run the float32
    path whatever the default dtype; float64 arrays injected under a float64 default take lev_exp's all-fp64
    GBM path and the inv1 files are float64."""
    c = _cfg(GBM, overrides)
    dev = T.device("cuda")
    n, h = c["investors"], c["horizon"]
    out: Dict[str, np.ndarray] = {}
    for x in range(len(c["drift"])):
        t0 = time.perf_counter()
        log_mean = float(T.tensor(c["drift"][x] - c["vol"][x] ** 2 / 2))     # fp32, like LOG_MEAN
        vol = float(T.tensor(c["vol"][x]))
        oc = outcomes[x] if outcomes is not None else engine.lev_draw("gbm", n, h, seed=seed, log_mean=log_mean,
                                                                      sigma=vol)
        lev_exp.gbm_fixed_final_lev(dev, oc, c["top"], c["value_0"], c["l0_l"][x], c["l0_h"][x], c["l0_i"][x])
        d, dT = lev_exp.gbm_smart_lev(dev, oc, n, h, c["top"], c["value_0"], c["l1_l"][x], c["l1_h"][x],
                                      c["l1_i"][x])
        _save(path_results, c["name"][x] + "_inv1_val", d, out)
        _save(path_results, c["name"][x] + "_inv1_val_T", dT, out)
        del oc
        _report(t0)
    return out


def inv1_plot_inputs(inv1_data: np.ndarray, inv1_data_T: np.ndarray, p4_max: float) -> Dict[str, np.ndarray]:
    """
    Every array `plot_inv1` derives from the two saved files before it draws
    (plotting/plots_multiverse.py:44-169), under the names used there.
    """
    with np.errstate(divide="ignore", invalid="ignore"):
        d = {}
        d["levs_num"] = inv1_data[:, -1, 0] * 100
        d["x_steps"] = np.arange(0, inv1_data.shape[2])
        d["mean_adj_v"] = np.log10(inv1_data[:, 2])                    # panel (a), y of panel (c)
        d["top_adj_v"] = np.log10(inv1_data[:, 1])                     # x of panel (c)
        d["vals"] = np.log10(inv1_data_T.T)                            # panel (b): [N, L] box-plot input
        lo_lim = 1e-39
        for j, grp in enumerate(("nor", "top", "adj")):
            mean, mad, std = inv1_data[:, j, -1], inv1_data[:, 3 + j, -1], inv1_data[:, 6 + j, -1]
            d[grp + "_mean"] = np.log10(mean)
            d[grp + "_mad_up"] = np.log10(np.minimum(p4_max, mean + mad))
            d[grp + "_mad_lo"] = np.log10(np.maximum(lo_lim, mean - mad))
            d[grp + "_std_up"] = np.log10(np.minimum(p4_max, mean + std))
            d[grp + "_med"] = np.log10(inv1_data[:, -4 + j, -1])
        vals_95 = np.percentile(inv1_data_T.T, 5, method="median_unbiased", axis=0)
        d["vals_95"] = vals_95
        d["log_vals_95"] = np.log10(vals_95)
    return d

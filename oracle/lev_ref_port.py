"""
TEST / BASELINE INFRASTRUCTURE ONLY - torch-CPU port of the reference's
`*_fixed_final_lev` loop, op for op, used as the CPU arm of bench.py
(`cpu_baseline`, `--impl reference`) on the GPU box, where /root/reference does
not exist.  The product (rlmd_b200/) never imports it.

It follows lev/lev_exp.py:56-104 (coin), :508-562 (dice), :935-984 (gbm),
:1121-1185 (dice_sh): for each leverage of the fp32 grid, materialise the
[N,H] factor matrix with torch.where / torch.exp, reduce it with
prod(dim=1), sort descending, split top / rest, and take std_mean, median and
the mean absolute deviation of the three groups - all torch CPU ops on all host
threads, as the reference runs with VRAM=False (lev/dice_roll.py:63,137).

Pinned against the unmodified reference in tests/test_oracle_ref_port.py
(identical printed statistics on the same outcomes as the reference's text in
tests/golden/final_text.json).
"""
import torch as T

from oracle.lev_oracle import param_range


def _grid(low, high, incr, up_r=None, down_r=None):
    g = T.tensor(param_range(low, high, incr))
    if up_r is not None and -down_r > up_r:
        g = -g
    return g


def _three_group_stats(value_T: T.Tensor, top: int):
    ordered = value_T.sort(descending=True)[0]
    out = []
    for grp in (value_T, ordered[0:top], ordered[top:]):
        std, mean = T.std_mean(grp, unbiased=False)
        med = T.median(grp)
        mad = T.mean(T.abs(grp - mean))
        out.append((mean, med, mad, std))
    return out


def fixed_final(kind, outcomes, top, value_0, returns, grid, sh=None):
    """
    kind: "coin" (outcomes fp32 {0,1}), "dice"/"dice_sh" (int64 {0,1,2}), "gbm" (fp32 x).
    returns: (up, down[, mid]); grid: (low, high, incr).  -> list over leverages of
    [(mean, med, mad, std) for all / top / adj] as 0-dim fp32 tensors, and the grid.
    """
    value_0 = T.as_tensor(value_0, dtype=T.float32)
    if kind == "gbm":
        levs = _grid(*grid)
    else:
        levs = _grid(*grid, returns[0], returns[1])
    if kind in ("dice", "dice_sh"):
        outcomes = outcomes.to(T.float32)
    rows = []
    for lev in levs:
        if kind == "coin":
            up_r, down_r = returns
            gambles = T.where(outcomes == 1, 1 + lev * up_r, 1 + lev * down_r)
        elif kind == "dice":
            up_r, down_r, mid_r = returns
            gambles = T.where(outcomes == 0, 1 + lev * up_r, outcomes)
            gambles = T.where(outcomes == 1, 1 + lev * down_r, gambles)
            gambles = T.where(outcomes == 2, 1 + lev * mid_r, gambles)
        elif kind == "dice_sh":
            up_r, down_r, mid_r = returns
            s_up, s_down, s_mid = sh
            gambles = T.where(outcomes == 0, 1 + lev * up_r + (1 - lev) * s_up, outcomes)
            gambles = T.where(outcomes == 1, 1 + lev * down_r + (1 - lev) * s_down, gambles)
            gambles = T.where(outcomes == 2, 1 + lev * mid_r + (1 - lev) * s_mid, gambles)
        else:
            gambles = T.exp(lev * outcomes)
        value_T = value_0 * gambles.prod(dim=1)
        rows.append(_three_group_stats(value_T, top))
    return rows, levs


def format_rows(rows, levs) -> str:
    fmt = """       lev {:1.0f}%:
                 avg mean/med/mad/std:  $ {:1.2e} / {:1.2e} / {:1.1e} / {:1.1e}
                 top mean/med/mad/std:  $ {:1.2e} / {:1.2e} / {:1.1e} / {:1.1e}
                 adj mean/med/mad/std:  $ {:1.2e} / {:1.2e} / {:1.1e} / {:1.1e}"""
    return "\n".join(fmt.format(float(l) * 100, *[float(x) for grp in r for x in grp]) for r, l in zip(rows, levs))

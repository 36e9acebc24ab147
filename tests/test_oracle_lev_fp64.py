"""
CPU checks of the float64 leverage path: the fp64 restatements of oracle/lev_oracle_f64.py
against the closed forms (SURVEY.md App. C, "all-fp64 run"), the fp32 overflow that
makes the fp64 run worth having, and the C ABI of the float64 entry points.
"""
import ctypes as C
import os
import subprocess

import numpy as np

from oracle import lev_oracle as lo
from oracle import lev_oracle_f64 as lo64

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "rlmd_b200.h")

# lev/gbm.py's second environment (gbm_snp): drift 0.054..., vol 0.1897...
SNP_LOG_MEAN = 0.0540025395205692 - 0.1897916175617430 ** 2 / 2
SNP_SIGMA = 0.1897916175617430


def test_coin_chain_f64_matches_closed_form():
    rs = np.random.RandomState(3)
    n, h, v0 = 500, 3000, 100.0
    oc = (rs.rand(n, h) < 0.5).astype(np.uint8)
    lev = lo64.lev_grid_f64(0.1, 1.0, 0.1, 0.5, -0.4)
    f = lo64.coin_factors_f64(lev, 0.5, -0.4)
    assert f.dtype == np.float64 and np.array_equal(f[:, 1], 1.0 + lev * 0.5)
    w = lo64.chain_discrete_f64(oc, f, v0)
    n_up = oc.sum(axis=1).astype(np.float64)
    # in the log domain: (1 - 0.4 l)^n_down alone leaves fp64 range at l = 1.0 (the interleaved product does not)
    log_w = n_up[None, :] * np.log(1 + lev[:, None] * 0.5) + (h - n_up)[None, :] * np.log(1 + lev[:, None] * -0.4)
    closed = v0 * np.exp(log_w)
    assert w.dtype == np.float64
    assert np.all(w > 0)      # l = 1.0 at H = 3000: the median wealth is ~e^-157, far inside fp64 range
    assert np.max(np.abs(w - closed) / closed) <= 1e-12


def test_gbm_chain_f64_matches_closed_form():
    rs = np.random.RandomState(4)
    n, h, v0 = 300, 2000, 100.0
    x = SNP_LOG_MEAN + SNP_SIGMA * rs.randn(n, h)
    lev = lo64.lev_grid_f64(0.2, 2.0, 0.2)
    w = lo64.chain_gbm_f64(x, lev, v0)
    closed = v0 * np.exp(lev[:, None] * x.sum(axis=1)[None, :])
    assert np.all(np.isfinite(w))
    assert np.max(np.abs(w - closed) / closed) <= 1e-15 * h


def test_gbm_h1e4_lev04_finite_in_fp64_inf_in_fp32():
    """App. C: at H = 1e4 every l >= 0.4 is inf in the reference's fp32 run; the fp64 run keeps l = 0.4 finite
    and still overflows at l = 2.0 (2 S passes ln DBL_MAX ~ 709.8 for most investors)."""
    rs = np.random.RandomState(5)
    n, h = 64, 10000
    x = SNP_LOG_MEAN + SNP_SIGMA * rs.randn(n, h)
    lev = np.array([0.4, 2.0])
    w64 = lo64.chain_gbm_f64(x, lev, 100.0)
    w32 = lo.chain_gbm(x.astype(np.float32), lev.astype(np.float32), 100.0)
    assert np.all(np.isfinite(w64[0])) and np.all(w64[0] > 0)
    assert np.all(np.isinf(w32[0]))
    assert np.mean(np.isinf(w64[1])) > 0.5
    closed = 100.0 * np.exp(0.4 * x.sum(axis=1))
    assert np.max(np.abs(w64[0] - closed) / closed) <= 1e-15 * h


def test_smart_and_final_f64_agree_with_chain():
    rs = np.random.RandomState(6)
    n, h, top = 257, 40, 3
    oc = (rs.rand(n, h) < 0.5).astype(np.uint8)
    lev = lo64.lev_grid_f64(0.5, 1.0, 0.25, 0.5, -0.4)
    f = lo64.coin_factors_f64(lev, 0.5, -0.4)
    data, data_T = lo64.smart_lev_f64(oc, f, lev, top, 100.0)
    assert data.shape == (len(lev), 13, h - 1) and data.dtype == np.float64
    assert np.array_equal(data_T, lo64.chain_discrete_f64(oc, f, 100.0))
    fin = lo64.fixed_final_lev_f64(oc, f, top, 100.0)
    assert np.array_equal(fin, data[:, :12, -1])
    assert np.array_equal(data[:, 12, 0], lev)
    # a subset of steps: the other columns stay nan
    part, _ = lo64.smart_lev_f64(oc, f, lev, top, 100.0, steps={1, h - 1})
    assert np.array_equal(part[:, :, -1], data[:, :, -1]) and np.isnan(part[:, 0, 1]).all()


def test_summary_stats_f64_empty_adj_group():
    s = lo64.summary_stats_f64(np.array([3.5]), 1)
    assert list(s[[0, 1, 3, 4, 6, 7, 9, 10]]) == [3.5, 3.5, 0.0, 0.0, 0.0, 0.0, 3.5, 3.5]
    assert np.isnan(s[[2, 5, 8, 11]]).all()
    v = np.array([1.0, -2.0, 5.0])
    assert np.array_equal(lo64.summary_stats_f64(v, 1), lo.summary_stats(v, 1))


# C ABI of the float64 entry points: (header type, ctypes type) of the result and of every argument
def _spec():
    from rlmd_b200 import _lib

    vp = C.c_void_p
    return {
        "b200_rowstats_f64_workspace_bytes": (("int64_t", C.c_int64), [("int64_t", C.c_int64)]),
        "b200_rowstats_f64": (("int", C.c_int), [("const double*", vp), ("int64_t", C.c_int64), ("int64_t", C.c_int64),
                                                 ("int64_t", C.c_int64), ("int64_t", C.c_int64), ("void*", vp),
                                                 ("double*", vp), ("void*", vp)]),
        "b200_lev_chunk_f64": (("int", C.c_int), [("const b200_lev_desc*", C.POINTER(_lib.LevDesc)),
                                                  ("const void*", vp), ("const double*", C.POINTER(C.c_double)),
                                                  ("int32_t", C.c_int32), ("int32_t", C.c_int32), ("double*", vp),
                                                  ("double*", vp), ("void*", vp)]),
    }


def test_f64_entry_points_bound_as_declared(tmp_path):
    """The header's prototypes are the spec's (a C compiler checks them) and _lib.py binds the same types."""
    from rlmd_b200 import _lib

    spec = _spec()
    lines = ["#include <stdio.h>", f'#include "{HEADER}"', "int main(void){"]
    for name, ((res, _), args) in spec.items():
        lines.append(f"{res} (*p_{name})({', '.join(a for a, _ in args)}) = {name};")
        lines.append(f'printf("%d\\n", p_{name} != 0);')
    lines.append("return 0;}")
    src = tmp_path / "sig.c"
    src.write_text("\n".join(lines))
    # only compiled, never linked or run against the library: a prototype mismatch is a compile error
    subprocess.check_call(["gcc", "-std=c99", "-Werror=incompatible-pointer-types", "-c", "-o",
                           str(tmp_path / "sig.o"), str(src)])
    for name, ((_, res), args) in spec.items():
        got_res, got_args = _lib._SIGNATURES[name]
        assert got_res == res, name
        assert list(got_args) == [t for _, t in args], name
        assert hasattr(_lib.lib, name)


"""
ctypes binding of librlmd_b200.so (include/rlmd_b200.h).

There is no CPU fallback: if the shared library is missing this module raises
at import, and every compute entry point fails loudly without a CUDA device.
Build it with `python -c "import __graft_entry__ as g; g.build()"` or `make`.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "librlmd_b200.so")

B200_OK, B200_EINVAL, B200_ECUDA, B200_ELIMIT = 0, -1, -2, -3
LEV_DISCRETE, LEV_GBM = 0, 1
SRC_STREAM, SRC_PHILOX = 0, 1
MODE_CHAIN, MODE_LOG = 1, 2
MAX_GRID, MAX_OUTCOMES = 64, 4


class LevDesc(C.Structure):
    _fields_ = [
        ("n_investors", C.c_int64),
        ("ld_outcomes", C.c_int64),
        ("investor_offset", C.c_int64),
        ("ld_out", C.c_int64),
        ("seed", C.c_uint64),
        ("horizon", C.c_int32),
        ("n_grid", C.c_int32),
        ("n_outcomes", C.c_int32),
        ("kind", C.c_int32),
        ("source", C.c_int32),
        ("mode", C.c_int32),
        ("value_0", C.c_float),
        ("log_mean", C.c_float),
        ("sigma", C.c_float),
        ("variant", C.c_int32),
        ("thresholds", C.c_uint32 * MAX_OUTCOMES),
        ("outcome_bits", C.c_int32),
        ("flags", C.c_int32),
    ]


LEV_FLAG_FINAL_ONLY, LEV_FLAG_STATE_OUT, LEV_FLAG_BESIDE_SWEEP, LEV_FLAG_RADIX_SELECT, LEV_FLAG_EARLY_START = 1, 2, 4, 8, 16
MAX_PEERS = 8


class PeerSet(C.Structure):
    _fields_ = [
        ("workspace", C.c_void_p * MAX_PEERS),
        ("flags", C.c_void_p * MAX_PEERS),
        ("stage", C.c_void_p * MAX_PEERS),
        ("stage_rows", C.c_int64),
        ("world", C.c_int32),
        ("rank", C.c_int32),
        ("epoch", C.c_uint32),
        ("reserved", C.c_uint32),
    ]


class TallyPlan(C.Structure):
    _fields_ = [
        ("rows_cap", C.c_int64),
        ("bins_cap", C.c_int64),
        ("grid_cap", C.c_int32),
        ("world", C.c_int32),
    ]


class TallyPeers(C.Structure):
    _fields_ = [
        ("exchange", C.c_void_p * MAX_PEERS),
        ("world", C.c_int32),
        ("rank", C.c_int32),
        ("epoch", C.c_uint32),
        ("reserved", C.c_uint32),
    ]


DT_U8, DT_I32, DT_I64, DT_F32, DT_F64 = 0, 1, 2, 3, 4
TALLY_INFO_WORDS = 8
TALLY_MAX_HORIZON = (1 << 21) - 1

ENV_COIN, ENV_DICE, ENV_GBM, ENV_DICE_SH = 0, 1, 2, 3
INV_A, INV_B, INV_C, INV_INSURED = 0, 1, 2, 3
ENV_MAX_GAMBLES = 8


class EnvDesc(C.Structure):
    _fields_ = [
        ("family", C.c_int32),
        ("investor", C.c_int32),
        ("n_gambles", C.c_int32),
        ("stop_abs", C.c_int32),
        ("max_value", C.c_double),
        ("initial_value", C.c_double),
        ("min_value", C.c_double),
        ("max_abs_action", C.c_double),
        ("min_reward", C.c_double),
        ("min_return", C.c_double),
        ("max_return", C.c_double),
        ("min_weight", C.c_double),
        ("lev_factor", C.c_double),
        ("returns", C.c_double * 3),
        ("probs", C.c_double * 3),
        ("sh_returns", C.c_double * 3),
        ("i_lev_factor", C.c_double),
        ("sh_lev_factor", C.c_double),
        ("log_mean", C.c_double),
        ("vol", C.c_double),
        ("seed", C.c_uint64),
    ]


REPLAY_MAX_STEPS = 64


class ReplayDesc(C.Structure):
    _fields_ = [
        ("mem_size", C.c_int64),
        ("state_dim", C.c_int32),
        ("action_dim", C.c_int32),
        ("state_memory", C.c_void_p),
        ("action_memory", C.c_void_p),
        ("reward_memory", C.c_void_p),
        ("next_state_memory", C.c_void_p),
        ("terminal_memory", C.c_void_p),
        ("episode_start", C.c_void_p),
        ("header", C.c_void_p),
    ]


class MarketDesc(C.Structure):
    _fields_ = [
        ("investor", C.c_int32),
        ("n_assets", C.c_int32),
        ("obs_days", C.c_int32),
        ("time_length", C.c_int32),
        ("max_value", C.c_double),
        ("initial_value", C.c_double),
        ("min_value", C.c_double),
        ("max_abs_action", C.c_double),
        ("min_reward", C.c_double),
        ("min_return", C.c_double),
        ("max_return", C.c_double),
        ("min_weight", C.c_double),
        ("lev_factor", C.c_double),
    ]


MARKET_MAX_ASSETS = 128


class CollectDesc(C.Structure):
    _fields_ = [
        ("env", EnvDesc),
        ("replay", ReplayDesc),
        ("n_envs", C.c_int64),
        ("lane_len", C.c_int64),
        ("reward_floor", C.c_double),
    ]


BB_COIN, BB_DICE, BB_MAX_POINTS = 0, 1, 128


class BigBrainDesc(C.Structure):
    _fields_ = [
        ("n_investors", C.c_int64),
        ("ld_outcomes", C.c_int64),
        ("horizon", C.c_int32),
        ("n_points", C.c_int32),
        ("kind", C.c_int32),
        ("reserved", C.c_int32),
        ("value_0", C.c_float),
        ("lev_factor32", C.c_float),
        ("lev_factor64", C.c_double),
        ("returns", C.c_double * 3),
    ]


class B200Error(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"rlmd_b200 error {code}: {msg}")
        self.code = code


if not os.path.isfile(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} is missing: build the CUDA library first (make, or __graft_entry__.build()); "
        "rlmd_b200 has no CPU fallback"
    )

lib = C.CDLL(LIB_PATH)

_vp, _i32, _i64 = C.c_void_p, C.c_int32, C.c_int64
_SIGNATURES = {
    "b200_last_error": (C.c_char_p, []),
    "b200_version": (C.c_int, []),
    "b200_device_info": (C.c_int, [C.POINTER(_i32)] * 3),
    "b200_lev_sweep": (C.c_int, [C.POINTER(LevDesc), _vp, C.POINTER(C.c_float), _vp, _vp, _vp, _vp]),
    "b200_lev_draw": (C.c_int, [C.POINTER(LevDesc), _vp, _vp]),
    "b200_lev_from_counts": (C.c_int, [C.POINTER(LevDesc), _vp, C.POINTER(C.c_float), _vp, _vp, _vp]),
    "b200_lev_pack": (C.c_int, [_vp, _i64, _i32, _i64, _vp, _i64, _vp]),
    "b200_lev_pack_bits": (C.c_int, [_vp, _i64, _i32, _i64, _vp, _i64, _i32, _vp]),
    "b200_lev_chunk": (C.c_int, [C.POINTER(LevDesc), _vp, C.POINTER(C.c_float), _i32, _i32, _vp, _vp, _vp]),
    "b200_menv_dims": (C.c_int, [C.POINTER(EnvDesc)] + [C.POINTER(_i32)] * 3),
    "b200_menv_reset": (C.c_int, [C.POINTER(EnvDesc), _i64, _vp, _vp, _vp, _vp, _vp]),
    "b200_menv_step": (C.c_int, [C.POINTER(EnvDesc), _i64, _vp, _vp, _vp, _vp, C.c_uint64, _vp, _vp, _vp, _vp, _vp]),
    "b200_replay_reset": (C.c_int, [C.POINTER(ReplayDesc), _vp]),
    "b200_replay_store": (C.c_int, [C.POINTER(ReplayDesc), _vp, _vp, _vp, _vp, _vp, _i64, _i32, _i64, C.c_double, _vp]),
    "b200_replay_store_host": (C.c_int, [C.POINTER(ReplayDesc), C.POINTER(C.c_double), C.POINTER(C.c_double),
                                         C.c_double, C.POINTER(C.c_double), _i32, _i64, C.c_double, _vp]),
    "b200_replay_sample": (C.c_int, [C.POINTER(ReplayDesc), _vp, _i64, _i32, _i64, _i32, C.POINTER(C.c_float), _i32,
                                     C.c_uint64, C.c_uint64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "b200_replay_sample_counted": (C.c_int, [C.POINTER(ReplayDesc), _i64, _i32, _i32, C.POINTER(C.c_float), _i32,
                                             C.c_uint64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "b200_exchange_pack": (C.c_int, [_vp, _i64, _i64, _i64, _i64, _i64, _i64, _vp, _vp]),
    "b200_exchange_unpack": (C.c_int, [_vp, _i64, _i64, _i64, _i64, _i64, _i64, _vp, _vp]),
    "b200_market_dims": (C.c_int, [C.POINTER(MarketDesc)] + [C.POINTER(_i32)] * 3),
    "b200_market_reset": (C.c_int, [C.POINTER(MarketDesc), _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "b200_market_step": (C.c_int, [C.POINTER(MarketDesc), _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "b200_collect_reset": (C.c_int, [C.POINTER(CollectDesc), _vp, _vp, _vp, _vp, _vp]),
    "b200_collect_step": (C.c_int, [C.POINTER(CollectDesc), _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "b200_collect_sample": (C.c_int, [C.POINTER(CollectDesc), _vp, _i64, _i32, _i32, C.POINTER(C.c_float), _i32,
                                      C.c_uint64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "b200_menv_rollout": (C.c_int, [C.POINTER(EnvDesc), _i64, _vp, _vp, C.c_uint64, _i32, _vp, _vp, _vp, _vp, _vp]),
    "b200_bigbrain_chunk": (C.c_int, [C.POINTER(BigBrainDesc), _vp, C.POINTER(C.c_float), C.POINTER(C.c_float),
                                      C.POINTER(C.c_double), _i32, _i32, _vp, _vp, _vp]),
    "b200_growth_workspace_bytes": (_i64, [_i64]),
    "b200_gbm_valid": (C.c_int, [_vp, _vp, _i64, _i64, C.POINTER(C.c_float), _i32, C.c_double, _vp, _vp]),
    "b200_gbm_growth_assemble": (C.c_int, [_vp, _vp, C.POINTER(C.c_float), _i32, _i32, _i32, _vp, _vp, _vp, _vp]),
    "b200_growth_exchange": (C.c_int, [_i32, C.POINTER(_i64)]),
    "b200_growth_summary": (C.c_int, [_vp, _vp, _i64, _i64, _i64, _i64, _i64, C.c_double, _i32, C.POINTER(C.c_double),
                                      _i32, _vp, _vp, _i32, _vp]),
    "b200_tally_workspace_bytes": (_i64, [C.POINTER(TallyPlan)]),
    "b200_tally_exchange_bytes": (_i64, [C.POINTER(TallyPlan)]),
    "b200_tally_reset": (C.c_int, [C.POINTER(TallyPlan), _vp, _vp]),
    "b200_lev_tally": (C.c_int, [C.POINTER(LevDesc), _vp, C.POINTER(TallyPlan), _vp, _vp, _vp]),
    "b200_lev_ingest": (C.c_int, [_vp, _i32, _i64, _i32, _i64, _i32, _vp, _i64, _vp, C.POINTER(TallyPlan), _vp, _vp]),
    "b200_tally_finalize": (C.c_int, [C.POINTER(TallyPlan), _vp, C.POINTER(TallyPeers), _i32, _vp]),
    "b200_tally_stats": (C.c_int, [C.POINTER(TallyPlan), _vp, C.POINTER(LevDesc), C.POINTER(C.c_float), _i64, _i64,
                                   _vp, _vp]),
    "b200_rowstats_workspace_bytes": (_i64, [_i64]),
    "b200_rowstats_stage_bytes": (_i64, [_i64, _i32]),
    "b200_rowstats": (C.c_int, [_vp, _i64, _i64, _i64, _i64, _i64, _vp, _vp, _i32, _vp]),
    "b200_rowstats_exchange": (C.c_int, [_i32, C.POINTER(_i64)]),
    "b200_rowstats_p2p": (C.c_int, [_vp, _i64, _i64, _i64, _i64, _i64, C.POINTER(PeerSet), _vp, _vp]),
    "b200_rowstats_f64_workspace_bytes": (_i64, [_i64]),
    "b200_rowstats_f64": (C.c_int, [_vp, _i64, _i64, _i64, _i64, _vp, _vp, _vp]),
    "b200_lev_chunk_f64": (C.c_int, [C.POINTER(LevDesc), _vp, C.POINTER(C.c_double), _i32, _i32, _vp, _vp, _vp]),
}
# extended below as entry points are added; tests/test_cabi.py checks that every
# symbol declared in include/rlmd_b200.h is listed here and exported.
EXPORTS = _SIGNATURES


def _bind():
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args


_bind()


def check(rc: int) -> None:
    if rc != 0:
        raise B200Error(rc, lib.b200_last_error().decode("utf-8", "replace"))


def require_cuda():
    import torch

    if not torch.cuda.is_available():
        raise B200Error(B200_ECUDA, "no CUDA device: rlmd_b200 has no CPU fallback")


def stream_ptr():
    """The current torch stream of the current device as a cudaStream_t (called on every launch: the raw
    accessor skips building a torch.cuda.Stream object)."""
    import torch

    raw = getattr(torch._C, "_cuda_getCurrentRawStream", None)
    if raw is not None:
        return C.c_void_p(raw(torch.cuda.current_device()))
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    """Raw device pointer of a torch tensor (None -> NULL)."""
    return C.c_void_p(0 if t is None else t.data_ptr())

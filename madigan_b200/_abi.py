"""ctypes mirror of ``include/madigan_b200.h`` (the C-ABI of the CUDA library).

Field order and types must match the header byte for byte; ``tests/test_abi.py``
checks the struct sizes against the compiled library (``mdg_sizeof``).
"""
import ctypes as C

MDG_ABI_VERSION = 16
FLAG_FORCE_EXACT_GATE = 1
FLAG_GENERIC_FILL = 2
XFORM_NONE, XFORM_PAIR_RATIO, XFORM_RETURNS = 0, 1, 2
MDG_MAX_ASSETS = 16
MDG_GEN_NPARAM = 10
MDG_BROKER_NPARAM = 7  # broker table rows, MdgParams field order (data_source.BROKER_SLOTS)
MDG_MAX_NSTEP = 64
MDG_MAX_SINE_COMPONENTS = 16
MDG_MAX_SINE_TRENDS = 4
MDG_STATS_NSCALAR = 8

MDG_OK, MDG_E_INVALID, MDG_E_UNSUPPORTED, MDG_E_CUDA = 0, -1, -2, -3

# RiskInfo (reference: environments/cpp/DataTypes.h:70-75)
RISK_GREEN, RISK_INSUFF_MARGIN, RISK_MARGIN_CALL, RISK_BLOWN_OUT = 0, 1, 2, 3

GEN_SYNTH, GEN_OU, GEN_OUPAIR, GEN_SIMPLETREND, GEN_TRENDOU, GEN_TRENDYOU = 0, 1, 2, 3, 4, 5
GEN_SAWTOOTH, GEN_TRIANGLE, GEN_GAUSSIAN = 6, 7, 8
GEN_SINEADDER, GEN_SINEDYNAMIC, GEN_SINEDYNAMICTREND = 9, 10, 11

SHAPER_OFF, SHAPER_SUM, SHAPER_DSR, SHAPER_DDR, SHAPER_COSINE = 0, 1, 2, 3, 4
SHAPER_SHARPE, SHAPER_SORTINO_A, SHAPER_SORTINO_B = 5, 6, 7

MODE_HOLD, MODE_MULTI, MODE_SINGLE = 0, 1, 2

NORM_NONE, NORM_LOOKBACK, NORM_LOOKBACK_LOG, NORM_LOG = 0, 1, 2, 3
NORM_STANDARD, NORM_LOG_STANDARD, NORM_EXPANDING = 4, 5, 6
DTYPE_F64, DTYPE_F32 = 0, 1
LAYOUT_NKF, LAYOUT_NFK = 0, 1

_dp = C.c_void_p  # device (or, for the oracle, host) pointer


class MdgAssetGen(C.Structure):
    _fields_ = [("type", C.c_int32), ("role", C.c_int32), ("nslot", C.c_int32),
                ("nslot_aux", C.c_int32), ("uslot", C.c_int32), ("gslot", C.c_int32),
                ("partner", C.c_int32), ("_pad", C.c_int32),
                ("p", C.c_double * MDG_GEN_NPARAM)]


class MdgParams(C.Structure):
    _fields_ = [("n_assets", C.c_int32), ("n_gstate", C.c_int32), ("n_normals", C.c_int32),
                ("n_uniforms", C.c_int32), ("init_cash", C.c_double),
                ("required_margin", C.c_double), ("maintenance_margin", C.c_double),
                ("slippage_rel", C.c_double), ("slippage_abs", C.c_double),
                ("tcost_rel", C.c_double), ("tcost_abs", C.c_double),
                ("gen", MdgAssetGen * MDG_MAX_ASSETS), ("gen_ext", _dp), ("n_gen_ext", C.c_int64)]


class MdgReward(C.Structure):
    _fields_ = [("shaper", C.c_int32), ("reduce_rewards", C.c_int32), ("nstep", C.c_int32),
                ("_pad", C.c_int32), ("discount", C.c_double), ("adaptation_rate", C.c_double),
                ("cosine_temp", C.c_double), ("sortino_exp", C.c_double),
                ("desired_portfolio", C.c_double * (MDG_MAX_ASSETS + 1)),
                ("discounts", C.c_double * MDG_MAX_NSTEP)]


class MdgState(C.Structure):
    _fields_ = [(n, _dp) for n in ("price", "ledger", "mean_entry", "borrowed", "cash", "gstate",
                                   "timestamp", "shaper_A", "shaper_B", "nstep_ring", "nstep_len", "reset_ts", "folds")]


class MdgStepIO(C.Structure):
    _fields_ = [(n, _dp) for n in ("units", "normals", "uniforms", "obs_price", "obs_port",
                                   "pre_price", "reward", "done", "trans_price", "trans_units",
                                   "trans_cost", "risk", "margin_call", "agent_reward",
                                   "shaped_reward", "n_popped", "actions", "weights")]


class MdgLaunch(C.Structure):
    _fields_ = [("n_envs", C.c_int64), ("env_offset", C.c_int64), ("seed", C.c_uint64),
                ("window", C.c_int32), ("head", C.c_int32), ("mode", C.c_int32),
                ("asset_idx", C.c_int32), ("nstep_pos", C.c_int32), ("action_atoms", C.c_int32),
                ("stream", C.c_void_p), ("unit_size", C.c_double), ("flags", C.c_int32), ("_pad", C.c_int32)]


class MdgWindow(C.Structure):
    _fields_ = [("ring", _dp), ("prefix", _dp), ("timestamp", _dp), ("reset_ts", _dp), ("n_envs", C.c_int64),
                ("n_feats", C.c_int32), ("window", C.c_int32), ("head", C.c_int32), ("n_valid", C.c_int32),
                ("norm_type", C.c_int32), ("flat_prefix", C.c_int32), ("out_dtype", C.c_int32),
                ("out_layout", C.c_int32), ("out", _dp), ("stream", _dp), ("transform", C.c_int32), ("stride", C.c_int32),
                ("age0", C.c_int32), ("out_feats_total", C.c_int32), ("out_feat_offset", C.c_int32), ("_pad", C.c_int32)]


class MdgDerived(C.Structure):
    _fields_ = [(n, _dp) for n in ("equity", "asset_value", "pnl", "balance", "available_margin",
                                   "used_margin", "borrowed_margin", "borrowed_asset_value", "risk",
                                   "position_values", "pnl_positions", "ledger_normed",
                                   "ledger_abs_normed", "ledger_normed_full",
                                   "ledger_abs_normed_full", "position_values_full", "ledger_full")]


# every symbol include/madigan_b200.h declares: name -> (restype, argtypes)
_P = C.POINTER
class MdgReplay(C.Structure):
    _fields_ = [(n, _dp) for n in ("t_env", "t_state_slot", "t_next_slot", "t_state_step", "t_done", "t_reward",
                                   "t_action", "cursor", "act_ring")] + \
               [("capacity", C.c_int64), ("depth", C.c_int32), ("nstep", C.c_int32), ("ra", C.c_int32),
                ("n_action", C.c_int32)]


class MdgReplayBatch(C.Structure):
    _fields_ = [(n, _dp) for n in ("idx", "state_price", "next_price", "state_port", "next_port", "action",
                                   "reward", "done")]


class MdgPrioritized(C.Structure):
    _fields_ = [(n, _dp) for n in ("sum_tree", "min_tree", "leaf_pos", "batch_pos", "dirty", "dirty_list", "ctl",
                                   "seen", "max_priority", "n_rejected")] + \
               [("capacity", C.c_int64), ("tree_size", C.c_int64), ("alpha", C.c_double)]


class MdgReplayRows(C.Structure):
    _fields_ = [(n, _dp) for n in ("rows", "row_end", "row_count", "last_ts")] + \
               [("n_rows", C.c_int64), ("n_feats", C.c_int32), ("window", C.c_int32)]


class MdgParamSets(C.Structure):
    _fields_ = [("p", _dp), ("set_of_env", _dp), ("n_sets", C.c_int32), ("_pad", C.c_int32)]


class MdgSetDraw(C.Structure):
    _fields_ = [("cdf", _dp), ("episode_set", _dp)]


RN_NULL, RN_SHARPE_FIXED, RN_SORTINO_A, RN_SORTINO_B, RN_SORTINO_C, RN_SHARPE_EWMA = range(6)


MDG_TS_MAX_OFFSETS = 8
MDG_TS_NFIXED = 7


class MdgTearsheet(C.Structure):
    _fields_ = [("n_envs", C.c_int64), ("n_assets", C.c_int32), ("n_offsets", C.c_int32)] + \
               [(n, _dp) for n in ("nsteps", "active", "sum_equity", "last_equity", "sum_reward", "peak", "min_valley",
                                   "sum_cost", "in_pos", "eq_ring", "ret_n", "ret_mean", "ret_m2", "ret_down")]


class MdgEpisodeResults(C.Structure):
    _fields_ = [("ts", MdgTearsheet), ("acc", _dp), ("ext", _dp), ("n_sets", C.c_int32), ("n_fields", C.c_int32)]


MDG_RES_DIGITS = 5  # base-2^30 digits of a quantised value (MdgEpisodeResults)


class MdgRewardNorm(C.Structure):
    _fields_ = [("kind", C.c_int32), ("window", C.c_int32), ("n_envs", C.c_int64), ("alpha", C.c_double)] + \
               [(n, _dp) for n in ("buffer", "size", "front", "count", "mean_est", "ssq", "ewma", "ewma_old",
                                   "ewssq_old", "ewssq", "w1", "w2")]


SYMBOLS = {
    "mdg_abi_version": (C.c_int, []),
    "mdg_last_error": (C.c_char_p, []),
    "mdg_sizeof": (C.c_int, [C.c_int]),
    "mdg_step": (C.c_int, [_P(MdgParams), _P(MdgReward), _P(MdgState), _P(MdgStepIO), _P(MdgLaunch)]),
    "mdg_reset": (C.c_int, [_P(MdgParams), _P(MdgState), _P(MdgStepIO), _P(MdgLaunch), C.c_void_p,
                            C.c_int, C.c_int]),
    "mdg_reset_ws": (C.c_int, [_P(MdgParams), _P(MdgState), _P(MdgStepIO), _P(MdgLaunch), C.c_void_p,
                               C.c_int, C.c_int, C.c_void_p, C.c_int64]),
    "mdg_reset_workspace_bytes": (C.c_int64, [_P(MdgParams), C.c_int64, C.c_int]),
    "mdg_step_autoreset": (C.c_int, [_P(MdgParams), _P(MdgReward), _P(MdgState), _P(MdgStepIO), _P(MdgLaunch),
                                     C.c_int, C.c_int, C.c_void_p, C.c_int64]),
    "mdg_init_state": (C.c_int, [_P(MdgParams), _P(MdgReward), _P(MdgState), _P(MdgLaunch)]),
    "mdg_step_sets": (C.c_int, [_P(MdgParams), _P(MdgReward), _P(MdgState), _P(MdgStepIO), _P(MdgLaunch),
                                _P(MdgParamSets)]),
    "mdg_step_autoreset_sets": (C.c_int, [_P(MdgParams), _P(MdgReward), _P(MdgState), _P(MdgStepIO), _P(MdgLaunch),
                                          C.c_int, C.c_int, C.c_void_p, C.c_int64, _P(MdgParamSets)]),
    "mdg_reset_ws_sets": (C.c_int, [_P(MdgParams), _P(MdgState), _P(MdgStepIO), _P(MdgLaunch), C.c_void_p,
                                    C.c_int, C.c_int, C.c_void_p, C.c_int64, _P(MdgParamSets)]),
    "mdg_init_state_sets": (C.c_int, [_P(MdgParams), _P(MdgReward), _P(MdgState), _P(MdgLaunch), _P(MdgParamSets)]),
    "mdg_step_sets_broker": (C.c_int, [_P(MdgParams), _P(MdgReward), _P(MdgState), _P(MdgStepIO), _P(MdgLaunch),
                                       _P(MdgParamSets), C.c_void_p]),
    "mdg_step_autoreset_sets_broker": (C.c_int, [_P(MdgParams), _P(MdgReward), _P(MdgState), _P(MdgStepIO),
                                                 _P(MdgLaunch), C.c_int, C.c_int, C.c_void_p, C.c_int64,
                                                 _P(MdgParamSets), C.c_void_p]),
    "mdg_reset_ws_sets_broker": (C.c_int, [_P(MdgParams), _P(MdgState), _P(MdgStepIO), _P(MdgLaunch), C.c_void_p,
                                           C.c_int, C.c_int, C.c_void_p, C.c_int64, _P(MdgParamSets), C.c_void_p]),
    "mdg_init_state_sets_broker": (C.c_int, [_P(MdgParams), _P(MdgReward), _P(MdgState), _P(MdgLaunch),
                                             _P(MdgParamSets), C.c_void_p]),
    "mdg_step_autoreset_sets_draw": (C.c_int, [_P(MdgParams), _P(MdgReward), _P(MdgState), _P(MdgStepIO),
                                               _P(MdgLaunch), C.c_int, C.c_int, C.c_void_p, C.c_int64,
                                               _P(MdgParamSets), C.c_void_p, _P(MdgSetDraw)]),
    "mdg_reset_ws_sets_draw": (C.c_int, [_P(MdgParams), _P(MdgState), _P(MdgStepIO), _P(MdgLaunch), C.c_void_p,
                                         C.c_int, C.c_int, C.c_void_p, C.c_int64, _P(MdgParamSets), C.c_void_p,
                                         _P(MdgSetDraw)]),
    "mdg_init_state_sets_draw": (C.c_int, [_P(MdgParams), _P(MdgReward), _P(MdgState), _P(MdgLaunch),
                                           _P(MdgParamSets), C.c_void_p, _P(MdgSetDraw)]),
    "mdg_refresh_folds": (C.c_int, [_P(MdgParams), _P(MdgState), _P(MdgLaunch)]),
    "mdg_derived": (C.c_int, [_P(MdgParams), _P(MdgState), _P(MdgDerived), _P(MdgLaunch)]),
    "mdg_derived_sets_broker": (C.c_int, [_P(MdgParams), _P(MdgState), _P(MdgDerived), _P(MdgLaunch),
                                          _P(MdgParamSets), C.c_void_p]),
    "mdg_materialise_window": (C.c_int, [_P(MdgWindow)]),
    "mdg_replay_append": (C.c_int, [_P(MdgReplay), C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.c_void_p, C.c_void_p]),
    "mdg_replay_sample": (C.c_int, [_P(MdgReplay), C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                    C.c_int32, C.c_int64, C.c_uint64, C.c_uint64, _P(MdgReplayBatch), C.c_void_p]),
    "mdg_per_ingest": (C.c_int, [_P(MdgPrioritized), _P(MdgReplay), C.c_int64, C.c_void_p]),
    "mdg_per_sample": (C.c_int, [_P(MdgPrioritized), _P(MdgReplay), C.c_int64, C.c_int64, C.c_void_p, C.c_void_p,
                                 C.c_int32, C.c_int32, C.c_int32, C.c_int64, C.c_double, C.c_uint64, C.c_uint64,
                                 _P(MdgReplayBatch), C.c_void_p, C.c_void_p, C.c_void_p]),
    "mdg_per_update": (C.c_int, [_P(MdgPrioritized), C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mdg_replay_rows_ingest": (C.c_int, [_P(MdgReplayRows), _P(MdgWindow), C.c_int64, C.c_int32]),
    "mdg_replay_sample_rows": (C.c_int, [_P(MdgReplay), _P(MdgReplayRows), C.c_int64, C.c_int64, C.c_void_p, C.c_int32,
                                         C.c_int32, C.c_int32, C.c_int64, C.c_uint64, C.c_uint64, _P(MdgReplayBatch),
                                         C.c_void_p]),
    "mdg_per_sample_rows": (C.c_int, [_P(MdgPrioritized), _P(MdgReplay), _P(MdgReplayRows), C.c_int64, C.c_int64,
                                      C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int64, C.c_double, C.c_uint64,
                                      C.c_uint64, _P(MdgReplayBatch), C.c_void_p, C.c_void_p, C.c_void_p]),
    "mdg_materialise_time": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p]),
    "mdg_episode_stats": (C.c_int, [_P(MdgParams), _P(MdgState), _P(MdgStepIO), _P(MdgLaunch),
                                    C.c_void_p]),
    "mdg_reward_norm_reset": (C.c_int, [_P(MdgRewardNorm), C.c_void_p, C.c_void_p]),
    "mdg_reward_norm_stream": (C.c_int, [_P(MdgRewardNorm), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mdg_tearsheet_reset": (C.c_int, [_P(MdgTearsheet), C.c_void_p, C.c_void_p]),
    "mdg_tearsheet_update": (C.c_int, [_P(MdgParams), _P(MdgState), _P(MdgStepIO), _P(MdgTearsheet), C.c_void_p]),
    "mdg_tearsheet_summary": (C.c_int, [_P(MdgTearsheet), C.c_void_p, C.c_void_p]),
    "mdg_step_autoreset_results": (C.c_int, [_P(MdgParams), _P(MdgReward), _P(MdgState), _P(MdgStepIO),
                                             _P(MdgLaunch), C.c_int, C.c_int, C.c_void_p, C.c_int64,
                                             _P(MdgParamSets), C.c_void_p, _P(MdgSetDraw), _P(MdgEpisodeResults)]),
    "mdg_episode_results_record": (C.c_int, [_P(MdgParams), _P(MdgState), _P(MdgStepIO), _P(MdgParamSets),
                                             C.c_void_p, _P(MdgEpisodeResults), C.c_void_p]),
}


def bind(lib):
    """Attach restype/argtypes for every declared symbol; raises AttributeError if one is missing."""
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    return lib


STRUCTS = (MdgAssetGen, MdgParams, MdgReward, MdgState, MdgStepIO, MdgLaunch, MdgDerived, MdgWindow, MdgReplay,
           MdgReplayBatch, MdgRewardNorm, MdgTearsheet, MdgPrioritized, MdgReplayRows, MdgParamSets,
           MdgSetDraw, MdgEpisodeResults)  # mdg_sizeof order

"""ctypes binding of ``csrc/libcrowdnav_b200.so`` (declared in ``include/crowdnav_b200.h``).

The product path has no CPU fallback: if the CUDA library is missing, ``load()`` raises, and every compute
entry point fails with ``CrowdNavError`` when no sm_100 device is usable.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libcrowdnav_b200.so")

CN_OK, CN_EINVAL, CN_ECUDA, CN_ENOMEM, CN_EUNSUPPORTED, CN_EVALUE = 0, -1, -2, -3, -4, -5
NOTHING, DANGER, REACHGOAL, COLLISION, TIMEOUT = 0, 1, 2, 3, 4
CIRCLE_CROSSING, SQUARE_CROSSING = 0, 1
PREC_F32, PREC_F16_TC = 0, 1
WORLD_ATTENTION, WORLD_MLP = 0, 1                    # learned human-motion models (CN_WORLD_*)
NET_SARL, NET_CADRL, NET_LSTM_RL = 0, 1, 2           # value network behind the lookahead (CN_NET_*)
KIN_HOLONOMIC, KIN_UNICYCLE, KIN_NONE = 0, 1, 2      # robot kinematics (CN_KIN_*); NONE = the fork as shipped (cadrl.py:66)
AGENT_STRIDE = 8

EXPORTS = [
    "cn_last_error", "cn_version", "cn_device_count", "cn_env_cfg_default", "cn_sarl_cfg_default",
    "cn_env_create", "cn_env_destroy", "cn_env_set_state", "cn_env_get_state", "cn_env_set_theta", "cn_env_get_theta", "cn_env_reset", "cn_env_orca",
    "cn_env_robot_orca", "cn_env_step", "cn_env_get_views", "cn_env_read_outputs", "cn_env_read_human_actions",
    "cn_env_read_next_obs", "cn_env_read_actions", "cn_env_set_actions", "cn_env_set_human_actions", "cn_env_read_stats", "cn_env_copy_outputs", "cn_env_copy_world_pairs", "cn_env_episode_table_bytes", "cn_env_read_episode_table", "cn_policy_create", "cn_policy_destroy",
    "cn_policy_param_count", "cn_policy_load_weights", "cn_policy_action_table", "cn_policy_lookahead",
    "cn_policy_read", "cn_policy_bad_count", "cn_policy_transform", "cn_policy_last_state", "cn_policy_forward", "cn_rollout_step", "cn_rollout_step_sharded", "cn_rollout_episodes", "cn_rollout_step_host", "cn_rollout_step_host_packed", "cn_rollout_step_host_packed_async", "cn_stream_sync", "cn_host_step_bytes",
    "cn_scenes_generate", "cn_world_create", "cn_world_destroy", "cn_world_param_count", "cn_world_load_weights", "cn_world_predict",
    "cn_world_load_weights_device", "cn_world_trainer_create", "cn_world_trainer_destroy", "cn_world_trainer_param_count",
    "cn_world_trainer_sync_weights", "cn_world_trainer_step", "cn_world_trainer_apply", "cn_world_trainer_eval",
    "cn_trainer_create", "cn_trainer_destroy", "cn_trainer_param_count", "cn_trainer_sync_weights", "cn_trainer_step", "cn_trainer_step_indexed", "cn_trainer_apply",
    "cn_launch_count", "cn_debug_trace", "cn_debug_trace_dump", "cn_selftest_umma", "cn_selftest_umma_bmn", "cn_selftest_umma_ts", "cn_selftest_umma_pair", "cn_debug_tc_timing", "cn_debug_kernel_ms",
]


class CrowdNavError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("libcrowdnav_b200 error %d: %s" % (code, msg))
        self.code = code


class EnvCfg(C.Structure):
    _fields_ = [("num_envs", C.c_int32), ("human_num", C.c_int32), ("time_limit", C.c_double),
                ("time_step", C.c_double), ("success_reward", C.c_double), ("collision_penalty", C.c_double),
                ("discomfort_dist", C.c_double), ("discomfort_penalty_factor", C.c_double),
                ("neighbor_dist", C.c_double), ("max_neighbors", C.c_int32), ("time_horizon", C.c_double),
                ("human_safety_space", C.c_double), ("robot_visible", C.c_int32), ("sim_rule", C.c_int32),
                ("circle_radius", C.c_double), ("square_width", C.c_double), ("human_radius", C.c_double),
                ("human_v_pref", C.c_double), ("robot_radius", C.c_double), ("robot_v_pref", C.c_double),
                ("seed", C.c_uint64), ("env_id_offset", C.c_int64), ("auto_reset", C.c_int32),
                ("gamma", C.c_double), ("randomize_attributes", C.c_int32), ("robot_kinematics", C.c_int32)]


class SarlCfg(C.Structure):
    _fields_ = [("input_dim", C.c_int32), ("self_state_dim", C.c_int32), ("mlp1_dims", C.c_int32 * 2),
                ("mlp2_dims", C.c_int32 * 2), ("attn_dims", C.c_int32 * 3), ("mlp3_dims", C.c_int32 * 4),
                ("speed_samples", C.c_int32), ("rotation_samples", C.c_int32), ("gamma", C.c_double),
                ("v_pref", C.c_double), ("precision", C.c_int32), ("kinematics", C.c_int32),
                ("network", C.c_int32), ("lstm_hidden", C.c_int32), ("lstm_mlp1_dims", C.c_int32 * 4),
                ("with_om", C.c_int32), ("cell_num", C.c_int32), ("cell_size", C.c_double), ("om_channel_size", C.c_int32),
                ("without_global_state", C.c_int32)]


class RolloutRecord(C.Structure):
    """cn_rollout_record: replay-side records of cn_rollout_episodes (device arrays of the caller)."""
    _fields_ = [("transform_policy", C.c_void_p), ("last_state", C.c_int32), ("states_dev", C.c_void_p),
                ("reward_dev", C.c_void_p), ("done_dev", C.c_void_p)]


ROBOT_POLICY, ROBOT_ORCA, ROBOT_KEEP = 0, 1, 2


class Stats(C.Structure):
    _fields_ = [("episodes", C.c_int64), ("success", C.c_int64), ("collision", C.c_int64),
                ("timeout", C.c_int64), ("steps", C.c_int64), ("too_close", C.c_int64),
                ("sum_min_dist", C.c_double), ("sum_success_time", C.c_double),
                ("sum_collision_time", C.c_double), ("sum_timeout_time", C.c_double),
                ("sum_return", C.c_double)]


class EnvViews(C.Structure):
    _fields_ = [("reward", C.c_void_p), ("done", C.c_void_p), ("info", C.c_void_p), ("dmin", C.c_void_p),
                ("human_v", C.c_void_p), ("next_obs", C.c_void_p), ("state", C.c_void_p), ("time", C.c_void_p),
                ("action_idx", C.c_void_p), ("action_xy", C.c_void_p)]


_lib = None


def load():
    """Load the CUDA library; raises if it has not been built (no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError("%s is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(nvcc, sm_100a). There is no CPU fallback." % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    vp, i32, i64, dbl = C.c_void_p, C.c_int32, C.c_int64, C.c_double
    L.cn_last_error.restype = C.c_char_p
    L.cn_launch_count.restype = i64
    L.cn_policy_param_count.restype = i64
    L.cn_policy_param_count.argtypes = [C.POINTER(SarlCfg)]
    L.cn_env_cfg_default.argtypes = [C.POINTER(EnvCfg)]
    L.cn_env_cfg_default.restype = None
    L.cn_sarl_cfg_default.argtypes = [C.POINTER(SarlCfg)]
    L.cn_sarl_cfg_default.restype = None
    L.cn_env_create.argtypes = [C.POINTER(EnvCfg), C.c_int, C.POINTER(vp)]
    L.cn_env_destroy.argtypes = [vp]
    L.cn_env_set_state.argtypes = [vp, vp, vp, vp]
    L.cn_env_get_state.argtypes = [vp, vp, vp, vp]
    L.cn_env_set_theta.argtypes = [vp, vp, vp]
    L.cn_env_get_theta.argtypes = [vp, vp, vp]
    L.cn_env_reset.argtypes = [vp, vp]
    L.cn_env_orca.argtypes = [vp, vp]
    L.cn_env_robot_orca.argtypes = [vp, dbl, vp]
    L.cn_env_step.argtypes = [vp, vp, C.c_int, vp]
    L.cn_env_get_views.argtypes = [vp, C.POINTER(EnvViews)]
    L.cn_env_read_outputs.argtypes = [vp, vp, vp, vp, vp, vp]
    L.cn_env_read_human_actions.argtypes = [vp, vp, vp]
    L.cn_env_read_next_obs.argtypes = [vp, vp, vp]
    L.cn_env_set_actions.argtypes = [vp, vp, vp]
    L.cn_env_set_human_actions.argtypes = [vp, vp, vp]
    L.cn_env_read_actions.argtypes = [vp, vp, vp, vp]
    L.cn_env_read_stats.argtypes = [vp, C.POINTER(Stats), C.c_int, vp]
    L.cn_env_copy_outputs.argtypes = [vp, vp, vp, vp, vp]
    L.cn_env_episode_table_bytes.argtypes = [vp]
    L.cn_env_episode_table_bytes.restype = i64
    L.cn_env_read_episode_table.argtypes = [vp, vp, vp, vp]
    L.cn_policy_create.argtypes = [C.POINTER(SarlCfg), C.c_int, C.POINTER(vp)]
    L.cn_policy_destroy.argtypes = [vp]
    L.cn_policy_load_weights.argtypes = [vp, vp, i64, vp]
    L.cn_policy_action_table.argtypes = [vp, vp, C.POINTER(i32)]
    L.cn_policy_lookahead.argtypes = [vp, vp, C.c_int, dbl, vp]
    L.cn_policy_read.argtypes = [vp, vp, vp, vp, vp]
    L.cn_policy_bad_count.argtypes = [vp, C.POINTER(i64), C.c_int, vp]
    L.cn_policy_transform.argtypes = [vp, vp, vp, vp]
    L.cn_policy_last_state.argtypes = [vp, vp, vp, vp]
    L.cn_policy_forward.argtypes = [vp, vp, i32, i32, vp, vp]
    L.cn_rollout_step.argtypes = [vp, vp, C.c_int, dbl, vp]
    L.cn_rollout_step_sharded.argtypes = [vp, vp, C.c_int, dbl, vp]
    L.cn_rollout_episodes.argtypes = [vp, vp, vp, C.c_int, dbl, C.c_int, dbl, C.c_int32, C.c_int32, C.POINTER(RolloutRecord),
                                      C.POINTER(C.c_int32), vp]
    L.cn_rollout_step_host.argtypes = [vp, vp, C.c_int, dbl, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    L.cn_rollout_step_host_packed.argtypes = [vp, vp, C.c_int, dbl, vp, vp, vp]
    L.cn_rollout_step_host_packed_async.argtypes = [vp, vp, C.c_int, dbl, vp, vp, vp]
    L.cn_stream_sync.argtypes = [C.c_int, vp]
    L.cn_host_step_bytes.argtypes = [vp, C.c_int]
    L.cn_scenes_generate.argtypes = [i32, vp, i32, i32, dbl, dbl, dbl, dbl, dbl, dbl, dbl, i32, vp]
    L.cn_world_create.argtypes = [i32, i32, C.c_int, C.POINTER(vp)]
    L.cn_world_destroy.argtypes = [vp]
    L.cn_world_param_count.argtypes = [vp]
    L.cn_world_param_count.restype = i64
    L.cn_world_load_weights.argtypes = [vp, vp, i64, vp]
    L.cn_world_predict.argtypes = [vp, vp, vp]
    L.cn_world_load_weights_device.argtypes = [vp, vp, i64, vp]
    L.cn_env_copy_world_pairs.argtypes = [vp, vp, vp, vp, vp]
    f32 = C.c_float
    L.cn_world_trainer_create.argtypes = [i32, i32, C.c_int, i32, f32, C.POINTER(vp)]
    L.cn_world_trainer_destroy.argtypes = [vp]
    L.cn_world_trainer_param_count.argtypes = [vp]
    L.cn_world_trainer_param_count.restype = i64
    L.cn_world_trainer_sync_weights.argtypes = [vp, vp, C.c_int, vp]
    L.cn_world_trainer_step.argtypes = [vp, vp, vp, vp, vp, i32, i32, f32, f32, f32, f32, C.c_uint64, vp, vp, vp, vp]
    L.cn_world_trainer_apply.argtypes = [vp, vp, vp, f32, f32, f32, f32, f32, vp]
    L.cn_world_trainer_eval.argtypes = [vp, vp, vp, vp, i32, i32, vp, vp]
    L.cn_trainer_create.argtypes = [C.POINTER(SarlCfg), C.c_int, i32, i32, C.POINTER(vp)]
    L.cn_trainer_destroy.argtypes = [vp]
    L.cn_trainer_param_count.argtypes = [vp]
    L.cn_trainer_param_count.restype = i64
    L.cn_trainer_sync_weights.argtypes = [vp, vp, C.c_int, vp]
    L.cn_trainer_step.argtypes = [vp, vp, vp, vp, i32, i32, C.c_float, C.c_float, vp, vp, vp]
    L.cn_trainer_step_indexed.argtypes = [vp, vp, vp, vp, vp, i32, i32, C.c_float, C.c_float, vp, vp, vp]
    L.cn_trainer_apply.argtypes = [vp, vp, vp, C.c_float, C.c_float, C.c_float, vp]
    L.cn_debug_trace.argtypes = [C.c_int]
    L.cn_debug_trace_dump.argtypes = [C.c_char_p, i64]
    L.cn_host_step_bytes.restype = i64
    L.cn_selftest_umma.argtypes = [i32, i32, vp, vp, vp, C.c_int]
    L.cn_selftest_umma_bmn.argtypes = [i32, i32, vp, vp, vp, C.c_int]
    L.cn_selftest_umma_pair.argtypes = [i32, i32, vp, vp, vp, i32, vp, C.c_int]
    L.cn_selftest_umma_ts.argtypes = [i32, i32, vp, vp, vp, C.c_int]
    L.cn_debug_tc_timing.argtypes = [vp, vp]
    L.cn_debug_kernel_ms.argtypes = [vp, C.c_int, vp]
    _lib = L
    return L


def check(rc):
    if rc != CN_OK:
        raise CrowdNavError(rc, load().cn_last_error().decode())
    return rc


def default_env_cfg(**kw):
    cfg = EnvCfg()
    load().cn_env_cfg_default(C.byref(cfg))
    for k, v in kw.items():
        if not hasattr(cfg, k):
            raise AttributeError("cn_env_cfg has no field %r" % k)
        setattr(cfg, k, v)
    return cfg


def default_sarl_cfg(**kw):
    cfg = SarlCfg()
    load().cn_sarl_cfg_default(C.byref(cfg))
    for k, v in kw.items():
        if not hasattr(cfg, k):
            raise AttributeError("cn_sarl_cfg has no field %r" % k)
        if isinstance(v, (list, tuple)):
            arr = getattr(cfg, k)
            if len(v) != len(arr):
                raise ValueError("cn_sarl_cfg.%s holds %d values, got %d" % (k, len(arr), len(v)))
            for i, x in enumerate(v):
                arr[i] = x
        else:
            setattr(cfg, k, v)
    return cfg

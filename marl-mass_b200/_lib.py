"""ctypes binding of include/marl_mass_b200.h.

There is no CPU fallback: if the CUDA library is missing this module raises, and every env call goes
through it.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MM_LIB_PATH") or os.path.join(_HERE, "_build", "libmarl_mass_b200.so")

MAXV = 12
NS = 30
NA = 5

F64_FIELDS = ("x", "y", "heading", "speed", "target_speed", "gvx", "rec1_x", "rec1_vx", "rec2_x", "rec2_vx",
              "act_steer", "act_acc", "safe_steer", "safe_acc", "timer", "min_headway", "steering_angle")
I32_FIELDS = ("kind", "lane", "target_lane", "speed_index", "crashed", "hl_action", "hist_len", "fg_set",
              "is_collaborating", "is_lc_safe", "collaborate_adj")
ENV_FIELDS = ("n_veh", "n_cav", "n_merge", "steps", "time")
SH_I = ("ran", "leader", "front_adj", "rear_adj", "constrain_adj", "active", "is_lc_safe", "moved", "hl_action", "lane")
SH_F = ("safe_acc", "safe_steer", "nom_acc", "nom_steer", "lc_margin", "x", "y", "heading", "speed", "min_headway")

_PD = C.POINTER(C.c_double)
_PF = C.POINTER(C.c_float)
_PI = C.POINTER(C.c_int32)
_PU8 = C.POINTER(C.c_uint8)
_PI8 = C.POINTER(C.c_int8)


ABI_VERSION = 9           # MM_ABI_VERSION of the header this binding was written against


class MMConfig(C.Structure):
    """mm_config; struct_size is filled in by __init__ (the library's ABI guard checks it)."""
    _fields_ = [("struct_size", C.c_int32), ("shield", C.c_int32), ("reward_kind", C.c_int32), ("traffic_density", C.c_int32),
                ("traffic_type", C.c_int32), ("duration_steps", C.c_int32), ("substeps", C.c_int32),
                ("dt", C.c_double), ("eta", C.c_double), ("tau", C.c_double),
                ("collision_reward", C.c_double), ("high_speed_reward", C.c_double), ("headway_cost", C.c_double),
                ("headway_time", C.c_double), ("merging_lane_cost", C.c_double), ("env_v0", C.c_int32),
                ("steer_vel", C.c_int32), ("couple_counts", C.c_int32), ("env_hdv", C.c_int32), ("supervisor", C.c_int32)]


    def __init__(self, *args, **kw):
        super().__init__(*args, **kw)
        self.struct_size = C.sizeof(MMConfig)


class MMStateHost(C.Structure):
    _fields_ = [(k, _PD) for k in F64_FIELDS] + [(k, _PI) for k in I32_FIELDS] + [(k, _PI) for k in ENV_FIELDS]


class MMBuffers(C.Structure):
    _fields_ = [("obs", C.c_void_p), ("reward", C.c_void_p), ("done", C.c_void_p), ("agents_rewards", C.c_void_p),
                ("regional_rewards", C.c_void_p), ("agents_dones", C.c_void_p), ("average_speed", C.c_void_p),
                ("traffic_speed", C.c_void_p), ("min_headway", C.c_void_p), ("merge_percent", C.c_void_p),
                ("n_agents", C.c_void_p), ("actions", C.c_void_p), ("action_mask", C.c_void_p), ("new_actions", C.c_void_p)]


class MMPackedHost(C.Structure):
    _fields_ = [("veh", C.c_void_p), ("nbr", C.c_void_p), ("n_veh", C.c_void_p), ("n_agents", C.c_void_p),
                ("reward", C.c_void_p), ("done", C.c_void_p), ("regional_rewards", C.c_void_p)]


class MMShieldQueryOut(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in ("safe_steer", "safe_acc", "min_headway", "ran", "leader", "front_adj", "rear_adj",
                                          "constrain_adj", "active", "is_lc_safe")]


class MMShieldDiagHost(C.Structure):
    _fields_ = [(k, _PI) for k in SH_I] + [(k, _PD) for k in SH_F]


class MMStats(C.Structure):
    _fields_ = [(k, C.c_double) for k in ("agent_steps", "env_steps", "episodes", "crashed_episodes", "reward_sum",
                                          "speed_sum", "merge_percent_sum", "shield_solves", "shield_active",
                                          "lane_change_vetoes", "min_headway")]


class MMPpoNet(C.Structure):
    """mm_ppo_net: parameter pointers of one network of the on-device PPO learner"""
    _fields_ = [(k, C.c_void_p) for k in ("w1", "b1", "w2", "b2", "w3", "b3", "w4", "b4")]


class MMPpoGrads(C.Structure):
    """mm_ppo_grads_out: one gradient buffer per parameter, same layout"""
    _fields_ = [(k, C.c_void_p) for k in ("w1", "b1", "w2", "b2", "w3", "b3", "w4", "b4")]


PPO_ACTOR, PPO_CRITIC, PPO_SHARED = 0, 1, 2     # MM_PPO_ACTOR / _CRITIC / _SHARED
# MM_PPO_STAT_*: the fields of mm_ppo_stats' output vector, in order; PPO_STATS_LEN = MM_PPO_STATS_LEN
PPO_STAT_FIELDS = ("n", "entropy", "k3", "clipped", "ratio_min", "ratio_max", "v", "v2", "g", "g2", "res2")
PPO_STATS_LEN = len(PPO_STAT_FIELDS)
PPO_STAT = {k: i for i, k in enumerate(PPO_STAT_FIELDS)}


class MMOptTensor(C.Structure):
    """mm_opt_tensor: one parameter of an optimiser group (device pointers; mirror_cols is host memory)"""
    _fields_ = [("param", C.c_void_p), ("grad", C.c_void_p), ("square_avg", C.c_void_p), ("numel", C.c_int64),
                ("mirror", C.c_void_p), ("mirror_cols", _PI), ("mirror_ncols", C.c_int32), ("mirror_ld", C.c_int64)]


class MMOptGroup(C.Structure):
    """mm_opt_group: one network stepped by mm_rmsprop_step"""
    _fields_ = [("tensors", C.POINTER(MMOptTensor)), ("n_tensors", C.c_int32)] + \
               [(k, C.c_float) for k in ("lr", "alpha", "one_minus_alpha", "eps", "max_norm", "grad_scale")] + \
               [("total_norm", C.c_void_p)]


OPT_MAX_GROUPS, OPT_MAX_TENSORS = 8, 16     # MM_OPT_MAX_GROUPS / MM_OPT_MAX_TENSORS


class MMEvalRecords(C.Structure):
    """mm_eval_records: the evaluation's per-episode records (device pointers) and their step capacity T"""
    _fields_ = [("T", C.c_int32)] + [(k, C.c_void_p) for k in ("n_agents", "active", "rewards", "steps", "avg_speed_sum",
                                                              "traffic_speed_sum", "min_headway", "merge_percent", "crashed",
                                                              "vehicle_speed", "vehicle_position")]


PROFILE_I = ("moved", "ran", "active", "is_lc_safe", "hl_action", "lane")
PROFILE_F = ("x", "y", "heading", "speed", "min_headway", "safe_acc", "safe_steer", "nom_acc", "nom_steer")
SHIELD_COUNTS = ("shield_solves", "shield_active", "lane_change_vetoes", "shield_interventions")
SHIELD_F64 = ("acc_correction_sum", "acc_correction_max", "steer_correction_max", "min_agent_acc")


class MMEvalShieldRecords(C.Structure):
    """mm_eval_shield_records: per-episode shield records and optional control profiles (device pointers)"""
    _fields_ = [("T", C.c_int32)] + [(k, C.c_void_p) for k in ("n_agents", "active") + SHIELD_COUNTS + SHIELD_F64 +
                                     ("profile_slot",) + tuple("profile_" + f for f in PROFILE_I + PROFILE_F)]


class MMError(RuntimeError):
    pass


_lib = None

SUPERVISOR_DRAWS = 32     # MM_SUPERVISOR_DRAWS
EXPORTS = ("mm_create", "mm_destroy", "mm_set_config", "mm_num_envs", "mm_reset", "mm_step", "mm_step_host",
           "mm_step_host_ragged", "mm_step_host_packed", "mm_expand_obs_rows",
           "mm_buffers_get", "mm_get_state", "mm_set_state", "mm_get_shield_diag", "mm_stats", "mm_shield_qp", "mm_shield_query",
           "mm_actor_sample", "mm_actor_sample_mlp", "mm_set_actor_impl", "mm_set_step_variant", "mm_step_build", "mm_abi_version", "mm_discounted_returns", "mm_lambda_returns", "mm_ppo_targets", "mm_ppo_grads", "mm_ppo_stats", "mm_rmsprop_step", "mm_supervise", "mm_set_supervisor_draws", "mm_supervisor_draws_used",
           "mm_reset_seeded", "mm_check_seeds", "mm_eval_record", "mm_eval_shield_record", "mm_kernel_launches", "mm_last_error", "mm_version")


def lib():
    """Load libmarl_mass_b200.so (built by marl_mass_b200.build).  Raises if it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise MMError("CUDA library %s is missing; run `python -m marl_mass_b200.build` "
                      "(there is no CPU fallback)" % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    L.mm_abi_version.restype = C.c_int
    if L.mm_abi_version() != ABI_VERSION:
        raise MMError("%s was built with MM_ABI_VERSION %d, this binding expects %d: rebuild with "
                      "`python -m marl_mass_b200.build`" % (LIB_PATH, L.mm_abi_version(), ABI_VERSION))
    h = C.c_void_p
    L.mm_create.argtypes = [C.POINTER(MMConfig), C.c_int, C.c_int, C.c_int, C.POINTER(h)]
    L.mm_destroy.argtypes = [h]
    L.mm_set_config.argtypes = [h, C.POINTER(MMConfig)]
    L.mm_num_envs.argtypes = [h]
    L.mm_reset.argtypes = [h, C.c_uint64, C.c_void_p, C.c_int, C.c_void_p]
    L.mm_step.argtypes = [h, C.c_void_p, C.c_int, C.c_void_p]
    L.mm_reset_seeded.argtypes = [h, C.c_void_p, C.c_void_p, C.c_void_p]
    L.mm_check_seeds.argtypes = [C.POINTER(MMConfig), C.c_int, C.c_void_p, C.c_void_p]
    L.mm_eval_record.argtypes = [h, C.POINTER(MMEvalRecords), C.c_int, C.c_void_p]
    L.mm_eval_shield_record.argtypes = [h, C.POINTER(MMEvalShieldRecords), C.c_int, C.c_void_p]
    L.mm_step_host.argtypes = [h, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.mm_step_host_ragged.argtypes = [h, C.c_void_p, C.c_int] + [C.c_void_p] * 6
    L.mm_step_host_packed.argtypes = [h, C.c_void_p, C.c_int, C.POINTER(MMPackedHost)]
    L.mm_expand_obs_rows.argtypes = [C.POINTER(MMPackedHost), C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int]
    L.mm_buffers_get.argtypes = [h, C.POINTER(MMBuffers)]
    L.mm_get_state.argtypes = [h, C.POINTER(MMStateHost)]
    L.mm_set_state.argtypes = [h, C.POINTER(MMStateHost)]
    L.mm_get_shield_diag.argtypes = [h, C.POINTER(MMShieldDiagHost)]
    L.mm_stats.argtypes = [h, C.POINTER(MMStats), C.c_int]
    L.mm_shield_query.argtypes = [h, C.c_void_p, C.c_void_p, C.POINTER(MMShieldQueryOut), C.c_void_p]
    L.mm_shield_qp.argtypes = [C.c_void_p] * 6 + [C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]
    L.mm_actor_sample.argtypes = [C.c_void_p, C.c_void_p, C.c_int64] + [C.c_void_p] * 6 + [C.c_uint64, C.c_uint64] + \
                                 [C.c_void_p] * 5
    L.mm_actor_sample_mlp.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int] + [C.c_void_p] * 8 + [C.c_uint64, C.c_uint64] + \
                                     [C.c_void_p] * 8
    L.mm_set_actor_impl.argtypes = [C.c_int]
    L.mm_set_step_variant.argtypes = [C.c_int]
    L.mm_step_build.argtypes = [h]
    L.mm_discounted_returns.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_int, C.c_int64, C.c_int,
                                        C.c_void_p, C.c_void_p]
    L.mm_lambda_returns.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_float, C.c_int, C.c_int64,
                                    C.c_int, C.c_void_p, C.c_void_p]
    L.mm_ppo_targets.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(MMPpoNet), C.c_void_p,
                                 C.c_void_p, C.c_void_p]
    L.mm_ppo_grads.argtypes = [C.c_int] + [C.c_void_p] * 6 + [C.c_int64, C.c_float, C.POINTER(MMPpoNet), C.POINTER(MMPpoGrads),
                                                             C.c_void_p, C.c_void_p]
    L.mm_ppo_stats.argtypes = [C.c_int] + [C.c_void_p] * 5 + [C.c_int64, C.c_float, C.POINTER(MMPpoNet), C.c_void_p, C.c_void_p]
    L.mm_rmsprop_step.argtypes = [C.POINTER(MMOptGroup), C.c_int, C.c_void_p]
    L.mm_kernel_launches.argtypes = [h]
    L.mm_kernel_launches.restype = C.c_int64
    L.mm_last_error.restype = C.c_char_p
    L.mm_version.restype = C.c_char_p
    L.mm_supervise.argtypes = [h, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.mm_set_supervisor_draws.argtypes = [h, C.c_void_p]
    L.mm_supervisor_draws_used.argtypes = [h, C.c_void_p]
    for name in EXPORTS:
        if name not in ("mm_kernel_launches", "mm_last_error", "mm_version"):
            getattr(L, name).restype = C.c_int
    _lib = L
    return L


def check(rc):
    if rc != 0:
        raise MMError("marl_mass_b200: %s (status %d)" % (lib().mm_last_error().decode(), rc))

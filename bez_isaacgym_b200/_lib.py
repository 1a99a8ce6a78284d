"""ctypes binding of libbezk.so (C ABI in ``include/bezk.h``).

The library is the product: if it is missing or fails to load this module raises -- there is no
Python / torch / CPU fallback for any op.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("BEZK_LIB", os.path.join(_HERE, "libbezk.so"))     # BEZK_LIB: A/B builds of the same library

NUM_DOF = 18

F_CLEATS = 1
F_WRITE_CONTACT_FILTER = 2
F_RESET_ROOT_STATES = 4
F_OBS_STREAMED = 8

PART_BOOKKEEP = 1
PART_OBS = 2
PART_REWARD = 4
PART_ALL = 7

TASK_KICK, TASK_WALK, TASK_ORIENT = 0, 1, 2


class BezkTaskCfg(C.Structure):
    _fields_ = [
        ("num_bodies", C.c_int32), ("imu_body", C.c_int32), ("left_foot_body", C.c_int32),
        ("right_foot_body", C.c_int32), ("max_episode_length", C.c_int32), ("flags", C.c_uint32),
        ("dt", C.c_float), ("imu_max_lin_acc", C.c_float), ("imu_max_ang_vel", C.c_float),
        ("clip_obs", C.c_float), ("clip_actions", C.c_float), ("bez_init_xy", C.c_float * 2),
        ("reset_pos_lo", C.c_float), ("reset_pos_span", C.c_float),
        ("reset_vel_lo", C.c_float), ("reset_vel_span", C.c_float),
        ("default_dof_pos", C.c_float * NUM_DOF), ("dof_lower", C.c_float * NUM_DOF),
        ("dof_upper", C.c_float * NUM_DOF),
    ]


class BezkNoiseCfg(C.Structure):
    _fields_ = [("distribution", C.c_int32), ("operation", C.c_int32), ("a", C.c_float), ("b", C.c_float),
                ("a_corr", C.c_float), ("b_corr", C.c_float)]


class BezkRolloutCfg(C.Structure):
    _fields_ = [("scale_value", C.c_float), ("shift_value", C.c_float), ("gamma", C.c_float), ("value_bootstrap", C.c_int32)]


class BezkPpoCfg(C.Structure):
    _fields_ = [
        ("e_clip", C.c_float), ("critic_coef", C.c_float), ("entropy_coef", C.c_float),
        ("bounds_loss_coef", C.c_float), ("soft_bound", C.c_float), ("clip_value", C.c_int32),
        ("bound_form", C.c_int32),
    ]


_P = C.c_void_p
_I64 = C.c_int64
_U64 = C.c_uint64

#: name -> (restype, argtypes); mirrors include/bezk.h one to one
SIGNATURES = {
    "bezk_version": (C.c_int, []),
    "bezk_last_error": (C.c_char_p, []),
    "bezk_set_l2_fetch_granularity": (C.c_int, [C.c_int32, C.POINTER(C.c_int32)]),
    "bezk_pre_physics": (C.c_int, [_P, _P, _P, C.POINTER(BezkTaskCfg), _I64, _P]),
    "bezk_compute_observations": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, C.POINTER(BezkTaskCfg), _P, _P, _I64, _P]),
    "bezk_compute_reward": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, C.POINTER(BezkTaskCfg), _P, _P, _I64, _P]),
    "bezk_reset_idx": (C.c_int, [_P, _I64, _P, _U64, _U64, _P, _P, _P, _P, _P, C.POINTER(BezkTaskCfg), _I64, _P]),
    "bezk_post_physics": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _U64, _U64, _P, _P, _P, _P,
                                    C.POINTER(BezkTaskCfg), _P, _P, _P, C.c_int, _I64, _P]),
    "bezk_post_physics_chunk": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _U64, _U64, _P, _P, _P, _P,
                                          C.POINTER(BezkTaskCfg), _P, _P, _P, C.c_int, _I64, _I64, _P, _P, _P]),
    "bezk_stage_sparse_rows": (C.c_int, [_P, _P, C.POINTER(BezkTaskCfg), _P, _P, _I64, _I64, _P]),
    "bezk_stage_sparse_rows_split": (C.c_int, [_P, _P, C.POINTER(BezkTaskCfg), _P, _P, _I64, _I64, _P, _P]),
    "bezk_host_pack_config": (C.c_int, [C.c_int32, C.c_int32, C.c_int32]),
    "bezk_host_pack_record_floats": (C.c_int, [C.c_int, C.POINTER(BezkTaskCfg)]),
    "bezk_host_pack_begin": (_I64, [C.c_int, _P, _P, _P, _P, _P, C.POINTER(BezkTaskCfg), _P, _I64, _I64]),
    "bezk_post_physics_packed": (C.c_int, [C.c_int, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _U64, _U64, _P, _P, _P, _P,
                                           C.POINTER(BezkTaskCfg), _P, _P, _P, C.c_int, _I64, _I64, _P, _P,
                                           C.POINTER(BezkRolloutCfg), _P, _P, _P, _P]),
    "bezk_host_pack_wait": (C.c_int, [_I64]),
    "bezk_post_physics_staged": (C.c_int, [C.c_int, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _U64, _U64, _P, _P, _P, _P,
                                           C.POINTER(BezkTaskCfg), _P, _P, _P, C.c_int, _I64, _I64, _P, _P,
                                           C.POINTER(BezkRolloutCfg), _P, _P, _P, _P]),
    "bezk_philox_uniforms": (C.c_int, [_U64, _U64, _P, _I64, _P]),
    "bezk_gae": (C.c_int, [_P, _P, _P, _P, _P, C.c_int, C.c_double, C.c_double, _P, _P, C.c_int32, _I64, _P]),
    "bezk_rms_scratch_doubles": (_I64, [C.c_int32]),
    "bezk_rms_moments": (C.c_int, [_P, _P, _P, _P, _I64, C.c_int32, _P]),
    "bezk_rms_merge": (C.c_int, [_P, _P, _P, _P, _P, C.c_int32, _P]),
    "bezk_rms_moments_slabs_batched": (C.c_int, [_P, _I64, _I64, _I64, _P, _P, _P, _I64, C.c_int32, C.c_int32, _P]),
    "bezk_rms_merge_sequence": (C.c_int, [_P, C.c_int32, _P, C.c_int32, _P, _P, _P, _P, _P, C.c_int32, _P]),
    "bezk_rms_normalize": (C.c_int, [_P, _P, _P, C.c_float, C.c_int, _P, _I64, C.c_int32, _P]),
    "bezk_rms_train_forward": (C.c_int, [_P, _I64, _I64, _P, _P, _P, C.c_float, _P, _P, _I64, C.c_int32, _P]),
    "bezk_rms_moments_ext": (C.c_int, [_P, _I64, _I64, _P, _P, _P, _P, _P, _I64, C.c_int32, _P]),
    "bezk_rms_merge_normalize": (C.c_int, [_P, _I64, _I64, _P, _P, _P, _P, C.c_float, _P, _I64, C.c_int32, _P]),
    "bezk_adv_normalize_fused": (C.c_int, [_P, _P, _P, _P, C.c_int, _I64, _P]),
    "bezk_adv_moments": (C.c_int, [_P, _P, _P, _P, _I64, _P]),
    "bezk_adv_normalize": (C.c_int, [_P, _P, _P, _P, C.c_int, _I64, _P]),
    "bezk_ppo_scratch_doubles": (_I64, []),
    "bezk_ppo_loss": (C.c_int, [_P] * 10 + [C.POINTER(BezkPpoCfg)] + [_P] * 6 + [_I64, _P]),
    "bezk_post_physics_task": (C.c_int, [C.c_int, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _U64, _U64, _P, _P, _P, _P,
                                         C.POINTER(BezkTaskCfg), _P, _P, _P, C.c_int, _I64, _P]),
    "bezk_post_physics_rollout": (C.c_int, [C.c_int, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _U64, _U64, _P, _P, _P, _P,
                                            C.POINTER(BezkTaskCfg), _P, _P, _P, C.POINTER(BezkRolloutCfg), _P, _P, _P, _I64, _I64, _P]),
    "bezk_post_physics_rollout_ep": (C.c_int, [C.c_int, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _U64, _U64, _P, _P, _P, _P,
                                               C.POINTER(BezkTaskCfg), _P, _P, _P, C.POINTER(BezkRolloutCfg), _P, _P, _P, _I64, _I64,
                                               _P, _P, _P, _P]),
    "bezk_episode_meter_update": (C.c_int, [_P, C.c_int, _I64, _I64, _P, _P, _P]),
    "bezk_post_physics_rollout_ep_norm": (C.c_int, [C.c_int, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _U64, _U64, _P, _P, _P, _P,
                                                    C.POINTER(BezkTaskCfg), _P, _P, _P, C.POINTER(BezkRolloutCfg), _P, _P, _P, _I64,
                                                    _I64, _P, _P, _P, _P, _P, C.c_float, _P, _P]),
    "bezk_player_tally_update": (C.c_int, [_P, C.c_int, _I64, _I64, _P, _P, _P]),
    "bezk_outcome_classes": (C.c_int, [C.c_int]),
    "bezk_post_physics_rollout_ep_outcome": (C.c_int, [C.c_int, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _U64, _U64, _P, _P, _P,
                                                       _P, C.POINTER(BezkTaskCfg), _P, _P, _P, C.POINTER(BezkRolloutCfg), _P, _P, _P,
                                                       _I64, _I64, _P, _P, _P, _P, _P, C.c_float, _P, _P, _P]),
    "bezk_outcome_meter_update": (C.c_int, [_P, C.c_int, _I64, C.c_int, _I64, _P, _P, _P]),
    "bezk_player_outcome_update": (C.c_int, [_P, C.c_int, _I64, C.c_int, _I64, _P, _P, _P]),
    "bezk_reward_terms": (C.c_int, [C.c_int]),
    "bezk_post_physics_rollout_ep_terms": (C.c_int, [C.c_int, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _U64, _U64, _P, _P, _P,
                                                     _P, C.POINTER(BezkTaskCfg), _P, _P, _P, C.POINTER(BezkRolloutCfg), _P, _P, _P,
                                                     _I64, _I64, _P, _P, _P, _P, _P, C.c_float, _P, _P, _P, _P]),
    "bezk_reward_terms_update": (C.c_int, [_P, C.c_int, _I64, C.c_int, _P, _P]),
    "bezk_post_physics_rollout_ep_game_terms": (C.c_int, [C.c_int, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _U64, _U64, _P, _P, _P,
                                                          _P, C.POINTER(BezkTaskCfg), _P, _P, _P, C.POINTER(BezkRolloutCfg), _P, _P,
                                                          _P, _I64, _I64, _P, _P, _P, _P, _P, C.c_float, _P, _P, _P, _P, _P, _P]),
    "bezk_game_terms_meter_update": (C.c_int, [_P, _P, C.c_int, _I64, C.c_int, _I64, _P, _P, _P]),
    "bezk_player_game_terms_update": (C.c_int, [_P, _P, C.c_int, _I64, C.c_int, _I64, _P, _P, _P]),
    "bezk_reset_idx_task": (C.c_int, [C.c_int, _P, _I64, _P, _P, _U64, _U64, _P, _P, _P, _P, _P, _P, C.POINTER(BezkTaskCfg), _I64, _I64,
                                      _P]),
    "bezk_goal_uniforms": (C.c_int, [_U64, _U64, _P, _P]),
    "bezk_l2_release": (C.c_int, [_P, _U64, _P]),
    "bezk_rms_moments_slabs": (C.c_int, [_P, _I64, _I64, _P, _P, _P, _I64, C.c_int32, _P]),
    "bezk_rms_normalize_slabs_batched": (C.c_int, [_P, _I64, _I64, _I64, _P, _P, _I64, C.c_float, _P, _I64, C.c_int32, C.c_int32, _P]),
    "bezk_rms_normalize_slabs": (C.c_int, [_P, _I64, _I64, _P, _P, C.c_float, C.c_int, _P, _I64, C.c_int32, _P]),
    "bezk_ppo_loss_slabs": (C.c_int, [_P] * 10 + [_I64, _I64, C.POINTER(BezkPpoCfg)] + [_P] * 6 + [_I64, _P]),
    "bezk_swap_and_flatten01": (C.c_int, [_P, _P, C.c_int32, _I64, _I64, _I64, C.c_int32, _P]),
    "bezk_policy_head": (C.c_int, [_P, _P, _P, _P, _P, C.c_float, _P, _U64, _U64, _P, _P, _P, _P, _P,
                                   C.POINTER(BezkTaskCfg), _P, _P, _I64, _I64, _P]),
    "bezk_normal_noise": (C.c_int, [_U64, _U64, _P, _I64, _I64, _P]),
    "bezk_dr_noise": (C.c_int, [_P, _P, _P, _U64, _U64, C.POINTER(BezkNoiseCfg), _P, _I64, _P]),
    "bezk_dr_noise_clip": (C.c_int, [_P, _P, _P, _U64, _U64, C.POINTER(BezkNoiseCfg), _P, _P, C.c_float, _I64, _P]),
    "bezk_quat_rotate": (C.c_int, [_P, _P, _P, C.c_int, _I64, _P]),
    "bezk_scale_transform": (C.c_int, [_P, _P, _P, _P, C.c_int, _I64, C.c_int32, _P]),
    "bezk_selftest_fastmath": (C.c_int, [_U64, _U64, _P, _P]),
    "bezk_dr_fill": (C.c_int, [_U64, _U64, C.c_int32, _P, _I64, _P]),
}

_lib = None


class BezkError(RuntimeError):
    pass


def load():
    """Load libbezk.so (once).  Raises if the CUDA extension has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise BezkError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C bez_isaacgym_b200/csrc`).  bez_isaacgym_b200 has no CPU / torch fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if a declared symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc, what=""):
    if rc != 0:
        msg = load().bezk_last_error().decode("utf-8", "replace")
        raise BezkError(f"{what or 'bezk call'} failed with code {rc}: {msg}")

"""ctypes binding of libodgsim.so — exactly the entry points include/odg.h declares.

The library is CUDA-only. If it is missing or no CUDA device is present this module raises; there is
no CPU or PyTorch fallback anywhere in the package.
"""
from __future__ import annotations

import ctypes as C
import os

from .model.compile import OdgModel

PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("ODG_LIB_PATH") or os.path.join(PKG, "libodgsim.so")   # override: tuning variants

# every symbol include/odg.h declares (tests check the .so exports all of them)
SYMBOLS = [
    "odg_default_config", "odg_create", "odg_destroy", "odg_num_envs", "odg_obs_dim", "odg_act_dim",
    "odg_nq", "odg_nv", "odg_reset", "odg_step", "odg_evaluate", "odg_get_state", "odg_set_state",
    "odg_get_env_state", "odg_set_env_state", "odg_launch_count", "odg_last_error", "odg_version", "odg_set_frame_skip",
    "odg_step_host",
    # rollout / policy entry points (include/odg_policy.h)
    "odg_policy_create", "odg_policy_create_hidden", "odg_policy_destroy", "odg_policy_load", "odg_policy_forward", "odg_gae",
    "odg_normalize_advantages", "odg_policy_launch_count", "odg_tanh_backward_bias", "odg_tanh_backward_bias_scratch_floats",
    "odg_ppo_loss", "odg_ppo_loss_scratch_floats", "odg_tanh_bf16",
    # QuadrupedEnv surface (include/odg_sim2real.h)
    "odg_s2r_default_config", "odg_s2r_create", "odg_s2r_destroy", "odg_s2r_reset", "odg_s2r_step",
    "odg_s2r_set_bookkeeping", "odg_s2r_default_config_for", "odg_s2r_obs_dim", "odg_s2r_act_dim",
    # the terrain trainer's height fields (include/odg_sim2real.h)
    "odg_terrain_create", "odg_terrain_destroy", "odg_terrain_generate", "odg_terrain_from_raw", "odg_terrain_height",
    "odg_terrain_data",
    # MPPI (include/odg_mppi.h)
    "odg_mppi_sample", "odg_mppi_accumulate", "odg_mppi_reduce", "odg_mppi_rollout",
    "odg_mppi_broadcast", "odg_mppi_rollout_groups", "odg_mppi_reduce_groups",
]


class OdgEnvConfig(C.Structure):
    _fields_ = [("task", C.c_int), ("frame_skip", C.c_int), ("max_episode_steps", C.c_int),
                ("auto_reset", C.c_int), ("solver_iterations", C.c_int), ("ls_iterations", C.c_int),
                ("solver_tolerance", C.c_float), ("ls_tolerance", C.c_float), ("reset_noise_scale", C.c_float),
                ("scale_actions", C.c_int), ("launch_lanes", C.c_int), ("first_env_id", C.c_int), ("obs_layout", C.c_int),
                ("launch_block", C.c_int), ("launch_lockstep", C.c_int), ("launch_fat", C.c_int)]


_vp = C.c_void_p


class OdgInfoPtrs(C.Structure):
    _fields_ = [(n, _vp) for n in (
        "x_position", "y_position", "distance_from_origin", "paw_contact_forces", "patterns_matches",
        "linear_vel_tracking_reward", "reward_ctrl", "terminal_obs", "paws_in_ground", "gait_reward",
        "qacc", "ncon", "contact_normal_force", "solver_iters", "ls_evals", "reward_unclipped", "cfrc_ext", "task_terms")]


class OdgPolicyWeights(C.Structure):
    _fields_ = [("actor_w", _vp * 3), ("actor_b", _vp * 3), ("critic_w", _vp * 3), ("critic_b", _vp * 3),
                ("action_log_std", _vp)]


class OdgS2RConfig(C.Structure):
    _fields_ = [("action_amplitude_rad", C.c_double), ("settle_steps", C.c_int), ("auto_reset", C.c_int),
                ("real_home_deg", C.c_double * 8), ("joint_scale", C.c_double * 8), ("max_steps", C.c_int), ("variant", C.c_int)]


class OdgError(RuntimeError):
    pass


_lib = None


def load():
    """Load libodgsim.so (building it with nvcc if the sources are newer). Raises if impossible."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        from . import build as _build
        _build.build()
    L = C.CDLL(LIB_PATH)
    L.odg_default_config.argtypes = [C.POINTER(OdgEnvConfig)]
    L.odg_default_config.restype = None
    L.odg_create.argtypes = [C.POINTER(OdgModel), C.POINTER(OdgEnvConfig), C.c_int, C.c_int, C.c_uint64,
                             C.POINTER(_vp)]
    L.odg_destroy.argtypes = [_vp]
    L.odg_destroy.restype = None
    for n in ("odg_num_envs", "odg_obs_dim", "odg_act_dim", "odg_nq", "odg_nv"):
        getattr(L, n).argtypes = [_vp]
    L.odg_launch_count.argtypes = [_vp]
    L.odg_set_frame_skip.argtypes = [_vp, C.c_int]
    L.odg_launch_count.restype = C.c_longlong
    L.odg_reset.argtypes = [_vp, _vp, _vp, _vp]
    L.odg_step.argtypes = [_vp, _vp, _vp, _vp, _vp, _vp, C.POINTER(OdgInfoPtrs), _vp]
    L.odg_step_host.argtypes = [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, C.POINTER(OdgInfoPtrs), _vp, _vp, C.c_size_t, _vp]
    L.odg_evaluate.argtypes = [_vp, _vp, _vp, _vp, _vp, _vp, C.POINTER(OdgInfoPtrs), _vp]
    L.odg_get_state.argtypes = [_vp, _vp, _vp, _vp]
    L.odg_set_state.argtypes = [_vp, _vp, _vp, _vp, _vp]
    L.odg_get_env_state.argtypes = [_vp] * 8
    L.odg_set_env_state.argtypes = [_vp] * 8
    L.odg_policy_create.argtypes = [C.c_int, C.c_int, C.c_int, C.POINTER(_vp)]
    L.odg_policy_create_hidden.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(_vp)]
    L.odg_policy_destroy.argtypes = [_vp]
    L.odg_policy_destroy.restype = None
    L.odg_policy_load.argtypes = [_vp, C.POINTER(OdgPolicyWeights), _vp]
    L.odg_policy_forward.argtypes = [_vp, _vp, C.c_int, _vp, _vp, _vp, _vp, C.c_uint64, C.c_uint32, _vp, C.c_int, _vp]
    L.odg_gae.argtypes = [_vp, _vp, _vp, C.c_int, C.c_int, C.c_float, C.c_float, _vp, _vp, _vp, _vp]
    L.odg_normalize_advantages.argtypes = [_vp, C.c_longlong, _vp, _vp]
    L.odg_tanh_backward_bias.argtypes = [_vp, _vp, _vp, _vp, _vp, C.c_longlong, C.c_int, _vp]
    L.odg_tanh_backward_bias_scratch_floats.argtypes = [C.c_int]
    L.odg_ppo_loss_scratch_floats.argtypes = []
    L.odg_tanh_bf16.argtypes = [_vp, _vp, C.c_longlong, _vp]
    L.odg_ppo_loss.argtypes = [_vp] * 7 + [C.c_longlong, C.c_int, C.c_float, C.c_float, C.c_float] + [_vp] * 7
    L.odg_policy_launch_count.argtypes = [_vp]
    L.odg_policy_launch_count.restype = C.c_longlong
    L.odg_s2r_default_config.argtypes = [C.POINTER(OdgS2RConfig)]
    L.odg_s2r_default_config.restype = None
    L.odg_s2r_create.argtypes = [_vp, C.POINTER(OdgModel), C.POINTER(OdgS2RConfig), C.POINTER(_vp)]
    L.odg_s2r_destroy.argtypes = [_vp]
    L.odg_s2r_destroy.restype = None
    L.odg_s2r_reset.argtypes = [_vp, _vp, _vp, _vp]
    L.odg_s2r_step.argtypes = [_vp] * 9
    L.odg_s2r_set_bookkeeping.argtypes = [_vp] * 8
    L.odg_s2r_default_config_for.argtypes = [C.POINTER(OdgS2RConfig), C.c_int]
    L.odg_s2r_default_config_for.restype = None
    L.odg_s2r_obs_dim.argtypes = [_vp]
    L.odg_s2r_act_dim.argtypes = [_vp]
    L.odg_terrain_create.argtypes = [C.c_int, C.c_int, C.c_uint64, C.c_int, C.POINTER(_vp)]
    L.odg_terrain_destroy.argtypes = [_vp]
    L.odg_terrain_destroy.restype = None
    L.odg_terrain_generate.argtypes = [_vp, _vp, _vp]
    L.odg_terrain_from_raw.argtypes = [_vp, _vp, _vp, _vp]
    L.odg_terrain_height.argtypes = [_vp, _vp, _vp, _vp]
    L.odg_terrain_data.argtypes = [_vp]
    L.odg_terrain_data.restype = _vp
    L.odg_mppi_sample.argtypes = [_vp, C.c_float, C.c_int, C.c_int, C.c_uint64, C.c_uint32, C.c_uint32, _vp, _vp]
    L.odg_mppi_accumulate.argtypes = [_vp, _vp, C.c_int, C.c_float, _vp, _vp, _vp]
    L.odg_mppi_rollout.argtypes = [_vp, _vp, C.c_float, C.c_int, C.c_uint64, C.c_uint32, _vp, C.c_float, _vp, _vp, _vp]
    L.odg_mppi_reduce.argtypes = [_vp, _vp, C.c_int, C.c_int, C.c_int, C.c_float, _vp, _vp, _vp]
    L.odg_mppi_broadcast.argtypes = [_vp, _vp, C.c_int, C.c_int, _vp]
    L.odg_mppi_rollout_groups.argtypes = [_vp, C.c_int, _vp, C.c_float, C.c_int, C.c_uint64, C.c_uint32, _vp, C.c_float, _vp, _vp,
                                          _vp]
    L.odg_mppi_reduce_groups.argtypes = [_vp, _vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, _vp, _vp, _vp]
    L.odg_last_error.restype = C.c_char_p
    L.odg_version.restype = C.c_char_p
    _lib = L
    return L


def check(rc: int, what: str):
    if rc != 0:
        raise OdgError(f"{what} failed ({rc}): {load().odg_last_error().decode()}")

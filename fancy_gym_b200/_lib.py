"""ctypes binding of the C-ABI library (include/fancy_gym_b200.h).

There is deliberately NO fallback: if the CUDA library has not been built, importing this module
raises, and so does every product entry point that needs it.
"""
from __future__ import annotations

import ctypes as C
import os

FG_MAX_DOF = 8
FG_MAX_OBS = 40
FG_MAX_PLANS = 32
# link counts the reacher rollout (fg_dispatch.cu) and env-step (fg_env_step.cu) kernels are instantiated for; resets and
# stand-alone trajectories take 1..FG_MAX_DOF
STEP_LINKS = range(2, 8)

# enums (include/fancy_gym_b200.h)
ENV_HOLE_REACHER, ENV_VIAPOINT_REACHER, ENV_SIMPLE_REACHER, ENV_TOY = 0, 1, 2, 3
MP_PROMP, MP_DMP, MP_PRODMP, MP_TRAJ = 0, 1, 2, 3
CTRL_VELOCITY, CTRL_POSITION, CTRL_MOTOR = 0, 1, 2
FLAG_TERMINATED, FLAG_TRUNCATED, FLAG_SUCCESS, FLAG_COLLIDED = 1, 2, 4, 8
OK, ERR_INVALID, ERR_UNSUPPORTED, ERR_CUDA, ERR_NOMEM = 0, -1, -2, -3, -4


class FgConfig(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32),
        ("env_kind", C.c_int32), ("mp_kind", C.c_int32), ("ctrl_kind", C.c_int32),
        ("n_dof", C.c_int32), ("n_steps", C.c_int32), ("n_basis", C.c_int32),
        ("max_episode_steps", C.c_int32),
        ("dt", C.c_double),
        ("p_gains", C.c_double * FG_MAX_DOF), ("d_gains", C.c_double * FG_MAX_DOF),
        ("tau", C.c_float), ("dmp_alpha", C.c_float), ("weights_scale", C.c_float), ("goal_scale", C.c_float),
        ("relative_goal", C.c_int32),
        ("allow_self_collision", C.c_int32), ("allow_wall_collision", C.c_int32),
        ("collision_penalty", C.c_double),
        ("rew_fct", C.c_int32), ("wall_mode", C.c_int32), ("time_aware", C.c_int32),
        ("n_obs_out", C.c_int32), ("obs_index", C.c_int32 * FG_MAX_OBS),
        ("tab_a", C.c_void_p), ("tab_b", C.c_void_p),
    ]


class FgRolloutIO(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32),
        ("params", C.c_void_p), ("ctx", C.c_void_p), ("traj_pos", C.c_void_p), ("traj_vel", C.c_void_p),
        ("q", C.c_void_p), ("v", C.c_void_p), ("steps", C.c_void_p), ("done", C.c_void_p),
        ("cond_pos", C.c_void_p), ("cond_vel", C.c_void_p),
        ("use_cond", C.c_int32), ("write_cond", C.c_int32),
        ("ret", C.c_void_p), ("length", C.c_void_p), ("flags", C.c_void_p), ("obs", C.c_void_p), ("info", C.c_void_p),
        ("dbg_actions", C.c_void_p), ("dbg_obs", C.c_void_p), ("dbg_rewards", C.c_void_p), ("flag_bytes", C.c_void_p), ("seg_steps_env", C.c_void_p), ("prev_obs", C.c_void_p), ("prev_info", C.c_void_p), ("keep_state", C.c_int32),
        ("n_plans", C.c_int32), ("plan_T", C.c_int32), ("plan_seg", C.c_int32 * FG_MAX_PLANS), ("plan_row0", C.c_int32 * FG_MAX_PLANS),
        ("dbg_state", C.c_void_p), ("peer_bufs", C.c_void_p), ("n_peers", C.c_int32), ("peer_offset", C.c_int64),
        ("phase", C.c_void_p), ("phase_tau", C.c_void_p), ("phase_delay", C.c_void_p), ("phase_times", C.c_void_p),
    ]


class FgResetCfg(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32),
        ("env_kind", C.c_int32), ("n_dof", C.c_int32), ("random_start", C.c_int32), ("time_aware", C.c_int32),
        ("device", C.c_int32),
        ("fixed", C.c_double * 4), ("has_fixed", C.c_int32 * 4),
        ("n_obs_out", C.c_int32), ("obs_index", C.c_int32 * FG_MAX_OBS),
    ]


class FgResetIO(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32),
        ("seeds", C.c_void_p), ("seed0", C.c_int64), ("reseed", C.c_int32), ("rng_state", C.c_void_p), ("mask", C.c_void_p),
        ("q", C.c_void_p), ("v", C.c_void_p), ("steps", C.c_void_p), ("done", C.c_void_p), ("ctx", C.c_void_p),
        ("obs", C.c_void_p),
    ]


class FgEnvStepCfg(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32),
        ("env_kind", C.c_int32), ("n_dof", C.c_int32), ("max_episode_steps", C.c_int32), ("dt", C.c_double),
        ("allow_self_collision", C.c_int32), ("allow_wall_collision", C.c_int32), ("collision_penalty", C.c_double),
        ("rew_fct", C.c_int32), ("action_f64", C.c_int32),
    ]


class FgEnvStepIO(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32),
        ("action", C.c_void_p), ("v_is_f32", C.c_int32),
        ("q", C.c_void_p), ("v", C.c_void_p), ("steps", C.c_void_p), ("done", C.c_void_p), ("ctx", C.c_void_p),
        ("latch", C.c_void_p),
        ("obs", C.c_void_p), ("reward", C.c_void_p), ("flag_bytes", C.c_void_p), ("info", C.c_void_p),
    ]


class FgPhaseBasis(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32), ("phase_kind", C.c_int32), ("alpha_phase", C.c_double),
        ("n_basis_total", C.c_int32), ("first_learnable", C.c_int32),
        ("centers", C.c_double * 16), ("bandwidth", C.c_double * 16),
        ("pc_pos", C.c_void_p), ("pc_vel", C.c_void_p), ("pc_y", C.c_void_p), ("n_pc", C.c_int32),
        ("scaled_dt", C.c_float), ("init_time", C.c_float), ("scale", C.c_double * 17),
        ("n_steps_env", C.c_void_p), ("times_table", C.c_void_p), ("times_stride", C.c_int32),
        ("exp_right_clip", C.c_int32), ("basis_scale", C.c_double), ("eval_f64", C.c_int32),
    ]


# every symbol include/fancy_gym_b200.h declares (tests check the library exports all of them)
EXPORTED_SYMBOLS = [
    "fg_last_error", "fg_abi_version", "fg_create", "fg_destroy", "fg_num_params", "fg_obs_full_dim",
    "fg_rollout", "fg_trajgen", "fg_trajgen_phase", "fg_reset", "fg_env_step", "fg_traj_cov", "fg_traj_cov_work_floats", "fg_ffma_probe",
]

LIB_PATH = os.environ.get("FG_LIB_PATH") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "lib", "libfancygym_b200.so")


class LibraryMissingError(ImportError):
    pass


def _load():
    if not os.path.exists(LIB_PATH):
        raise LibraryMissingError(
            f"{LIB_PATH} not found: build it with `make` (or `python -c 'import __graft_entry__ as g; g.build()'`). "
            "fancy_gym_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    lib.fg_last_error.restype = C.c_char_p
    lib.fg_abi_version.restype = C.c_int32
    lib.fg_create.argtypes = [C.POINTER(FgConfig), C.c_int32, C.POINTER(C.c_void_p)]
    lib.fg_create.restype = C.c_int
    lib.fg_destroy.argtypes = [C.c_void_p]
    lib.fg_destroy.restype = C.c_int
    lib.fg_num_params.argtypes = [C.c_void_p]
    lib.fg_num_params.restype = C.c_int32
    lib.fg_obs_full_dim.argtypes = [C.c_void_p]
    lib.fg_obs_full_dim.restype = C.c_int32
    lib.fg_rollout.argtypes = [C.c_void_p, C.POINTER(FgRolloutIO), C.c_int64, C.c_int32, C.c_void_p]
    lib.fg_rollout.restype = C.c_int
    lib.fg_trajgen.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                               C.c_void_p]
    lib.fg_trajgen.restype = C.c_int
    lib.fg_trajgen_phase.argtypes = [C.c_void_p, C.POINTER(FgPhaseBasis)] + [C.c_void_p] * 8 + [C.c_int64, C.c_void_p]
    lib.fg_trajgen_phase.restype = C.c_int
    lib.fg_traj_cov_work_floats.argtypes = [C.c_void_p, C.c_int64]
    lib.fg_traj_cov_work_floats.restype = C.c_int64
    lib.fg_traj_cov.argtypes = [C.c_void_p, C.c_void_p, C.c_float, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                C.c_int64, C.c_void_p]
    lib.fg_traj_cov.restype = C.c_int
    lib.fg_reset.argtypes = [C.POINTER(FgResetCfg), C.POINTER(FgResetIO), C.c_int64, C.c_void_p]
    lib.fg_reset.restype = C.c_int
    lib.fg_env_step.argtypes = [C.POINTER(FgEnvStepCfg), C.POINTER(FgEnvStepIO), C.c_int64, C.c_void_p]
    lib.fg_env_step.restype = C.c_int
    lib.fg_ffma_probe.argtypes = [C.c_int32, C.c_int32, C.c_void_p, C.POINTER(C.c_double), C.c_void_p]
    lib.fg_ffma_probe.restype = C.c_int
    return lib


lib = _load()
assert lib.fg_abi_version() == 2, "ABI version mismatch between fancy_gym_b200/_lib.py and the shared library"


def check_step_links(env_kind: int, n_links: int):
    """Refuses a step of a reacher whose link count has no step kernel, before the caller changes any state (the library
    refuses it too, but only once the host has counted the plan and flipped its result buffers)."""
    if env_kind != ENV_TOY and n_links not in STEP_LINKS:
        raise NotImplementedError(f"n_links={n_links}: the reacher step kernels are instantiated for "
                                  f"{STEP_LINKS[0]}..{STEP_LINKS[-1]} links")


def check(status: int):
    """Maps fg_status to the exception types the reference raises for the same conditions."""
    if status == OK:
        return
    msg = lib.fg_last_error().decode()
    if status == ERR_INVALID:
        raise ValueError(msg)
    if status == ERR_UNSUPPORTED:
        raise NotImplementedError(msg)
    if status == ERR_NOMEM:
        raise MemoryError(msg)
    raise RuntimeError(msg)

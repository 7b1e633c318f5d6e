"""ctypes binding of libmr_rl_b200.so (the C ABI in include/mr_rl_b200.h).

There is deliberately no fallback: if the CUDA library has not been built, importing any
compute entry point raises.  Build it with ``python -m mr_rl_b200.build`` (nvcc, sm_100a).
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MR_LIB_PATH") or os.path.join(HERE, "_lib", "libmr_rl_b200.so")   # MR_LIB_PATH: tuning variants

ABI_VERSION = 2
MR_F64, MR_F32 = 0, 1
NOISE_NONE, NOISE_TABLE, NOISE_PHILOX = 0, 1, 2
ACTIONS_TENSOR, ACTIONS_PHILOX, ACTIONS_ACTOR, ACTIONS_BROADCAST = 0, 1, 2, 3
REWARD_CONST10, REWARD_SHAPED = 0, 1
ENV_SOLVER_FAILED, ENV_NONFINITE, ENV_NOISE_OVERFLOW, ENV_ATTEMPT_CAP = 1, 2, 4, 8
STATS_LEN = 8
STAT_NAMES = ("episodes", "sum_length", "sum_reward", "goal", "out_of_bounds", "timeout", "env_steps", "failed")


class SimParams(C.Structure):
    _fields_ = [
        ("a0", C.c_double), ("noise_var", C.c_double),
        ("is_mismatched", C.c_int32), ("mism_at_reset", C.c_int32),
        ("time_span", C.c_double), ("rtol", C.c_double), ("atol", C.c_double),
        ("max_timesteps", C.c_int32), ("reward_mode", C.c_int32),
        ("min_dist2goal", C.c_double), ("bound_xy", C.c_double), ("bound_d", C.c_double),
        ("auto_reset", C.c_int32), ("action_f32", C.c_int32),
        ("init_low", C.c_double * 2), ("init_high", C.c_double * 2), ("action_high", C.c_double * 2),
    ]


class EnvState(C.Structure):
    _fields_ = [("x", C.c_void_p), ("y", C.c_void_p), ("fx", C.c_void_p), ("fy", C.c_void_p), ("h", C.c_void_p),
                ("counter", C.c_void_p), ("cursor", C.c_void_p), ("status", C.c_void_p),
                ("a0", C.c_void_p), ("noise_var", C.c_void_p), ("is_mismatched", C.c_void_p)]


class ResetParams(C.Structure):
    _fields_ = [("a0", C.c_void_p), ("noise_var", C.c_void_p), ("is_mismatched", C.c_void_p)]


class Noise(C.Structure):
    _fields_ = [("mode", C.c_int32), ("reserved", C.c_int32), ("table", C.c_void_p), ("table_len", C.c_int64),
                ("seed", C.c_uint64), ("offset", C.c_uint64), ("env_base", C.c_uint64), ("offset_dev", C.c_void_p)]


class TimeTable(C.Structure):
    _fields_ = [("t", C.c_void_p), ("len", C.c_int32), ("reserved", C.c_int32)]


class StepOut(C.Structure):
    _fields_ = [("obs", C.c_void_p), ("rew", C.c_void_p), ("done", C.c_void_p), ("state_prime", C.c_void_p),
                ("row_stride", C.c_int64), ("skip_goal_rows", C.c_int32), ("out_f32", C.c_int32)]


class RolloutIO(C.Structure):
    _fields_ = [("action_source", C.c_int32), ("k_steps", C.c_int32), ("actions", C.c_void_p), ("actor", C.c_void_p),
                ("traj_xy", C.c_void_p), ("traj_state_prime", C.c_void_p), ("traj_done", C.c_void_p),
                ("stats", C.c_void_p), ("traj_actions", C.c_void_p), ("traj_rew", C.c_void_p), ("traj_reset_xy", C.c_void_p),
                ("traj_episode", C.c_void_p), ("traj_step", C.c_void_p), ("episode_counter", C.c_void_p),
                ("reset_init", C.c_void_p), ("reset_init_len", C.c_int32), ("reserved", C.c_int32)]


class GPModel(C.Structure):
    _fields_ = [("x_train_scaled", C.c_void_p), ("alpha", C.c_void_p), ("linv", C.c_void_p), ("n_train", C.c_int32),
                ("n_pad", C.c_int32), ("dim", C.c_int32), ("proj_rows", C.c_int32),
                ("length_scale", C.c_double), ("noise_level", C.c_double)]


class HostStepIO(C.Structure):
    _fields_ = [("actions_host", C.c_void_p), ("actions_dev", C.c_void_p), ("obs_host", C.c_void_p), ("rew_host", C.c_void_p),
                ("done_host", C.c_void_p), ("host_row_stride", C.c_int64), ("copy_goal_rows", C.c_int32), ("io_f32", C.c_int32)]


class DDPGState(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("actor", "actor_target", "critic", "critic_target", "adam_actor_m", "adam_actor_v",
                                          "adam_critic_m", "adam_critic_v", "grad_actor", "grad_critic")]


class Replay(C.Structure):
    _fields_ = [("s", C.c_void_p), ("a", C.c_void_p), ("r", C.c_void_p), ("d", C.c_void_p), ("s2", C.c_void_p),
                ("capacity", C.c_int64)]


class DDPGHyper(C.Structure):
    _fields_ = [("gamma", C.c_double), ("tau", C.c_double), ("lr_actor", C.c_double), ("lr_critic", C.c_double),
                ("action_bound", C.c_double * 2), ("adam_beta1", C.c_double), ("adam_beta2", C.c_double), ("adam_eps", C.c_double)]


GP_PAD = 128


EXPORTS = ("mr_abi_version", "mr_last_error", "mr_default_params", "mr_fill_time_table_host", "mr_env_reset",
           "mr_env_step", "mr_env_rollout", "mr_gp_predict", "mr_gp_workspace_bytes", "mr_gp_correct_heading", "mr_gp_fit", "mr_gp_fit_workspace_bytes", "mr_actor_param_count",
           "mr_critic_param_count", "mr_replay_add", "mr_ou_noise_add", "mr_ddpg_update", "mr_learn_preprocess",
           "mr_learn_workspace_bytes", "mr_ddpg_workspace_bytes", "mr_replay_sample", "mr_actor_forward_env", "mr_ddpg_gradients", "mr_ddpg_apply", "mr_gp_correct_heading_cheb", "mr_host_pipeline_create", "mr_host_pipeline_destroy", "mr_env_step_host",
           "mr_actor_forward", "mr_set_step_path", "mr_env_reset_ex", "mr_counter_set", "mr_set_actor_path",
           "mr_host_register", "mr_host_unregister", "mr_philox_normals", "mr_gp_correct_action_2d")

_lib = None


class MRLibraryError(RuntimeError):
    pass


def load():
    """Load the CUDA library; raises MRLibraryError if it is missing (no CPU fallback exists)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise MRLibraryError(
            f"{LIB_PATH} not found: mr_rl_b200 has no CPU fallback — build the CUDA library with "
            "`python -m mr_rl_b200.build` (needs nvcc; targets sm_100a)")
    lib = C.CDLL(LIB_PATH)
    P = C.POINTER
    lib.mr_abi_version.restype = C.c_int
    lib.mr_last_error.restype = C.c_char_p
    lib.mr_default_params.argtypes = [P(SimParams)]
    lib.mr_default_params.restype = None
    lib.mr_fill_time_table_host.argtypes = [C.c_void_p, C.c_int32, C.c_double]
    lib.mr_fill_time_table_host.restype = None
    lib.mr_env_reset.argtypes = [P(EnvState), C.c_int64, C.c_int32, P(SimParams), P(Noise), C.c_void_p, C.c_void_p,
                                 C.c_int32, P(StepOut), C.c_void_p]
    lib.mr_env_reset_ex.argtypes = [P(EnvState), C.c_int64, C.c_int32, P(SimParams), P(Noise), C.c_void_p, C.c_void_p,
                                    C.c_int32, P(ResetParams), P(StepOut), C.c_void_p]
    lib.mr_env_reset_ex.restype = C.c_int
    lib.mr_counter_set.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p]
    lib.mr_counter_set.restype = C.c_int
    lib.mr_env_step.argtypes = [P(EnvState), C.c_int64, C.c_int32, P(SimParams), P(Noise), P(TimeTable), C.c_void_p,
                                P(StepOut), C.c_void_p]
    lib.mr_env_rollout.argtypes = [P(EnvState), C.c_int64, C.c_int32, P(SimParams), P(Noise), P(TimeTable),
                                   P(RolloutIO), P(StepOut), C.c_void_p]
    lib.mr_gp_predict.argtypes = [P(GPModel), C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                                  C.c_void_p]
    lib.mr_gp_correct_heading.argtypes = [P(GPModel), P(GPModel), C.c_void_p, C.c_int64, C.c_double, C.c_double, C.c_double,
                                          C.c_double, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.mr_gp_correct_heading.restype = C.c_int
    lib.mr_gp_correct_action_2d.argtypes = [P(GPModel), P(GPModel), C.c_void_p, C.c_int64, C.c_double, C.c_double * 2,
                                            C.c_double * 2, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.mr_gp_correct_action_2d.restype = C.c_int
    lib.mr_gp_fit.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_double, C.c_double, C.c_double,
                              C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                              C.c_void_p]
    lib.mr_gp_fit.restype = C.c_int
    lib.mr_host_pipeline_create.argtypes = [C.c_int32, P(C.c_void_p)]
    lib.mr_host_pipeline_create.restype = C.c_int
    lib.mr_host_pipeline_destroy.argtypes = [C.c_void_p]
    lib.mr_host_pipeline_destroy.restype = None
    lib.mr_env_step_host.argtypes = [C.c_void_p, P(EnvState), C.c_int64, C.c_int32, P(SimParams), P(Noise), P(TimeTable),
                                     P(HostStepIO), P(StepOut), C.c_int32, C.c_void_p]
    lib.mr_env_step_host.restype = C.c_int
    lib.mr_learn_preprocess.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_double, C.c_double,
                                        C.c_void_p, C.c_double, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
    lib.mr_learn_preprocess.restype = C.c_int
    lib.mr_learn_workspace_bytes.argtypes = [C.c_int32]
    lib.mr_learn_workspace_bytes.restype = C.c_int64
    lib.mr_critic_param_count.restype = C.c_int32
    lib.mr_replay_add.argtypes = [P(Replay), C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                  C.c_int64, C.c_int64, C.c_int32, C.c_void_p]
    lib.mr_replay_add.restype = C.c_int
    lib.mr_ou_noise_add.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_double, C.c_double, C.c_double,
                                    C.c_double, C.c_uint64, C.c_uint64, C.c_uint64, C.c_void_p]
    lib.mr_ou_noise_add.restype = C.c_int
    lib.mr_ddpg_update.argtypes = [P(DDPGState), P(Replay), C.c_int64, C.c_int32, C.c_void_p, C.c_uint64, C.c_int64,
                                   P(DDPGHyper), C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
    lib.mr_actor_forward_env.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int32, C.c_double * 2, C.c_void_p,
                                         C.c_void_p]
    lib.mr_actor_forward_env.restype = C.c_int
    lib.mr_gp_correct_heading_cheb.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.c_double, C.c_double,
                                               C.c_double, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.mr_gp_correct_heading_cheb.restype = C.c_int
    lib.mr_ddpg_gradients.argtypes = [P(DDPGState), P(Replay), C.c_int64, C.c_int32, C.c_void_p, C.c_uint64, C.c_int64,
                                      P(DDPGHyper), C.c_int32, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
    lib.mr_ddpg_gradients.restype = C.c_int
    lib.mr_ddpg_apply.argtypes = [P(DDPGState), C.c_int32, C.c_void_p, C.c_double, C.c_int64, P(DDPGHyper), C.c_void_p]
    lib.mr_ddpg_apply.restype = C.c_int
    lib.mr_ddpg_workspace_bytes.argtypes = [C.c_int32]
    lib.mr_ddpg_workspace_bytes.restype = C.c_int64
    lib.mr_replay_sample.argtypes = [C.c_int64, C.c_int32, C.c_uint64, C.c_int64, C.c_void_p, C.c_void_p]
    lib.mr_replay_sample.restype = C.c_int
    lib.mr_ddpg_update.restype = C.c_int
    lib.mr_gp_fit_workspace_bytes.argtypes = [C.c_int32]
    lib.mr_gp_fit_workspace_bytes.restype = C.c_int64
    lib.mr_gp_workspace_bytes.argtypes = [P(GPModel), C.c_int64, C.c_int32]
    lib.mr_gp_workspace_bytes.restype = C.c_int64
    lib.mr_actor_param_count.restype = C.c_int32
    lib.mr_philox_normals.argtypes = [C.c_uint64, C.c_uint64, C.c_uint64, C.c_int32, C.c_int32, C.c_int64, C.c_void_p, C.c_void_p]
    lib.mr_philox_normals.restype = C.c_int
    lib.mr_host_register.argtypes = [C.c_void_p, C.c_int64]
    lib.mr_host_register.restype = C.c_int
    lib.mr_host_unregister.argtypes = [C.c_void_p]
    lib.mr_host_unregister.restype = C.c_int
    lib.mr_set_actor_path.argtypes = [C.c_int32]
    lib.mr_set_actor_path.restype = C.c_int
    lib.mr_set_step_path.argtypes = [C.c_int32]
    lib.mr_set_step_path.restype = C.c_int
    lib.mr_actor_forward.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int32, C.c_double * 2, C.c_void_p,
                                     C.c_void_p]
    for f in ("mr_env_reset", "mr_env_step", "mr_env_rollout", "mr_gp_predict", "mr_actor_forward"):
        getattr(lib, f).restype = C.c_int
    if lib.mr_abi_version() != ABI_VERSION:
        raise MRLibraryError(f"ABI version mismatch: library {lib.mr_abi_version()}, binding {ABI_VERSION}")
    _lib = lib
    return lib


STEP_PATHS = {"default": 0, "tma": 1, "vec": 2, "scalar": 3, "ws": 4, "tmap": 5}   # tma: 1-D bulk copies only; tmap = default


def set_step_path(name):
    """Force the kernel variant mr_env_step launches (tests / A-B timing); returns the previous name."""
    old = load().mr_set_step_path(STEP_PATHS[name])
    if old < 0:
        check(old, "mr_set_step_path")
    return {v: k for k, v in STEP_PATHS.items()}[old]


ACTOR_PATHS = {"default": 0, "simt": 1, "tf32": 2}


def set_actor_path(name):
    """Force the in-rollout actor implementation (tests / A-B timing); returns the previous name."""
    old = load().mr_set_actor_path(ACTOR_PATHS[name])
    if old < 0:
        check(old, "mr_set_actor_path")
    return {v: k for k, v in ACTOR_PATHS.items()}[old]


def check(rc, what=""):
    if rc != 0:
        msg = load().mr_last_error().decode(errors="replace")
        raise MRLibraryError(f"{what or 'mr_rl_b200'} failed ({rc}): {msg}")


def default_params() -> SimParams:
    p = SimParams()
    load().mr_default_params(C.byref(p))
    return p

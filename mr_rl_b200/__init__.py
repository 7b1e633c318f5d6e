"""mr_rl_b200 — B200-native batched implementation of MR_RL's rolling-microrobot environment.

Public surface (mirrors the reference's names):
    VecMREnv                      batched device env (reset / step / rollout)
    MR_Env, Simulator             single-env façades with the reference's class surface
    run_sim                       utils.run_sim as one fused rollout launch
    LearningModule, LearningModule2D, DeviceGP, DeviceGPR   GP disturbance model: fit, inference and heading correction on the device
    HeadingTrackingPolicy         LearningModule.tracking_policy: GP-corrected heading control inside VecMREnv.rollout
    DDPGLearner, ReplayBuffer, OUNoise, ddpg.train   the DDPG learner of RL/MR_ddpg.py on the device
    ddpg.collect                  its acting loop (actor + OU noise + env step + replay add) fused into one rollout launch
    DDPGPopulation, PopulationReplay, ddpg.train_population   many independent learners, one update and one collect launch
    evaluate_population, evaluate, pbt_plan, pbt_population   greedy evaluation of every member in one launch, and PBT on it
    init_actor / pack_actor / actor_forward   DDPG actor forward for the in-loop policy
    experiment_dict / save_experiment          recorded rollouts in the reference's MRExperiment pickle layout

All compute runs in hand-written sm_100a kernels behind the C ABI in include/mr_rl_b200.h;
there is no CPU fallback (importing is cheap, the first compute call loads the library).
"""
from ._lib import MRLibraryError, load as load_library  # noqa: F401
from .actor import actor_forward, init_actor, pack_actor  # noqa: F401
from .ddpg import (DDPGLearner, DDPGPopulation, OUNoise, PopulationEvaluation, PopulationReplay, ReplayBuffer, evaluate,  # noqa: F401
                   evaluate_population, pbt_plan, pbt_population)
from .gp import DeviceGP  # noqa: F401
from .gpr import DeviceGPR  # noqa: F401
from .learning_module import HeadingTrackingPolicy, LearningModule  # noqa: F401
from .learning_module_2d import LearningModule2D  # noqa: F401
from .mr_env import MR_Env, Simulator  # noqa: F401
from .recording import MRExperiment, experiment_dict, experiment_from_rollout, load_experiment, save_experiment  # noqa: F401
from .spaces import Box  # noqa: F401
from .utils import run_sim  # noqa: F401
from .vec_env import VecMREnv, shard_range  # noqa: F401

__version__ = "0.1.0"

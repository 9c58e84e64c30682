"""rl_rocket_6dof_b200 — B200-native batched 6DOF rocket-landing environment step.

Public surface (all CUDA-backed; importing the env classes without a built libr6dof.so or without a
GPU raises — there is no CPU path):

    load_config, derive_params          config.yaml -> kernel constants
    Rocket6DOFBatch                     N envs on one GPU, torch tensors in / out
    Rocket6DOFVecEnv                    stable-baselines3 VecEnv protocol + pinned-host fast path
    Rocket6DOF                          single-env gym contract of the reference
    make_env / make_vec_env             what main_6DOF.py:44-53 builds, batched
    TrajectoryRecorder                  [T, N] record of states / actions / times (SIM.states, .actions, .times)
    ActorCriticParams, PPOConfig,       PPO training on the device (SB3 1.6 PPO.train / learn): flat actor-critic
    PPOTrainer                          parameters, hyper-parameters, collect + update loop
"""
from .params import EnvParams, derive_params, load_config  # noqa: F401

__all__ = ["EnvParams", "derive_params", "load_config", "Rocket6DOFBatch", "Rocket6DOFVecEnv", "Rocket6DOF",
           "make_env", "make_vec_env", "make_annealed_env", "make_annealed_vec_env", "TrajectoryRecorder",
           "ActorCriticParams", "PPOConfig", "PPOTrainer"]


def __getattr__(name):  # lazy: params are usable without torch / CUDA
    if name == "Rocket6DOFBatch":
        from .batch import Rocket6DOFBatch
        return Rocket6DOFBatch
    if name == "Rocket6DOFVecEnv":
        from .vec_env import Rocket6DOFVecEnv
        return Rocket6DOFVecEnv
    if name == "Rocket6DOF":
        from .gym_env import Rocket6DOF
        return Rocket6DOF
    if name == "TrajectoryRecorder":
        from .recorder import TrajectoryRecorder
        return TrajectoryRecorder
    if name in ("ActorCriticParams", "PPOConfig", "PPOTrainer"):
        from . import ppo
        return getattr(ppo, name)
    if name in ("make_env", "make_vec_env", "make_annealed_env", "make_annealed_vec_env"):
        from . import factory
        return getattr(factory, name)
    raise AttributeError(name)

"""B200-native batched RendezvousEnv (step/reset hot path of cfdeinza/reinforcement-learning-rendezvous).

Public surface (mirrors the reference, see INTEGRATION.md):

* ``RendezvousEnv``           single-env Gym object (rendezvous_env.py)
* ``RendezvousVecEnv``        SB3 VecEnv with N GPU envs (replaces DummyVecEnv([...]), main.py:33-34)
* ``BatchedRendezvousEnv``    device-tensor API under both
* ``make_env`` / ``copy_env`` factory with the reference signature (utils/environment_utils.py)
* ``MlpPolicy``               fused fp32 policy forward (model.predict, monte_carlo.py:128-133)
* ``PolicyTable``             several MlpPolicy actors in one fused rollout (one per 128-env tile)
* ``evaluate`` / ``evaluate_batch``  Monte-Carlo evaluator (monte_carlo.py:94-207)
* ``ppo.PPO``                 device-tensor PPO loop with main.py's hyper-parameters (main.py:39-48, :114-118)

Importing the package needs neither a GPU nor the built library; using it does.  There is
no CPU fallback.
"""
from . import _native
from ._native import build as build_native
from .params import make_params


def __getattr__(name):
    # lazy: these import torch
    if name in ("BatchedRendezvousEnv",):
        from .batched_env import BatchedRendezvousEnv
        return BatchedRendezvousEnv
    if name == "RendezvousEnv":
        from .rendezvous_env import RendezvousEnv
        return RendezvousEnv
    if name == "RendezvousVecEnv":
        from .vec_env import RendezvousVecEnv
        return RendezvousVecEnv
    if name in ("make_env", "make_vec_env", "copy_env"):
        from . import environment_utils
        return getattr(environment_utils, name)
    if name in ("MlpPolicy", "PolicyTable"):
        from . import policy
        return getattr(policy, name)
    if name in ("evaluate", "evaluate_batch", "evaluate_sweep", "sensitivity_grid"):
        from . import monte_carlo
        return getattr(monte_carlo, name)
    raise AttributeError(name)


__all__ = ["BatchedRendezvousEnv", "RendezvousEnv", "RendezvousVecEnv", "make_env", "make_vec_env", "copy_env",
           "MlpPolicy", "PolicyTable", "evaluate", "evaluate_batch", "evaluate_sweep", "sensitivity_grid", "make_params", "build_native"]

"""marlnav_b200 -- the batched MARL-nav environment step as one fused sm_100a kernel.

Drop-in for ``marlnav.environment.Env`` (JussiM01/MARL-nav); see env.py.
"""
from ._lib import MarlnavError, LIB_PATH          # noqa: F401
from .env import Env, HostStepper, Observations, split_observations   # noqa: F401
from .params import default_env_params, template_env_params, ring_template   # noqa: F401
from .rollout import (FusedActor, FusedCritic, MappoRollout, RolloutGraph, StepGraph,   # noqa: F401
                      discounted_returns, gae, collect_rollout)
from .sharding import shard_bounds, shard_env_params, reduce_episode_stats, global_episode_stats  # noqa: F401

__all__ = ["Env", "HostStepper", "Observations", "split_observations", "default_env_params",
           "template_env_params", "ring_template", "shard_bounds", "shard_env_params",
           "reduce_episode_stats", "global_episode_stats", "MarlnavError", "LIB_PATH",
           "FusedActor", "FusedCritic", "MappoRollout", "RolloutGraph", "StepGraph", "discounted_returns",
           "gae", "collect_rollout"]

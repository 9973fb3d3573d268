"""B200-native batched simulator for the ``delivery_drone`` landing environment.

The per-instance Python ``DroneGame.step()/reset()`` loop of the reference
(/root/reference/delivery_drone/game/game_engine.py) is replaced by hand-written sm_100a CUDA
kernels (``csrc/``) behind a plain C ABI (``include/drone_b200.h``); this package is the thin
Python host: ``BatchedDroneEnv`` (gym-style batched surface), ``compat`` (per-index ``DroneGame``
view, in-process ``DroneGameClient``, socket shim) and the rollout-side device ops.

The directory name is not a Python identifier; import it with
``importlib.import_module("reinforcement-learning-101_b200")``.
"""
from . import _native as native
from ._native import build_native
from .distributed import (allreduce_moments, allreduce_stats, allreduce_stats_by_set, bind_to_gpu_numa, init_from_env,
                          mean_std_from_moments, shard_range, stats_dict)

__all__ = ["native", "build_native", "BatchedDroneEnv", "ShardedDroneEnv", "StepInfo", "gae", "discounted_returns", "advantage_moments",
           "normalize_advantages", "allreduce_stats", "allreduce_stats_by_set", "allreduce_moments", "shard_range", "stats_dict",
           "mean_std_from_moments", "init_from_env", "bind_to_gpu_numa", "PolicyBlob", "ValueBlob", "policy_forward", "value_forward",
           "rollout_values", "policy_rollout",
           "step_schedule", "collect_episodes", "curriculum_sweep"]


def __getattr__(name):
    # env / ppo_ops need the built CUDA library; resolve them lazily so that `build_native`
    # itself is importable on a tree that has not been built yet.
    if name in ("BatchedDroneEnv", "StepInfo"):
        from . import env
        return getattr(env, name)
    if name == "ShardedDroneEnv":
        from . import sharded
        return sharded.ShardedDroneEnv
    if name in ("gae", "discounted_returns", "advantage_moments", "normalize_advantages"):
        from . import ppo_ops
        return getattr(ppo_ops, name)
    if name in ("PolicyBlob", "ValueBlob", "policy_forward", "value_forward", "rollout_values", "policy_rollout"):
        from . import policy
        return getattr(policy, name)
    if name in ("step_schedule", "collect_episodes", "curriculum_sweep"):
        from . import curriculum
        return getattr(curriculum, name)
    if name in ("compat", "env", "ppo_ops", "policy", "curriculum", "sharded"):
        import importlib
        return importlib.import_module("." + name, __name__)
    raise AttributeError(name)

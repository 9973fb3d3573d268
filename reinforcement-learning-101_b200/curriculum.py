"""Curriculum rollouts (BASELINE.json configs[4]): the notebooks grow the episode cap ``max_steps``
over training (``step_schedule``, Actor_Critic_PPO.ipynb c19:L13-17; README.md:55 quotes 75 -> 250)
and, per iteration, let every game play exactly ONE episode until done or the cap
(``collect_episodes_ppo``, c16:L38-108), then report success rate / average reward / average length
(c21:L94-95,L158-169).  Here one "collect" is: reset every env, one launch of ``max_steps`` fused steps
with freeze-after-done (so each env plays exactly one episode), statistics reduced on the device and
all-reduced over ranks (NCCL) -- 8 words per stage, no other communication.
"""
from __future__ import annotations

from typing import Dict, Iterable, List, Optional

import numpy as np
import torch

from .env import BatchedDroneEnv


def step_schedule(num_iterations: int, start: int = 300, end: int = 500, steepness: float = 0.65) -> np.ndarray:
    """``np.round(start + (end - start) * x**steepness).astype(np.int32)``, x = linspace(0, 1, num)
    (Actor_Critic_PPO.ipynb c19:L13-17; Policy_Gradients.ipynb c25:L1-6)."""
    x = np.linspace(0, 1, num=int(num_iterations))
    return np.round(start + (end - start) * x ** steepness).astype(np.int32)


def _collect_keys(max_steps: int, s: Dict[str, float]) -> Dict[str, float]:
    return {"max_steps": int(max_steps), "num_games": s["episodes"], "num_successes": s["landed"],
            "success_rate": s["landing_rate"], "avg_reward": s["mean_return"], "avg_steps": s["mean_length"],
            "crashed": s["crashed"], "timed_out": s["truncated"], "env_steps": s["sum_length"]}


def collect_episodes(env: BatchedDroneEnv, max_steps: int, policy: str = "random", blob=None, sample: bool = True,
                     reduce: bool = True, t0: Optional[int] = None, by_set: bool = False) -> Dict[str, float]:
    """One curriculum iteration: every env plays one episode of at most ``max_steps`` steps.
    ``policy``: 'random' / 'bangbang' (scripted, in-kernel) or 'network' with a ``PolicyBlob``.
    ``t0``: offset of the in-kernel noise streams; ``None`` continues the env's running counter, so every stage /
    iteration explores with fresh noise (include/drone_b200.h, t0 contract).
    Returns the (all-reduced) statistics dict: success_rate, avg_reward (engine return), avg_steps, ...
    ``by_set=True`` (an env with ``set_param_sets(..., stats_by_set=True)``): the dict also holds ``"by_set"``, one dict
    with the same keys per parameter set -- one policy evaluated on several worlds in one launch."""
    if by_set and not env.stats_by_set:
        raise ValueError("by_set=True needs an env with set_param_sets(..., stats_by_set=True)")
    if env.auto_reset:
        raise ValueError("collect_episodes needs an env built with auto_reset=False (one episode per env)")
    env.max_steps = int(max_steps)
    env.reset(want_obs=False)                      # the rollout launch reads the state, not the observation buffer
    env.reset_stats()
    if policy == "network":
        if blob is None:
            raise ValueError("policy='network' needs a PolicyBlob")
        from .policy import policy_rollout
        policy_rollout(env, blob, int(max_steps), sample=sample, t0=t0, want="")
    else:
        env.rollout(int(max_steps), policy, t0=t0)
    out = _collect_keys(max_steps, env.stats(reduce=reduce))
    if by_set:
        out["by_set"] = [_collect_keys(max_steps, s) for s in env.stats(reduce=reduce, by_set=True)]
    return out


def curriculum_sweep(env: BatchedDroneEnv, caps: Iterable[int], policy: str = "random", blob=None,
                     sample: bool = True, reduce: bool = True, by_set: bool = False) -> List[Dict[str, float]]:
    """``collect_episodes`` for each cap in ``caps`` (e.g. ``step_schedule(8, 75, 250)``)."""
    out = []
    for cap in caps:        # t0=None: each stage continues the env's noise counter (stage j starts at sum(caps[:j]))
        out.append(collect_episodes(env, int(cap), policy=policy, blob=blob, sample=sample, reduce=reduce, by_set=by_set))
    return out

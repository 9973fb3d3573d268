"""Multi-GPU plumbing: environments shard by contiguous global id, one process per GPU, and the
only collectives are two tiny all-reduces (SURVEY.md 8e):

  * episode statistics  -- 8 int64 words        (Actor_Critic_PPO.ipynb c21:L94-95,L158-159,L169),
                           or count x 8 with statistics per parameter set
  * advantage moments   -- n, sum x, sum x^2     (Actor_Critic_PPO.ipynb c21:L105)

There is no per-step communication.  Integer sums make the statistics independent of the GPU
count; Philox spawns are keyed by the GLOBAL env id, so trajectories are too.  Everything here
works on any ``torch.distributed`` backend (NCCL on the GPU box, gloo in the CPU tests).
"""
from __future__ import annotations

import os
from typing import Dict, Tuple

import torch
import torch.distributed as dist

from ._native import RETURN_FIXED_SCALE

STAT_NAMES = ("episodes", "landed", "crashed", "truncated", "sum_return_fx", "sum_length", "env_steps", "reserved")


def world() -> Tuple[int, int]:
    """(rank, world_size) of the default group, or (0, 1) when not initialised."""
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def init_from_env(backend: str = "nccl") -> Tuple[int, int, int]:
    """torchrun-style initialisation (RANK / LOCAL_RANK / WORLD_SIZE / MASTER_*).
    Returns (rank, local_rank, world_size); a no-op single-process answer when WORLD_SIZE is unset."""
    ws = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if ws > 1 and not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29500")
        if backend == "nccl":
            torch.cuda.set_device(local)
            dist.init_process_group(backend, rank=rank, world_size=ws, device_id=torch.device("cuda", local))
        else:
            dist.init_process_group(backend, rank=rank, world_size=ws)
    return rank, local, ws


def bind_to_gpu_numa(device_index: int):
    """Pin the calling thread to the CPUs NVML reports as local to this GPU (same NUMA node / PCIe root), so that
    pinned host buffers allocated afterwards are first-touched next to the GPU and the host side of host<->device
    copies does not cross sockets.  Matters for host-buffer stepping at several ranks per box; returns the CPU list, or
    None when NVML / affinity control is unavailable (never raises)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        uuid = str(torch.cuda.get_device_properties(device_index).uuid)
        try:
            h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid).encode())
        except Exception:
            h = pynvml.nvmlDeviceGetHandleByIndex(device_index)
        pynvml.nvmlDeviceSetCpuAffinity(h)
        return sorted(os.sched_getaffinity(0))
    except Exception:
        return None


def shard_range(total_envs: int, rank: int, world_size: int) -> Tuple[int, int]:
    """Contiguous block [env_id_base, env_id_base + n_local) of global env ids owned by ``rank``.
    The first ``total % world`` ranks get one extra env."""
    if not (0 <= rank < world_size):
        raise ValueError("rank out of range")
    q, r = divmod(int(total_envs), int(world_size))
    n_local = q + (1 if rank < r else 0)
    base = rank * q + min(rank, r)
    return base, n_local


def allreduce_stats(words: torch.Tensor) -> torch.Tensor:
    """Sum the int64[8] statistics block over all ranks (in place; returns it)."""
    if words.dtype != torch.int64 or words.numel() != len(STAT_NAMES):
        raise ValueError("stats block must be int64[8]")
    if world()[1] > 1:
        dist.all_reduce(words, op=dist.ReduceOp.SUM)
    return words


def allreduce_stats_by_set(words: torch.Tensor) -> torch.Tensor:
    """Sum an int64[count, 8] statistics block per parameter set over all ranks, in one collective (in place; returns
    it).  Every rank must hold the same count."""
    if words.dtype != torch.int64 or words.dim() != 2 or words.shape[1] != len(STAT_NAMES) or words.shape[0] < 1:
        raise ValueError("per-set stats block must be int64[count, 8]")
    if world()[1] > 1:
        dist.all_reduce(words, op=dist.ReduceOp.SUM)
    return words


def stats_dict(words: torch.Tensor) -> Dict[str, float]:
    """Host view of a statistics block with the notebook's derived rates."""
    w = [int(v) for v in words.detach().cpu().tolist()]
    d = dict(zip(STAT_NAMES, w))
    ep = max(d["episodes"], 1)
    d["sum_return"] = d.pop("sum_return_fx") / RETURN_FIXED_SCALE
    d["landing_rate"] = d["landed"] / ep            # num_successes / num_games
    d["mean_return"] = d["sum_return"] / ep         # avg_reward
    d["mean_length"] = d["sum_length"] / ep         # avg_steps
    d.pop("reserved")
    return d


def allreduce_moments(m: torch.Tensor) -> torch.Tensor:
    """Sum the float64[3] block (n, sum x, sum x^2) over all ranks (in place; returns it)."""
    if m.dtype != torch.float64 or m.numel() != 3:
        raise ValueError("moments block must be float64[3]")
    if world()[1] > 1:
        dist.all_reduce(m, op=dist.ReduceOp.SUM)
    return m


def mean_std_from_moments(m: torch.Tensor) -> Tuple[float, float]:
    """mean and UNBIASED std (torch.std default, as the notebook uses) from (n, sum, sumsq)."""
    n, s, q = (float(v) for v in m.detach().cpu().tolist())
    if n <= 0:
        return 0.0, 0.0
    mean = s / n
    var = (q - s * mean) / (n - 1.0) if n > 1 else 0.0
    return mean, max(var, 0.0) ** 0.5

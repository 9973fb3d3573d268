"""K5 host side: the fused policy rollout (``csrc/policy_rollout.cu``).

``PolicyBlob`` packs the fp32 parameters of the notebook's policy network ``DroneGamerBoi``
(Actor_Critic_PPO.ipynb c11:L5-17 -- ``nn.Sequential`` indices 0/3/6/9 are the Linears, 1/4/7 the
LayerNorms) into the bf16 tensor-core operand images the kernel keeps in shared memory.
``policy_forward`` runs just the network (parity hook against eager torch); ``policy_rollout``
runs T steps of {observe, policy, act, step} in one launch on a ``BatchedDroneEnv`` and fills
on-device rollout buffers (obs, action, log-prob, reward, done -- what ``collect_episodes_ppo``,
c16:L42-108, appends per step).
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Mapping, Optional

import torch

from . import _native as nv
from .env import BatchedDroneEnv

BLOB_BYTES = 67616
_OPERANDS = {"auto": nv.OPERANDS_AUTO, "bf16": nv.OPERANDS_BF16, "fp16": nv.OPERANDS_FP16}
ACTION_THRESHOLD, ACTION_SAMPLE = 0, 1
_KEYS = ("network.0.weight", "network.0.bias", "network.1.weight", "network.1.bias",
         "network.3.weight", "network.3.bias", "network.4.weight", "network.4.bias",
         "network.6.weight", "network.6.bias", "network.7.weight", "network.7.bias",
         "network.9.weight", "network.9.bias")
_SHAPES = ((128, 15), (128,), (128,), (128,), (128, 128), (128,), (128,), (128,),
           (64, 128), (64,), (64,), (64,), (3, 64), (3,))


class PolicyBlob:
    """Device-resident packed network (67,616 bytes) + its host-side per-column constants.
    ``head=3``: the policy ``DroneGamerBoi`` (sigmoid probabilities); ``head=1``: the critic
    ``DroneTeacherBoi`` (same trunk, ``Linear(64, 1)``, raw scalar) -- see ``ValueBlob``."""

    def __init__(self, state_dict: Mapping[str, torch.Tensor], device="cuda", head: int = 3, operands: str = "auto"):
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise ValueError("PolicyBlob lives on a CUDA device")
        if head not in (1, 3):
            raise ValueError("head must be 3 (policy) or 1 (critic)")
        if operands not in _OPERANDS:
            raise ValueError("operands must be 'auto', 'bf16' or 'fp16'")
        self.head = head
        shapes = _SHAPES[:-2] + ((head, 64), (head,))
        params = []
        for key, shape in zip(_KEYS, shapes):
            if key not in state_dict and key[len("network."):] in state_dict:
                key = key[len("network."):]                 # a bare nn.Sequential: '0.weight', ...
            if key not in state_dict:
                raise KeyError(f"state_dict lacks {key!r} (expected the DroneGamerBoi layout)")
            t = state_dict[key].detach()
            if tuple(t.shape) != shape:
                raise ValueError(f"{key}: shape {tuple(t.shape)} != {shape}")
            params.append(t)
        if all(not t.is_cuda for t in params):
            # host state_dict: one staging buffer and ONE host->device copy instead of 14 small ones
            flat = torch.cat([t.to(torch.float32).reshape(-1) for t in params]).to(self.device)
            offs = [0]
            for t in params:
                offs.append(offs[-1] + t.numel())
            params = [flat[offs[j]:offs[j + 1]] for j in range(len(params))]    # every offset is a multiple of 4 bytes
            self._flat = flat
        else:
            params = [t.to(device=self.device, dtype=torch.float32).contiguous() for t in params]
        self._params = params                              # keep alive until the pack kernel has run
        self.blob = torch.empty(BLOB_BYTES, dtype=torch.uint8, device=self.device)
        self.consts = nv.DDPolicyConsts()                  # host side: rides in the kernel-argument constant bank
        pol = nv.DDPolicy(*[t.data_ptr() for t in params])
        # 'auto': fp16 operand images when the network provably fits the fp16 range (checked on the device from the
        # parameters, include/drone_b200.h DD_OPERANDS_*), else bf16; 'fp16' raises when it does not fit
        nv.check(nv.lib().dd_policy_pack_ex(C.byref(pol), head, _OPERANDS[operands], self.blob.data_ptr(), C.byref(self.consts),
                                            torch.cuda.current_stream(self.device).cuda_stream), "dd_policy_pack_ex")
        self.operand_dtype = "fp16" if self.consts.operands == nv.OPERANDS_FP16 else "bf16"

    @classmethod
    def from_module(cls, module: torch.nn.Module, device="cuda", head: int = 3, operands: str = "auto") -> "PolicyBlob":
        return cls(module.state_dict(), device=device, head=head, operands=operands)


def ValueBlob(state_dict: Mapping[str, torch.Tensor], device="cuda", operands: str = "auto") -> PolicyBlob:
    """The critic ``DroneTeacherBoi`` (Actor_Critic_PPO.ipynb: 15-128-128-64-1, LayerNorm + ReLU) packed for
    ``value_forward``."""
    return PolicyBlob(state_dict, device=device, head=1, operands=operands)


def _rows(obs: torch.Tensor) -> torch.Tensor:
    if not obs.is_cuda or obs.dtype != torch.float32 or obs.dim() < 2 or obs.shape[-1] != 15:
        raise ValueError("obs must be a CUDA float32 tensor of shape [..., 15]")
    return obs.contiguous().view(-1, 15)


def policy_forward(blob: PolicyBlob, obs: torch.Tensor) -> torch.Tensor:
    """probs [..., 3] = sigmoid(policy(obs [..., 15])) on the tensor-core path (persistent over the rows)."""
    if blob.head != 3:
        raise ValueError("policy_forward needs a policy blob (head=3)")
    rows = _rows(obs)
    probs = torch.empty(rows.shape[0], 3, dtype=torch.float32, device=obs.device)
    nv.check(nv.lib().dd_policy_forward(blob.blob.data_ptr(), C.byref(blob.consts), rows.data_ptr(), probs.data_ptr(), rows.shape[0],
                                        torch.cuda.current_stream(obs.device).cuda_stream), "dd_policy_forward")
    return probs.view(*obs.shape[:-1], 3)


def value_forward(blob: PolicyBlob, obs: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """values [...] = critic(obs [..., 15]) -- ``values = critic(states_tensor)`` of the PPO training loop
    (Actor_Critic_PPO.ipynb, PHASE 2) for a whole rollout buffer in one launch."""
    if blob.head != 1:
        raise ValueError("value_forward needs a critic blob (ValueBlob / head=1)")
    rows = _rows(obs)
    if out is None:
        out = torch.empty(obs.shape[:-1], dtype=torch.float32, device=obs.device)
    elif out.dtype != torch.float32 or not out.is_contiguous() or out.numel() != rows.shape[0] or out.device != obs.device:
        raise ValueError("out must be a contiguous float32 tensor with one element per observation row")
    nv.check(nv.lib().dd_value_forward(blob.blob.data_ptr(), C.byref(blob.consts), rows.data_ptr(), out.data_ptr(), rows.shape[0],
                                       torch.cuda.current_stream(obs.device).cuda_stream), "dd_value_forward")
    return out


def rollout_values(vblob: PolicyBlob, obs_tn: torch.Tensor, final_obs: torch.Tensor) -> torch.Tensor:
    """values [T+1, N] for ``gae``: the critic on the rollout's observations obs_tn [T, N, 15] plus the bootstrap
    row on the observation after the last step (final_obs [N, 15], e.g. ``env.observe()``)."""
    T, n = obs_tn.shape[0], obs_tn.shape[1]
    v = torch.empty(T + 1, n, dtype=torch.float32, device=obs_tn.device)
    value_forward(vblob, obs_tn, out=v[:T])
    value_forward(vblob, final_obs, out=v[T])
    return v


def policy_rollout(env: BatchedDroneEnv, blob: PolicyBlob, T: int, sample: bool = True, t0: Optional[int] = None,
                   want: str = "arld", out: Optional[Dict[str, torch.Tensor]] = None, stats: bool = True,
                   temperature: float = 1.0) -> Dict[str, torch.Tensor]:
    """T fused steps on ``env`` (float32 envs only).  ``want`` picks the [T,N] buffers to fill:
    a=actions (uint8 DD_ACT bits), l=logp, r=reward, d=done flags, o=obs [T,N,15], p=probs [T,N,3],
    s=shaped (the notebook's client-side training reward, Actor_Critic_PPO.ipynb c7 + c16:L89-93).
    ``t0``: offset of the Bernoulli noise stream (include/drone_b200.h: uniforms = Philox(seed, env id, t0 + t)); the
    default ``None`` continues the env's own running counter (``env.t_rollout``, advanced by T), so that successive PPO
    iterations explore with fresh noise.  ``obs[t]`` is the observation BEFORE step t (the network input).
    ``temperature``: the evaluation sampling of the notebooks' ``evaluate_policy_simple`` (c18) -- actions drawn from
    ``p**(1/t) / (p**(1/t) + (1-p)**(1/t))``; 0 means ``probs > 0.5`` (like ``sample=False``), 1 the policy itself.
    Returns the dict of buffers (allocated unless passed in ``out``)."""
    if temperature < 0:
        raise ValueError("temperature must be >= 0")
    if temperature == 0:
        sample, temperature = False, 1.0
    if env.dtype != torch.float32:
        raise ValueError("policy_rollout needs a float32 env")
    if env.param_sets is not None:
        raise ValueError("policy_rollout does not take per-env parameter sets: the fused policy kernel runs one DDParams "
                         "per launch (call env.set_param_sets(None) first)")
    if env._needs_reset:
        raise RuntimeError("call reset() before policy_rollout()")
    n, dev = env.num_envs, env.device
    spec = {"a": ("actions", (T, n), torch.uint8), "l": ("logp", (T, n), torch.float32),
            "r": ("reward", (T, n), torch.float32), "d": ("done", (T, n), torch.uint8),
            "o": ("obs", (T, n, 15), torch.float32), "p": ("probs", (T, n, 3), torch.float32),
            "s": ("shaped", (T, n), torch.float32)}
    bufs: Dict[str, torch.Tensor] = dict(out or {})
    for ch in want:
        name, shape, dtype = spec[ch]
        if name not in bufs:
            bufs[name] = torch.empty(shape, dtype=dtype, device=dev)
        b = bufs[name]
        if tuple(b.shape) != shape or b.dtype != dtype or not b.is_contiguous() or b.device != dev:
            raise ValueError(f"{name} must be a contiguous {dtype} tensor of shape {shape} on {dev}")
    ptr = lambda k: bufs[k].data_ptr() if k in bufs else None
    if "shaped" in bufs:
        env._fresh_prev_dist()
    t0 = env._take_t0(t0, T)
    nv.check(nv.lib().dd_policy_rollout(
        C.byref(env._state), C.byref(env._params), C.byref(env._cfg), blob.blob.data_ptr(), C.byref(blob.consts),
        ACTION_SAMPLE if sample else ACTION_THRESHOLD, float(temperature), int(t0), int(T), ptr("actions"), ptr("logp"), ptr("reward"),
        ptr("done"), ptr("obs"), ptr("probs"), ptr("shaped"), env.stats_slots.data_ptr() if stats else None, n,
        env._stream()),
        "dd_policy_rollout")
    return bufs

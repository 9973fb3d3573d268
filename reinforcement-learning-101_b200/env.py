"""``BatchedDroneEnv`` -- the gym-style ``reset()/step()`` surface of the reference ``DroneGame``
(/root/reference/delivery_drone/game/game_engine.py:14-298) for N environments at once, stepped by
the sm_100a kernels behind the C ABI of ``include/drone_b200.h``.

PyTorch is plumbing here: it owns the device buffers and the stream.  Every numeric result comes
from ``libdrone_b200.so``; there is no Python / torch fallback for any of it.

Semantics kept from the reference (file:line are under /root/reference/delivery_drone/game/):
  * observation = the first 15 keys of ``get_state()`` in policy order (game_engine.py:146-177,
    Actor_Critic_PPO.ipynb c10:L3-19); with ``obs_stride=16`` column 15 is ``steps`` (16th key)
  * reward / termination priority of ``_calculate_reward`` (game_engine.py:179-216)
  * ``auto_reset=False``: frozen after done -- reward 0, done stays True, no state change
    (game_engine.py:107-111)
  * action = any truthy value per thruster (game_engine.py:114-118)
New, because the reference has neither: same-step auto-reset with Philox spawns, ``max_steps``
truncation (the notebooks' time-out, Actor_Critic_PPO.ipynb c16:L89-93, without its client-side
-500), and on-device episode statistics.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional

import torch

from . import _native as nv

_STATE_KEYS = ("x", "y", "vx", "vy", "angle", "angular_velocity", "fuel", "total_reward",
               "platform_x", "platform_y", "steps", "episode", "flags", "prev_dist")
POLICIES = {"trace": nv.POLICY_TRACE, "random": nv.POLICY_RANDOM, "bangbang": nv.POLICY_BANGBANG}
# observation element dtype -> DDEnvConfig.obs_format (16-bit formats: float32 state only)
_OBS_FORMATS = {torch.float16: nv.OBS_F16, torch.bfloat16: nv.OBS_BF16}
# single-set entry point -> its per-env parameter-set counterpart (include/drone_b200.h DDParamSets)
_SETS_ENTRY = {"dd_reset": "dd_reset_sets", "dd_step": "dd_step_sets", "dd_step_plan": "dd_step_plan_sets",
               "dd_rollout_shaped": "dd_rollout_sets"}


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


# The raw cudaStream_t of torch's current stream on a device, without building a torch.cuda.Stream object first
# (1.5-2 us of the ~7 us a planned step costs on the host).  Private torch entry point (what torch's own compiled code
# calls); falls back to the public API when a torch build lacks it.
_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def _current_stream_handle(device: torch.device) -> int:
    if _raw_stream is not None:
        return _raw_stream(device.index)
    return torch.cuda.current_stream(device).cuda_stream


def _out_layout(n: int, stride: int, dtype: torch.dtype, obs_dtype: Optional[torch.dtype] = None):
    """Byte offsets of (obs, reward, step_flags, end) inside the packed per-step output block.  ``dtype`` is the state
    (and reward) dtype, ``obs_dtype`` the observation's (default: ``dtype``)."""
    isz = 4 if dtype == torch.float32 else 8
    osz = torch.empty((), dtype=obs_dtype or dtype).element_size()
    up = lambda b: -(-b // 256) * 256
    o_rew = up(n * stride * osz)
    o_flg = o_rew + up(n * isz)
    return 0, o_rew, o_flg, max(o_flg + up(n), 256)


def _carve(block: torch.Tensor, layout, n: int, stride: int, dtype: torch.dtype, obs_dtype: Optional[torch.dtype] = None):
    isz = 4 if dtype == torch.float32 else 8
    obs_dtype = obs_dtype or dtype
    osz = torch.empty((), dtype=obs_dtype).element_size()
    o_obs, o_rew, o_flg, _ = layout
    obs = block[o_obs:o_obs + n * stride * osz].view(obs_dtype).view(n, stride)
    reward = block[o_rew:o_rew + n * isz].view(dtype)
    flags = block[o_flg:o_flg + n]
    return obs, reward, flags


class StepInfo(dict):
    """``info`` of a batched step.  ``flags`` (uint8 DD_* bits of THIS step) is always present;
    the derived boolean / counter views are materialised only when asked for."""

    def __init__(self, env: "BatchedDroneEnv", flags: torch.Tensor):
        super().__init__(flags=flags)
        self._env = env

    def __missing__(self, key):
        f = dict.__getitem__(self, "flags")
        if key == "landed":
            v = (f & nv.LANDED) != 0
        elif key == "crashed":
            v = (f & nv.CRASHED) != 0
        elif key == "truncated":
            v = (f & nv.TRUNCATED) != 0
        elif key == "cause":
            v = (f & nv.CAUSE_MASK) >> 4
        elif key == "steps":
            v = self._env.steps
        elif key == "episode_return":
            v = self._env.att_fuel[:, 3]
        elif key == "final_obs":
            v = self._env.final_obs
        else:
            raise KeyError(key)
        self[key] = v
        return v


class BatchedDroneEnv:
    """N ``DroneGame`` instances on one GPU.

    ``DroneGame(render_mode=None, randomize_drone=False, randomize_platform=True)`` defaults are
    kept (game_engine.py:14).  ``dtype=torch.float64`` selects the exact-parity instantiation of the
    kernels (the reference computes in float64); ``torch.float32`` is the throughput one.

    ``obs_dtype``: element dtype of the observations the env hands out (``obs``, ``final_obs``, ``step_host``'s
    ``io['obs']``, ``rollout(obs_out=...)``).  ``None`` / ``torch.float32``: the state dtype.  ``torch.float16`` /
    ``torch.bfloat16`` (float32 state only): the kernels write 16-bit rows, each value exactly the float32 one
    rounded to nearest even (``obs32.to(obs_dtype)``, bit for bit), at half the observation bytes; state, rewards,
    flags and statistics stay as they are.  With ``obs_stride=16`` the ``steps`` column is converted too: exact up to
    2048 steps in float16, 256 in bfloat16.  ``policy_rollout`` ignores it (its ``obs`` rows are always float32).

    ``param_sets`` / ``param_index`` / ``resample_param_sets``: per-env physics (domain randomisation, curricula per env
    group), see ``set_param_sets``.
    """

    def __init__(self, num_envs: int, device="cuda", seed: int = 0, randomize_drone: bool = False,
                 randomize_platform: bool = True, max_steps: Optional[int] = None, auto_reset: bool = True,
                 dtype: torch.dtype = torch.float32, env_id_base: int = 0, obs_stride: int = nv.OBS_DIM,
                 want_final_obs: bool = False, params: Optional[nv.DDParams] = None, launch_flags: int = 0,
                 shaping: str = "ppo", obs_dtype: Optional[torch.dtype] = None, param_sets=None,
                 param_index: Optional[torch.Tensor] = None, resample_param_sets: bool = False):
        if dtype not in (torch.float32, torch.float64):
            raise ValueError("dtype must be torch.float32 or torch.float64")
        if obs_dtype is None or obs_dtype == dtype or (obs_dtype == torch.float32 and dtype == torch.float32):
            obs_dtype, obs_format = dtype, nv.OBS_NATIVE
        elif obs_dtype in _OBS_FORMATS:
            if dtype != torch.float32:
                raise ValueError("16-bit observations (obs_dtype float16 / bfloat16) need dtype=torch.float32")
            obs_format = _OBS_FORMATS[obs_dtype]
        else:
            raise ValueError("obs_dtype must be None, torch.float32, torch.float16 or torch.bfloat16")
        if obs_stride not in (15, 16):
            raise ValueError("obs_stride must be 15 or 16")
        if num_envs < 0:
            raise ValueError("num_envs must be >= 0")
        if shaping not in ("ppo", "pg"):
            raise ValueError("shaping must be 'ppo' (Actor_Critic_PPO / Actor_Critic_Basic calc_reward) or 'pg' "
                             "(Policy_Gradients calc_reward)")
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise ValueError("BatchedDroneEnv runs on a CUDA device only (there is no CPU fallback)")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self._lib = nv.lib()
        self.num_envs = n = int(num_envs)
        self.dtype = dtype
        self.obs_dtype = obs_dtype
        self.obs_stride = int(obs_stride)
        self._params = nv.DDParams.from_buffer_copy(params if params is not None else nv.default_params())
        dev = self.device
        # ---- state in HBM (layout: include/drone_b200.h DDState) ----
        self.pos_vel = torch.zeros(n, 4, dtype=dtype, device=dev)      # x, y, vx, vy
        self.att_fuel = torch.zeros(n, 4, dtype=dtype, device=dev)     # angle, angvel, fuel, ep_return
        self.platform = torch.zeros(n, 2, dtype=dtype, device=dev)     # px, py
        self.steps = torch.zeros(n, dtype=torch.int32, device=dev)
        self.episode = torch.zeros(n, dtype=torch.int32, device=dev)   # uint32 bit pattern
        self.flags = torch.zeros(n, dtype=torch.uint8, device=dev)
        self.prev_dist = torch.full((n,), float("nan"), dtype=dtype, device=dev)   # N2 shaping bookkeeping
        # ---- per-step outputs: ONE block [obs | reward | step_flags] (256-byte aligned parts), so that the
        #      host-buffer step moves them with a single device->host copy ----
        self._out_layout = _out_layout(n, self.obs_stride, dtype, obs_dtype)
        self._out_block = torch.zeros(self._out_layout[-1], dtype=torch.uint8, device=dev)
        self.obs, self.reward, self.step_flags = _carve(self._out_block, self._out_layout, n, self.obs_stride, dtype, obs_dtype)
        self.final_obs = torch.zeros(n, self.obs_stride, dtype=obs_dtype, device=dev) if want_final_obs else None
        self._packed = torch.zeros(n, dtype=torch.uint8, device=dev)
        # ---- episode statistics (K3) ----
        self.stats_slots = torch.zeros(nv.STATS_SLOTS, nv.STATS_WORDS, dtype=torch.int64, device=dev)
        self._stats_out = torch.zeros(nv.STATS_WORDS, dtype=torch.int64, device=dev)

        self._state = nv.DDState(self.pos_vel.data_ptr(), self.att_fuel.data_ptr(), self.platform.data_ptr(),
                                 self.steps.data_ptr(), self.episode.data_ptr(), self.flags.data_ptr(),
                                 nv.F32 if dtype == torch.float32 else nv.F64, 0, self.prev_dist.data_ptr())
        self._cfg = nv.DDEnvConfig(int(seed) & (2 ** 64 - 1), int(env_id_base), int(max_steps or 0),
                                   int(bool(auto_reset)), int(bool(randomize_drone)), int(bool(randomize_platform)),
                                   int(launch_flags), nv.SHAPING_PG if shaping == "pg" else nv.SHAPING_PPO, obs_format)
        self.shaping = shaping
        self._needs_reset = True
        self._plans: Dict[tuple, "nv.DDStepPlan"] = {}       # resolved dd_step launches (dd_step_plan), by (want_obs, stats)
        self._planned = self._lib.dd_step_planned
        self._prev_dist_stale = False                      # dd_step does not advance prev_dist (include/drone_b200.h)
        self.t_rollout = 0                                 # running step offset of the in-kernel RNG streams (t0 contract)
        # per-env parameter sets (set_param_sets): None = every env runs under self._params
        self._sets = None
        self._ps = None
        self._ps_table = None
        self.param_index: Optional[torch.Tensor] = None
        if param_sets is not None:
            self.set_param_sets(param_sets, param_index, resample_param_sets)
        elif param_index is not None or resample_param_sets:
            raise ValueError("param_index / resample_param_sets need param_sets")

    # ---- configuration ------------------------------------------------------------------------
    @property
    def seed(self) -> int:
        return self._cfg.seed

    @property
    def env_id_base(self) -> int:
        return self._cfg.env_id_base

    @property
    def max_steps(self) -> int:
        return self._cfg.max_steps

    @max_steps.setter
    def max_steps(self, v: Optional[int]) -> None:
        """Curriculum knob (Actor_Critic_PPO.ipynb c19:L13-17): takes effect on the next step."""
        self._cfg.max_steps = int(v or 0)
        self._plans.clear()

    @property
    def params(self) -> "nv.DDParams":
        """A COPY of the physics parameters (``DDParams``).  Writing a field of the returned struct changes nothing;
        assign a whole struct instead (``p = env.params; p.gravity = 0.5; env.params = p``): the setter copies it and
        drops the resolved step launches, which carry the derived constants, so that every later call -- ``step``,
        ``reset``, ``observe``, the rollouts -- runs with the new values."""
        return nv.DDParams.from_buffer_copy(self._params)

    @params.setter
    def params(self, p: "nv.DDParams") -> None:
        if not isinstance(p, nv.DDParams):
            raise TypeError("params must be a DDParams struct")
        if self._sets is not None:
            raise RuntimeError("per-env parameter sets are active, so params would not be used: call "
                               "set_param_sets(None) first, or set_param_sets(...) with the new sets")
        self._params = nv.DDParams.from_buffer_copy(p)
        self._plans.clear()

    # ---- per-env parameter sets --------------------------------------------------------------------
    def set_param_sets(self, sets, index: Optional[torch.Tensor] = None, resample: bool = False) -> None:
        """Give env i the physics of ``sets[min(param_index[i], len(sets) - 1)]`` (include/drone_b200.h, DDParamSets).

        ``sets``: a sequence of 1-64 ``DDParams`` structs (copied), or None to return every env to ``params``.
        ``index``: the set of each env (``[N]`` integers in [0, 255]); None means ``i % len(sets)``.  The env keeps it as
        ``param_index`` (uint8 ``[N]`` on the device): editing that tensor in place takes effect at the next call.
        ``resample``: every reset of an env -- ``reset`` and same-step auto-resets -- draws its next set from
        Philox(seed, env id, episode, stream 3), writes it to ``param_index`` and spawns under it; the step that ends an
        episode keeps the old set.  Drops the resolved step launches, like the ``params`` setter."""
        self._plans.clear()
        if sets is None:
            if index is not None or resample:
                raise ValueError("index / resample need sets")
            self._sets = self._ps = self._ps_table = self.param_index = None
            return
        sets = [nv.DDParams.from_buffer_copy(p) if isinstance(p, nv.DDParams) else p for p in sets]
        dt = nv.F32 if self.dtype == torch.float32 else nv.F64
        table = nv.build_param_table(sets, dt)            # validates count and types
        n = self.num_envs
        if index is None:
            idx = (torch.arange(n, device=self.device) % len(sets)).to(torch.uint8)
        else:
            idx = torch.as_tensor(index, device=self.device)
            if tuple(idx.shape) != (n,):
                raise ValueError("param_index must have shape [num_envs]")
            if idx.dtype != torch.uint8:
                if idx.numel() and (int(idx.min()) < 0 or int(idx.max()) > 255):
                    raise ValueError("param_index values must be in [0, 255]")
                idx = idx.to(torch.uint8)
            idx = idx.contiguous().clone()
        self._ps_table = torch.frombuffer(bytearray(table), dtype=torch.uint8).to(self.device)
        self._sets = sets
        self.param_index = idx
        self._ps = nv.DDParamSets(self._ps_table.data_ptr(), idx.data_ptr(), len(sets), dt,
                                  nv.PARAM_SETS_RESAMPLE if resample else 0, 0)

    @property
    def param_sets(self):
        """Copies of the active ``DDParams`` sets, or None when every env runs under ``params``."""
        return None if self._sets is None else [nv.DDParams.from_buffer_copy(p) for p in self._sets]

    @property
    def resample_param_sets(self) -> bool:
        return self._ps is not None and bool(self._ps.flags & nv.PARAM_SETS_RESAMPLE)

    def _pargs(self, name: str):
        """The C entry point ``name`` (or its _sets twin while sets are active) and its parameter argument."""
        if self._ps is None:
            return getattr(self._lib, name), C.byref(self._params)
        return getattr(self._lib, _SETS_ENTRY[name]), C.byref(self._ps)

    @property
    def launch_flags(self) -> int:
        return self._cfg.launch_flags

    @launch_flags.setter
    def launch_flags(self, v: int) -> None:
        """``native.LAUNCH_PDL`` etc. (include/drone_b200.h DD_LAUNCH_*)."""
        self._cfg.launch_flags = int(v)
        self._plans.clear()

    @property
    def auto_reset(self) -> bool:
        return bool(self._cfg.auto_reset)

    def _stream(self) -> int:
        return _current_stream_handle(self.device)

    # ---- DroneGame.reset ------------------------------------------------------------------------
    def reset(self, mask: Optional[torch.Tensor] = None, want_obs: bool = True) -> Optional[torch.Tensor]:
        """``DroneGame.reset()`` (game_engine.py:59-93) for all envs, or those with ``mask[i]`` set.
        Returns the observation tensor ``[N, obs_stride]`` (rows of unmasked envs are refreshed too);
        ``want_obs=False`` skips writing it (half of the reset's memory traffic) and returns None -- for callers
        that go straight into a rollout launch."""
        if not want_obs:
            m = None
            if mask is not None:
                m = mask.to(device=self.device).ne(0).to(torch.uint8).contiguous()
                if m.shape != (self.num_envs,):
                    raise ValueError("mask must have shape [num_envs]")
            fn, pa = self._pargs("dd_reset")
            nv.check(fn(C.byref(self._state), pa, C.byref(self._cfg), _ptr(m),
                        None, self.obs_stride, self.num_envs, self._stream()), "dd_reset")
            self._needs_reset = False
            return None
        m = None
        if mask is not None:
            m = mask.to(device=self.device).ne(0).to(torch.uint8).contiguous()
            if m.shape != (self.num_envs,):
                raise ValueError("mask must have shape [num_envs]")
            self.observe()                     # rows of unmasked envs: current state
        fn, pa = self._pargs("dd_reset")
        nv.check(fn(C.byref(self._state), pa, C.byref(self._cfg), _ptr(m),
                    self.obs.data_ptr(), self.obs_stride, self.num_envs, self._stream()), "dd_reset")
        self._needs_reset = False
        return self.obs

    def observe(self) -> torch.Tensor:
        """``get_state()`` (game_engine.py:140-177) of every env without stepping."""
        self._packed.fill_(nv.ACT_SKIP)
        fn, pa = self._pargs("dd_step")
        nv.check(fn(C.byref(self._state), pa, C.byref(self._cfg),
                                   self._packed.data_ptr(), self.obs.data_ptr(), self.obs_stride, None, None, None,
                                   None, self.num_envs, self._stream()), "dd_step(observe)")
        return self.obs

    # ---- actions ----------------------------------------------------------------------------------
    def pack_actions(self, actions: torch.Tensor) -> torch.Tensor:
        """``[N]`` uint8 bit-packed actions pass through; ``[N,3]`` (main, left, right; any non-zero
        value = pressed, game_engine.py:114-118) is packed on the device."""
        a = actions
        if a.device != self.device:
            a = a.to(self.device, non_blocking=True)
        if a.dim() == 1:
            if a.dtype != torch.uint8:
                a = a.to(torch.uint8)
            if a.shape[0] != self.num_envs:
                raise ValueError("actions must have shape [num_envs] or [num_envs, 3]")
            return a.contiguous()
        if a.shape != (self.num_envs, 3):
            raise ValueError("actions must have shape [num_envs] or [num_envs, 3]")
        if a.dtype == torch.bool:
            a3 = a.contiguous().view(torch.uint8)
        elif a.dtype == torch.uint8:
            a3 = a.contiguous()
        else:
            a3 = a.ne(0).contiguous().view(torch.uint8)
        nv.check(self._lib.dd_pack_actions(a3.data_ptr(), self._packed.data_ptr(), self.num_envs, self._stream()),
                 "dd_pack_actions")
        return self._packed

    # ---- DroneGame.step -----------------------------------------------------------------------------
    def step_raw(self, packed: torch.Tensor, want_obs: bool = True, stats: bool = True):
        """One ``DroneGame.step`` per env: exactly one kernel launch, no other device work.
        ``packed``: uint8 ``[N]`` on this device.  Returns ``(obs, reward, step_flags)`` -- the
        env's own output buffers, overwritten by the next call."""
        if self._needs_reset:
            raise RuntimeError("call reset() before step()")
        plan = self._plans.get((want_obs, stats))
        if plan is None:
            plan = self._make_plan(want_obs, stats)
        rc = self._planned(plan, packed.data_ptr(), _current_stream_handle(self.device))
        if rc:
            nv.check(rc, "dd_step_planned")
        self._prev_dist_stale = True
        return self.obs, self.reward, self.step_flags

    def _make_plan(self, want_obs: bool, stats: bool, obs=None, reward=None, flags=None, key=None):
        """Resolve the dd_step launch for this env's buffers once (include/drone_b200.h dd_step_plan): a step is then
        a 3-argument call.  ``obs`` / ``reward`` / ``flags`` override the destination addresses (e.g. device-mapped
        pinned host memory for ``step_host(zero_copy=True)``)."""
        plan = nv.DDStepPlan()
        fn, pa = self._pargs("dd_step_plan")
        nv.check(fn(
            C.byref(self._state), pa, C.byref(self._cfg),
            (self.obs.data_ptr() if obs is None else obs) if want_obs else None, self.obs_stride,
            self.reward.data_ptr() if reward is None else reward, self.step_flags.data_ptr() if flags is None else flags,
            _ptr(self.final_obs), self.stats_slots.data_ptr() if stats else None, self.num_envs, C.byref(plan)), "dd_step_plan")
        ref = C.pointer(plan)                              # a ctypes pointer object keeps the storage alive
        self._plans[(want_obs, stats) if key is None else key] = ref
        return ref

    def step(self, actions: torch.Tensor):
        """Gym-style: ``(obs [N,obs_stride], reward [N], done [N] bool, info)``.

        ``auto_reset=True``: on the terminating step ``reward``/``done``/``info`` describe the finished
        episode while ``obs`` is the first observation of the next one (``info['final_obs']`` holds the
        terminal observation when the env was built with ``want_final_obs=True``).
        ``auto_reset=False``: reference behaviour, frozen after done until ``reset()``."""
        packed = self.pack_actions(actions)
        obs, reward, flags = self.step_raw(packed)
        done = (flags & nv.DONE) != 0
        return obs, reward, done, StepInfo(self, flags)

    # ---- T steps in one launch ---------------------------------------------------------------------
    def _take_t0(self, t0: Optional[int], T: int) -> int:
        """The t0 contract of include/drone_b200.h: the in-kernel RNG streams (random actions, Bernoulli uniforms) are
        pure functions of (seed, env id, t0 + t).  ``t0=None`` uses this env's running counter and advances it by T, so
        consecutive rollouts draw fresh noise; an explicit ``t0`` is used as given and leaves the counter alone."""
        if t0 is not None:
            return int(t0) & 0xffffffff
        t = self.t_rollout
        self.t_rollout = (t + int(T)) & 0xffffffff
        return t

    def _fresh_prev_dist(self) -> None:
        """Before a shaped-reward rollout: if dd_step ran since the last one, prev_dist is stale -> 'no previous state'."""
        if self._prev_dist_stale:
            self.prev_dist.fill_(float("nan"))
            self._prev_dist_stale = False

    def rollout(self, T: int, policy: str = "random", actions: Optional[torch.Tensor] = None, t0: Optional[int] = None,
                reward_out: Optional[torch.Tensor] = None, done_out: Optional[torch.Tensor] = None,
                obs_out: Optional[torch.Tensor] = None, shaped_out: Optional[torch.Tensor] = None, stats: bool = True):
        """T steps per launch with the env state in registers (one state round trip per launch).
        ``policy``: 'trace' (``actions`` uint8 ``[T,N]``), 'random' (Philox, p=0.5 per thruster;
        examples/random_agent.py:27-31; ``t0=None`` continues this env's noise stream, see ``_take_t0``) or
        'bangbang' (main = vy > 1.5).  Optional ``[T,N]`` outputs (``obs_out[t]`` = observation AFTER step t, in
        ``obs_dtype``; ``reward_out`` / ``shaped_out`` in the state dtype);
        ``shaped_out`` receives the PPO notebook's client-side training reward (``calc_reward`` +
        time-out penalty, Actor_Critic_PPO.ipynb c7, c16:L89-93) computed in the same launch."""
        if self._needs_reset:
            raise RuntimeError("call reset() before rollout()")
        pol = POLICIES[policy]
        n = self.num_envs
        if pol == nv.POLICY_TRACE:
            if actions is None or actions.dtype != torch.uint8 or tuple(actions.shape) != (T, n):
                raise ValueError("policy='trace' needs uint8 actions of shape [T, num_envs]")
            actions = actions.contiguous()
        for name, t, shape in (("reward_out", reward_out, (T, n)), ("done_out", done_out, (T, n)),
                               ("shaped_out", shaped_out, (T, n)), ("obs_out", obs_out, (T, n, self.obs_stride))):
            if t is not None and (tuple(t.shape) != shape or not t.is_contiguous() or t.device != self.device):
                raise ValueError(f"{name} must be a contiguous {shape} tensor on {self.device}")
        for t in (reward_out, shaped_out):
            if t is not None and t.dtype != self.dtype:
                raise ValueError("reward_out / shaped_out must have the env dtype")
        if obs_out is not None and obs_out.dtype != self.obs_dtype:
            raise ValueError("obs_out must have the env's obs_dtype")
        if done_out is not None and done_out.dtype != torch.uint8:
            raise ValueError("done_out must be uint8")
        if shaped_out is not None:
            self._fresh_prev_dist()
        t0 = self._take_t0(t0, T) if pol == nv.POLICY_RANDOM else int(t0 or 0)
        fn, pa = self._pargs("dd_rollout_shaped")
        nv.check(fn(
            C.byref(self._state), pa, C.byref(self._cfg), pol, _ptr(actions), int(t0), int(T),
            _ptr(reward_out), _ptr(done_out), _ptr(obs_out), self.obs_stride, _ptr(shaped_out),
            self.stats_slots.data_ptr() if stats else None, n, self._stream()), "dd_rollout")

    def random_actions(self, T: int, t0: int = 0, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """The ``[T,N]`` uint8 trace that ``policy='random'`` draws in-kernel."""
        if out is None:
            out = torch.empty(T, self.num_envs, dtype=torch.uint8, device=self.device)
        nv.check(self._lib.dd_fill_random_actions(out.data_ptr(), self._cfg.seed, self._cfg.env_id_base, int(t0),
                                                  int(T), self.num_envs, self._stream()), "dd_fill_random_actions")
        return out

    # ---- episode statistics (K3) --------------------------------------------------------------------
    def stats_tensor(self) -> torch.Tensor:
        """int64[8] on device: episodes, landed, crashed, truncated, sum_return (2^-20 units),
        sum_length, env_steps (= sum_length + steps so far of the running episodes), reserved --
        accumulated since the last ``reset_stats()``."""
        nv.check(self._lib.dd_stats_collapse(self.stats_slots.data_ptr(), self.steps.data_ptr(), self.flags.data_ptr(),
                                             self.num_envs, self._stats_out.data_ptr(), self._stream()),
                 "dd_stats_collapse")
        return self._stats_out

    def reset_stats(self) -> None:
        self.stats_slots.zero_()

    def stats(self, reduce: bool = False) -> Dict[str, float]:
        """Host dict of the episode statistics (Actor_Critic_PPO.ipynb c21:L94-95,L158-159,L169);
        ``reduce=True`` all-reduces the 8 words over the default process group first."""
        from .distributed import allreduce_stats, stats_dict
        w = self.stats_tensor()
        if reduce:
            w = allreduce_stats(w.clone())
        return stats_dict(w)

    # ---- checkpoint / injection -----------------------------------------------------------------------
    def get_state(self) -> Dict[str, torch.Tensor]:
        """Copies of the raw (un-normalised) state, reference attribute names (drone.py:19-32,
        platform.py:19-20, game_engine.py:50-53); with parameter sets active also ``param_index``."""
        pv, af, pf = self.pos_vel, self.att_fuel, self.platform
        st = {
            "x": pv[:, 0].clone(), "y": pv[:, 1].clone(), "vx": pv[:, 2].clone(), "vy": pv[:, 3].clone(),
            "angle": af[:, 0].clone(), "angular_velocity": af[:, 1].clone(), "fuel": af[:, 2].clone(),
            "total_reward": af[:, 3].clone(), "platform_x": pf[:, 0].clone(), "platform_y": pf[:, 1].clone(),
            "steps": self.steps.clone(), "episode": self.episode.clone(), "flags": self.flags.clone(),
            "prev_dist": self.prev_dist.clone(),
        }
        if self.param_index is not None:
            st["param_index"] = self.param_index.clone()
        return st

    def set_state(self, state: Dict[str, torch.Tensor]) -> None:
        """Overwrite any subset of the state tensors (each ``[N]``)."""
        cols = {"x": (self.pos_vel, 0), "y": (self.pos_vel, 1), "vx": (self.pos_vel, 2), "vy": (self.pos_vel, 3),
                "angle": (self.att_fuel, 0), "angular_velocity": (self.att_fuel, 1), "fuel": (self.att_fuel, 2),
                "total_reward": (self.att_fuel, 3), "platform_x": (self.platform, 0), "platform_y": (self.platform, 1)}
        for k, v in state.items():
            if k not in _STATE_KEYS and not (k == "param_index" and self.param_index is not None):
                raise KeyError(k)
            v = torch.as_tensor(v, device=self.device)
            if k in cols:
                buf, j = cols[k]
                buf[:, j] = v.to(self.dtype)
            else:
                getattr(self, k).copy_(v.to(getattr(self, k).dtype))
        self._needs_reset = False

    def inject(self, x, y, platform_x, platform_y) -> torch.Tensor:
        """``g.reset(); g.drone.reset(x, y); g.platform.reset(px, py)`` for every env (the parity
        tests' way of starting from identical states).  Returns the observation."""
        n, dev = self.num_envs, self.device
        z = torch.zeros(n, dtype=self.dtype, device=dev)
        self.set_state({
            "x": x, "y": y, "platform_x": platform_x, "platform_y": platform_y,
            "vx": z, "vy": z, "angle": z, "angular_velocity": z, "total_reward": z,
            "fuel": self._max_fuel(),
            "steps": torch.zeros(n, dtype=torch.int32, device=dev),
            "flags": torch.zeros(n, dtype=torch.uint8, device=dev),
            "episode": self.episode + 1,
        })
        self.prev_dist.fill_(float("nan"))
        return self.observe()

    def _max_fuel(self) -> torch.Tensor:
        """``[N]``: each env's ``max_fuel`` (its parameter set's, when sets are active)."""
        if self._sets is None:
            return torch.full((self.num_envs,), float(self._params.max_fuel), dtype=self.dtype, device=self.device)
        mf = torch.tensor([p.max_fuel for p in self._sets], dtype=self.dtype, device=self.device)
        return mf[self.param_index.long().clamp(max=len(self._sets) - 1)]

    # ---- host-buffer entry point (what a CPU-side caller such as the socket shim uses) -----------------
    def make_host_io(self):
        """Pinned host buffers for ``step_host``: ``actions`` (packed uint8 in) and ONE packed output block with the
        same layout as the device's, of which ``obs`` / ``reward`` / ``flags`` are views."""
        n = self.num_envs
        block = torch.zeros(self._out_layout[-1], dtype=torch.uint8, pin_memory=True)
        obs, reward, flags = _carve(block, self._out_layout, n, self.obs_stride, self.dtype, self.obs_dtype)
        return {"actions": torch.zeros(n, dtype=torch.uint8, pin_memory=True), "block": block,
                "obs": obs, "reward": reward, "flags": flags}

    def step_host(self, io, mode: str = "copy", actions: Optional[torch.Tensor] = None, wait: bool = True):
        """HOST in / HOST out step: copies ``actions`` (pinned host memory, packed uint8 [N]; default
        ``io['actions']``) to the device, steps, and returns with obs / reward / flags of the step in ``io``
        (pinned host memory).  ``wait=False`` returns at once with a ``torch.cuda.Event`` instead; ``io`` holds the
        step's results once ``event.synchronize()`` returns -- a caller that owns several envs (shards) can so keep
        the device->host copy of one env's step in flight while the next env's actions go up and its kernel runs
        (call it under ``torch.cuda.stream(...)`` with one stream per env in flight).

        ``mode='copy'``      the kernel writes its packed output block in HBM, ONE device->host copy brings it back
                             (65 B per env-step with float32 observations, 35 B with 16-bit ones: this copy is what
                             bounds the call, PCIe);
        ``mode='zero_copy'`` the kernel's obs / reward / flags destinations ARE the pinned host buffers (device-mapped
                             under UVA): the observation tile of each CTA leaves the SM as one TMA bulk store straight
                             over PCIe, there is no HBM round trip and no separate copy."""
        stream = torch.cuda.current_stream(self.device)
        self._packed.copy_(io["actions"] if actions is None else actions, non_blocking=True)
        if mode == "copy":
            self.step_raw(self._packed)
            io["block"].copy_(self._out_block, non_blocking=True)
        elif mode == "zero_copy":
            if self._needs_reset:
                raise RuntimeError("call reset() before step()")
            key = ("host", io["block"].data_ptr())
            plan = self._plans.get(key)
            if plan is None:
                plan = self._make_plan(True, True, obs=io["obs"].data_ptr(), reward=io["reward"].data_ptr(),
                                       flags=io["flags"].data_ptr(), key=key)
            rc = self._planned(plan, self._packed.data_ptr(), stream.cuda_stream)
            if rc:
                nv.check(rc, "dd_step_planned")
            self._prev_dist_stale = True
        else:
            raise ValueError("mode must be 'copy' or 'zero_copy'")
        if wait:
            stream.synchronize()
            return None
        ev = torch.cuda.Event()
        ev.record(stream)
        return ev

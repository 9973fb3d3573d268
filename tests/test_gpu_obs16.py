"""16-bit observation outputs on the GPU (``BatchedDroneEnv(obs_dtype=torch.float16 / torch.bfloat16)``).

Every test runs twin envs with the same seed and inputs, one with float32 observations and one with a 16-bit format.
The 16-bit rows must be the float32 rows converted with round-to-nearest-even (``obs32.to(fmt)``, bit for bit), and
everything else -- reward, flags, state, Philox spawns, statistics -- bit-identical."""
import ctypes as C
import importlib
import os

import numpy as np
import pytest
import torch

from param_reference import HARD, make_params

pytestmark = pytest.mark.gpu
dd = importlib.import_module("reinforcement-learning-101_b200")
envmod = importlib.import_module("reinforcement-learning-101_b200.env")
nv = dd.native
DEV = "cuda:0"
FMTS = {"f16": torch.float16, "bf16": torch.bfloat16}
BLOCKS = {128: nv.LAUNCH_BLOCK_128, 256: 0, 512: nv.LAUNCH_BLOCK_512}


def _bits(t):
    return t.contiguous().view(torch.int16) if t.element_size() == 2 else t.contiguous().view(torch.int32)


def _eq16(o16, o32, fmt):
    """o16 (16-bit) == o32 converted to fmt, bit for bit."""
    assert o16.dtype == fmt and o32.dtype == torch.float32
    return torch.equal(_bits(o16), _bits(o32.to(fmt)))


def _same_state(a, b):
    for k in ("pos_vel", "att_fuel", "platform", "prev_dist"):
        assert torch.equal(_bits(getattr(a, k)), _bits(getattr(b, k))), k
    for k in ("steps", "episode", "flags", "stats_slots"):
        assert torch.equal(getattr(a, k), getattr(b, k)), k


def _twins(n, fmt, **kw):
    return (dd.BatchedDroneEnv(n, device=DEV, **kw), dd.BatchedDroneEnv(n, device=DEV, obs_dtype=fmt, **kw))


def _actions(T, n, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    a = torch.randint(0, 8, (T, n), device=DEV, dtype=torch.uint8, generator=g)
    a[(torch.rand(T, n, device=DEV, generator=g) < 0.02)] = nv.ACT_SKIP
    return a


def test_obs_dtype_arguments():
    e = dd.BatchedDroneEnv(8, device=DEV)
    assert e.obs_dtype == torch.float32 and e.obs.dtype == torch.float32
    assert dd.BatchedDroneEnv(8, device=DEV, obs_dtype=torch.float32).obs_dtype == torch.float32
    assert dd.BatchedDroneEnv(8, device=DEV, dtype=torch.float64).obs_dtype == torch.float64
    b = dd.BatchedDroneEnv(8, device=DEV, obs_dtype=torch.bfloat16, want_final_obs=True, obs_stride=16)
    assert b.obs.dtype == b.final_obs.dtype == torch.bfloat16 and b.reward.dtype == torch.float32
    with pytest.raises(ValueError):
        dd.BatchedDroneEnv(8, device=DEV, obs_dtype=torch.float16, dtype=torch.float64)
    for bad in (torch.float64, torch.int16, torch.uint8, "float16"):
        with pytest.raises(ValueError):
            dd.BatchedDroneEnv(8, device=DEV, obs_dtype=bad)
    b.reset()
    with pytest.raises(ValueError, match="obs_dtype"):
        b.rollout(4, obs_out=torch.zeros(4, 8, 16, device=DEV))
    with pytest.raises(ValueError):
        b.rollout(4, reward_out=torch.zeros(4, 8, device=DEV, dtype=torch.bfloat16))


@pytest.mark.parametrize("fmt", list(FMTS))
@pytest.mark.parametrize("block", list(BLOCKS))
@pytest.mark.parametrize("auto_reset", [True, False])
@pytest.mark.parametrize("stride", [15, 16])
@pytest.mark.parametrize("n", [1, 255, 257, 5000, 1 << 20])
def test_step_every_step(fmt, block, auto_reset, stride, n):
    f = FMTS[fmt]
    T = 300
    a, b = _twins(n, f, seed=3, randomize_drone=True, randomize_platform=True, max_steps=90, auto_reset=auto_reset,
                  obs_stride=stride, want_final_obs=True, launch_flags=BLOCKS[block] | nv.LAUNCH_PDL)
    assert _eq16(b.reset(), a.reset(), f)
    acts = _actions(T, n, seed=n + stride)
    for t in range(T):
        oa, ra, fa = a.step_raw(acts[t]); ob, rb, fb = b.step_raw(acts[t])
        assert _eq16(ob, oa, f), t
        assert torch.equal(_bits(ra), _bits(rb)) and torch.equal(fa, fb), t
        assert _eq16(b.final_obs, a.final_obs, f), t
    _same_state(a, b)
    sa = a.stats()
    assert sa == b.stats() and sa["episodes"] > 0
    if stride == 16:                                     # final_obs keeps no `steps` column, as with float32 rows
        assert not b.final_obs[:, 15].any()


@pytest.mark.parametrize("fmt", list(FMTS))
@pytest.mark.parametrize("stride", [15, 16])
def test_reset_observe_and_planned_step(fmt, stride):
    f = FMTS[fmt]
    n = 4097
    a, b = _twins(n, f, seed=9, randomize_drone=True, randomize_platform=True, max_steps=40, obs_stride=stride,
                  want_final_obs=True)
    assert _eq16(b.reset(), a.reset(), f)
    acts = _actions(60, n, seed=1)
    lib = nv.lib()
    for t in range(60):
        if t % 2:
            a.step_raw(acts[t]); b.step_raw(acts[t])            # dd_step_planned
        else:                                                   # dd_step with the same buffers
            for e in (a, b):
                nv.check(lib.dd_step(C.byref(e._state), C.byref(e._params), C.byref(e._cfg), acts[t].data_ptr(),
                                     e.obs.data_ptr(), stride, e.reward.data_ptr(), e.step_flags.data_ptr(),
                                     e.final_obs.data_ptr(), e.stats_slots.data_ptr(), n, e._stream()), "dd_step")
        assert _eq16(b.obs, a.obs, f) and _eq16(b.final_obs, a.final_obs, f), t
        assert torch.equal(a.reward, b.reward) and torch.equal(a.step_flags, b.step_flags)
    assert _eq16(b.observe(), a.observe(), f)
    m = (torch.arange(n, device=DEV) % 3 == 0)
    assert _eq16(b.reset(mask=m), a.reset(mask=m), f)
    _same_state(a, b)
    # planned == unplanned on one env
    c = dd.BatchedDroneEnv(n, device=DEV, seed=9, randomize_drone=True, randomize_platform=True, max_steps=40,
                           obs_stride=stride, want_final_obs=True, obs_dtype=f)
    c.set_state({k: v for k, v in b.get_state().items()})
    c.stats_slots.copy_(b.stats_slots)
    b.step_raw(acts[0])
    nv.check(lib.dd_step(C.byref(c._state), C.byref(c._params), C.byref(c._cfg), acts[0].data_ptr(), c.obs.data_ptr(),
                         stride, c.reward.data_ptr(), c.step_flags.data_ptr(), c.final_obs.data_ptr(),
                         c.stats_slots.data_ptr(), n, c._stream()), "dd_step")
    assert torch.equal(_bits(b.obs), _bits(c.obs)) and torch.equal(b.step_flags, c.step_flags)


@pytest.mark.parametrize("fmt", list(FMTS))
@pytest.mark.parametrize("policy", ["trace", "random", "bangbang"])
@pytest.mark.parametrize("n", [1000, 1001, 4096 + 4])
@pytest.mark.parametrize("stride", [15, 16])
def test_rollout_obs_tn(fmt, policy, n, stride):
    """obs_tn of dd_rollout (no other outputs) and dd_rollout_shaped: n % 8 == 0 takes the TMA bulk store, the others
    the fallback."""
    f = FMTS[fmt]
    T = 37
    a, b = _twins(n, f, seed=4, randomize_drone=True, randomize_platform=True, max_steps=25, obs_stride=stride)
    a.reset(want_obs=False); b.reset(want_obs=False)
    acts = _actions(T, n, seed=2) if policy == "trace" else None
    oa = torch.full((T, n, stride), 7.0, device=DEV); ob = torch.full((T, n, stride), 7.0, device=DEV, dtype=f)
    a.rollout(T, policy, actions=acts, obs_out=oa, t0=0); b.rollout(T, policy, actions=acts, obs_out=ob, t0=0)
    assert _eq16(ob, oa, f)
    _same_state(a, b)
    ra, rb = torch.empty(T, n, device=DEV), torch.empty(T, n, device=DEV)
    da, db = torch.empty(T, n, device=DEV, dtype=torch.uint8), torch.empty(T, n, device=DEV, dtype=torch.uint8)
    sa, sb = torch.empty(T, n, device=DEV), torch.empty(T, n, device=DEV)
    a.rollout(T, policy, actions=acts, obs_out=oa, reward_out=ra, done_out=da, shaped_out=sa, t0=T)
    b.rollout(T, policy, actions=acts, obs_out=ob, reward_out=rb, done_out=db, shaped_out=sb, t0=T)
    assert _eq16(ob, oa, f)
    assert torch.equal(_bits(ra), _bits(rb)) and torch.equal(da, db) and torch.equal(_bits(sa), _bits(sb))
    _same_state(a, b)
    assert (da != 0).any()


@pytest.mark.parametrize("fmt", list(FMTS))
def test_sharded_graphs_eager_and_fp32(fmt):
    f = FMTS[fmt]
    S, N, k = 3, 5000, 41
    kw = dict(seed=12, randomize_drone=True, randomize_platform=True, max_steps=30, trace_len=7)
    g16 = dd.ShardedDroneEnv(S, N, device=DEV, obs_dtype=f, **kw)
    e16 = dd.ShardedDroneEnv(S, N, device=DEV, obs_dtype=f, use_graphs=False, **kw)
    g32 = dd.ShardedDroneEnv(S, N, device=DEV, **kw)
    for e in (g16, e16, g32):
        e.reset(); e.random_trace()
        e.run(k); e.run(k)
        e.join()
    assert g16.graph_replays > 0 and e16.eager_launches == 2 * k
    for s in range(S):
        assert torch.equal(_bits(g16.shards[s].obs), _bits(e16.shards[s].obs))
        assert _eq16(g16.shards[s].obs, g32.shards[s].obs, f)
        _same_state(g16.shards[s], e16.shards[s]); _same_state(g16.shards[s], g32.shards[s])
    assert g16.stats() == g32.stats()
    obs, rew, fl = g16.step_all(torch.ones(S, N, dtype=torch.uint8, device=DEV))
    obs32, rew32, fl32 = g32.step_all(torch.ones(S, N, dtype=torch.uint8, device=DEV))
    for s in range(S):
        assert _eq16(obs[s], obs32[s], f) and torch.equal(rew[s], rew32[s]) and torch.equal(fl[s], fl32[s])


@pytest.mark.parametrize("fmt", list(FMTS))
@pytest.mark.parametrize("mode", ["copy", "zero_copy"])
@pytest.mark.parametrize("stride", [15, 16])
def test_step_host(fmt, mode, stride):
    f = FMTS[fmt]
    n = 3001
    a = dd.BatchedDroneEnv(n, device=DEV, seed=8, randomize_drone=True, max_steps=50, obs_stride=stride, obs_dtype=f)
    b = dd.BatchedDroneEnv(n, device=DEV, seed=8, randomize_drone=True, max_steps=50, obs_stride=stride, obs_dtype=f)
    c32 = dd.BatchedDroneEnv(n, device=DEV, seed=8, randomize_drone=True, max_steps=50, obs_stride=stride)
    a.reset(); b.reset(); c32.reset()
    io = a.make_host_io()
    assert io["obs"].dtype == f and io["reward"].dtype == torch.float32 and io["obs"].is_pinned()
    acts = _actions(80, n, seed=5)
    for t in range(80):
        io["actions"].copy_(acts[t].cpu())
        a.step_host(io, mode=mode)
        ob, rb, fb = b.step_raw(acts[t]); oc, rc, fc = c32.step_raw(acts[t])
        assert torch.equal(_bits(io["obs"]), _bits(ob.cpu())), t
        assert torch.equal(io["reward"], rb.cpu()) and torch.equal(io["flags"], fb.cpu()), t
        assert _eq16(ob, oc, f), t
    _same_state(a, b)


@pytest.mark.parametrize("fmt", list(FMTS))
def test_hard_physics_generic_kernels(fmt):
    """Non-default parameters (the generic, constant-bank builds): the same conversion rule."""
    f = FMTS[fmt]
    n, T = 20000, 150
    p = make_params(nv, **HARD)
    a, b = _twins(n, f, seed=21, randomize_drone=True, randomize_platform=True, max_steps=80, want_final_obs=True,
                  params=p)
    assert _eq16(b.reset(), a.reset(), f)
    acts = _actions(T, n, seed=11)
    for t in range(T):
        oa, ra, fa = a.step_raw(acts[t]); ob, rb, fb = b.step_raw(acts[t])
        assert _eq16(ob, oa, f) and _eq16(b.final_obs, a.final_obs, f), t
        assert torch.equal(_bits(ra), _bits(rb)) and torch.equal(fa, fb), t
    oa = torch.empty(20, n, 15, device=DEV); ob = torch.empty(20, n, 15, device=DEV, dtype=f)
    a.rollout(20, "random", obs_out=oa); b.rollout(20, "random", obs_out=ob)
    assert _eq16(ob, oa, f)
    _same_state(a, b)
    assert a.stats()["episodes"] > 0


@pytest.mark.parametrize("fmt", list(FMTS))
def test_policy_rollout_keeps_fp32_obs(golden_dir, fmt):
    d = np.load(os.path.join(golden_dir, "policy_v1.npz"))
    sd = {k: torch.from_numpy(d[k]) for k in d.files if k.startswith("network")}
    blob = dd.PolicyBlob(sd, device=DEV)
    n, T = 3000, 16
    a, b = _twins(n, FMTS[fmt], seed=2, randomize_drone=True, randomize_platform=True, max_steps=40)
    a.reset(); b.reset()
    oa = dd.policy_rollout(a, blob, T, sample=True, t0=1, want="arldo")
    ob = dd.policy_rollout(b, blob, T, sample=True, t0=1, want="arldo")
    assert ob["obs"].dtype == torch.float32
    for k in oa:
        assert torch.equal(_bits(oa[k]) if oa[k].is_floating_point() else oa[k],
                           _bits(ob[k]) if ob[k].is_floating_point() else ob[k]), k
    _same_state(a, b)


# ---- guard bands (the pattern of test_gpu_guardbands.py) -------------------------------------------------------------
CANARY, GAP = 0xA5, 1024


class Arena:
    def __init__(self, nbytes):
        self.buf = torch.full((nbytes,), CANARY, dtype=torch.uint8, device=DEV)
        self.off, self.used = GAP, []

    def carve(self, shape, dtype, fill=0):
        nb = int(np.prod(shape)) * torch.empty((), dtype=dtype).element_size()
        lo = -(-self.off // 256) * 256
        v = self.buf[lo:lo + nb].view(dtype).view(*shape)
        if fill is not None:
            v.fill_(fill)
        self.used.append((lo, lo + nb))
        self.off = lo + nb + GAP
        assert self.off + GAP <= self.buf.numel(), "arena too small"
        return v

    def check(self, what=""):
        mask = torch.ones(self.buf.numel(), dtype=torch.bool, device=DEV)
        for lo, hi in self.used:
            mask[lo:hi] = False
        bad = (self.buf != CANARY) & mask
        assert not bool(bad.any()), f"{what}: guard bytes overwritten at {bad.nonzero().flatten()[:8].tolist()}"


def _armour(env, arena):
    n, dt, st = env.num_envs, env.dtype, env.obs_stride
    env.pos_vel = arena.carve((n, 4), dt); env.att_fuel = arena.carve((n, 4), dt); env.platform = arena.carve((n, 2), dt)
    env.steps = arena.carve((n,), torch.int32); env.episode = arena.carve((n,), torch.int32)
    env.flags = arena.carve((n,), torch.uint8); env.prev_dist = arena.carve((n,), dt, fill=float("nan"))
    env._out_block = arena.carve((env._out_layout[-1],), torch.uint8)
    env.obs, env.reward, env.step_flags = envmod._carve(env._out_block, env._out_layout, n, st, dt, env.obs_dtype)
    env.final_obs = arena.carve((n, st), env.obs_dtype)
    env._packed = arena.carve((n,), torch.uint8)
    env.stats_slots = arena.carve((nv.STATS_SLOTS, nv.STATS_WORDS), torch.int64)
    env._stats_out = arena.carve((nv.STATS_WORDS,), torch.int64)
    env._state = nv.DDState(env.pos_vel.data_ptr(), env.att_fuel.data_ptr(), env.platform.data_ptr(), env.steps.data_ptr(),
                            env.episode.data_ptr(), env.flags.data_ptr(), nv.F32, 0, env.prev_dist.data_ptr())
    env._plans.clear()
    return env


@pytest.mark.parametrize("fmt", list(FMTS))
@pytest.mark.parametrize("stride", [15, 16])
@pytest.mark.parametrize("n", [1, 255, 1000, 1024, 4097, 8192])
def test_16bit_outputs_stay_inside_their_buffers(fmt, stride, n):
    f = FMTS[fmt]
    kw = dict(seed=6, randomize_drone=True, randomize_platform=True, max_steps=25, auto_reset=True, want_final_obs=True,
              obs_stride=stride, obs_dtype=f)
    arena = Arena(32 << 20)
    a = _armour(dd.BatchedDroneEnv(n, device=DEV, **kw), arena)
    b = dd.BatchedDroneEnv(n, device=DEV, **kw)
    a.reset(); b.reset()
    arena.check("dd_reset")
    T = 40
    acts = _actions(T, n, seed=n)
    for t in range(T):
        oa, ra, fa = a.step_raw(acts[t]); ob, rb, fb = b.step_raw(acts[t])
        assert torch.equal(_bits(oa), _bits(ob)) and torch.equal(_bits(a.final_obs), _bits(b.final_obs))
    arena.check("dd_step")
    m = (torch.arange(n, device=DEV) % 3 == 0)
    a.reset(mask=m); b.reset(mask=m)
    arena.check("masked dd_reset + observe")
    obs = arena.carve((T, n, stride), f)
    a.rollout(T, "random", obs_out=obs)
    arena.check("dd_rollout")
    sh = arena.carve((T, n), torch.float32)
    a.rollout(T, "bangbang", obs_out=obs, shaped_out=sh)
    arena.check("dd_rollout_shaped")
    ob = torch.empty(T, n, stride, device=DEV, dtype=f)
    b.rollout(T, "random", obs_out=ob)
    b.rollout(T, "bangbang", obs_out=ob)
    assert torch.equal(_bits(obs), _bits(ob))

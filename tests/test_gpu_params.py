"""The kernels under non-default physics parameters.  GPU only (``-m gpu``).

Every env kernel exists twice: with config.py's defaults baked in as immediates (DEF = true) and reading ``Consts`` from
the kernel argument (DEF = false); ``params_are_default`` (and ``pol_params_default`` for the fused policy kernel) picks
one per launch.  Three parameter sets reach the generic instantiations:

  * the defaults with ``spawn_x_count = 601.0000001``: the derived constants are identical in both precisions, only the
    byte comparison fails, so every output must be BIT-IDENTICAL to the default-parameter run;
  * "hard" and "large" (tests/param_reference.py): checked against the float64 reference of tests/param_reference.py --
    float64 flags / counters exact and values to 1e-11, float32 under the fp32 rule of tests/test_gpu_parity.py with
    the band scaled by the world size;
  * the fused policy kernel under them must replay bit for bit through dd_rollout, and its landing shortcut must decide
    like the exact evaluation even where one float32 ulp of the coordinates exceeds its default 1e-3 px margin.

And: assigning new parameters to an env that already holds resolved step launches (or captured graphs) takes effect.
"""
import ctypes as C
import importlib
import os

import numpy as np
import pytest
import torch

from oracle import c_oracle as co
from param_reference import PARAM_SETS, ParamRef, make_params, world_scale

pytestmark = pytest.mark.gpu

dd = importlib.import_module("reinforcement-learning-101_b200")
nv = dd.native
DEV = "cuda:0"
BAND = 2e-4


def _eq(a, b):
    """torch.equal that treats NaN == NaN (prev_dist uses NaN for 'no previous state')."""
    if a.is_floating_point():
        a, b = torch.nan_to_num(a, nan=-12345.0), torch.nan_to_num(b, nan=-12345.0)
    return torch.equal(a, b)


def _same_state(a, b):
    sa, sb = a.get_state(), b.get_state()
    for k in sa:
        assert _eq(sa[k], sb[k]), k


def _close32(a, b):
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    return np.abs(a - b) <= 1e-5 * np.maximum(np.abs(b), 1.0)


def _generic_defaults():
    """config.py's values through the generic kernels: (uint32) 601.0000001 == 601, but the bytes differ."""
    p = nv.default_params()
    p.spawn_x_count = 601.0000001
    return p


def _pair(n, dtype, **kw):
    a = dd.BatchedDroneEnv(n, device=DEV, dtype=dtype, **kw)
    b = dd.BatchedDroneEnv(n, device=DEV, dtype=dtype, params=_generic_defaults(), **kw)
    return a, b


def _t(a):
    return torch.as_tensor(np.ascontiguousarray(a), device=DEV)


@pytest.fixture(scope="module")
def policy_sd(golden_dir):
    d = np.load(os.path.join(golden_dir, "policy_v1.npz"))
    return {k: torch.from_numpy(d[k]) for k in d.files if k.startswith("network")}


# =================================================================================================
# generic instantiations at the default values: bit-identical to the immediates
# =================================================================================================
_STEP_CASES = [(dt, auto, obs, stride, blk) for dt in (torch.float32, torch.float64) for auto in (False, True)
               for obs in (False, True) for stride in (15, 16) for blk in ((0, 0x10, 0x20) if dt == torch.float32 else (0,))]


@pytest.mark.parametrize("dtype,auto,want_obs,stride,block", _STEP_CASES)
def test_generic_step_bit_identical(dtype, auto, want_obs, stride, block):
    n, T = 3001, 40
    kw = dict(seed=8, randomize_drone=True, randomize_platform=True, max_steps=25, auto_reset=auto, obs_stride=stride,
              want_final_obs=True, launch_flags=block)
    a, b = _pair(n, dtype, **kw)
    a.reset(); b.reset()
    A = a.random_actions(T)
    A[:, 5::11] |= nv.ACT_SKIP
    L = nv.lib()
    for t in range(T):
        for e in (a, b):
            if t % 2 == 0:                                      # dd_step_planned
                e.step_raw(A[t], want_obs=want_obs)
            else:                                               # dd_step
                nv.check(L.dd_step(C.byref(e._state), C.byref(e._params), C.byref(e._cfg), A[t].data_ptr(),
                                   e.obs.data_ptr() if want_obs else None, e.obs_stride, e.reward.data_ptr(),
                                   e.step_flags.data_ptr(), e.final_obs.data_ptr(), e.stats_slots.data_ptr(), n,
                                   e._stream()), "dd_step")
        assert torch.equal(a.step_flags, b.step_flags) and torch.equal(a.reward, b.reward), t
        if want_obs:
            assert torch.equal(a.obs, b.obs), t
        assert torch.equal(a.final_obs, b.final_obs), t
    _same_state(a, b)
    assert a.stats() == b.stats() and a.stats()["episodes"] > 0


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("policy", ["trace", "random", "bangbang"])
@pytest.mark.parametrize("outs", [False, True])
@pytest.mark.parametrize("shaping", ["ppo", "pg"])
def test_generic_rollout_bit_identical(dtype, policy, outs, shaping):
    n, T = 2049, 90
    kw = dict(seed=4, randomize_drone=True, randomize_platform=True, max_steps=60, auto_reset=True, shaping=shaping)
    a, b = _pair(n, dtype, **kw)
    a.reset(); b.reset()
    acts = a.random_actions(T, t0=500) if policy == "trace" else None
    res = []
    for e in (a, b):
        o = {}
        if outs:
            o = dict(reward_out=torch.empty(T, n, dtype=dtype, device=DEV), done_out=torch.empty(T, n, dtype=torch.uint8, device=DEV),
                     obs_out=torch.empty(T, n, 15, dtype=dtype, device=DEV), shaped_out=torch.empty(T, n, dtype=dtype, device=DEV))
        e.rollout(T, policy, actions=acts, t0=3, **o)
        res.append(o)
    for k in res[0]:
        assert torch.equal(res[0][k], res[1][k]), k
    _same_state(a, b)
    assert a.stats() == b.stats()


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_generic_reset_bit_identical(dtype):
    n = 5000
    a, b = _pair(n, dtype, seed=12, randomize_drone=True, randomize_platform=True, auto_reset=True)
    assert torch.equal(a.reset(), b.reset())
    a.rollout(30, "random"); b.rollout(30, "random")
    m = (torch.arange(n, device=DEV) % 3 == 0)
    assert torch.equal(a.reset(mask=m), b.reset(mask=m))
    a.reset(want_obs=False); b.reset(want_obs=False)
    _same_state(a, b)


def test_generic_policy_rollout_bit_identical(policy_sd):
    blob = dd.PolicyBlob(policy_sd, device=DEV)
    n, T = 1000, 60
    kw = dict(seed=21, randomize_drone=True, randomize_platform=True, max_steps=40, auto_reset=True, env_id_base=5000)
    for sample, want in ((True, "arldo"), (True, "arldops"), (False, "arldops")):
        a, b = _pair(n, torch.float32, **kw)
        a.reset(); b.reset()
        oa = dd.policy_rollout(a, blob, T, sample=sample, t0=3, want=want)
        ob = dd.policy_rollout(b, blob, T, sample=sample, t0=3, want=want)
        for k in oa:
            assert torch.equal(oa[k], ob[k]), (want, sample, k)
        _same_state(a, b)
        assert a.stats() == b.stats()


# =================================================================================================
# "hard" and "large" parameters against the float64 reference
# =================================================================================================
def _fixed_trace(T, n):
    A = co.random_actions(31, 0, 0, T, n)
    return np.where(co.random_actions(32, 0, 0, T, n) < 3, A & 1, A).astype(np.uint8)   # fewer spins: landings


@pytest.mark.parametrize("which", sorted(PARAM_SETS))
@pytest.mark.parametrize("n", [1, 257, 5000])
@pytest.mark.parametrize("policy", ["trace", "random"])
@pytest.mark.parametrize("auto", [False, True])
def test_f64_step_vs_reference(which, n, policy, auto):
    p = make_params(nv, **PARAM_SETS[which])
    T = 250
    kw = dict(seed=19, randomize_drone=True, randomize_platform=True, max_steps=150 if auto else 0, auto_reset=auto,
              env_id_base=300)
    r = ParamRef(n, p, **kw)
    e = dd.BatchedDroneEnv(n, device=DEV, dtype=torch.float64, params=p, want_final_obs=True, **kw)
    obs0 = e.reset().cpu().numpy()
    ro = r.reset()
    assert np.array_equal(e.pos_vel[:, :2].cpu().numpy(), np.stack([r.x, r.y], 1))
    assert np.array_equal(e.platform.cpu().numpy(), np.stack([r.px, r.py], 1))
    np.testing.assert_allclose(obs0, ro, rtol=1e-15, atol=0)
    A = _fixed_trace(T, n) if policy == "trace" else e.random_actions(T).cpu().numpy()
    Ad = _t(A)
    for t in range(T):
        was_done = (r.flags & nv.DONE) > 0                     # frozen envs report their flags but write no final obs
        obs, rew, fl = e.step_raw(Ad[t])
        oo, orr, od, of = r.step(A[t], want_final=True)
        fl = fl.cpu().numpy()
        assert np.array_equal(fl, od), t
        assert np.array_equal(e.steps.cpu().numpy(), r.steps) and np.array_equal(e.episode.cpu().numpy().astype(np.uint32), r.episode)
        np.testing.assert_allclose(obs.cpu().numpy(), oo, rtol=1e-11, atol=1e-11)
        np.testing.assert_allclose(rew.cpu().numpy(), orr, rtol=1e-11, atol=1e-11)
        d = ((fl & nv.DONE) > 0) & ~was_done
        np.testing.assert_allclose(e.final_obs.cpu().numpy()[d], of[d], rtol=1e-11, atol=1e-11)
    s = e.stats()
    assert (s["episodes"], s["landed"], s["crashed"], s["truncated"], s["sum_length"]) == r.stats.as_tuple()
    assert s["sum_return"] == pytest.approx(r.stats.sum_return, rel=1e-9, abs=1e-5 * max(1, s["episodes"]))


@pytest.mark.parametrize("which", sorted(PARAM_SETS))
def test_f32_step_vs_reference(which):
    p = make_params(nv, **PARAM_SETS[which])
    n, T = 8192, 250
    kw = dict(seed=29, randomize_drone=True, randomize_platform=True, auto_reset=False)
    r = ParamRef(n, p, **kw)
    e = dd.BatchedDroneEnv(n, device=DEV, dtype=torch.float32, params=p, **kw)
    obs0 = e.reset().cpu().numpy()
    ro = r.reset()
    assert np.array_equal(e.pos_vel[:, :2].cpu().numpy().astype(np.float64), np.stack([r.x, r.y], 1))
    assert np.array_equal(e.platform.cpu().numpy().astype(np.float64), np.stack([r.px, r.py], 1))
    assert _close32(obs0, ro).all()
    A = _fixed_trace(T, n)
    Ad = _t(A)
    band = BAND * world_scale(p)
    valid = np.ones(n, bool)
    flips = []
    for t in range(T):
        obs, rew, fl = e.step_raw(Ad[t])
        oo, orr, od = r.step(A[t])
        fl = fl.cpu().numpy()
        bad = valid & (fl != od)
        if bad.any():
            mg = r.threshold_margin()
            for i in np.nonzero(bad)[0]:
                assert mg[i] < band, f"env {i} step {t}: flags {fl[i]:#x} vs {od[i]:#x}, float64 margin {mg[i]:.3g}"
                flips.append((int(i), t, float(mg[i])))
            valid &= ~bad
        assert np.array_equal(e.steps.cpu().numpy()[valid], r.steps[valid])
        assert _close32(obs.cpu().numpy(), oo)[valid].all(), f"step {t}: obs outside fp32 tolerance"
        assert _close32(rew.cpu().numpy(), orr)[valid].all(), f"step {t}: reward outside fp32 tolerance"
    assert len(flips) <= 4, flips
    print(f"{which}: {len(flips)} float32 threshold flips {flips}")


@pytest.mark.parametrize("which", sorted(PARAM_SETS))
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_rollout_equals_stepping_under_params(which, dtype):
    p = make_params(nv, **PARAM_SETS[which])
    n, T = 4097, 120
    kw = dict(seed=3, randomize_drone=True, randomize_platform=True, max_steps=70, auto_reset=True, params=p, dtype=dtype)
    a = dd.BatchedDroneEnv(n, device=DEV, **kw); a.reset()
    b = dd.BatchedDroneEnv(n, device=DEV, obs_stride=16, **kw); b.reset()
    A = a.random_actions(T)
    rew = torch.empty(T, n, dtype=dtype, device=DEV)
    don = torch.empty(T, n, dtype=torch.uint8, device=DEV)
    obs = torch.empty(T, n, 16, dtype=dtype, device=DEV)
    b.rollout(T, policy="random", reward_out=rew, done_out=don, obs_out=obs)
    for t in range(T):
        o_, r_, f_ = a.step_raw(A[t])
        assert torch.equal(r_, rew[t]) and torch.equal(f_, don[t]) and torch.equal(o_, obs[t, :, :15]), t
    _same_state(a, b)
    assert a.stats() == b.stats() and a.stats()["episodes"] > 0


@pytest.mark.parametrize("which", sorted(PARAM_SETS))
def test_policy_rollout_replays_under_params(which, policy_sd):
    """K5 under non-default parameters: its actions replayed through dd_rollout give its rewards, flags, observations,
    final state and statistics bit for bit; obs[0] is reset()'s observation; the FAST instantiation equals the generic."""
    p = make_params(nv, **PARAM_SETS[which])
    blob = dd.PolicyBlob(policy_sd, device=DEV)
    n, T = 1000, 70
    kw = dict(seed=21, randomize_drone=True, randomize_platform=True, max_steps=50, auto_reset=True, dtype=torch.float32,
              env_id_base=5000, params=p)
    a = dd.BatchedDroneEnv(n, device=DEV, **kw); a.reset()
    b = dd.BatchedDroneEnv(n, device=DEV, **kw); b.reset()
    out = dd.policy_rollout(a, blob, T, sample=True, t0=3, want="arldop")
    rew = torch.empty(T, n, device=DEV); don = torch.empty(T, n, dtype=torch.uint8, device=DEV)
    obs = torch.empty(T, n, 15, device=DEV)
    b.rollout(T, "trace", actions=out["actions"], reward_out=rew, done_out=don, obs_out=obs)
    assert torch.equal(out["reward"], rew) and torch.equal(out["done"], don)
    _same_state(a, b)
    assert a.stats() == b.stats() and a.stats()["episodes"] > 0
    c = dd.BatchedDroneEnv(n, device=DEV, **kw)
    assert torch.equal(out["obs"][0], c.reset())
    assert torch.equal(out["obs"][1:], obs[:-1])
    f = dd.BatchedDroneEnv(n, device=DEV, **kw); f.reset()
    fast = dd.policy_rollout(f, blob, T, sample=True, t0=3, want="arldo")
    for k in ("actions", "reward", "logp", "done", "obs"):
        assert torch.equal(fast[k], out[k]), k
    _same_state(a, f)
    # threshold mode too
    g = dd.BatchedDroneEnv(n, device=DEV, **kw); g.reset()
    h = dd.BatchedDroneEnv(n, device=DEV, **kw); h.reset()
    thr = dd.policy_rollout(g, blob, T, sample=False, want="ard")
    h.rollout(T, "trace", actions=thr["actions"], reward_out=rew, done_out=don)
    assert torch.equal(thr["reward"], rew) and torch.equal(thr["done"], don)
    _same_state(g, h)


def test_policy_landing_shortcut_at_platform_edges_in_a_large_world(policy_sd):
    """K5 decides most landings from angle-addition sin / cos and falls back to the exact evaluation only near a platform
    edge.  Around x = 20,000 one float32 ulp is 1.95e-3 px, more than config.py's 1e-3 px margin, so the two can round
    the bottom centre to different sides of an edge.  Envs are placed with the post-update bottom centre within +-8 ulps
    of each of the four edges (turning, slow, upright); one K5 step without thrust must decide like dd_step."""
    p = make_params(nv, **PARAM_SETS["large"])
    n = 1 << 20
    rng = np.random.default_rng(2024)
    edge = np.arange(n) % 4                                   # left, right, top, bottom
    # target offset in ulps: half of the envs within one ulp of the edge, where a one-ulp disagreement flips the side
    k = np.where(rng.random(n) < 0.5, rng.integers(-1, 2, n), rng.integers(-8, 9, n))
    px = rng.integers(20100, 20700, n).astype(np.float64); py = rng.integers(20100, 20550, n).astype(np.float64)
    a1 = rng.uniform(-12, 12, n); w = rng.choice([-1, 1], n) * rng.uniform(0.5, 7.5, n)    # |w| <= 8: shortcut taken
    a0 = a1 - w
    vx = rng.uniform(-1.5, 1.5, n); vy = rng.uniform(-1.5, 1.2, n)
    hw, hh, half = p.platform_w / 2, p.platform_h / 2, p.drone_height / 2
    # bottom centre target (post-update): on the chosen edge, well inside along the other axis
    bx = np.where(edge == 0, px - hw, np.where(edge == 1, px + hw, px + rng.uniform(-0.8, 0.8, n) * hw))
    by = np.where(edge == 2, py - hh, np.where(edge == 3, py + hh, py + rng.uniform(-0.8, 0.8, n) * hh))
    vx1, vy1 = vx * p.drag, (vy + p.gravity) * p.drag
    rad = np.radians(a1)
    x0 = (bx + half * np.sin(rad) - vx1).astype(np.float32)
    y0 = (by - half * np.cos(rad) - vy1).astype(np.float32)
    f32 = lambda v: torch.tensor(np.asarray(v, np.float32), device=DEV)
    kw = dict(randomize_drone=False, randomize_platform=False, auto_reset=False, dtype=torch.float32, params=p)

    def state(x, y):
        return {"x": f32(x), "y": f32(y), "vx": f32(vx), "vy": f32(vy), "angle": f32(a0), "angular_velocity": f32(w),
                "fuel": f32(np.full(n, p.max_fuel)), "total_reward": f32(np.zeros(n)), "platform_x": f32(px),
                "platform_y": f32(py), "steps": torch.zeros(n, dtype=torch.int32, device=DEV),
                "flags": torch.zeros(n, dtype=torch.uint8, device=DEV), "episode": torch.ones(n, dtype=torch.int32, device=DEV)}

    zero = torch.zeros(n, dtype=torch.uint8, device=DEV)
    # one exact (dd_step) step from the first guess; measure where the bottom centre lands, in ulps of the coordinate
    probe = dd.BatchedDroneEnv(n, device=DEV, **kw)
    probe.set_state(state(x0, y0))
    probe.step_raw(zero)
    st = probe.get_state()
    x1, y1, ang1 = (st[c].cpu().numpy().astype(np.float64) for c in ("x", "y", "angle"))
    ulp = np.spacing(np.float32(20000.0)).astype(np.float64)
    assert np.all((np.abs(np.stack([x0, y0, x1, y1])) >= 16384) & (np.abs(np.stack([x0, y0, x1, y1])) < 32768))   # one binade
    r1 = np.radians(ang1)
    miss_x = np.rint((bx - (x1 - half * np.sin(r1))) / ulp)
    miss_y = np.rint((by - (y1 + half * np.cos(r1))) / ulp)
    on_x = edge < 2
    x0 = np.where(on_x, x0 + (miss_x + k) * ulp, x0).astype(np.float32)
    y0 = np.where(on_x, y0, y0 + (miss_y + k) * ulp).astype(np.float32)
    sd = {kk: v.clone() for kk, v in policy_sd.items()}
    sd["network.9.weight"].zero_(); sd["network.9.bias"].fill_(-50.0)      # probabilities ~0: never thrust
    blob = dd.PolicyBlob(sd, device=DEV)
    ref = dd.BatchedDroneEnv(n, device=DEV, **kw); ref.set_state(state(x0, y0))
    k5 = dd.BatchedDroneEnv(n, device=DEV, **kw); k5.set_state(state(x0, y0))
    _, rew_d, fl_d = ref.step_raw(zero)
    out = dd.policy_rollout(k5, blob, 1, sample=False, want="ard")
    assert torch.equal(out["actions"][0], zero)
    st = ref.get_state()
    bx1 = st["x"].double().cpu().numpy() - half * np.sin(np.radians(st["angle"].double().cpu().numpy()))
    by1 = st["y"].double().cpu().numpy() + half * np.cos(np.radians(st["angle"].double().cpu().numpy()))
    off = np.where(on_x, bx1 - bx, by1 - by) / ulp
    assert np.abs(off).max() <= 9.5                          # the envs sit where the shortcut's margin matters
    fl_d = fl_d.cpu().numpy(); fl_k = out["done"][0].cpu().numpy()
    diverged = np.nonzero(fl_d != fl_k)[0]
    landed = (fl_d & nv.LANDED) != 0
    print(f"landing shortcut: {diverged.size} of {n} envs decided differently from dd_step "
          f"({landed.sum()} landed, edges {np.bincount(edge[diverged], minlength=4).tolist()})")
    assert diverged.size == 0, [(int(i), int(edge[i]), int(k[i]), int(fl_d[i]), int(fl_k[i])) for i in diverged[:10]]
    assert 0.25 * n < landed.sum() < 0.75 * n
    assert torch.equal(out["reward"][0], rew_d)
    _same_state(ref, k5)


# =================================================================================================
# new parameters on a live env take effect
# =================================================================================================
def _moved(p0, **kw):
    p = nv.DDParams.from_buffer_copy(p0)
    for key, v in kw.items():
        setattr(p, key, v)
    return p


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_params_assignment_reaches_planned_steps(dtype):
    n = 1000
    kw = dict(seed=6, randomize_drone=True, randomize_platform=True, max_steps=80, auto_reset=True, dtype=dtype)
    e = dd.BatchedDroneEnv(n, device=DEV, **kw)
    e.reset()
    A = e.random_actions(20)
    e.step_raw(A[0]); e.step(A[1])                          # the step launches are resolved and cached
    e.params.gravity = 0.5                                  # a field write on the returned copy changes nothing
    assert e.params.gravity == nv.default_params().gravity
    for new in (_moved(e.params, gravity=0.5), _moved(nv.default_params(), drag=0.9, main_thrust=1.1, land_speed=2.7)):
        e.params = new
        fresh = dd.BatchedDroneEnv(n, device=DEV, params=new, **kw)
        fresh.set_state(e.get_state())
        for t in range(2, 12):
            o1, r1, f1 = e.step_raw(A[t])
            o2, r2, f2 = fresh.step_raw(A[t])
            assert torch.equal(o1, o2) and torch.equal(r1, r2) and torch.equal(f1, f2), t
        _same_state(e, fresh)
        assert e.params.gravity == new.gravity
    with pytest.raises(TypeError):
        e.params = {"gravity": 0.5}


def test_params_assignment_reaches_sharded_graphs():
    S, N = 2, 512
    kw = dict(seed=7, randomize_drone=True, randomize_platform=True, max_steps=80, auto_reset=True, dtype=torch.float64)
    s = dd.ShardedDroneEnv(S, N, device=DEV, chains=2, **kw)
    s.reset()
    A = torch.stack([torch.stack([sh.random_actions(1, t0=t)[0] for sh in s.shards]) for t in range(12)])
    s.step_all(A[0]); s.step_all(A[1])
    assert s.graphs_cached > 0
    new = _moved(nv.default_params(), gravity=0.45, angular_drag=0.8)
    s.params = new
    assert s.graphs_cached == 0 and all(sh.params.gravity == 0.45 for sh in s.shards)
    fresh = [dd.BatchedDroneEnv(N, device=DEV, env_id_base=i * N, params=new, **kw) for i in range(S)]
    for f, sh in zip(fresh, s.shards):
        f.set_state(sh.get_state())
    for t in range(2, 12):
        obs, rew, fl = s.step_all(A[t])
        for i, f in enumerate(fresh):
            o2, r2, f2 = f.step_raw(A[t, i])
            assert torch.equal(obs[i], o2) and torch.equal(rew[i], r2) and torch.equal(fl[i], f2), (t, i)
    for f, sh in zip(fresh, s.shards):
        _same_state(f, sh)

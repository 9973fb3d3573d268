"""The fused policy rollout (K5) under per-env physics parameter sets (dd_policy_rollout_sets, ``policy_rollout`` on an env
with ``set_param_sets``).

The central check, as for the env kernels: envs are independent and keep their env ids, so for every set s the rows with
index == s of a mixed K5 run are bit-identical to a K5 run of all N envs under ``params = sets[s]`` -- actions, log-probs,
rewards, flags, observations, probabilities, shaped rewards and the final state.  With resampling, K5's actions replayed
through dd_rollout_sets give its rewards, flags, observations, indices and statistics bit for bit."""
import importlib
import os

import numpy as np
import pytest
import torch

from param_reference import LARGE, make_params
from test_gpu_guardbands import Arena, _armour
from test_gpu_param_sets import _index, _rows_equal, _sets, _state
from test_param_sets_cpu import resample_draw

dd = importlib.import_module("reinforcement-learning-101_b200")
nv = dd.native

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
KW = dict(seed=31, randomize_drone=True, randomize_platform=True, max_steps=90, auto_reset=True, dtype=torch.float32,
          env_id_base=700)
OUTS = ("actions", "logp", "reward", "done", "obs", "probs", "shaped")
# (want, sample, temperature): the FAST instantiation (PPO collection), the generic one with every output and a tempered
# distribution, and threshold actions
MODES = {"fast": ("arldo", True, 1.0), "generic": ("arldops", True, 0.7), "threshold": ("arldops", False, 1.0)}


@pytest.fixture(scope="module")
def policy_sd(golden_dir):
    d = np.load(os.path.join(golden_dir, "policy_v1.npz"))
    return {k: torch.from_numpy(d[k]) for k in d.files if k.startswith("network")}


def _k5(env, blob, T, mode, t0=3, out=None):
    want, sample, temp = MODES[mode]
    return dd.policy_rollout(env, blob, T, sample=sample, temperature=temp, t0=t0, want=want, out=out)


def _same(a, b, what=""):
    for k in a:
        assert torch.equal(a[k], b[k]), (what, k)


@pytest.mark.parametrize("n,mode,operands", [(3001, "fast", "fp16"), (3001, "generic", "bf16"), (3001, "threshold", "fp16"),
                                             (65536, "fast", "bf16"), (65536, "generic", "fp16"),
                                             (65536, "threshold", "bf16")])
def test_selection_equals_per_set_runs(policy_sd, n, mode, operands):
    T, count = 160, 5
    blob = dd.PolicyBlob(policy_sd, device=DEV, operands=operands)
    assert blob.operand_dtype == operands
    sets, idx = _sets(count), _index(n, count, "random", seed=17)
    mixed = dd.BatchedDroneEnv(n, device=DEV, param_sets=sets, param_index=idx, **KW)
    mixed.reset(want_obs=False)
    got = _k5(mixed, blob, T, mode)
    assert int(mixed.stats_tensor()[0]) > 0
    for s in range(count):
        single = dd.BatchedDroneEnv(n, device=DEV, params=sets[s], **KW)
        single.reset(want_obs=False)
        ref = _k5(single, blob, T, mode)
        rows = idx.long() == s
        for k in got:
            _rows_equal(got[k].transpose(0, 1), ref[k].transpose(0, 1), rows, f"{k} set {s}")
        for a, b in zip(_state(mixed) + [mixed.prev_dist], _state(single) + [single.prev_dist]):
            _rows_equal(torch.nan_to_num(a.float(), nan=-7.0) if a.is_floating_point() else a,
                        torch.nan_to_num(b.float(), nan=-7.0) if b.is_floating_point() else b, rows, f"state set {s}")
    assert torch.equal(mixed.param_index, idx)                    # read only without resampling


@pytest.mark.parametrize("resample", [False, True])
@pytest.mark.parametrize("mode", ["fast", "generic"])
def test_replay_through_the_rollout_kernel(policy_sd, resample, mode):
    """K5's actions through env.rollout("trace") of a twin env with the same sets (dd_rollout_sets)."""
    n, T, count = 4000, 200, 16
    blob = dd.PolicyBlob(policy_sd, device=DEV)
    sets, idx = _sets(count), _index(n, count, "random", seed=5)
    kw = dict(KW, param_sets=sets, resample_param_sets=resample)
    a = dd.BatchedDroneEnv(n, device=DEV, param_index=idx.clone(), **kw)
    b = dd.BatchedDroneEnv(n, device=DEV, param_index=idx.clone(), **kw)
    c = dd.BatchedDroneEnv(n, device=DEV, param_index=idx.clone(), **kw)
    a.reset(want_obs=False); b.reset(want_obs=False)
    out = _k5(a, blob, T, mode)
    rep = dict(reward_out=torch.empty(T, n, device=DEV), done_out=torch.empty(T, n, dtype=torch.uint8, device=DEV),
               obs_out=torch.empty(T, n, 15, device=DEV))
    if "shaped" in out:
        rep["shaped_out"] = torch.empty(T, n, device=DEV)
    b.rollout(T, "trace", actions=out["actions"], **rep)
    assert torch.equal(out["reward"], rep["reward_out"]) and torch.equal(out["done"], rep["done_out"])
    if "shaped" in out:
        assert torch.equal(out["shaped"], rep["shaped_out"])
    assert torch.equal(out["obs"][0], c.reset())
    assert torch.equal(out["obs"][1:], rep["obs_out"][:-1])
    for x, y in zip(_state(a), _state(b)):
        assert torch.equal(x, y)
    assert torch.equal(a.param_index, b.param_index)
    assert a.stats() == b.stats() and a.stats()["episodes"] > 500
    if resample:
        assert not torch.equal(a.param_index, idx)


def test_resampling_writes_the_stream_3_draw_and_only_then(policy_sd):
    n, T, count = 5000, 150, 16
    blob = dd.PolicyBlob(policy_sd, device=DEV)
    big = torch.where(torch.arange(n, device=DEV) % 7 == 0, torch.full((n,), 200, dtype=torch.uint8, device=DEV),
                      _index(n, count, "random", seed=9))
    e = dd.BatchedDroneEnv(n, device=DEV, param_sets=_sets(count), param_index=big.clone(), resample_param_sets=True, **KW)
    e.reset(want_obs=False)                                      # the reset draws too (dd_reset_sets)
    ep0 = e.episode.cpu().numpy().view(np.uint32).copy()
    idx0 = e.param_index.cpu().numpy().copy()
    _k5(e, blob, T, "fast")
    ep1 = e.episode.cpu().numpy().view(np.uint32)
    ended = ep1 != ep0
    want = idx0.copy()
    want[ended] = resample_draw(KW["seed"], KW["env_id_base"] + np.nonzero(ended)[0], ep1[ended] - 1, count)
    assert ended.sum() > 1000                                    # (with max_steps = 90 < T: every env, some twice)
    assert np.array_equal(e.param_index.cpu().numpy(), want)
    # without the flag param_index is only read: the same bytes, out-of-range values included
    f = dd.BatchedDroneEnv(n, device=DEV, param_sets=_sets(count), param_index=big.clone(), **KW)
    f.reset(want_obs=False)
    _k5(f, blob, T, "generic")
    assert int(f.stats_tensor()[0]) > 1000
    assert torch.equal(f.param_index, big)


def test_one_set_equals_the_single_set_run(policy_sd):
    n, T = 3001, 120
    blob = dd.PolicyBlob(policy_sd, device=DEV)
    hard = _sets(2)[1]
    a = dd.BatchedDroneEnv(n, device=DEV, param_sets=[hard], param_index=torch.zeros(n, dtype=torch.uint8, device=DEV), **KW)
    b = dd.BatchedDroneEnv(n, device=DEV, params=hard, **KW)
    a.reset(want_obs=False); b.reset(want_obs=False)
    for mode in ("fast", "generic"):
        _same(_k5(a, blob, T, mode, t0=None), _k5(b, blob, T, mode, t0=None), mode)
    for x, y in zip(_state(a), _state(b)):
        assert torch.equal(x, y)
    assert a.stats() == b.stats()


def test_out_of_range_indices_clamp(policy_sd):
    n, T, count = 2000, 120, 3
    blob = dd.PolicyBlob(policy_sd, device=DEV)
    idx = _index(n, count, "random", seed=4)
    big = torch.where(idx == count - 1, torch.randint(count - 1, 256, (n,), device=DEV, dtype=torch.int32).to(torch.uint8), idx)
    assert int(big.max()) > count
    a = dd.BatchedDroneEnv(n, device=DEV, param_sets=_sets(count), param_index=idx, **KW)
    b = dd.BatchedDroneEnv(n, device=DEV, param_sets=_sets(count), param_index=big, **KW)
    a.reset(want_obs=False); b.reset(want_obs=False)
    _same(_k5(a, blob, T, "generic"), _k5(b, blob, T, "generic"))
    for x, y in zip(_state(a), _state(b)):
        assert torch.equal(x, y)


def test_sixty_four_sets(policy_sd):
    n, T, count = 8192, 100, 64
    blob = dd.PolicyBlob(policy_sd, device=DEV)
    sets, idx = _sets(count), _index(n, count, "random", seed=64)
    mixed = dd.BatchedDroneEnv(n, device=DEV, param_sets=sets, param_index=idx, **KW)
    mixed.reset(want_obs=False)
    got = _k5(mixed, blob, T, "fast")
    for s in (0, 2, 31, 47, 63):
        single = dd.BatchedDroneEnv(n, device=DEV, params=sets[s], **KW)
        single.reset(want_obs=False)
        ref = _k5(single, blob, T, "fast")
        rows = idx.long() == s
        assert int(rows.sum()) > 50
        for k in got:
            _rows_equal(got[k].transpose(0, 1), ref[k].transpose(0, 1), rows, f"{k} set {s}")


def test_in_place_index_edits_reach_the_next_call(policy_sd):
    n, T, count = 4096, 60, 4
    blob = dd.PolicyBlob(policy_sd, device=DEV)
    sets = _sets(count)
    a = dd.BatchedDroneEnv(n, device=DEV, param_sets=sets, **KW)
    b = dd.BatchedDroneEnv(n, device=DEV, param_sets=sets, **KW)
    a.reset(want_obs=False); b.reset(want_obs=False)
    _same(_k5(a, blob, T, "fast", t0=None), _k5(b, blob, T, "fast", t0=None), "before")
    a.param_index.copy_(torch.flip(a.param_index, [0]))          # in place: the env keeps the pointer
    b.set_param_sets(sets, torch.flip(b.param_index, [0]))        # a fresh table and index
    _same(_k5(a, blob, T, "fast", t0=None), _k5(b, blob, T, "fast", t0=None), "after")
    for x, y in zip(_state(a), _state(b)):
        assert torch.equal(x, y)


def _edge_states(p, n, rng, px_lo, px_hi, py_lo, py_hi):
    """Upright, slow, turning envs whose post-update bottom centre lands on one of the four platform edges of params p
    (before the ulp correction); the shape of test_gpu_params' large-world landing test."""
    edge = np.arange(n) % 4                                   # left, right, top, bottom
    k = np.where(rng.random(n) < 0.5, rng.integers(-1, 2, n), rng.integers(-8, 9, n))
    px = rng.integers(px_lo, px_hi, n).astype(np.float64); py = rng.integers(py_lo, py_hi, n).astype(np.float64)
    a1 = rng.uniform(-12, 12, n); w = rng.choice([-1, 1], n) * rng.uniform(0.5, 7.5, n)
    vx = rng.uniform(-1.5, 1.5, n); vy = rng.uniform(-1.5, 1.2, n)
    hw, hh, half = p.platform_w / 2, p.platform_h / 2, p.drone_height / 2
    bx = np.where(edge == 0, px - hw, np.where(edge == 1, px + hw, px + rng.uniform(-0.8, 0.8, n) * hw))
    by = np.where(edge == 2, py - hh, np.where(edge == 3, py + hh, py + rng.uniform(-0.8, 0.8, n) * hh))
    vx1, vy1 = vx * p.drag, (vy + p.gravity) * p.drag
    rad = np.radians(a1)
    x0 = bx + half * np.sin(rad) - vx1
    y0 = by - half * np.cos(rad) - vy1
    return dict(edge=edge, k=k, px=px, py=py, a0=a1 - w, w=w, vx=vx, vy=vy, bx=bx, by=by, x0=x0, y0=y0, half=half)


def test_landing_shortcut_in_a_mixed_world_decides_like_dd_step_sets(policy_sd):
    """Default and LARGE sets in one launch, the LARGE envs' bottom centre within +-8 float ulps of a platform edge: the
    landing shortcut's margin must be the env's own set's (1.95e-3 px ulps there, above the default world's 1e-3 px)."""
    large = make_params(nv, **LARGE)
    sets = [nv.default_params(), large]
    n = 1 << 20
    rng = np.random.default_rng(2025)
    idx = (np.arange(n) // 4 % 2).astype(np.uint8)                 # alternating blocks of the four edges
    g0 = _edge_states(sets[0], n, rng, 150, 650, 150, 500)
    g1 = _edge_states(large, n, rng, 20100, 20700, 20100, 20550)
    g = {key: np.where(idx == 1, g1[key], g0[key]) for key in g0 if key != "half"}
    half = np.where(idx == 1, g1["half"], g0["half"])
    f32 = lambda v: torch.tensor(np.asarray(v, np.float32), device=DEV)
    fuel = np.array([s.max_fuel for s in sets])[idx]
    kw = dict(randomize_drone=False, randomize_platform=False, auto_reset=False, dtype=torch.float32, param_sets=sets,
              param_index=torch.as_tensor(idx, device=DEV))

    def state(x, y):
        return {"x": f32(x), "y": f32(y), "vx": f32(g["vx"]), "vy": f32(g["vy"]), "angle": f32(g["a0"]),
                "angular_velocity": f32(g["w"]), "fuel": f32(fuel), "total_reward": f32(np.zeros(n)),
                "platform_x": f32(g["px"]), "platform_y": f32(g["py"]), "steps": torch.zeros(n, dtype=torch.int32, device=DEV),
                "flags": torch.zeros(n, dtype=torch.uint8, device=DEV), "episode": torch.ones(n, dtype=torch.int32, device=DEV)}

    zero = torch.zeros(n, dtype=torch.uint8, device=DEV)
    x0, y0 = g["x0"].astype(np.float32), g["y0"].astype(np.float32)
    probe = dd.BatchedDroneEnv(n, device=DEV, **kw)
    probe.set_state(state(x0, y0))
    probe.step_raw(zero)
    st = probe.get_state()
    x1, y1, ang1 = (st[c].cpu().numpy().astype(np.float64) for c in ("x", "y", "angle"))
    on_x = g["edge"] < 2
    ulp = np.spacing(np.abs(np.where(on_x, x1, y1)).astype(np.float32)).astype(np.float64)
    r1 = np.radians(ang1)
    miss_x = np.rint((g["bx"] - (x1 - half * np.sin(r1))) / ulp)
    miss_y = np.rint((g["by"] - (y1 + half * np.cos(r1))) / ulp)
    x0 = np.where(on_x, x0 + (miss_x + g["k"]) * ulp, x0).astype(np.float32)
    y0 = np.where(on_x, y0, y0 + (miss_y + g["k"]) * ulp).astype(np.float32)
    sd = {kk: v.clone() for kk, v in policy_sd.items()}
    sd["network.9.weight"].zero_(); sd["network.9.bias"].fill_(-50.0)      # probabilities ~0: never thrust
    blob = dd.PolicyBlob(sd, device=DEV)
    ref = dd.BatchedDroneEnv(n, device=DEV, **kw); ref.set_state(state(x0, y0))
    k5 = dd.BatchedDroneEnv(n, device=DEV, **kw); k5.set_state(state(x0, y0))
    _, rew_d, fl_d = ref.step_raw(zero)                              # dd_step_sets
    out = dd.policy_rollout(k5, blob, 1, sample=False, want="ard")
    assert torch.equal(out["actions"][0], zero)
    st = ref.get_state()
    bx1 = st["x"].double().cpu().numpy() - half * np.sin(np.radians(st["angle"].double().cpu().numpy()))
    by1 = st["y"].double().cpu().numpy() + half * np.cos(np.radians(st["angle"].double().cpu().numpy()))
    off = np.where(on_x, bx1 - g["bx"], by1 - g["by"]) / ulp
    assert np.abs(off[idx == 1]).max() <= 9.5                      # the LARGE envs sit where the margin matters
    fl_d = fl_d.cpu().numpy(); fl_k = out["done"][0].cpu().numpy()
    diverged = np.nonzero(fl_d != fl_k)[0]
    assert diverged.size == 0, [(int(i), int(idx[i]), int(g["edge"][i]), int(fl_d[i]), int(fl_k[i])) for i in diverged[:10]]
    for s in (0, 1):
        landed = (fl_d[idx == s] & nv.LANDED) != 0
        assert 0.25 * landed.size < landed.sum() < 0.75 * landed.size
    assert torch.equal(out["reward"][0], rew_d)
    for x, y in zip(_state(ref), _state(k5)):
        assert torch.equal(x, y)


@pytest.mark.parametrize("n", [1001, 1024])                       # ragged (per-row observation stores) / TMA tile stores
def test_sets_kernel_stays_inside_its_buffers_and_repeats_exactly(policy_sd, n):
    count, T = 5, 40
    arena = Arena(64 << 20)
    blob = dd.PolicyBlob(policy_sd, device=DEV)
    packed = arena.carve((blob.blob.numel(),), torch.uint8)
    packed.copy_(blob.blob); blob.blob = packed
    e = _armour(dd.BatchedDroneEnv(n, device=DEV, param_sets=_sets(count), resample_param_sets=True,
                                   **dict(KW, max_steps=25)), arena)
    idx = arena.carve((n,), torch.uint8)
    idx.copy_(_index(n, count, "random", seed=2))
    table = arena.carve((nv.PARAM_TABLE_BYTES,), torch.uint8, fill=None)
    table.copy_(e._ps_table)
    e.param_index, e._ps_table = idx, table
    e._ps.index, e._ps.table = idx.data_ptr(), table.data_ptr()
    e.reset(want_obs=False)
    out = {"actions": arena.carve((T, n), torch.uint8), "logp": arena.carve((T, n), torch.float32),
           "reward": arena.carve((T, n), torch.float32), "done": arena.carve((T, n), torch.uint8),
           "obs": arena.carve((T, n, 15), torch.float32), "probs": arena.carve((T, n, 3), torch.float32),
           "shaped": arena.carve((T, n), torch.float32)}
    state0, stats0 = e.get_state(), e.stats_slots.clone()
    first = None
    for rep in range(3):                                              # same state, same noise: identical buffers
        e.set_state(state0); e.stats_slots.copy_(stats0)
        e.prev_dist.copy_(state0["prev_dist"]); e._prev_dist_stale = False
        _k5(e, blob, T, "generic", t0=11, out=out)
        arena.check(f"dd_policy_rollout_sets n={n} rep={rep}")
        snap = {k: torch.nan_to_num(v.float(), nan=-1.0) for k, v in out.items()}
        snap.update(state=torch.cat([e.pos_vel.flatten(), e.att_fuel.flatten()]), index=e.param_index.clone(),
                    stats=e.stats_slots.clone())
        if first is None:
            first = snap
        else:
            _same(snap, first, f"rep {rep}")
    assert not torch.equal(first["index"], state0["param_index"])     # the resampling write-back ran
    fast = {k: out[k] for k in ("actions", "logp", "reward", "done", "obs")}
    _k5(e, blob, T, "fast", out=fast)
    arena.check("dd_policy_rollout_sets (FAST)")
    assert int(e.stats_tensor()[0]) > 0


def test_collect_episodes_with_a_network_on_sets_equals_the_replay(policy_sd):
    n, cap, count = 6000, 150, 8
    blob = dd.PolicyBlob(policy_sd, device=DEV)
    sets, idx = _sets(count), _index(n, count, "random", seed=21)
    kw = dict(KW, auto_reset=False, param_sets=sets)
    a = dd.BatchedDroneEnv(n, device=DEV, param_index=idx.clone(), **kw)
    got = dd.collect_episodes(a, cap, policy="network", blob=blob, t0=0, reduce=False)
    b = dd.BatchedDroneEnv(n, device=DEV, param_index=idx.clone(), **kw)        # the same actions, kept
    b.max_steps = cap; b.reset(want_obs=False)
    acts = dd.policy_rollout(b, blob, cap, t0=0, want="a")["actions"]
    c = dd.BatchedDroneEnv(n, device=DEV, param_index=idx.clone(), **kw)
    c.max_steps = cap; c.reset(want_obs=False)
    c.rollout(cap, "trace", actions=acts)
    s = c.stats()
    assert got["num_games"] == s["episodes"] == n
    assert (got["num_successes"], got["crashed"], got["timed_out"], got["env_steps"]) == \
           (s["landed"], s["crashed"], s["truncated"], s["sum_length"])
    assert got["avg_reward"] == s["mean_return"] and got["success_rate"] == s["landing_rate"]
    sweep = dd.curriculum_sweep(dd.BatchedDroneEnv(n, device=DEV, param_index=idx.clone(), **kw), [40, 80], policy="network",
                                blob=blob, reduce=False)
    assert [r["num_games"] for r in sweep] == [n, n]


def test_a_critic_blob_is_refused(policy_sd, golden_dir):
    c = np.load(os.path.join(golden_dir, "critic_v1.npz"))
    vblob = dd.ValueBlob({k: torch.from_numpy(c[k]) for k in c.files if k.startswith("network")}, device=DEV)
    for sets in (None, _sets(3)):
        e = dd.BatchedDroneEnv(256, device=DEV, param_sets=sets, **KW)
        e.reset(want_obs=False)
        with pytest.raises(ValueError, match="head=3"):
            dd.policy_rollout(e, vblob, 4)
        with pytest.raises(ValueError, match="parameter sets" if sets else "PolicyBlob"):
            dd.policy_rollout(e, None, 4)

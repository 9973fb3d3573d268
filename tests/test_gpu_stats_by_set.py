"""Episode statistics per parameter set (DD_PARAM_SETS_STATS_BY_SET) on the GPU.

Every by-set run is checked against a plain run from the same state: all outputs, the state and ``param_index`` are
bit-identical and the per-set blocks sum to the plain totals in all 8 words.  The blocks themselves are checked against
a numpy attribution of a step-by-step dd_step_sets replay (an episode counts under the set its ending step ran under),
across launch shapes and shards, inside a canary arena, and through ``collect_episodes(by_set=True)``."""
import ctypes as C
import importlib
import os

import numpy as np
import pytest
import torch

from test_gpu_guardbands import Arena
from test_gpu_param_sets import _index, _sets, _state

dd = importlib.import_module("reinforcement-learning-101_b200")
nv = dd.native

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
KW = dict(seed=41, randomize_drone=True, randomize_platform=True, max_steps=90, env_id_base=300)


@pytest.fixture(scope="module")
def policy_sd(golden_dir):
    d = np.load(os.path.join(golden_dir, "policy_v1.npz"))
    return {k: torch.from_numpy(d[k]) for k in d.files if k.startswith("network")}


def _pair(n, count, resample, idx_seed=7, **kw):
    """Two envs from one state: plain statistics and statistics per set (the index may exceed count - 1)."""
    sets = _sets(count)
    idx = torch.as_tensor(np.random.default_rng(idx_seed).integers(0, count + 3, n).astype(np.uint8), device=DEV)
    a = dd.BatchedDroneEnv(n, device=DEV, **dict(KW, **kw))
    b = dd.BatchedDroneEnv(n, device=DEV, **dict(KW, **kw))
    a.set_param_sets(sets, idx.clone(), resample)
    b.set_param_sets(sets, idx.clone(), resample, stats_by_set=True)
    a.reset(want_obs=False); b.reset(want_obs=False)
    assert b.stats_by_set and tuple(b.stats_slots.shape) == (count, nv.STATS_SLOTS, nv.STATS_WORDS)
    return a, b


def _same_everything(a, b):
    for x, y in zip(_state(a) + [a.param_index], _state(b) + [b.param_index]):
        assert torch.equal(x, y)
    plain, rows = a.stats_tensor().clone(), b.stats_tensor(by_set=True).clone()
    assert torch.equal(rows.sum(0), plain) and torch.equal(b.stats_tensor(), plain)
    assert a.stats() == b.stats()
    return rows


def _attribute(log, count):
    """numpy attribution of a step-by-step run: words 0-5 per set."""
    want = np.zeros((count, 6), np.int64)
    for idx, ret0, steps0, fl0, rew, fl, dtype in log:
        end = (fl != 0) & ((fl0 & nv.DONE) == 0)
        s = np.minimum(idx[end], count - 1).astype(np.int64)
        f = fl[end]
        ret = (ret0[end].astype(dtype) + rew[end].astype(dtype)).astype(dtype)
        fx = np.rint(ret.astype(np.float64) * nv.RETURN_FIXED_SCALE).astype(np.int64)
        for w, v in enumerate((np.ones_like(s), (f & nv.LANDED) != 0, (f & nv.CRASHED) != 0, (f & nv.TRUNCATED) != 0,
                               fx, steps0[end].astype(np.int64) + 1)):
            np.add.at(want[:, w], s, np.asarray(v, np.int64))
    return want


def _log_step(env, actions, log, step):
    before = (env.param_index.cpu().numpy(), env.att_fuel[:, 3].cpu().numpy(), env.steps.cpu().numpy(),
              env.flags.cpu().numpy())
    out = step(actions)
    torch.cuda.synchronize()
    log.append(before + (env.reward.cpu().numpy(), env.step_flags.cpu().numpy(),
                         np.float32 if env.dtype == torch.float32 else np.float64))
    return out


def _direct_step(env, actions, obs=True):
    """dd_step_sets itself (not the plan): the env's buffers, stats block and sets."""
    nv.check(env._lib.dd_step_sets(C.byref(env._state), C.byref(env._ps), C.byref(env._cfg), actions.data_ptr(),
                                   env.obs.data_ptr() if obs else None, env.obs_stride, env.reward.data_ptr(),
                                   env.step_flags.data_ptr(), None, env.stats_slots.data_ptr(), env.num_envs,
                                   env._stream()), "dd_step_sets")


# =================================================================================================
# totals unchanged, and the blocks are the attribution
# =================================================================================================
@pytest.mark.parametrize("resample", [False, True])
@pytest.mark.parametrize("dtype,auto,obs,flags", [
    (torch.float32, True, True, 0), (torch.float32, True, False, nv.LAUNCH_BLOCK_128), (torch.float32, False, True, 0),
    (torch.float32, False, False, nv.LAUNCH_BLOCK_512), (torch.float64, True, True, 0), (torch.float64, False, False, 0)])
def test_step_sets_totals_unchanged_and_blocks_are_the_attribution(resample, dtype, auto, obs, flags):
    n, T, count = 20000, 200, 16
    a, b = _pair(n, count, resample, dtype=dtype, auto_reset=auto, launch_flags=flags, max_steps=150 if auto else T)
    acts = torch.randint(0, 8, (T, n), dtype=torch.uint8, device=DEV, generator=torch.Generator(DEV).manual_seed(3))
    log = []
    for t in range(T):
        if t % 2:                                          # planned (dd_step_planned) and unplanned (dd_step_sets) steps
            a.step_raw(acts[t], want_obs=obs)
            _log_step(b, acts[t], log, lambda x: b.step_raw(x, want_obs=obs))
        else:
            _direct_step(a, acts[t], obs)
            _log_step(b, acts[t], log, lambda x: _direct_step(b, x, obs))
        assert torch.equal(a.reward, b.reward) and torch.equal(a.step_flags, b.step_flags)
        if obs:
            assert torch.equal(a.obs, b.obs)
    rows = _same_everything(a, b)
    assert torch.equal(rows[:, :6].cpu(), torch.from_numpy(_attribute(log, count)))
    assert int(rows[:, 0].sum()) > 1000 and bool((rows[:, 0] > 0).all())
    # word 6: sum_length + the live steps grouped by the clamped index
    st, fl, ix = b.steps.cpu().numpy(), b.flags.cpu().numpy(), np.minimum(b.param_index.cpu().numpy(), count - 1)
    live = np.bincount(ix, weights=np.where(fl & nv.DONE, 0, st), minlength=count).astype(np.int64)
    assert np.array_equal(rows[:, 6].cpu().numpy(), rows[:, 5].cpu().numpy() + live)


@pytest.mark.parametrize("resample", [False, True])
@pytest.mark.parametrize("policy,shaped", [("trace", False), ("random", True), ("bangbang", False), ("random", False)])
def test_rollout_sets_totals_unchanged_and_equal_the_step_by_step_blocks(resample, policy, shaped):
    n, T, count = 30000, 160, 16
    a, b = _pair(n, count, resample, auto_reset=True, max_steps=120)
    c = _pair(n, count, resample, auto_reset=True, max_steps=120)[1]
    acts = torch.randint(0, 8, (T, n), dtype=torch.uint8, device=DEV, generator=torch.Generator(DEV).manual_seed(4))
    outs = []
    for e in (a, b):
        o = dict(reward_out=torch.empty(T, n, device=DEV), done_out=torch.empty(T, n, dtype=torch.uint8, device=DEV))
        if shaped:
            o["shaped_out"] = torch.empty(T, n, device=DEV)
        e.rollout(T, policy, actions=acts if policy == "trace" else None, t0=9, **o)
        outs.append(o)
    for k in outs[0]:
        assert torch.equal(outs[0][k], outs[1][k]), k
    rows = _same_everything(a, b)
    assert int(rows[:, 0].sum()) > 1000
    if policy != "bangbang":                               # the same actions stepped one launch at a time through K1
        trace = acts if policy == "trace" else c.random_actions(T, t0=9)
        for t in range(T):
            c.step_raw(trace[t], want_obs=False)
        assert torch.equal(c.stats_tensor(by_set=True), rows)


# =================================================================================================
# the fused policy rollout (K5)
# =================================================================================================
@pytest.mark.parametrize("resample", [False, True])
@pytest.mark.parametrize("want,sample,temp,operands", [("arldo", True, 1.0, "fp16"), ("arldo", True, 1.0, "bf16"),
                                                       ("arldops", True, 0.7, "fp16"), ("arldops", False, 1.0, "bf16")])
def test_policy_rollout_sets_totals_unchanged_and_replay(policy_sd, resample, want, sample, temp, operands):
    n, T, count = 12000, 180, 16
    blob = dd.PolicyBlob(policy_sd, device=DEV, operands=operands)
    a, b = _pair(n, count, resample, auto_reset=True, max_steps=90)
    c = _pair(n, count, resample, auto_reset=True, max_steps=90)[1]
    oa = dd.policy_rollout(a, blob, T, sample=sample, temperature=temp, t0=5, want=want)
    ob = dd.policy_rollout(b, blob, T, sample=sample, temperature=temp, t0=5, want=want)
    for k in oa:
        assert torch.equal(oa[k], ob[k]), k
    rows = _same_everything(a, b)
    c.rollout(T, "trace", actions=oa["actions"])              # its actions through dd_rollout_sets: the same blocks
    assert torch.equal(c.stats_tensor(by_set=True), rows) and int(rows[:, 0].sum()) > 500


@pytest.mark.parametrize("n", [65536, 65536 + 77, 200000])
def test_policy_rollout_blocks_do_not_depend_on_the_launch_shape(policy_sd, n):
    """Spread (n below the SM count x 4 tiles), packed and ragged-last-tile launches: the blocks equal a K1 replay."""
    T, count = 120, 16
    blob = dd.PolicyBlob(policy_sd, device=DEV)
    _, b = _pair(n, count, True, auto_reset=True, max_steps=70)
    _, c = _pair(n, count, True, auto_reset=True, max_steps=70)
    acts = dd.policy_rollout(b, blob, T, t0=0, want="arldo")["actions"]
    for t in range(T):
        c.step_raw(acts[t], want_obs=False)
    assert torch.equal(b.stats_tensor(by_set=True), c.stats_tensor(by_set=True))


# =================================================================================================
# invariance
# =================================================================================================
def test_blocks_do_not_depend_on_cta_size_and_repeat():
    n, T, count = 50000, 150, 16
    got = []
    for flags in (0, nv.LAUNCH_BLOCK_128, nv.LAUNCH_BLOCK_512, 0, 0):
        _, b = _pair(n, count, True, auto_reset=True, max_steps=100, launch_flags=flags)
        acts = torch.randint(0, 8, (T, n), dtype=torch.uint8, device=DEV, generator=torch.Generator(DEV).manual_seed(8))
        for t in range(T):
            b.step_raw(acts[t])
        got.append(b.stats_tensor(by_set=True).clone())
    assert all(torch.equal(g, got[0]) for g in got) and int(got[0][:, 0].sum()) > 1000


def test_two_shards_equal_one_env():
    N, T, count = 40000, 100, 8
    sets = _sets(count)
    idx = _index(N, count, "random", seed=9)
    kw = dict(seed=5, randomize_drone=True, randomize_platform=True, max_steps=60)
    one = dd.BatchedDroneEnv(N, device=DEV, **kw)
    one.set_param_sets(sets, idx.clone(), True, stats_by_set=True)
    sh = dd.ShardedDroneEnv(2, N // 2, device=DEV, **kw)
    sh.set_param_sets(sets, idx.clone().view(2, N // 2), True, stats_by_set=True)
    one.reset(); sh.reset()
    acts = torch.randint(0, 8, (T, N), dtype=torch.uint8, device=DEV, generator=torch.Generator(DEV).manual_seed(2))
    for t in range(T):
        one.step_raw(acts[t])
        sh.step_all(acts[t].view(2, N // 2))
    assert torch.equal(sh.stats_tensor(by_set=True), one.stats_tensor(by_set=True))
    assert torch.equal(sh.stats_tensor(), one.stats_tensor())
    assert sh.stats(by_set=True) == one.stats(by_set=True)


def test_three_launches_from_one_state_give_the_same_blocks(policy_sd):
    n, T, count = 30000, 100, 16
    blob = dd.PolicyBlob(policy_sd, device=DEV)
    _, b = _pair(n, count, True, auto_reset=True)
    st = b.get_state()
    got = []
    for _ in range(3):
        b.set_state(st); b.reset_stats()
        b.rollout(T, "random", t0=1)
        dd.policy_rollout(b, blob, T, t0=2, want="arldo")
        got.append(b.stats_tensor(by_set=True).clone())
    assert torch.equal(got[0], got[1]) and torch.equal(got[0], got[2])


def test_freeze_rollout_word6_is_sum_length_plus_live_steps_by_index():
    n, count = 30000, 16
    _, b = _pair(n, count, False, auto_reset=False, max_steps=500)
    b.rollout(60, "random", t0=0)                          # stopped mid-episode: most envs still run
    rows = b.stats_tensor(by_set=True).cpu().numpy()
    st, fl = b.steps.cpu().numpy(), b.flags.cpu().numpy()
    ix = np.minimum(b.param_index.cpu().numpy(), count - 1)
    live = np.bincount(ix, weights=np.where(fl & nv.DONE, 0, st), minlength=count).astype(np.int64)
    assert live.sum() > 0 and np.array_equal(rows[:, 6], rows[:, 5] + live)
    assert (b.param_index.cpu().numpy() >= count).any()      # indices >= count counted under count - 1


# =================================================================================================
# guard bands
# =================================================================================================
@pytest.mark.parametrize("count", [3, 64])
def test_by_set_blocks_stay_inside_their_buffer(policy_sd, count):
    n, T = 9000, 80
    _, b = _pair(n, count, True, auto_reset=True, max_steps=50)
    arena = Arena(count * nv.STATS_SLOTS * nv.STATS_WORDS * 8 + count * 64 + 4096)
    blk = arena.carve((count, nv.STATS_SLOTS, nv.STATS_WORDS), torch.int64)
    out = arena.carve((count, nv.STATS_WORDS), torch.int64)
    b.stats_slots = blk
    b._plans.clear()
    b.rollout(T, "random", t0=0)
    dd.policy_rollout(b, dd.PolicyBlob(policy_sd, device=DEV), T, t0=1, want="arldo")
    for t in range(T):
        b.step_raw(torch.randint(0, 8, (n,), dtype=torch.uint8, device=DEV))
    nv.check(nv.lib().dd_stats_collapse_sets(blk.data_ptr(), count, b.steps.data_ptr(), b.flags.data_ptr(),
                                             b.param_index.data_ptr(), n, out.data_ptr(), None), "collapse")
    torch.cuda.synchronize()
    arena.check(f"count {count}")
    assert int(out[:, 0].sum()) > 100


# =================================================================================================
# evaluation: one policy on 16 worlds in one launch
# =================================================================================================
@pytest.mark.parametrize("policy", ["network", "bangbang"])
def test_collect_episodes_by_set(policy_sd, policy):
    n, count, cap = 16 * 1500, 16, 250
    sets = _sets(count)
    idx = _index(n, count, "random", seed=21)
    env = dd.BatchedDroneEnv(n, device=DEV, seed=3, randomize_drone=True, randomize_platform=True, auto_reset=False)
    env.set_param_sets(sets, idx.clone(), stats_by_set=True)
    blob = dd.PolicyBlob(policy_sd, device=DEV) if policy == "network" else None
    r = dd.collect_episodes(env, cap, policy=policy, blob=blob, by_set=True)
    per = r["by_set"]
    assert len(per) == count
    for k in ("num_games", "num_successes", "crashed", "timed_out", "env_steps"):
        assert sum(p[k] for p in per) == r[k], k
    counts = np.bincount(idx.cpu().numpy(), minlength=count)
    assert [p["num_games"] for p in per] == counts.tolist()          # one episode per env, under its set
    fl, ix = env.flags.cpu().numpy(), idx.cpu().numpy()
    ret, steps = env.att_fuel[:, 3].double().cpu().numpy(), env.steps.cpu().numpy()
    for s in range(count):
        m = ix == s
        assert per[s]["num_successes"] == int(((fl[m] & nv.LANDED) != 0).sum())
        assert per[s]["crashed"] == int(((fl[m] & nv.CRASHED) != 0).sum())
        assert per[s]["timed_out"] == int(((fl[m] & nv.TRUNCATED) != 0).sum())
        assert per[s]["env_steps"] == int(steps[m].sum())
        fx = int(np.rint(ret[m] * nv.RETURN_FIXED_SCALE).astype(np.int64).sum())
        assert per[s]["avg_reward"] == fx / nv.RETURN_FIXED_SCALE / counts[s]
    with pytest.raises(ValueError):
        dd.collect_episodes(dd.BatchedDroneEnv(64, device=DEV, auto_reset=False), cap, by_set=True)

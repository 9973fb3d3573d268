"""Per-env physics parameter sets on the GPU (dd_*_sets, BatchedDroneEnv.set_param_sets, ShardedDroneEnv).

The central check: envs are independent and keep their env ids, so for every set s the rows with index == s of a mixed
run must be bit-identical to an ordinary run of all N envs under ``params = sets[s]``."""
import ctypes as C
import importlib

import numpy as np
import pytest
import torch

from oracle import c_oracle as co
from param_reference import HARD, LARGE, make_params
from test_gpu_guardbands import Arena, _armour
from test_param_sets_cpu import MixedRef, resample_draw

dd = importlib.import_module("reinforcement-learning-101_b200")
nv = dd.native

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
OBS_DTYPES = {"native": None, "f16": torch.float16, "bf16": torch.bfloat16}
BLOCKS = {128: nv.LAUNCH_BLOCK_128, 256: 0, 512: nv.LAUNCH_BLOCK_512}


def _sets(count):
    """``count`` distinct sets: defaults, HARD, LARGE, then HARD / defaults with gravity, spawn ranges, tank and landing
    tolerance moved per set."""
    base = [nv.default_params(), make_params(nv, **HARD), make_params(nv, **LARGE)]
    out = base[:count]
    for j in range(len(out), count):
        src = dict(HARD) if j % 2 else {}
        src.update(gravity=0.2 + 0.004 * j, max_fuel=300.0 + 10 * j, land_speed=2.2 + 0.05 * (j % 16),
                   platform_w=70.0 + 2 * j, spawn_y_min=40.0 + j, r_land=90.0 + j)
        out.append(make_params(nv, **src))
    return out


def _index(n, count, kind, seed=3):
    if kind == "contiguous":
        return torch.as_tensor((np.arange(n) * count // max(n, 1)).astype(np.uint8), device=DEV)
    return torch.as_tensor(np.random.default_rng(seed).integers(0, count, n).astype(np.uint8), device=DEV)


def _rows_equal(a, b, rows, what):
    a, b = a[rows], b[rows]
    if a.dtype in (torch.float16, torch.bfloat16):
        a, b = a.view(torch.int16), b.view(torch.int16)
    assert torch.equal(a, b), what


def _state(e):
    return [e.pos_vel, e.att_fuel, e.platform, e.steps, e.episode, e.flags]


def _run_pair(n, count, kind, dtype=torch.float32, auto=True, block=256, stride=15, obs="native", T=300,
              planned=True, final=True):
    sets = _sets(count)
    idx = _index(n, count, kind)
    kw = dict(seed=11, randomize_drone=True, randomize_platform=True, max_steps=120, auto_reset=auto, dtype=dtype,
              obs_stride=stride, obs_dtype=OBS_DTYPES[obs], launch_flags=BLOCKS[block], want_final_obs=final,
              env_id_base=5)
    mixed = dd.BatchedDroneEnv(n, device=DEV, param_sets=sets, param_index=idx, **kw)
    single = [dd.BatchedDroneEnv(n, device=DEV, params=p, **kw) for p in sets]
    sel = idx.long()
    rows = [sel == s for s in range(count)]
    live = [s for s in range(count) if bool(rows[s].any())]
    o = mixed.reset()
    for s in live:
        _rows_equal(o, single[s].reset(), rows[s], "reset")
    A = torch.as_tensor(co.random_actions(11, 5, 0, T, n), device=DEV)
    for t in range(T):
        if t == T // 2:                                          # masked reset and observe
            m = torch.arange(n, device=DEV) % 3 == 0
            o = mixed.reset(m)
            for s in live:
                _rows_equal(o, single[s].reset(m), rows[s], "masked reset")
            o = mixed.observe()
            for s in live:
                _rows_equal(o, single[s].observe(), rows[s], "observe")
        if planned:
            out = [x.clone() for x in mixed.step_raw(A[t])]
        else:                                                    # dd_step_sets, no plan
            fn, pa = mixed._pargs("dd_step")
            nv.check(fn(C.byref(mixed._state), pa, C.byref(mixed._cfg), A[t].data_ptr(), mixed.obs.data_ptr(), stride,
                        mixed.reward.data_ptr(), mixed.step_flags.data_ptr(),
                        None if mixed.final_obs is None else mixed.final_obs.data_ptr(), mixed.stats_slots.data_ptr(), n,
                        mixed._stream()), "dd_step_sets")
            out = [x.clone() for x in (mixed.obs, mixed.reward, mixed.step_flags)]
        if final:
            out.append(mixed.final_obs.clone())
        for s in live:
            ref = list(single[s].step_raw(A[t]))
            if final:
                ref.append(single[s].final_obs)
            for a, b in zip(out, ref):
                _rows_equal(a, b, rows[s], f"step {t} set {s}")
    for s in live:
        for a, b in zip(_state(mixed), _state(single[s])):
            _rows_equal(a, b, rows[s], "state")
    return mixed, single, rows


@pytest.mark.parametrize("count,kind,n", [(1, "random", 257), (3, "random", 5000), (16, "contiguous", 5000),
                                          (16, "random", 255), (64, "random", 5000), (3, "random", 1)])
def test_selection_equals_per_set_runs(count, kind, n):
    _run_pair(n, count, kind)


@pytest.mark.parametrize("dtype,auto,block,stride,obs", [
    (torch.float64, True, 256, 16, "native"), (torch.float64, False, 256, 15, "native"),
    (torch.float32, False, 128, 16, "native"), (torch.float32, True, 512, 15, "native"),
    (torch.float32, True, 256, 16, "f16"), (torch.float32, False, 128, 15, "bf16"), (torch.float32, True, 512, 16, "bf16")])
def test_selection_over_kernel_variants(dtype, auto, block, stride, obs):
    mixed, single, _ = _run_pair(2053, 3, "random", dtype=dtype, auto=auto, block=block, stride=stride, obs=obs)
    assert int(sum(int(e.stats_tensor()[0]) for e in single)) > 0


def test_selection_unplanned_and_without_final_obs():
    _run_pair(777, 3, "random", planned=False, final=False, T=120)


def test_selection_at_2_20_envs():
    _run_pair(1 << 20, 16, "random", T=40)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("policy", ["trace", "random", "bangbang"])
@pytest.mark.parametrize("outs", ["none", "all"])
@pytest.mark.parametrize("shaping", ["ppo", "pg"])
def test_rollout_selection_equals_per_set_runs(dtype, policy, outs, shaping):
    n, T, count = 3000, 300, 3
    sets, idx = _sets(count), _index(n, count, "random", seed=8)
    obs_dtype = torch.bfloat16 if (dtype == torch.float32 and shaping == "pg" and outs == "all") else None
    kw = dict(seed=4, randomize_drone=True, randomize_platform=True, max_steps=110, auto_reset=True, dtype=dtype,
              obs_stride=16, shaping=shaping, obs_dtype=obs_dtype)
    mixed = dd.BatchedDroneEnv(n, device=DEV, param_sets=sets, param_index=idx, **kw)
    single = [dd.BatchedDroneEnv(n, device=DEV, params=p, **kw) for p in sets]
    A = torch.as_tensor(co.random_actions(4, 0, 0, T, n), device=DEV) if policy == "trace" else None

    def go(e):
        e.reset(want_obs=False)
        if outs == "none":
            e.rollout(T, policy, actions=A, t0=0)
            return {}
        o = dict(reward_out=torch.zeros(T, n, dtype=dtype, device=DEV), done_out=torch.zeros(T, n, dtype=torch.uint8, device=DEV),
                 shaped_out=torch.zeros(T, n, dtype=dtype, device=DEV),
                 obs_out=torch.zeros(T, n, 16, dtype=e.obs_dtype, device=DEV))
        e.rollout(T, policy, actions=A, t0=0, **o)
        return o

    got = go(mixed)
    for s, e in enumerate(single):
        ref = go(e)
        r = idx.long() == s
        for k in got:
            _rows_equal(got[k].transpose(0, 1), ref[k].transpose(0, 1), r, k)
        for a, b in zip(_state(mixed), _state(e)):
            _rows_equal(a, b, r, "state")


def test_stats_with_contiguous_blocks_equal_separate_envs():
    n, count = 4096, 16
    sets = _sets(count)
    idx = _index(n, count, "contiguous")
    kw = dict(seed=9, randomize_drone=True, randomize_platform=True, max_steps=100, auto_reset=True)
    mixed = dd.BatchedDroneEnv(n, device=DEV, param_sets=sets, param_index=idx, **kw)
    blk = n // count
    parts = [dd.BatchedDroneEnv(blk, device=DEV, params=sets[s], env_id_base=s * blk, **kw) for s in range(count)]
    A = torch.as_tensor(co.random_actions(9, 0, 0, 250, n), device=DEV)
    mixed.reset()
    for e in parts:
        e.reset()
    for t in range(250):
        mixed.step_raw(A[t])
        for s, e in enumerate(parts):
            e.step_raw(A[t, s * blk:(s + 1) * blk].contiguous())
    mixed.rollout(50, "random")
    for e in parts:
        e.rollout(50, "random")
    tot = sum(e.stats_tensor().clone() for e in parts)
    assert torch.equal(mixed.stats_tensor(), tot) and int(tot[0]) > 0


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_single_default_set_equals_the_default_kernel(dtype):
    n, T = 3000, 200
    kw = dict(seed=2, randomize_drone=True, randomize_platform=True, max_steps=90, auto_reset=True, dtype=dtype)
    a = dd.BatchedDroneEnv(n, device=DEV, **kw)
    b = dd.BatchedDroneEnv(n, device=DEV, param_sets=[nv.default_params()], **kw)
    assert torch.equal(a.reset(), b.reset())
    A = torch.as_tensor(co.random_actions(2, 0, 0, T, n), device=DEV)
    for t in range(T):
        for x, y in zip(a.step_raw(A[t]), b.step_raw(A[t])):
            assert torch.equal(x, y), t
    a.rollout(60, "bangbang"); b.rollout(60, "bangbang")
    for x, y in zip(_state(a), _state(b)):
        assert torch.equal(x, y)
    assert torch.equal(a.stats_tensor(), b.stats_tensor())


def test_out_of_range_index_is_clamped():
    n, T = 1500, 150
    sets = _sets(3)
    idx = _index(n, 3, "random")
    big = torch.where(idx == 2, torch.randint(2, 256, (n,), device=DEV, dtype=torch.int32).to(torch.uint8), idx)
    kw = dict(seed=7, randomize_drone=True, randomize_platform=True, max_steps=80, auto_reset=True, want_final_obs=True)
    a = dd.BatchedDroneEnv(n, device=DEV, param_sets=sets, param_index=idx, **kw)
    b = dd.BatchedDroneEnv(n, device=DEV, param_sets=sets, param_index=big, **kw)
    assert int(big.max()) > 2
    assert torch.equal(a.reset(), b.reset())
    A = torch.as_tensor(co.random_actions(7, 0, 0, T, n), device=DEV)
    for t in range(T):
        for x, y in zip(a.step_raw(A[t]), b.step_raw(A[t])):
            assert torch.equal(x, y)
    a.rollout(40, "random"); b.rollout(40, "random")
    for x, y in zip(_state(a), _state(b)):
        assert torch.equal(x, y)
    assert torch.equal(b.param_index, big)                       # read only without resampling


def test_resampling_f64_matches_the_per_env_reference():
    n, T, count = 2000, 320, 3
    sets = _sets(count)
    idx = _index(n, count, "random", seed=12)
    kw = dict(seed=13, randomize_drone=True, randomize_platform=True, max_steps=130, auto_reset=True, env_id_base=21)
    e = dd.BatchedDroneEnv(n, device=DEV, dtype=torch.float64, param_sets=sets, param_index=idx, resample_param_sets=True,
                           want_final_obs=True, obs_stride=16, **kw)
    r = MixedRef(n, sets, idx.cpu().numpy(), resample=True, **kw)
    np.testing.assert_allclose(e.reset().cpu().numpy(), r.reset(stride=16), rtol=1e-11, atol=1e-11)
    A = co.random_actions(13, 21, 0, T, n)
    Ad = torch.as_tensor(A, device=DEV)
    ends = 0
    for t in range(T):
        obs, rew, fl = (x.cpu().numpy() for x in e.step_raw(Ad[t]))
        oo, orr, od, of = r.step(A[t], 16)
        assert np.array_equal(fl, od), t
        assert np.array_equal(e.param_index.cpu().numpy(), r.index.astype(np.uint8)), t
        assert np.array_equal(e.episode.cpu().numpy().view(np.uint32), r.refs[0].episode)
        np.testing.assert_allclose(obs, oo, rtol=1e-11, atol=1e-11)
        np.testing.assert_allclose(rew, orr, rtol=1e-11, atol=1e-11)
        d = (fl & nv.DONE) > 0
        np.testing.assert_allclose(e.final_obs.cpu().numpy()[d, :15], of[d, :15], rtol=1e-11, atol=1e-11)
        ends += int(d.sum())
    assert ends > 500


@pytest.mark.parametrize("path", ["step", "rollout"])
def test_resampling_f32_writes_the_philox_index_sequence(path):
    n, T, count = 5000, 300, 16
    kw = dict(seed=14, randomize_drone=True, randomize_platform=True, max_steps=70, auto_reset=True, env_id_base=3)
    e = dd.BatchedDroneEnv(n, device=DEV, param_sets=_sets(count), resample_param_sets=True, **kw)
    ep = e.episode.cpu().numpy().view(np.uint32).copy()
    e.reset()
    assert np.array_equal(e.param_index.cpu().numpy(), resample_draw(14, 3 + np.arange(n), ep, count))
    for t in range(T // 10):
        ep = e.episode.cpu().numpy().view(np.uint32).copy()
        prev = e.param_index.cpu().numpy().copy()
        if path == "step":
            for j in range(10):
                e0 = e.episode.cpu().numpy().view(np.uint32).copy()
                p0 = e.param_index.cpu().numpy().copy()
                _, _, fl = e.step_raw(torch.as_tensor(co.random_actions(14, 3, 10 * t + j, 1, n)[0], device=DEV))
                d = (fl.cpu().numpy() & nv.DONE) != 0
                p0[d] = resample_draw(14, 3 + np.nonzero(d)[0], e0[d], count)
                assert np.array_equal(e.param_index.cpu().numpy(), p0)
        else:
            done = torch.zeros(10, n, dtype=torch.uint8, device=DEV)
            e.rollout(10, "bangbang", done_out=done)
            # an env's last reset in the window drew from the counter before it: episode - 1
            ep1 = e.episode.cpu().numpy().view(np.uint32)
            reset = ep1 != ep
            want = prev.copy()
            want[reset] = resample_draw(14, 3 + np.nonzero(reset)[0], ep1[reset] - 1, count)
            assert np.array_equal(e.param_index.cpu().numpy(), want)
            assert np.array_equal((done.cpu().numpy() & nv.DONE).sum(0), ep1 - ep)
    assert len(np.unique(e.param_index.cpu().numpy())) == count


def test_resampled_bangbang_episodes_equal_fixed_index_episodes():
    """The bang-bang policy depends on the state only: an episode drawn under set s equals the episode with the same
    counter of a fixed-index run under s."""
    n, T, count = 1024, 400, 4
    sets = _sets(count)
    kw = dict(seed=15, randomize_drone=True, randomize_platform=True, max_steps=90, auto_reset=True)
    e = dd.BatchedDroneEnv(n, device=DEV, param_sets=sets, resample_param_sets=True, **kw)
    e.reset()
    rew = torch.zeros(T, n, device=DEV); done = torch.zeros(T, n, dtype=torch.uint8, device=DEV)
    idx_hist = []
    for t in range(T):                                           # step by step to record the set of every episode
        idx_hist.append(e.param_index.clone())
        e.rollout(1, "bangbang", reward_out=rew[t:t + 1], done_out=done[t:t + 1])
    fixed = []
    for s in range(count):
        f = dd.BatchedDroneEnv(n, device=DEV, param_sets=sets, param_index=torch.full((n,), s, dtype=torch.uint8, device=DEV), **kw)
        f.reset()
        fr = torch.zeros(T * 3, n, device=DEV); fd = torch.zeros(T * 3, n, dtype=torch.uint8, device=DEV)
        f.rollout(T * 3, "bangbang", reward_out=fr, done_out=fd)
        fixed.append((fr.cpu().numpy(), fd.cpu().numpy()))
    R, D, I = rew.cpu().numpy(), done.cpu().numpy(), torch.stack(idx_hist).cpu().numpy()
    checked = 0
    for i in range(0, n, 37):
        ends = np.nonzero(D[:, i] & nv.DONE)[0]
        starts = np.concatenate([[0], ends[:-1] + 1])
        for k, (a, b) in enumerate(zip(starts, ends)):          # complete episodes only; episode counter k + 1
            s = int(I[a, i])
            fr, fd = fixed[s]
            fe = np.nonzero(fd[:, i] & nv.DONE)[0]
            if k >= len(fe):
                continue
            fa = 0 if k == 0 else fe[k - 1] + 1
            assert np.array_equal(R[a:b + 1, i], fr[fa:fe[k] + 1, i]) and np.array_equal(D[a:b + 1, i], fd[fa:fe[k] + 1, i])
            checked += 1
    assert checked > 100


def test_in_place_index_edits_reach_planned_steps_and_sharded_graphs():
    n, count = 4096, 4
    sets = _sets(count)
    kw = dict(seed=1, randomize_drone=True, randomize_platform=True, max_steps=60, auto_reset=True)
    a = dd.BatchedDroneEnv(n, device=DEV, param_sets=sets, **kw)
    b = dd.BatchedDroneEnv(n, device=DEV, param_sets=sets, **kw)
    a.reset(); b.reset()
    A = torch.as_tensor(co.random_actions(1, 0, 0, 80, n), device=DEV)
    for t in range(80):
        if t == 30:
            a.param_index.copy_(torch.flip(a.param_index, [0]))      # in place: the plan keeps the pointer
            b.set_param_sets(sets, torch.flip(b.param_index, [0]))   # a fresh plan
        for x, y in zip(a.step_raw(A[t]), b.step_raw(A[t])):
            assert torch.equal(x, y), t

    S, N = 3, 2048
    sh = dd.ShardedDroneEnv(S, N, device=DEV, chains=2, trace_len=8, param_sets=sets, **kw)
    eager = dd.ShardedDroneEnv(S, N, device=DEV, chains=2, trace_len=8, use_graphs=False, param_sets=sets, **kw)
    one = dd.BatchedDroneEnv(S * N, device=DEV, param_sets=sets, launch_flags=nv.LAUNCH_PDL, **kw)
    for e in (sh, eager):
        e.reset()
        e.random_trace()
    one.reset()
    idx2 = _index(S * N, count, "random", seed=6).view(S, N)
    sh.set_param_sets(sets, idx2); eager.set_param_sets(sets, idx2); one.set_param_sets(sets, idx2.reshape(-1))
    tr = sh.trace
    for rnd in range(3):
        if rnd == 2:
            sh.join(); eager.join()
            for e in (sh, eager):
                for s in range(S):
                    e.shards[s].param_index.copy_((e.shards[s].param_index + 1) % count)
            one.param_index.copy_((one.param_index + 1) % count)
        sh.run(S * 8); eager.run(S * 8)                             # every shard steps trace rows 0 .. 7 in order
        for row in range(8):
            one.step_raw(tr[row].reshape(-1))
        sh.join(); eager.join()
        for s in range(S):
            for x, y, z in zip(_state(sh.shards[s]), _state(eager.shards[s]), _state(one)):
                assert torch.equal(x, y)
                assert torch.equal(x, z[s * N:(s + 1) * N])
    assert sh.graph_replays > 0


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_sets_kernels_stay_inside_their_buffers(dtype):
    n, count = 1000, 5
    arena = Arena(16 * 1024 * 1024)
    e = dd.BatchedDroneEnv(n, device=DEV, dtype=dtype, param_sets=_sets(count), resample_param_sets=True, want_final_obs=True,
                           seed=6, randomize_drone=True, randomize_platform=True, max_steps=25, auto_reset=True)
    _armour(e, arena)
    idx = arena.carve((n,), torch.uint8)
    table = arena.carve((nv.PARAM_TABLE_BYTES,), torch.uint8, fill=None)
    table.copy_(e._ps_table)
    e.param_index, e._ps_table = idx, table
    e._ps.index, e._ps.table = idx.data_ptr(), table.data_ptr()
    e.reset()
    A = torch.as_tensor(co.random_actions(6, 0, 0, 60, n), device=DEV)
    for t in range(60):
        e.step_raw(A[t])
    e.reset(torch.arange(n, device=DEV) % 2 == 0)
    e.observe()
    T = 40
    e.rollout(T, "random", reward_out=arena.carve((T, n), dtype), done_out=arena.carve((T, n), torch.uint8),
              obs_out=arena.carve((T, n, 15), dtype), shaped_out=arena.carve((T, n), dtype))
    torch.cuda.synchronize()
    arena.check("per-env parameter-set kernels")
    assert int(e.stats_tensor()[0]) > 0


def test_refusals():
    e = dd.BatchedDroneEnv(256, device=DEV, param_sets=_sets(2))
    with pytest.raises(RuntimeError, match="set_param_sets"):
        e.params = nv.default_params()
    from importlib import import_module
    pol = import_module("reinforcement-learning-101_b200.policy")
    with pytest.raises(ValueError, match="parameter sets"):
        pol.policy_rollout(e, None, 4)
    with pytest.raises(ValueError):
        dd.BatchedDroneEnv(16, device=DEV, param_sets=_sets(2) * 40)          # 80 sets
    with pytest.raises(ValueError):
        dd.BatchedDroneEnv(16, device=DEV, param_index=torch.zeros(16, dtype=torch.uint8))
    e.set_param_sets(None)
    e.params = nv.default_params()                                            # allowed again
    assert e.param_sets is None and e.param_index is None


def test_get_set_state_and_inject_carry_the_sets():
    n = 600
    sets = _sets(3)
    e = dd.BatchedDroneEnv(n, device=DEV, param_sets=sets, seed=3, randomize_drone=True)
    e.reset()
    st = e.get_state()
    assert torch.equal(st["param_index"], e.param_index)
    new = (st["param_index"] + 1) % 3
    e.set_state({"param_index": new})
    assert torch.equal(e.param_index, new)
    e.inject(torch.full((n,), 300.0), torch.full((n,), 200.0), torch.full((n,), 400.0), torch.full((n,), 500.0))
    mf = torch.tensor([p.max_fuel for p in sets], device=DEV)[new.long()]
    assert torch.equal(e.att_fuel[:, 2], mf.float())
    assert len(e.param_sets) == 3 and e.param_sets[1].gravity == sets[1].gravity

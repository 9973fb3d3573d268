"""Non-default physics parameters on a machine without a GPU.

``tests/param_reference.py`` restates the environment for any ``DDParams`` in float64.  It is pinned here first -- at
the default parameters it must equal the C oracle and the golden vectors recorded from the reference -- and then used as
the reference for the HOST instantiation of the kernels' source (csrc/drone_core.cuh via tests/hosttwin.py) under
parameter sets that move every constant the kernels derive from ``DDParams``:

  * float64 twin: flags and counters exact, values to 1e-11;
  * float32 twin: the fp32 rule of tests/test_gpu_parity.py (``|a - b| <= 1e-5 max(|b|, 1)`` on observations and
    rewards, flags exact except for listed envs whose float64 state lies within the band of a termination threshold),
    with the band scaled by the world size (``param_reference.world_scale``).
"""
import json
import os

import numpy as np
import pytest

from corpus import N_CORPUS, N_TRAJ, T_CORPUS, corpus_actions, corpus_spawns
from hosttwin import HostBatch, nv
from oracle import c_oracle as co
from oracle.shaping_port import EpisodeShaper
from param_reference import PARAM_SETS, POL_BANGBANG, POL_RANDOM, ParamRef, make_params, world_scale

BAND = 2e-4


def _close32(a, b):
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    return np.abs(a - b) <= 1e-5 * np.maximum(np.abs(b), 1.0)


# =================================================================================================
# the reference pinned at the default parameters
# =================================================================================================
@pytest.mark.parametrize("n", [1, 257, 3000])
def test_reference_equals_c_oracle_autoreset_truncation(n):
    kw = dict(seed=11, randomize_drone=True, randomize_platform=True, max_steps=60, auto_reset=True, env_id_base=1000)
    o = co.OracleBatch(n, **kw)
    r = ParamRef(n, nv.default_params(), **kw)
    assert np.array_equal(r.reset(), o.reset())
    T = 150
    A = co.random_actions(11, 1000, 0, T, n)
    A[:, 3::7] |= nv.ACT_SKIP                                # skipped envs keep their state
    for t in range(T):
        oo, orr, od, of = o.step(A[t], want_final=True)
        obs, rew, fl, fin = r.step(A[t], want_final=True)
        assert np.array_equal(fl, od), t
        assert np.array_equal(r.steps, o.steps) and np.array_equal(r.episode, o.episode)
        np.testing.assert_allclose(obs, oo, rtol=1e-12, atol=1e-12)
        np.testing.assert_allclose(rew, orr, rtol=1e-12, atol=1e-12)
        d = (fl & nv.DONE) > 0
        np.testing.assert_allclose(fin[d], of[d], rtol=1e-12, atol=1e-12)
    s = o.stats
    assert r.stats.as_tuple() == (s.episodes, s.landed, s.crashed, s.truncated, int(s.sum_length))
    assert r.stats.sum_return == pytest.approx(s.sum_return, rel=1e-12, abs=1e-9)
    assert s.episodes > 0


def test_reference_equals_c_oracle_rollout_policies():
    n, T = 500, 130
    kw = dict(seed=5, randomize_drone=True, randomize_platform=True, max_steps=100, auto_reset=True, env_id_base=77)
    for pol in (POL_RANDOM, POL_BANGBANG):
        o = co.OracleBatch(n, **kw); o.reset()
        r = ParamRef(n, nv.default_params(), **kw); r.reset()
        orew, odon, ostats = o.rollout(T, policy=pol, t0=7, record=True)
        rew, don, _ = r.rollout(T, pol, t0=7)
        assert np.array_equal(don, odon)
        np.testing.assert_allclose(rew, orew, rtol=1e-12, atol=1e-12)
        assert r.stats.as_tuple() == (ostats.episodes, ostats.landed, ostats.crashed, ostats.truncated, int(ostats.sum_length))


def test_reference_matches_golden_corpus(golden_dir):
    """4096 envs x 250 steps, freeze-after-done, against the vectors recorded from the reference (the tolerances of
    tests/test_oracle_golden.py)."""
    gs = np.load(os.path.join(golden_dir, "corpus_summary.npz"))
    gt = np.load(os.path.join(golden_dir, "corpus_traj.npz"))
    sx, sy, spx, spy = corpus_spawns()
    A = corpus_actions()
    r = ParamRef(N_CORPUS, nv.default_params(), randomize_drone=False, randomize_platform=False)
    r.inject(sx, sy, spx, spy)
    done_step = np.zeros(N_CORPUS, np.int16)
    for t in range(T_CORPUS):
        obs, rew, fl = r.step(A[t])
        d = (fl & nv.DONE) > 0
        np.testing.assert_allclose(obs.sum(0), gs["obs_sum"][t], rtol=1e-12, atol=1e-9)
        np.testing.assert_allclose(rew.sum(), gs["rew_sum"][t], rtol=1e-12, atol=1e-9)
        assert int(d.sum()) == gs["done_cnt"][t]
        np.testing.assert_allclose(obs[:N_TRAJ], gt["obs"][t], rtol=1e-12, atol=1e-13)
        np.testing.assert_allclose(rew[:N_TRAJ], gt["reward"][t], rtol=1e-12, atol=1e-13)
        assert np.array_equal(d[:N_TRAJ], gt["done"][t].astype(bool))
        newly = d & (done_step == 0)
        done_step[newly] = r.steps[newly]
    assert np.array_equal(done_step, gs["done_step"])
    assert np.array_equal(r.flags & 7, gs["flags"])
    np.testing.assert_allclose(r.ret, gs["total"], rtol=1e-12, atol=1e-12)
    fin = np.stack([r.x, r.y, r.vx, r.vy, r.angle, r.angvel, r.fuel], 1)
    np.testing.assert_allclose(fin, gs["final"], rtol=1e-12, atol=1e-12)


def test_reference_matches_golden_kats(golden_dir):
    kat = json.load(open(os.path.join(golden_dir, "kat.json")))
    names = ["KAT1_no_thrust", "KAT2_main", "KAT3_all", "KAT4_right", "KAT5_main_right", "KAT6_bangbang"]
    fixed = {"KAT1_no_thrust": 0, "KAT2_main": 1, "KAT3_all": 7, "KAT4_right": 4, "KAT5_main_right": 5}
    r = ParamRef(len(names), nv.default_params(), randomize_drone=False, randomize_platform=False)
    r.reset()
    last_r, last_f, obs = np.zeros(len(names)), np.zeros(len(names), np.uint8), None
    head = [[] for _ in names]
    for _ in range(3000):
        a = np.array([fixed[k] if k in fixed else int(r.vy[j] > 1.5) for j, k in enumerate(names)], np.uint8)
        obs, rew, fl = r.step(a)
        live = (fl & nv.DONE) == 0
        fresh = rew != 0
        last_r[fresh] = rew[fresh]; last_f[fresh] = fl[fresh]
        for j in range(len(names)):
            if r.steps[j] <= 3 and (live[j] or fresh[j]) and len(head[j]) < r.steps[j]:
                head[j].append(float(rew[j]))
        if not live.any():
            break
    tol = dict(rel=1e-13, abs=1e-12)
    for j, k in enumerate(names):
        ref = kat[k]
        assert r.steps[j] == ref["steps"], k
        assert bool(last_f[j] & nv.LANDED) == ref["landed"] and bool(last_f[j] & nv.CRASHED) == ref["crashed"], k
        assert last_r[j] == pytest.approx(ref["last_reward"], **tol)
        assert r.ret[j] == pytest.approx(ref["total_reward"], **tol)
        for a, rk in ((r.x, "x"), (r.y, "y"), (r.vx, "vx"), (r.vy, "vy"), (r.angle, "angle"), (r.angvel, "angvel"),
                      (r.fuel, "fuel")):
            assert a[j] == pytest.approx(ref[rk], **tol), (k, rk)
        for jj, key in enumerate(("drone_x", "drone_y", "drone_vx", "drone_vy", "drone_angle", "drone_angular_vel",
                                  "drone_fuel", "platform_x", "platform_y", "distance_to_platform", "dx_to_platform",
                                  "dy_to_platform", "speed", "landed", "crashed")):
            assert obs[j, jj] == pytest.approx(float(ref["final_state"][key]), **tol), (k, key)
        assert head[j] == pytest.approx([h["r"] for h in ref["head"]], **tol)


def test_reference_spawn_words_and_ranges():
    """Spawns are min + mulhi32(Philox word, count): equal to the C oracle's at the defaults, and cover exactly
    [min, min + count) under other ranges."""
    n = 20000
    r = ParamRef(n, nv.default_params(), seed=7, randomize_drone=True, randomize_platform=True, env_id_base=3)
    o = co.OracleBatch(n, seed=7, randomize_drone=True, randomize_platform=True, env_id_base=3)
    r.reset(); o.reset()
    for a, b in ((r.x, o.x), (r.y, o.y), (r.px, o.px), (r.py, o.py)):
        assert np.array_equal(a, b)
    p = make_params(nv, **PARAM_SETS["hard"])
    r = ParamRef(n, p, seed=7, randomize_drone=True, randomize_platform=True)
    r.reset()
    for a, lo, cnt in ((r.x, p.spawn_x_min, p.spawn_x_count), (r.y, p.spawn_y_min, p.spawn_y_count),
                       (r.px, p.plat_x_min, p.plat_x_count), (r.py, p.plat_y_min, p.plat_y_count)):
        assert a.min() == lo and a.max() == lo + cnt - 1


# =================================================================================================
# the host instantiation of drone_core.cuh under non-default parameters
# =================================================================================================
def _copy_state(h, r):
    """Reference state -> host twin buffers (exact in float64; rounded once in float32)."""
    h.pos_vel[:] = np.stack([r.x, r.y, r.vx, r.vy], 1); h.att_fuel[:] = np.stack([r.angle, r.angvel, r.fuel, r.ret], 1)
    h.platform[:] = np.stack([r.px, r.py], 1); h.steps[:] = r.steps; h.episode[:] = r.episode; h.flags[:] = r.flags


@pytest.mark.parametrize("which", sorted(PARAM_SETS))
@pytest.mark.parametrize("auto", [False, True])
def test_f64_twin_vs_reference(which, auto):
    p = make_params(nv, **PARAM_SETS[which])
    n, T = 1000, 250
    kw = dict(seed=17, randomize_drone=True, randomize_platform=True, max_steps=120 if auto else 0, auto_reset=auto,
              env_id_base=40)
    r = ParamRef(n, p, **kw)
    h = HostBatch(n, np.float64, params=p, **kw)
    obs0 = h.reset(stride=16)
    ro0 = r.reset(stride=16)
    assert np.array_equal(obs0, ro0)                                     # spawns exact, obs under the new norms
    A = co.random_actions(17, 40, 0, T, n)
    A[:, 1::2] = np.where(co.random_actions(18, 40, 0, T, n)[:, 1::2] < 3, A[:, 1::2] & 1, A[:, 1::2])   # fewer spins
    causes = 0
    for t in range(T):
        obs, rew, fl, fin = h.step(A[t], want_final=True, stride=16)
        oo, orr, od, of = r.step(A[t], stride=16, want_final=True)
        assert np.array_equal(fl, od), t
        assert np.array_equal(h.steps, r.steps) and np.array_equal(h.episode, r.episode)
        np.testing.assert_allclose(obs, oo, rtol=1e-11, atol=1e-11)
        np.testing.assert_allclose(rew, orr, rtol=1e-11, atol=1e-11)
        d = (fl & nv.DONE) > 0
        np.testing.assert_allclose(fin[d, :15], of[d, :15], rtol=1e-11, atol=1e-11)
        causes |= int(np.bitwise_or.reduce(fl))
    s = h.stats
    assert (int(s[0]), int(s[1]), int(s[2]), int(s[3]), int(s[5])) == r.stats.as_tuple()
    assert s[0] > 0
    if which == "hard":                                                 # the sets reach the branches they are for
        assert causes & nv.LANDED and (causes & nv.CAUSE_MASK) == nv.CAUSE_MASK
        if auto:
            assert causes & nv.TRUNCATED


@pytest.mark.parametrize("which", sorted(PARAM_SETS))
def test_f32_twin_vs_reference(which):
    p = make_params(nv, **PARAM_SETS[which])
    n, T = 2000, 250
    kw = dict(seed=23, randomize_drone=True, randomize_platform=True)
    r = ParamRef(n, p, **kw)
    h = HostBatch(n, np.float32, params=p, **kw)
    obs0, ro0 = h.reset(), r.reset()
    for a, b in ((h.pos_vel[:, 0], r.x), (h.pos_vel[:, 1], r.y), (h.platform[:, 0], r.px), (h.platform[:, 1], r.py)):
        assert np.array_equal(a, b)                                     # integer spawns: exact in float32 too
    assert _close32(obs0, ro0).all()
    A = co.random_actions(23, 0, 0, T, n)
    A[:, 1::2] = np.where(co.random_actions(24, 0, 0, T, n)[:, 1::2] < 3, A[:, 1::2] & 1, A[:, 1::2])
    band = BAND * world_scale(p)
    valid = np.ones(n, bool)
    flips = []
    for t in range(T):
        obs, rew, fl = h.step(A[t])
        oo, orr, od = r.step(A[t])
        bad = valid & (fl != od)
        if bad.any():
            mg = r.threshold_margin()
            for i in np.nonzero(bad)[0]:
                assert mg[i] < band, f"env {i} step {t}: flags {fl[i]:#x} vs {od[i]:#x}, float64 margin {mg[i]:.3g}"
                flips.append((int(i), t, float(mg[i])))
            valid &= ~bad
        assert np.array_equal(h.steps[valid], r.steps[valid])
        assert _close32(obs, oo)[valid].all(), f"step {t}: obs outside fp32 tolerance"
        assert _close32(rew, orr)[valid].all(), f"step {t}: reward outside fp32 tolerance"
    assert len(flips) <= 3, flips
    assert ((r.flags & nv.DONE) > 0).sum() > (n // 4 if which == "hard" else 0)
    print(f"{which}: {len(flips)} float32 threshold flips {flips}")


@pytest.mark.parametrize("which", sorted(PARAM_SETS))
@pytest.mark.parametrize("variant", ["ppo", "pg"])
def test_f64_twin_shaped_reward_under_params(which, variant):
    """The fused shaped reward reads its normalised inputs through the parameters' reciprocals: against the notebook
    port applied to the reference's observations."""
    p = make_params(nv, **PARAM_SETS[which])
    n, T, ms = 64, 150, 120
    kw = dict(seed=4, randomize_drone=True, randomize_platform=True, max_steps=ms, auto_reset=False)
    h = HostBatch(n, np.float64, params=p, shaping=variant, **kw)
    r = ParamRef(n, p, **kw)
    obs0 = h.reset()
    np.testing.assert_array_equal(obs0, r.reset())
    out = h.rollout(T, nv.POLICY_BANGBANG, want=("reward", "done", "obs", "shaped"))
    rrew, rdon, robs = r.rollout(T, POL_BANGBANG)
    assert np.array_equal(out["done"], rdon)
    np.testing.assert_allclose(out["obs"], robs, rtol=1e-11, atol=1e-11)
    exp = np.zeros((T, n))
    for i in range(n):
        sh = EpisodeShaper(ms, variant=variant)
        cur = obs0[i]
        for t in range(T):
            exp[t, i], _ = sh.step(cur, robs[t, i])
            cur = robs[t, i]
            if rdon[t, i]:
                break
    np.testing.assert_allclose(out["shaped"], exp, rtol=1e-9, atol=1e-9)
    assert (rdon & nv.DONE).any()

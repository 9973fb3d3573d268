"""Per-env physics parameter sets (DDParamSets, include/drone_b200.h) without a GPU: the header against the ctypes
binding, dd_param_sets_build, the argument codes of the _sets entry points (device library and host twin), and the
host twin of the per-env kernels against (a) the single-set host twin run once per set and (b) a float64 per-env
reference composed of one ``ParamRef`` per set, including the resampling rule."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from hosttwin import HostBatch, dd, lib as twin_lib, nv
from oracle import c_oracle as co
from param_reference import HARD, LARGE, ParamRef, make_params

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SETS3 = [nv.default_params(), make_params(nv, **HARD), make_params(nv, **LARGE)]


def _header():
    with open(os.path.join(ROOT, "include", "drone_b200.h")) as f:
        return f.read()


def _twin():
    L = twin_lib()
    if not hasattr(L, "_sets_bound"):
        vp, i32, i64, u32 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint32
        PS, PSS, PC = C.POINTER(nv.DDState), C.POINTER(nv.DDParamSets), C.POINTER(nv.DDEnvConfig)
        L.dd_param_sets_build_host.argtypes = [C.POINTER(nv.DDParams), i32, i32, vp]
        L.dd_reset_sets_host.argtypes = [PS, PSS, PC, vp, vp, i32, i64]
        L.dd_step_sets_host.argtypes = [PS, PSS, PC, vp, vp, i32, vp, vp, vp, vp, i64]
        L.dd_rollout_sets_host.argtypes = [PS, PSS, PC, i32, vp, u32, i32, vp, vp, vp, i32, vp, vp, i64]
        L._sets_bound = True
    return L


def _build(sets, dtype, device_lib=None):
    """The table bytes from the host twin's build, or from the device library's dd_param_sets_build."""
    arr = (nv.DDParams * len(sets))(*sets)
    out = C.create_string_buffer(nv.PARAM_TABLE_BYTES)
    f = _twin().dd_param_sets_build_host if device_lib is None else device_lib.dd_param_sets_build
    assert f(arr, len(sets), dtype, out) == 0
    return out.raw


def _p(a):
    return None if a is None else a.ctypes.data


class SetsBatch(HostBatch):
    """HostBatch stepped through the _sets twins: ``index`` (uint8 [n]) and the table are host arrays."""

    def __init__(self, n, sets, index, resample=False, **kw):
        super().__init__(n, **kw)
        dt = nv.F32 if self.dtype == np.float32 else nv.F64
        self.table = np.frombuffer(_build(sets, dt), np.uint8).copy()     # numpy data is 16-byte aligned
        self.index = np.ascontiguousarray(index, np.uint8).copy()
        self.ps = nv.DDParamSets(self.table.ctypes.data, self.index.ctypes.data, len(sets), dt,
                                 nv.PARAM_SETS_RESAMPLE if resample else 0, 0)

    def reset(self, mask=None, stride=15):
        obs = np.zeros((self.n, stride), self.dtype)
        m = None if mask is None else np.ascontiguousarray(mask, np.uint8)
        self._check(_twin().dd_reset_sets_host(C.byref(self.state), C.byref(self.ps), C.byref(self.cfg), _p(m), _p(obs),
                                               stride, self.n), "dd_reset_sets_host")
        return obs

    def step(self, actions, want_obs=True, want_final=False, stride=15):
        a = np.ascontiguousarray(actions, np.uint8)
        obs = np.zeros((self.n, stride), self.dtype) if want_obs else None
        rew = np.zeros(self.n, self.dtype); fl = np.zeros(self.n, np.uint8)
        fin = np.zeros((self.n, stride), self.dtype) if want_final else None
        self._check(_twin().dd_step_sets_host(C.byref(self.state), C.byref(self.ps), C.byref(self.cfg), _p(a), _p(obs),
                                              stride, _p(rew), _p(fl), _p(fin), _p(self.stats), self.n), "dd_step_sets_host")
        return (obs, rew, fl, fin) if want_final else (obs, rew, fl)

    def rollout(self, T, policy, actions=None, t0=0, want=("reward", "done"), stride=15):
        out = {}
        if "reward" in want: out["reward"] = np.zeros((T, self.n), self.dtype)
        if "done" in want: out["done"] = np.zeros((T, self.n), np.uint8)
        if "obs" in want: out["obs"] = np.zeros((T, self.n, stride), self.dtype)
        if "shaped" in want: out["shaped"] = np.zeros((T, self.n), self.dtype)
        a = None if actions is None else np.ascontiguousarray(actions, np.uint8)
        self._check(_twin().dd_rollout_sets_host(C.byref(self.state), C.byref(self.ps), C.byref(self.cfg), int(policy), _p(a),
                                                 int(t0), int(T), _p(out.get("reward")), _p(out.get("done")),
                                                 _p(out.get("obs")), stride, _p(out.get("shaped")), _p(self.stats), self.n),
                    "dd_rollout_sets_host")
        return out


def resample_draw(seed, env_ids, episodes, count):
    """The DD_PARAM_SETS_RESAMPLE rule restated: mulhi32(Philox4x32-10((id lo, id hi, episode, 3), seed).a, count)."""
    key = (seed & 0xffffffff, seed >> 32)
    a = np.array([co.philox((int(g) & 0xffffffff, int(g) >> 32, int(e), 3), key)[0] for g, e in zip(env_ids, episodes)],
                 np.uint64)
    return ((a * np.uint64(count)) >> np.uint64(32)).astype(np.uint8)


_STATE = ("x", "y", "vx", "vy", "angle", "angvel", "fuel", "ret", "px", "py", "steps", "episode", "flags")


class MixedRef:
    """float64 per-env reference: env i follows ``ParamRef(sets[min(index[i], count-1)])``.  One ParamRef per set runs
    over all n envs; after every call env i's state is copied from its own set's ref into the others."""

    def __init__(self, n, sets, index, resample=False, **kw):
        self.n, self.count, self.resample = n, len(sets), resample
        self.refs = [ParamRef(n, p, **kw) for p in sets]
        self.index = np.minimum(np.asarray(index, np.int64), self.count - 1)
        self.seed, self.base = int(kw.get("seed", 0)), int(kw.get("env_id_base", 0))

    def _pick(self, arrays):
        return np.stack(arrays)[self.index, np.arange(self.n)]

    def _sync(self):
        for a in _STATE:
            v = self._pick([getattr(r, a) for r in self.refs])
            for r in self.refs:
                setattr(r, a, v.copy())

    def obs(self, stride):
        return self._pick([r.obs(stride) for r in self.refs])

    def _respawn(self, idx, ep):
        """Resampling: envs ``idx`` draw their next set from the counter ``ep`` and spawn under it."""
        if not self.resample or len(idx) == 0:
            return
        self.index[idx] = resample_draw(self.seed, self.base + idx, ep[idx], self.count)
        for s, r in enumerate(self.refs):
            sel = idx[self.index[idx] == s]
            r.episode[sel] = ep[sel]
            r._reset_idx(sel)
        self._sync()

    def reset(self, mask=None, stride=15):
        ep = self.refs[0].episode.copy()
        for r in self.refs:
            r.reset(mask)
        self._sync()
        self._respawn(np.arange(self.n) if mask is None else np.nonzero(np.asarray(mask))[0], ep)
        return self.obs(stride)

    def step(self, actions, stride=15):
        ep = self.refs[0].episode.copy()
        res = [r.step(actions, stride, want_final=True) for r in self.refs]
        obs, rew, fl, fin = (self._pick([x[j] for x in res]) for j in range(4))
        self._sync()
        if self.refs[0].auto_reset:                    # every DONE flag is an episode that ended on this step
            self._respawn(np.nonzero((fl & nv.DONE) != 0)[0], ep)
            obs = self.obs(stride)
        return obs, rew, fl, fin


def _mixed_index(n, count, seed=5):
    return np.random.default_rng(seed).integers(0, count, n).astype(np.uint8)


# =================================================================================================
# header, binding, table build
# =================================================================================================
def test_header_matches_binding_and_both_libraries_export_the_sets_entry_points():
    h = _header()
    for name, v in (("DD_MAX_PARAM_SETS", nv.MAX_PARAM_SETS), ("DD_PARAM_TABLE_BYTES", nv.PARAM_TABLE_BYTES),
                    ("DD_PARAM_SETS_RESAMPLE", nv.PARAM_SETS_RESAMPLE)):
        assert int(re.search(rf"#define {name}\s+(0x[0-9a-fA-F]+|\d+)", h).group(1), 0) == v
    body = re.search(r"typedef struct DDParamSets \{(.*?)\} DDParamSets;", h, re.S).group(1)
    fields = re.findall(r"(\w+);", re.sub(r"/\*.*?\*/", "", body, flags=re.S))
    assert fields == [f for f, _ in nv.DDParamSets._fields_]
    assert C.sizeof(nv.DDParamSets) == 32
    dd.build_native()
    L, H = nv.lib(), twin_lib()
    for s in ("dd_param_sets_build", "dd_reset_sets", "dd_step_sets", "dd_step_plan_sets", "dd_rollout_sets"):
        assert s in nv.EXPORTS and hasattr(L, s)
    for s in ("dd_param_sets_build_host", "dd_reset_sets_host", "dd_step_sets_host", "dd_rollout_sets_host"):
        assert s in nv.HOST_TWIN_EXPORTS and hasattr(H, s)
    assert nv.ABI_VERSION == 6 == L.dd_abi_version() == H.dd_host_abi_version()


def test_param_sets_build_codes_counts_and_determinism():
    dd.build_native()
    L, H = nv.lib(), _twin()
    sets64 = [make_params(nv, gravity=0.2 + 0.005 * j, land_speed=2.0 + 0.03 * j) for j in range(64)]
    arr = (nv.DDParams * 65)(*(sets64 + sets64[:1]))
    out = C.create_string_buffer(nv.PARAM_TABLE_BYTES)
    for f in (L.dd_param_sets_build, H.dd_param_sets_build_host):
        assert f(None, 1, nv.F32, out) == -1
        assert f(arr, 1, nv.F32, None) == -1
        assert f(arr, 0, nv.F32, out) == -2
        assert f(arr, 65, nv.F32, out) == -2
        assert f(arr, 1, 7, out) == -3
    for dt in (nv.F32, nv.F64):
        for sets in (sets64[:1], sets64):
            a, b, c = _build(sets, dt, L), _build(sets, dt), _build(sets, dt)
            assert a == b == c and len(a) == nv.PARAM_TABLE_BYTES
    # count 1 leaves every other slot zero; a set's words do not depend on the other sets
    t1 = np.frombuffer(_build(sets64[:1], nv.F32), np.uint32).reshape(-1, 64)
    t64 = np.frombuffer(_build(sets64, nv.F32), np.uint32).reshape(-1, 64)
    assert not t1[:, 1:].any() and np.array_equal(t1[:, 0], t64[:, 0])
    assert np.array_equal(np.frombuffer(_build(sets64[5:6], nv.F64), np.uint64).reshape(-1, 64)[:, 0],
                          np.frombuffer(_build(sets64, nv.F64), np.uint64).reshape(-1, 64)[:, 5])


def test_sets_entry_point_argument_codes():
    """Checked before any CUDA call, device library and host twin alike."""
    dd.build_native()
    L, H = nv.lib(), _twin()
    table = np.zeros(nv.PARAM_TABLE_BYTES + 16, np.uint8)
    t0 = table.ctypes.data
    cases = [(None, nv.F32, 0, -1)]
    for dtype in (nv.F32, nv.F64):
        cases += [
            (nv.DDParamSets(None, 4096, 1, dtype, 0, 0), dtype, 0, -1),         # NULL table
            (nv.DDParamSets(t0, None, 1, dtype, 0, 0), dtype, 0, -1),           # NULL index
            (nv.DDParamSets(t0, 4096, 0, dtype, 0, 0), dtype, 0, -2),           # count 0
            (nv.DDParamSets(t0, 4096, 65, dtype, 0, 0), dtype, 0, -2),          # count 65
            (nv.DDParamSets(t0, 4096, 2, dtype, 2, 0), dtype, 0, -2),           # unknown flag bit
            (nv.DDParamSets(t0, 4096, 2, 1 - dtype, 0, 0), dtype, 0, -3),       # table of the other dtype
            (nv.DDParamSets(t0 + 8, 4096, 2, dtype, 1, 0), dtype, 0, -4),       # misaligned table
            (nv.DDParamSets(t0, 4096, 2, dtype, 1, 0), dtype, 9, -2),           # obs_format out of range
        ]
    cases.append((nv.DDParamSets(t0, 4096, 2, nv.F64, 0, 0), nv.F64, nv.OBS_BF16, -3))   # 16-bit obs, float64 state
    for ps, dtype, fmt, want in cases:
        st = nv.DDState(16, 32, 48, 64, 80, 96, dtype)
        cfg = nv.DDEnvConfig()
        cfg.obs_format = fmt
        S, P, Cf = C.byref(st), (None if ps is None else C.byref(ps)), C.byref(cfg)
        assert L.dd_reset_sets(S, P, Cf, None, None, 15, 8, None) == want
        assert L.dd_step_sets(S, P, Cf, 112, 128, 15, None, None, None, None, 8, None) == want
        plan = nv.DDStepPlan()
        assert L.dd_step_plan_sets(S, P, Cf, 128, 15, None, None, None, None, 8, C.byref(plan)) == want
        assert all(w == 0 for w in plan.opaque)
        assert L.dd_rollout_sets(S, P, Cf, nv.POLICY_RANDOM, None, 0, 4, None, None, 128, 15, None, None, 8, None) == want
        assert H.dd_reset_sets_host(S, P, Cf, None, None, 15, 8) == want
        assert H.dd_step_sets_host(S, P, Cf, 112, 128, 15, None, None, None, None, 8) == want
        assert H.dd_rollout_sets_host(S, P, Cf, nv.POLICY_RANDOM, None, 0, 4, None, None, 128, 15, None, None, 8) == want
    # the single-set checks still apply (obs stride, shaping mode), with the same codes
    ps = nv.DDParamSets(t0, 4096, 2, nv.F32, 0, 0)
    st, cfg = nv.DDState(16, 32, 48, 64, 80, 96, nv.F32), nv.DDEnvConfig()
    assert L.dd_step_sets(C.byref(st), C.byref(ps), C.byref(cfg), 112, 128, 14, None, None, None, None, 8, None) == -2
    assert H.dd_step_sets_host(C.byref(st), C.byref(ps), C.byref(cfg), 112, 128, 14, None, None, None, None, 8) == -2
    cfg.shaping = 5
    st.prev_dist = 112
    assert L.dd_rollout_sets(C.byref(st), C.byref(ps), C.byref(cfg), 1, None, 0, 4, None, None, None, 15, 256, None, 8,
                             None) == -2
    assert H.dd_rollout_sets_host(C.byref(st), C.byref(ps), C.byref(cfg), 1, None, 0, 4, None, None, None, 15, 256, None,
                                  8) == -2
    # n == 0 needs no buffers
    ps0 = nv.DDParamSets(None, None, 1, nv.F32, 0, 0)
    st0 = nv.DDState(None, None, None, None, None, None, nv.F32)
    assert L.dd_step_sets(C.byref(st0), C.byref(ps0), C.byref(nv.DDEnvConfig()), None, None, 15, None, None, None, None,
                          0, None) == 0


# =================================================================================================
# selection: the per-env twin equals the single-set twin on each set's rows
# =================================================================================================
KW = dict(seed=23, randomize_drone=True, randomize_platform=True, env_id_base=7)


def _state_rows(h, rows):
    return [a[rows].copy() for a in (h.pos_vel, h.att_fuel, h.platform, h.steps, h.episode, h.flags)]


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("auto", [False, True])
def test_twin_selection_equals_per_set_runs(dtype, auto):
    n, T = 600, 320
    idx = _mixed_index(n, 4)                                  # 3 = out of range: clamped to set 2
    kw = dict(KW, max_steps=150 if auto else 0, auto_reset=auto, dtype=dtype)
    mixed = SetsBatch(n, SETS3, idx, **kw)
    single = [HostBatch(n, params=p, **kw) for p in SETS3]
    sel = np.minimum(idx, 2)
    rows = [sel == s for s in range(3)]
    o = mixed.reset(stride=16)
    for s, h in enumerate(single):
        assert np.array_equal(h.reset(stride=16)[rows[s]], o[rows[s]])
    A = co.random_actions(23, 7, 0, T, n)
    for t in range(T):
        if t == 200:                                          # masked reset
            m = (np.arange(n) % 3 == 0).astype(np.uint8)
            o = mixed.reset(m, stride=16)
            for s, h in enumerate(single):
                assert np.array_equal(h.reset(m, stride=16)[rows[s]], o[rows[s]])
        out = mixed.step(A[t], want_final=True, stride=16)
        for s, h in enumerate(single):
            ref = h.step(A[t], want_final=True, stride=16)
            for a, b in zip(out, ref):
                assert np.array_equal(a[rows[s]], b[rows[s]]), (t, s)
    for s, h in enumerate(single):
        for a, b in zip(_state_rows(mixed, rows[s]), _state_rows(h, rows[s])):
            assert np.array_equal(a, b)
    assert np.array_equal(mixed.index, idx)                   # read only without RESAMPLE
    assert int(sum(h.stats[0] for h in single)) > 0


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("policy", [nv.POLICY_TRACE, nv.POLICY_RANDOM, nv.POLICY_BANGBANG])
@pytest.mark.parametrize("shaping", ["ppo", "pg"])
def test_twin_rollout_selection_equals_per_set_runs(dtype, policy, shaping):
    n, T = 300, 300
    idx = _mixed_index(n, 3, seed=9)
    kw = dict(KW, max_steps=120, auto_reset=True, dtype=dtype, shaping=shaping)
    mixed = SetsBatch(n, SETS3, idx, **kw)
    single = [HostBatch(n, params=p, **kw) for p in SETS3]
    mixed.reset()
    for h in single:
        h.reset()
    A = co.random_actions(3, 7, 0, T, n) if policy == nv.POLICY_TRACE else None
    want = ("reward", "done", "obs", "shaped")
    out = mixed.rollout(T, policy, A, t0=5, want=want, stride=16)
    for s, h in enumerate(single):
        ref = h.rollout(T, policy, A, t0=5, want=want, stride=16)
        r = idx == s
        for k in want:
            assert np.array_equal(out[k][:, r], ref[k][:, r]), (s, k)


# =================================================================================================
# float64 against the per-env reference; resampling
# =================================================================================================
def test_mixed_reference_at_count_one_is_param_ref():
    n, T = 200, 200
    p = make_params(nv, **HARD)
    kw = dict(KW, max_steps=90, auto_reset=True)
    m, r = MixedRef(n, [p], np.zeros(n, np.uint8), **kw), ParamRef(n, p, **kw)
    assert np.array_equal(m.reset(stride=16), r.reset(stride=16))
    A = co.random_actions(4, 7, 0, T, n)
    for t in range(T):
        for a, b in zip(m.step(A[t], 16), r.step(A[t], 16, want_final=True)):
            assert np.array_equal(a, b)


@pytest.mark.parametrize("resample", [False, True])
def test_f64_twin_vs_per_env_reference(resample):
    n, T = 800, 320
    idx = _mixed_index(n, 3, seed=11)
    kw = dict(KW, max_steps=140, auto_reset=True)
    h = SetsBatch(n, SETS3, idx, resample=resample, dtype=np.float64, **kw)
    r = MixedRef(n, SETS3, idx, resample=resample, **kw)
    np.testing.assert_allclose(h.reset(stride=16), r.reset(stride=16), rtol=1e-11, atol=1e-11)
    assert np.array_equal(h.index, r.index.astype(np.uint8))
    A = co.random_actions(11, 7, 0, T, n)
    ends = 0
    for t in range(T):
        obs, rew, fl, fin = h.step(A[t], want_final=True, stride=16)
        oo, orr, od, of = r.step(A[t], 16)
        assert np.array_equal(fl, od), t
        assert np.array_equal(h.index, r.index.astype(np.uint8)), t
        assert np.array_equal(h.steps, r.refs[0].steps) and np.array_equal(h.episode, r.refs[0].episode)
        np.testing.assert_allclose(obs, oo, rtol=1e-11, atol=1e-11)
        np.testing.assert_allclose(rew, orr, rtol=1e-11, atol=1e-11)
        d = (fl & nv.DONE) > 0
        np.testing.assert_allclose(fin[d, :15], of[d, :15], rtol=1e-11, atol=1e-11)
        ends += int(d.sum())
    assert ends > 200
    if resample:
        assert not np.array_equal(h.index, idx)


@pytest.mark.parametrize("count", [1, 3, 64])
def test_resampled_indices_follow_the_philox_rule(count):
    n, T = 500, 260
    sets = (SETS3 * 22)[:count]
    idx0 = np.zeros(n, np.uint8)
    h = SetsBatch(n, sets, idx0, resample=True, dtype=np.float32, **dict(KW, max_steps=60, auto_reset=True))
    ep = h.episode.copy()
    h.reset()
    want = resample_draw(KW["seed"], KW["env_id_base"] + np.arange(n), ep, count)
    assert np.array_equal(h.index, want)
    A = co.random_actions(2, 7, 0, T, n)
    seen = set()
    for t in range(T):
        ep = h.episode.copy()
        prev = h.index.copy()
        _, _, fl = h.step(A[t])
        d = (fl & nv.DONE) != 0
        want = prev.copy()
        want[d] = resample_draw(KW["seed"], KW["env_id_base"] + np.nonzero(d)[0], ep[d], count)
        assert np.array_equal(h.index, want), t
        seen.update(np.unique(h.index).tolist())
    assert len(seen) == count
    # rollout: the index is written back once, with the same draws
    h2 = SetsBatch(n, sets, idx0, resample=True, dtype=np.float32, **dict(KW, max_steps=60, auto_reset=True))
    h3 = SetsBatch(n, sets, idx0, resample=True, dtype=np.float32, **dict(KW, max_steps=60, auto_reset=True))
    h2.reset(); h3.reset()
    out = h2.rollout(T, nv.POLICY_TRACE, A, want=("reward", "done"))
    for t in range(T):
        h3.step(A[t])
    assert np.array_equal(h2.index, h3.index) and np.array_equal(h2.episode, h3.episode)
    assert out["done"].any()

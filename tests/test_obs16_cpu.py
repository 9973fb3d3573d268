"""16-bit observation outputs (DDEnvConfig.obs_format) without a GPU: the C ABI and its ctypes binding agree, arguments
are validated before any CUDA call, and the host twin -- the kernels' own per-environment source, with the portable
round-to-nearest-even routine standing in for the hardware conversion -- writes exactly numpy's float16 / torch's
bfloat16 of the float32 rows, while everything else stays bit-identical to the float32-observation env."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

from corpus import N_CORPUS, T_CORPUS, corpus_actions, corpus_spawns
from hosttwin import HostBatch, lib as twin_lib, nv

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FORMATS = {"f16": nv.OBS_F16, "bf16": nv.OBS_BF16}


def _header():
    return open(os.path.join(ROOT, "include", "drone_b200.h")).read()


def _ref16(x32, fmt):
    """numpy float16 / torch CPU bfloat16 of float32 values, as uint16 bit patterns."""
    x32 = np.ascontiguousarray(x32, np.float32)
    if fmt == nv.OBS_F16:
        with np.errstate(over="ignore"):
            return x32.astype(np.float16).view(np.uint16)
    return torch.from_numpy(x32).to(torch.bfloat16).view(torch.int16).numpy().view(np.uint16)


def _p(a):
    return None if a is None else a.ctypes.data


def _convert():
    f = twin_lib().dd_obs16_convert_host
    f.restype, f.argtypes = C.c_int, [C.c_int32, C.c_void_p, C.c_void_p, C.c_int64]
    return f


def test_env_config_and_obs_formats_match_the_header():
    h = _header()
    body = re.search(r"typedef struct DDEnvConfig \{(.*?)\} DDEnvConfig;", h, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields = [(t, f.strip()) for t, decl in re.findall(r"(u?int\d+_t) ([^;]+);", body) for f in decl.split(",")]
    ctypes_of = {"uint64_t": C.c_uint64, "int32_t": C.c_int32}
    assert [f for _, f in fields] == [k for k, _ in nv.DDEnvConfig._fields_]
    assert [ctypes_of[t] for t, _ in fields] == [t for _, t in nv.DDEnvConfig._fields_]
    assert fields[-2:] == [("int32_t", "obs_format"), ("int32_t", "reserved2")]
    assert C.sizeof(nv.DDEnvConfig) == 48
    for name, val in (("DD_OBS_NATIVE", nv.OBS_NATIVE), ("DD_OBS_F16", nv.OBS_F16), ("DD_OBS_BF16", nv.OBS_BF16)):
        m = re.search(rf"#define {name}\s+(\d+)", h)
        assert m and int(m.group(1)) == val, name
    # positional construction (env.py, tests/hosttwin.py) leaves the new fields zero: the native format
    c = nv.DDEnvConfig(1, 2, 3, 1, 0, 1, 0, nv.SHAPING_PG)
    assert c.obs_format == nv.OBS_NATIVE and c.reserved2 == 0 and c.shaping == nv.SHAPING_PG


def test_abi_version_6_everywhere():
    import importlib
    dd = importlib.import_module("reinforcement-learning-101_b200")
    dd.build_native()
    assert int(re.search(r"#define DD_ABI_VERSION (\d+)", _header()).group(1)) == 6 == nv.ABI_VERSION
    assert nv.lib().dd_abi_version() == 6
    assert twin_lib().dd_host_abi_version() == 6


def test_obs_format_argument_codes():
    """Validated before any CUDA call: a 16-bit format with float64 state -> DD_E_DTYPE (-3), an unknown value ->
    DD_E_RANGE (-2); device library and host twin alike."""
    import importlib
    dd = importlib.import_module("reinforcement-learning-101_b200")
    dd.build_native()
    L, H = nv.lib(), twin_lib()
    p = nv.default_params()
    for dtype, fmt, want in ((nv.F64, nv.OBS_F16, -3), (nv.F64, nv.OBS_BF16, -3), (nv.F32, 7, -2), (nv.F64, 7, -2),
                             (nv.F32, -1, -2)):
        st = nv.DDState(16, 32, 48, 64, 80, 96, dtype)
        cfg = nv.DDEnvConfig()
        cfg.obs_format = fmt
        S, P, Cf = C.byref(st), C.byref(p), C.byref(cfg)
        assert L.dd_reset(S, P, Cf, None, None, 15, 8, None) == want
        assert L.dd_step(S, P, Cf, 112, 128, 15, None, None, None, None, 8, None) == want
        plan = nv.DDStepPlan()
        assert L.dd_step_plan(S, P, Cf, 128, 15, None, None, None, None, 8, C.byref(plan)) == want
        assert all(w == 0 for w in plan.opaque)
        assert L.dd_rollout(S, P, Cf, nv.POLICY_RANDOM, None, 0, 4, None, None, 128, 15, None, 8, None) == want
        assert L.dd_rollout_shaped(S, P, Cf, nv.POLICY_RANDOM, None, 0, 4, None, None, 128, 15, None, None, 8, None) == want
        assert H.dd_reset_host(S, P, Cf, None, None, 15, 8) == want
        assert H.dd_step_host(S, P, Cf, 112, 128, 15, None, None, None, None, 8) == want
        assert H.dd_rollout_host(S, P, Cf, nv.POLICY_RANDOM, None, 0, 4, None, None, 128, 15, None, None, 8) == want


def _rne_sample():
    rng = np.random.default_rng(7)
    f16 = np.arange(0, 1 << 16, dtype=np.uint32).astype(np.uint16).view(np.float16)
    f16 = f16[np.isfinite(f16)].astype(np.float32)
    nxt = np.nextafter(f16[:-1], f16[1:])                                          # neighbours of fp16 values
    ties16 = ((f16[:-1].astype(np.float64) + f16[1:].astype(np.float64)) / 2).astype(np.float32)   # exact midpoints
    vals = [f16, nxt, ties16, np.nextafter(ties16, np.float32(np.inf)), np.nextafter(ties16, np.float32(-np.inf))]
    b = rng.integers(0, 1 << 16, 1 << 15, dtype=np.uint32) << 16
    vals += [(b | 0x8000).view(np.float32), (b | 0x8001).view(np.float32), (b | 0x7fff).view(np.float32),  # bf16 ties
             ((b + 0x10000) | 0x8000).view(np.float32)]
    tiny = np.float32(2.0 ** -24)
    vals += [np.array([2.0 ** -25, 2.0 ** -25 * 1.0000001, 2.0 ** -26, 3 * 2.0 ** -25, 2.0 ** -14 - 2.0 ** -26,
                       2.0 ** -14 - 2.0 ** -25, 65504, 65519.996, 65520, 65536, 1e6, 3.4e38, -65520, -2.0 ** -25,
                       np.inf, -np.inf, 0.0, -0.0, 1e-30, -1e-30], np.float32),
             (rng.uniform(-1, 1, 1 << 16) * tiny * 2048).astype(np.float32),      # the fp16 subnormal range
             rng.integers(0, 1 << 32, 1 << 17, dtype=np.uint64).astype(np.uint32).view(np.float32),
             rng.normal(0, 1, 1 << 16).astype(np.float32)]
    x = np.concatenate([np.ravel(v).astype(np.float32) for v in vals])
    return x[~np.isnan(x)]


@pytest.mark.parametrize("fmt", list(FORMATS))
def test_rne_helper_matches_numpy_and_torch(fmt):
    x = _rne_sample()
    out = np.zeros(x.shape, np.uint16)
    assert _convert()(FORMATS[fmt], _p(x), _p(out), x.size) == 0
    ref = _ref16(x, FORMATS[fmt])
    bad = np.nonzero(out != ref)[0]
    assert bad.size == 0, [(float(x[i]), hex(x[i:i + 1].view(np.uint32)[0]), hex(out[i]), hex(ref[i])) for i in bad[:5]]
    assert _convert()(3, _p(x), _p(out), 1) == -2


class Twin16(HostBatch):
    """HostBatch whose observation outputs are in format `fmt` (uint16 buffers for the 16-bit formats)."""

    def __init__(self, n, fmt, **kw):
        super().__init__(n, np.float32, **kw)
        self.cfg.obs_format = fmt
        self.odt = np.float32 if fmt == nv.OBS_NATIVE else np.uint16

    def reset(self, mask=None, stride=15):
        obs = np.zeros((self.n, stride), self.odt)
        m = None if mask is None else np.ascontiguousarray(mask, np.uint8)
        self._check(twin_lib().dd_reset_host(C.byref(self.state), C.byref(self.params), C.byref(self.cfg), _p(m), _p(obs),
                                             stride, self.n), "dd_reset_host")
        return obs

    def step(self, actions, stride=15):
        a = np.ascontiguousarray(actions, np.uint8)
        obs = np.zeros((self.n, stride), self.odt)
        fin = np.zeros((self.n, stride), self.odt)
        rew = np.zeros(self.n, np.float32); fl = np.zeros(self.n, np.uint8)
        self._check(twin_lib().dd_step_host(C.byref(self.state), C.byref(self.params), C.byref(self.cfg), _p(a), _p(obs),
                                            stride, _p(rew), _p(fl), _p(fin), _p(self.stats), self.n), "dd_step_host")
        return obs, rew, fl, fin

    def rollout(self, T, policy, stride=15, t0=0):
        obs = np.zeros((T, self.n, stride), self.odt)
        rew = np.zeros((T, self.n), np.float32); don = np.zeros((T, self.n), np.uint8); shp = np.zeros((T, self.n), np.float32)
        self._check(twin_lib().dd_rollout_host(C.byref(self.state), C.byref(self.params), C.byref(self.cfg), int(policy), None,
                                               int(t0), int(T), _p(rew), _p(don), _p(obs), stride, _p(shp), _p(self.stats),
                                               self.n), "dd_rollout_host")
        return obs, rew, don, shp


def _same_state(a, b):
    for k in ("pos_vel", "att_fuel", "platform", "steps", "episode", "flags", "prev_dist", "stats"):
        x, y = getattr(a, k), getattr(b, k)
        assert np.array_equal(x.view(np.uint8), y.view(np.uint8)), k


@pytest.mark.parametrize("fmt", list(FORMATS))
def test_twin_corpus_16bit_obs_are_the_rounded_fp32_obs(fmt):
    """The golden corpus (4096 envs x 250 steps): 16-bit rows == numpy float16 / torch bfloat16 of the float32 twin's
    rows, bit for bit; rewards, flags, state and statistics bit-identical."""
    f = FORMATS[fmt]
    sx, sy, spx, spy = corpus_spawns()
    A = corpus_actions()
    a = Twin16(N_CORPUS, nv.OBS_NATIVE, randomize_drone=False, randomize_platform=False)
    b = Twin16(N_CORPUS, f, randomize_drone=False, randomize_platform=False)
    a.inject(sx, sy, spx, spy); b.inject(sx, sy, spx, spy)
    for t in range(T_CORPUS):
        oa, ra, fa, _ = a.step(A[t])
        ob, rb, fb, _ = b.step(A[t])
        assert np.array_equal(ob, _ref16(oa, f)), t
        assert np.array_equal(ra.view(np.uint32), rb.view(np.uint32)) and np.array_equal(fa, fb), t
    _same_state(a, b)
    assert (a.flags & nv.DONE).any()


@pytest.mark.parametrize("fmt", list(FORMATS))
@pytest.mark.parametrize("stride", [15, 16])
def test_twin_autoreset_final_obs_reset_and_rollout(fmt, stride):
    """Auto-reset with truncation (final_obs rows), masked reset rows, the 16th `steps` column, and the T-step rollout
    (obs_tn), against the float32 twin converted."""
    f = FORMATS[fmt]
    n, T = 3000, 120
    kw = dict(seed=5, randomize_drone=True, randomize_platform=True, max_steps=70, auto_reset=True, env_id_base=77)
    a, b = Twin16(n, nv.OBS_NATIVE, **kw), Twin16(n, f, **kw)
    assert np.array_equal(b.reset(stride=stride), _ref16(a.reset(stride=stride), f))
    A = np.random.default_rng(3).integers(0, 8, (T, n)).astype(np.uint8)
    A[5, ::7] = nv.ACT_SKIP
    ends = 0
    for t in range(T):
        oa, ra, fa, fina = a.step(A[t], stride=stride)
        ob, rb, fb, finb = b.step(A[t], stride=stride)
        assert np.array_equal(ob, _ref16(oa, f)), t
        assert np.array_equal(ra.view(np.uint32), rb.view(np.uint32)) and np.array_equal(fa, fb), t
        d = (fa & nv.DONE) != 0
        assert np.array_equal(finb[d, :15], _ref16(fina[d, :15], f)), t
        assert not finb[:, 15:].any() and not finb[~d].any()              # the steps column of final_obs stays untouched
        ends += int(d.sum())
        if t == 60:
            m = (np.arange(n) % 5 == 0).astype(np.uint8)
            assert np.array_equal(b.reset(mask=m, stride=stride)[m != 0], _ref16(a.reset(mask=m, stride=stride)[m != 0], f))
    _same_state(a, b)
    assert ends > n // 2
    oa, ra, da, sa = a.rollout(50, nv.POLICY_RANDOM, stride=stride, t0=9)
    ob, rb, db, sb = b.rollout(50, nv.POLICY_RANDOM, stride=stride, t0=9)
    assert np.array_equal(ob, _ref16(oa, f))
    assert np.array_equal(ra.view(np.uint32), rb.view(np.uint32)) and np.array_equal(da, db)
    assert np.array_equal(sa.view(np.uint32), sb.view(np.uint32))
    _same_state(a, b)
    if stride == 16:                                                      # steps column: small integers, exact
        assert np.array_equal(ob[..., 15], _ref16(oa[..., 15], f)) and oa[..., 15].max() >= 69

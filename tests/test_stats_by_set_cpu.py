"""Episode statistics per parameter set (DD_PARAM_SETS_STATS_BY_SET, include/drone_b200.h) without a GPU: the flag and
dd_stats_collapse_sets' argument codes in both libraries, the host twin's per-set blocks against a numpy attribution of
its own step-by-step outputs, the Python surface's shapes and errors, and the per-set all-reduce under gloo."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

from hosttwin import dd, nv
from param_reference import HARD, LARGE, make_params
from test_param_sets_cpu import SetsBatch, _twin

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BY_SET = nv.PARAM_SETS_STATS_BY_SET
N, T, COUNT = 4096, 250, 16


def _sets16():
    base = [nv.default_params(), make_params(nv, **HARD), make_params(nv, **LARGE)]
    return [make_params(nv, gravity=0.25 + 0.02 * j, land_speed=1.5 + 0.1 * j) if j >= 3 else base[j] for j in range(COUNT)]


# =================================================================================================
# argument codes
# =================================================================================================
def test_flag_is_declared_and_accepted_by_every_sets_entry_point():
    h = open(os.path.join(ROOT, "include", "drone_b200.h")).read()
    assert int(re.search(r"#define DD_PARAM_SETS_STATS_BY_SET\s+(0x[0-9a-fA-F]+)", h).group(1), 16) == BY_SET == 0x04
    dd.build_native()
    L, H = nv.lib(), _twin()
    table = np.zeros(nv.PARAM_TABLE_BYTES + 16, np.uint8)
    t0 = table.ctypes.data
    # each call has one later fault (the table's dtype): DD_E_DTYPE shows the flags passed, DD_E_RANGE that they did not
    for flags, want in ((BY_SET, -3), (BY_SET | nv.PARAM_SETS_RESAMPLE, -3), (2, -2), (BY_SET | 2, -2), (8, -2)):
        for dtype in (nv.F32, nv.F64):
            ps = nv.DDParamSets(t0, 4096, 2, 1 - dtype, flags, 0)
            st, cfg = nv.DDState(16, 32, 48, 64, 80, 96, dtype), nv.DDEnvConfig()
            S, P, Cf = C.byref(st), C.byref(ps), C.byref(cfg)
            assert L.dd_reset_sets(S, P, Cf, None, None, 15, 8, None) == want
            assert L.dd_step_sets(S, P, Cf, 112, 128, 15, None, None, None, None, 8, None) == want
            plan = nv.DDStepPlan()
            assert L.dd_step_plan_sets(S, P, Cf, 128, 15, None, None, None, None, 8, C.byref(plan)) == want
            assert L.dd_rollout_sets(S, P, Cf, nv.POLICY_RANDOM, None, 0, 4, None, None, 128, 15, None, None, 8, None) == want
            assert H.dd_reset_sets_host(S, P, Cf, None, None, 15, 8) == want
            assert H.dd_step_sets_host(S, P, Cf, 112, 128, 15, None, None, None, None, 8) == want
            assert H.dd_rollout_sets_host(S, P, Cf, nv.POLICY_RANDOM, None, 0, 4, None, None, 128, 15, None, None, 8) == want
        ps = nv.DDParamSets(t0, 4096, 2, nv.F64, flags, 0)                 # K5: float32 state, float64 table
        st, cfg, consts = nv.DDState(16, 32, 48, 64, 80, 96, nv.F32, 0, 112), nv.DDEnvConfig(), nv.DDPolicyConsts()
        consts.operands = nv.OPERANDS_BF16
        assert L.dd_policy_rollout_sets(C.byref(st), C.byref(ps), C.byref(cfg), 16384, C.byref(consts), 1, 1.0, 0, 4, None,
                                        None, None, None, 128, None, None, None, 8, None) == want
    # n == 0 with the flag: nothing to do, no device touched
    ps0 = nv.DDParamSets(None, None, 1, nv.F32, BY_SET, 0)
    st0 = nv.DDState(None, None, None, None, None, None, nv.F32)
    assert L.dd_step_sets(C.byref(st0), C.byref(ps0), C.byref(nv.DDEnvConfig()), None, None, 15, None, None, None, None,
                          0, None) == 0


def test_stats_collapse_sets_codes_without_a_gpu():
    dd.build_native()
    L = nv.lib()
    assert "dd_stats_collapse_sets" in nv.EXPORTS and hasattr(L, "dd_stats_collapse_sets")
    f = L.dd_stats_collapse_sets
    assert f.restype == C.c_int and len(f.argtypes) == 8
    S, O, st, fl, ix = 4096, 8192, 12288, 16384, 20480
    for args, want in (
        ((None, 4, st, fl, ix, 8, O), -1),          # NULL stats
        ((S, 4, st, fl, ix, 8, None), -1),          # NULL out
        ((S, 0, st, fl, ix, 8, O), -2),             # count 0
        ((S, 65, st, fl, ix, 8, O), -2),            # count 65
        ((S, -1, st, fl, ix, 8, O), -2),
        ((S, 4, st, fl, ix, -1, O), -2),            # n < 0
        ((S, 4, st, None, ix, 8, O), -1),           # steps without flags
        ((S, 4, None, fl, ix, 8, O), -1),           # flags without steps
        ((S, 4, st, fl, None, 8, O), -1),           # running steps need the index
    ):
        assert f(*args, None) == want, args


# =================================================================================================
# host twin: attribution
# =================================================================================================
def _fx(ret):
    return np.rint(ret.astype(np.float64) * nv.RETURN_FIXED_SCALE).astype(np.int64)


def _run(dtype, resample, by_set, auto_reset=True, max_steps=120):
    """T steps of a 16-set batch through dd_step_sets_host; what a numpy attribution needs is read before every step."""
    rng = np.random.default_rng(11)
    b = SetsBatch(N, _sets16(), rng.integers(0, 20, N), resample=resample, dtype=dtype, seed=3, randomize_drone=True,
                  randomize_platform=True, auto_reset=auto_reset, max_steps=max_steps, env_id_base=5)
    b.ps.flags |= BY_SET if by_set else 0
    if by_set:
        b.stats = np.zeros((COUNT, nv.STATS_WORDS), np.uint64)
    b.reset()
    acts = np.random.default_rng(12).integers(0, 8, (T, N)).astype(np.uint8)
    log = []
    for t in range(T):
        before = (b.index.copy(), b.att_fuel[:, 3].copy(), b.steps.copy(), b.flags.copy())
        _, rew, fl = b.step(acts[t], want_obs=False)
        log.append((before, rew.copy(), fl.copy()))
    return b, log


def _attribute(log, dtype):
    """numpy attribution: an episode ends where the step's flags are set and the env was not frozen before it, under
    min(index before the step, count - 1); its return is the state's return before the step plus the step's reward in
    the state's precision."""
    want = np.zeros((COUNT, 6), np.int64)
    for (idx, ret0, steps0, fl0), rew, fl in log:
        end = (fl != 0) & ((fl0 & nv.DONE) == 0)
        s = np.minimum(idx[end], COUNT - 1).astype(np.int64)
        f = fl[end]
        ret = (ret0[end].astype(dtype) + rew[end].astype(dtype)).astype(dtype)
        for w, v in enumerate((np.ones_like(s), (f & nv.LANDED) != 0, (f & nv.CRASHED) != 0, (f & nv.TRUNCATED) != 0,
                               _fx(ret), steps0[end].astype(np.int64) + 1)):
            np.add.at(want[:, w], s, np.asarray(v, np.int64))
    return want


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("resample", [False, True])
def test_twin_step_blocks_equal_the_attribution_and_sum_to_the_totals(dtype, resample):
    b, log = _run(dtype, resample, True)
    blocks = b.stats.view(np.int64)
    assert np.array_equal(blocks[:, :6], _attribute(log, dtype))
    assert not blocks[:, 6:].any()
    assert blocks[:, 0].sum() > 500 and (blocks[:, 0] > 0).sum() == COUNT      # every set saw episodes end
    plain, plain_log = _run(dtype, resample, False)
    assert np.array_equal(blocks.sum(0).view(np.uint64), plain.stats)
    assert all(np.array_equal(x[2], y[2]) and np.array_equal(x[1], y[1]) for x, y in zip(log, plain_log))
    assert np.array_equal(b.index, plain.index) and np.array_equal(b.att_fuel, plain.att_fuel)
    if resample:                                          # the index moved: the ending step's set is not the next one's
        assert any((x[0][0] != y[0][0]).any() for x, y in zip(log[1:], log[:-1]))


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("resample", [False, True])
def test_twin_rollout_blocks_equal_the_step_by_step_blocks(dtype, resample):
    """dd_rollout_sets_host over T steps (trace policy) writes the blocks the T dd_step_sets_host calls write."""
    stepped, _ = _run(dtype, resample, True)
    rng = np.random.default_rng(11)
    b = SetsBatch(N, _sets16(), rng.integers(0, 20, N), resample=resample, dtype=dtype, seed=3, randomize_drone=True,
                  randomize_platform=True, auto_reset=True, max_steps=120, env_id_base=5)
    b.ps.flags |= BY_SET
    b.stats = np.zeros((COUNT, nv.STATS_WORDS), np.uint64)
    b.reset()
    acts = np.random.default_rng(12).integers(0, 8, (T, N)).astype(np.uint8)
    b.rollout(T, nv.POLICY_TRACE, actions=acts, want=())
    assert np.array_equal(b.stats, stepped.stats)
    assert np.array_equal(b.index, stepped.index) and np.array_equal(b.pos_vel, stepped.pos_vel)


def test_twin_freeze_mode_counts_each_env_once_under_its_index():
    b, log = _run(np.float32, False, True, auto_reset=False, max_steps=T)
    blocks = b.stats.view(np.int64)
    idx = np.minimum(log[0][0][0], COUNT - 1)
    assert np.array_equal(blocks[:, 0], np.bincount(idx, minlength=COUNT))       # every env ends once, within T steps
    assert np.array_equal(blocks[:, :6], _attribute(log, np.float32))


# =================================================================================================
# Python surface
# =================================================================================================
def test_stats_dict_rows_and_allreduce_by_set_checks():
    w = torch.zeros(3, 8, dtype=torch.int64)
    w[1] = torch.tensor([10, 3, 6, 1, int(-12.5 * nv.RETURN_FIXED_SCALE), 1500, 1600, 0])
    rows = [dd.stats_dict(r) for r in w]
    assert rows[1]["landing_rate"] == 0.3 and rows[1]["mean_return"] == -1.25 and rows[0]["episodes"] == 0
    assert dd.allreduce_stats_by_set(w) is w                      # one process: nothing to reduce
    for bad in (torch.zeros(8, dtype=torch.int64), torch.zeros(3, 7, dtype=torch.int64), torch.zeros(3, 8),
                torch.zeros(0, 8, dtype=torch.int64)):
        with pytest.raises(ValueError):
            dd.allreduce_stats_by_set(bad)
    with pytest.raises(ValueError):                               # the totals function keeps what it accepts
        dd.allreduce_stats(w)


def test_env_refuses_by_set_without_sets_on_a_cpu_machine():
    """BatchedDroneEnv refuses CPU devices, so the option's errors are checked through the class without an instance."""
    env = dd.BatchedDroneEnv.__new__(dd.BatchedDroneEnv)
    env._stats_by_set, env._plans = False, {}
    with pytest.raises(ValueError, match="stats_by_set"):
        env.stats_tensor(by_set=True)
    with pytest.raises(ValueError, match="stats_by_set"):
        dd.BatchedDroneEnv.set_param_sets(env, None, stats_by_set=True)


_WORKER = r"""
import importlib, sys
sys.path.insert(0, %(root)r)
import torch, torch.distributed as dist
dd = importlib.import_module('reinforcement-learning-101_b200')
rank, local, ws = dd.init_from_env('gloo')
w = torch.arange(3 * 8, dtype=torch.int64).reshape(3, 8) * (rank + 1)
w[2, 4] = -(rank + 1) * (1 << 20)
dd.allreduce_stats_by_set(w)
if rank == 0:
    print('RESULT', w.tolist())
dist.barrier()
dist.destroy_process_group()
"""


def test_gloo_world_size_2_by_set(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(_WORKER % {"root": ROOT})
    port = 31000 + os.getpid() % 2000
    out = subprocess.run(
        [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
         "--master-addr", "127.0.0.1", "--master-port", str(port), str(script)],
        capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = [l for l in out.stdout.splitlines() if l.startswith("RESULT")][0]
    want = (torch.arange(24, dtype=torch.int64).reshape(3, 8) * 3)
    want[2, 4] = -3 * (1 << 20)
    assert line == f"RESULT {want.tolist()}", line

"""CPU-side checks: the C-ABI library loads and exports every symbol of include/drone_b200.h, the
ctypes structs match the header, argument errors come back as codes, and the multi-GPU host
logic (sharding, statistics / moments all-reduce) works over gloo with world_size 2."""
import ctypes as C
import importlib
import os
import re
import subprocess
import sys
import types

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
dd = importlib.import_module("reinforcement-learning-101_b200")
nv = dd.native


@pytest.fixture(scope="module")
def lib():
    dd.build_native()
    return nv.lib()


def _header():
    return open(os.path.join(ROOT, "include", "drone_b200.h")).read()


def test_library_exports_every_declared_symbol(lib):
    declared = set(re.findall(r"^\s*(?:int|void|const char \*)\s*\*?(dd_\w+)\s*\(", _header(), re.M))
    assert declared >= set(nv.EXPORTS) and len(declared) >= 12
    for sym in declared:
        assert hasattr(lib, sym), f"{sym} declared in include/drone_b200.h but not exported"
    assert lib.dd_abi_version() == int(re.search(r"#define DD_ABI_VERSION (\d+)", _header()).group(1))


def test_header_constants_match_binding():
    h = _header()
    for name, val in (("DD_DONE", nv.DONE), ("DD_LANDED", nv.LANDED), ("DD_CRASHED", nv.CRASHED),
                      ("DD_TRUNCATED", nv.TRUNCATED), ("DD_CAUSE_GROUND", nv.CAUSE_GROUND),
                      ("DD_CAUSE_FUEL", nv.CAUSE_FUEL), ("DD_CAUSE_OOB", nv.CAUSE_OOB), ("DD_ACT_MAIN", nv.ACT_MAIN),
                      ("DD_ACT_LEFT", nv.ACT_LEFT), ("DD_ACT_RIGHT", nv.ACT_RIGHT), ("DD_ACT_SKIP", nv.ACT_SKIP),
                      ("DD_OBS_DIM", nv.OBS_DIM), ("DD_STATS_SLOTS", nv.STATS_SLOTS), ("DD_STATS_WORDS", nv.STATS_WORDS)):
        m = re.search(rf"#define {name}\s+(0x[0-9a-fA-F]+|\d+)u?", h)
        assert m and int(m.group(1), 0) == val, name
    # DDParams field order == header order
    body = re.search(r"typedef struct DDParams \{(.*?)\} DDParams;", h, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields = [f.strip() for decl in re.findall(r"double ([^;]+);", body) for f in decl.split(",")]
    assert fields == [k for k, _ in nv.DDParams._fields_]


def test_policy_binding_matches_header():
    """K5 binding constants: blob size, DDPolicyConsts image, per-game record length."""
    import ctypes as C
    h = _header()
    pol = importlib.import_module("reinforcement-learning-101_b200.policy")
    assert int(re.search(r"#define DD_POLICY_BLOB_BYTES (\d+)", h).group(1)) == pol.BLOB_BYTES
    assert int(re.search(r"#define DD_ENV_RECORD_DOUBLES (\d+)", h).group(1)) == nv.ENV_RECORD_DOUBLES
    body = re.search(r"typedef struct DDPolicyConsts \{(.*?)\} DDPolicyConsts;", h, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    words = 0
    for decl in re.findall(r"(?:float|int32_t) ([^;]+);", body):
        for f in decl.split(","):
            n = 1
            for d in re.findall(r"\[(\d+)\]", f):
                n *= int(d)
            words += n
    assert words * 4 == C.sizeof(nv.DDPolicyConsts) == 520 * 4
    assert nv.DDPolicyConsts.operands.offset == 516 * 4
    for name, val in (("DD_OPERANDS_AUTO", nv.OPERANDS_AUTO), ("DD_OPERANDS_BF16", nv.OPERANDS_BF16), ("DD_OPERANDS_FP16", nv.OPERANDS_FP16)):
        assert int(re.search(rf"#define {name} (\d+)", h).group(1)) == val
    assert C.sizeof(nv.DDPolicy) == 14 * C.sizeof(C.c_void_p)


def test_default_params_are_the_reference_config(lib):
    """config.py:4-5,18-68 and game_engine.py:66-85,156-177,214,254."""
    p = nv.default_params()
    got = {k: getattr(p, k) for k, _ in nv.DDParams._fields_}
    want = dict(width=800, height=600, gravity=0.3, drag=0.99, angular_drag=0.95, drone_height=20, main_thrust=0.6,
                side_thrust=0.3, max_fuel=1000, fuel_main=2, fuel_side=1, platform_w=100, platform_h=20,
                land_speed=3.0, land_angle=20.0, oob_margin=50, ground_margin=50, r_land=100, r_crash=-100,
                r_fuel=-50, r_oob=-50, r_step=-0.1, shape_offset=500, shape_div=5000, start_x=400, start_y=100,
                plat_default_x=400, plat_default_y=500, spawn_x_min=100, spawn_x_count=601, spawn_y_min=50,
                spawn_y_count=201, plat_x_min=100, plat_x_count=600, plat_y_min=100, plat_y_count=450,
                vel_norm=10, angle_norm=180, angvel_norm=10)
    assert got == {k: float(v) for k, v in want.items()}


NULL, RANGE, DTYPE, ALIGN = -1, -2, -3, -4
RESET = ("dd_reset", "dd_reset_sets")
STEP = ("dd_step", "dd_step_sets", "dd_step_plan", "dd_step_plan_sets")
ROLL = ("dd_rollout", "dd_rollout_shaped", "dd_rollout_sets")
SHAPED = ("dd_rollout_shaped", "dd_rollout_sets", "dd_policy_rollout")
ENV = RESET + STEP + ROLL
SETS = tuple(e for e in ENV if e.endswith("_sets"))
SINGLE = tuple(e for e in ENV if not e.endswith("_sets"))
K5, GATHER = ("dd_policy_rollout",), ("dd_gather_env",)

# Each entry point called with the arguments of a namespace `a` (_env_call_args): fake device pointers, real host structs.
_ENV_CALLS = {
    "dd_reset": lambda L, a: L.dd_reset(a.s, a.p, a.c, None, a.obs, a.stride, a.n, None),
    "dd_reset_sets": lambda L, a: L.dd_reset_sets(a.s, a.ps, a.c, None, a.obs, a.stride, a.n, None),
    "dd_step": lambda L, a: L.dd_step(a.s, a.p, a.c, a.actions, a.obs, a.stride, None, None, a.final_obs, None, a.n, None),
    "dd_step_sets": lambda L, a: L.dd_step_sets(a.s, a.ps, a.c, a.actions, a.obs, a.stride, None, None, a.final_obs, None,
                                                a.n, None),
    "dd_step_plan": lambda L, a: L.dd_step_plan(a.s, a.p, a.c, a.obs, a.stride, None, None, a.final_obs, None, a.n, C.byref(a.plan)),
    "dd_step_plan_sets": lambda L, a: L.dd_step_plan_sets(a.s, a.ps, a.c, a.obs, a.stride, None, None, a.final_obs, None,
                                                          a.n, C.byref(a.plan)),
    "dd_rollout": lambda L, a: L.dd_rollout(a.s, a.p, a.c, a.policy, a.actions_tn, 0, a.T, None, None, a.obs, a.stride,
                                            None, a.n, None),
    "dd_rollout_shaped": lambda L, a: L.dd_rollout_shaped(a.s, a.p, a.c, a.policy, a.actions_tn, 0, a.T, None, None, a.obs,
                                                          a.stride, a.shaped, None, a.n, None),
    "dd_rollout_sets": lambda L, a: L.dd_rollout_sets(a.s, a.ps, a.c, a.policy, a.actions_tn, 0, a.T, None, None, a.obs,
                                                      a.stride, a.shaped, None, a.n, None),
    "dd_policy_rollout": lambda L, a: L.dd_policy_rollout(a.s, a.p, a.c, a.blob, a.consts, a.mode, a.temperature, 0, a.T,
                                                          None, None, None, None, a.obs, None, a.shaped, None, a.n, None),
    "dd_gather_env": lambda L, a: L.dd_gather_env(a.s, a.obs, a.stride, None, None, a.i, a.n, a.out, None),
}


def _env_call_args(**kw):
    """A call that passes validation, but for the single fault in `kw`: `state_<field>`, `sets_<field>`, `cfg_<field>` and
    `consts_<field>` set one struct field; `s`, `p`, `ps`, `c`, `consts` or `out` = None pass NULL for the struct."""
    state = nv.DDState(16, 32, 48, 64, 80, 96, kw.get("state_dtype", nv.F32), 0, 112)
    sets = nv.DDParamSets(4096, 8192, 2, state.dtype, 0, 0)           # the table is built for the state's dtype
    cfg, consts = nv.DDEnvConfig(), nv.DDPolicyConsts()
    consts.operands = nv.OPERANDS_BF16
    for key, v in list(kw.items()):
        for prefix, struct in (("state_", state), ("sets_", sets), ("cfg_", cfg), ("consts_", consts)):
            if key.startswith(prefix):
                setattr(struct, key[len(prefix):], v)
                del kw[key]
    a = dict(s=C.byref(state), p=C.byref(nv.default_params()), ps=C.byref(sets), c=C.byref(cfg), consts=C.byref(consts),
             out=(C.c_double * nv.ENV_RECORD_DOUBLES)(), plan=nv.DDStepPlan(), n=8, T=4, obs=128, stride=15,
             final_obs=None, actions=192, policy=nv.POLICY_RANDOM, actions_tn=None, shaped=None, blob=16384, mode=1,
             temperature=1.0, i=0)
    a.update(kw)
    return types.SimpleNamespace(**a)


_STATE_FIELDS = ("pos_vel", "att_fuel", "platform", "steps", "episode", "flags")
_ARGUMENT_CASES = [
    # NULL structs
    (ENV + K5 + GATHER, dict(s=None), NULL),
    (SINGLE + K5, dict(p=None), NULL),
    (SETS, dict(ps=None), NULL),
    (ENV + K5, dict(c=None), NULL),
    (K5, dict(blob=None), NULL),
    (K5, dict(consts=None), NULL),
    (GATHER, dict(out=None), NULL),
    # dtypes
    (ENV + K5 + GATHER, dict(state_dtype=5), DTYPE),
    (K5, dict(state_dtype=nv.F64), DTYPE),
    (SETS, dict(sets_dtype=nv.F64), DTYPE),
    (SETS, dict(state_dtype=nv.F64, sets_dtype=nv.F32), DTYPE),
    # env counts
    (ENV + K5, dict(n=-1), RANGE),
    (ENV + K5, dict(n=0x7fffff01), RANGE),                             # DD_MAX_ENVS_PER_CALL + 1
    (GATHER, dict(i=-1), RANGE),
    (GATHER, dict(i=8), RANGE),
    (GATHER, dict(n=-1), RANGE),
    # state buffers
    *[(ENV + K5 + GATHER, {"state_" + f: None}, NULL) for f in _STATE_FIELDS],
    (ENV + K5, dict(state_pos_vel=24), ALIGN),
    (ENV + K5, dict(state_att_fuel=40), ALIGN),
    (ENV + K5, dict(state_platform=52), ALIGN),
    (ENV, dict(state_dtype=nv.F64, state_platform=56), ALIGN),
    # observations
    (ENV + GATHER, dict(stride=14), RANGE),
    (ENV + GATHER, dict(stride=17), RANGE),
    (STEP, dict(obs=None, final_obs=256, stride=14), RANGE),
    (ENV, dict(cfg_obs_format=3), RANGE),
    (ENV, dict(cfg_obs_format=-1), RANGE),
    (ENV, dict(state_dtype=nv.F64, cfg_obs_format=nv.OBS_F16), DTYPE),
    (ENV, dict(state_dtype=nv.F64, cfg_obs_format=nv.OBS_BF16), DTYPE),
    # actions and policies
    (("dd_step", "dd_step_sets"), dict(actions=None), NULL),
    (ROLL, dict(policy=3), RANGE),
    (ROLL, dict(policy=-1), RANGE),
    (ROLL + K5, dict(T=-1), RANGE),
    (ROLL, dict(policy=nv.POLICY_TRACE), NULL),
    # shaped training reward
    (SHAPED, dict(shaped=256, state_prev_dist=None), NULL),
    (SHAPED, dict(shaped=256, cfg_shaping=2), RANGE),
    # the fused policy rollout
    (K5, dict(mode=2), RANGE),
    (K5, dict(mode=-1), RANGE),
    (K5, dict(temperature=0.0), RANGE),
    (K5, dict(temperature=-1.0), RANGE),
    (K5, dict(temperature=float("nan")), RANGE),
    (K5, dict(consts_operands=nv.OPERANDS_AUTO), RANGE),
    (K5, dict(consts_operands=3), RANGE),
    (K5, dict(blob=16392), ALIGN),
    # parameter sets
    (SETS, dict(sets_table=None), NULL),
    (SETS, dict(sets_index=None), NULL),
    (SETS, dict(sets_count=0), RANGE),
    (SETS, dict(sets_count=65), RANGE),
    (SETS, dict(sets_flags=2), RANGE),
    (SETS, dict(sets_table=4104), ALIGN),
    # nothing to do: no buffer is needed and no CUDA call is made
    (RESET + ("dd_step", "dd_step_sets") + ROLL + K5, dict(n=0, **{"state_" + f: None for f in _STATE_FIELDS}), 0),
    (ROLL + K5, dict(T=0), 0),
]


def test_argument_errors_without_a_gpu(lib):
    """Validation happens before any CUDA call, so it is testable here: one call per check, each with a single fault,
    pins the code every env entry point returns for it."""
    for entries, fault, want in _ARGUMENT_CASES:
        for name in entries:
            a = _env_call_args(**fault)
            assert _ENV_CALLS[name](lib, a) == want, (name, fault)
            if name.startswith("dd_step_plan"):
                assert all(w == 0 for w in a.plan.opaque), (name, fault)
    assert lib.dd_step_planned(None, 192, None) == NULL
    assert lib.dd_step_planned(C.byref(nv.DDStepPlan()), 192, None) == RANGE      # zeroed: not a plan
    assert lib.dd_step(None, None, None, None, None, 15, None, None, None, None, 8, None) == -1
    assert lib.dd_reset(None, None, None, None, None, 15, 8, None) == -1
    assert lib.dd_moments(None, 4, None, None) == -1
    assert lib.dd_gae(None, None, None, None, None, 0.99, 0.95, 4, 4, None) == -1
    assert lib.dd_pack_actions(None, None, 4, None) == -1
    for code, word in ((0, b"ok"), (-1, b"null"), (-2, b"range"), (-3, b"dtype"), (-4, b"align")):
        assert word in lib.dd_error_string(code)


def test_env_refuses_cpu_device():
    with pytest.raises(ValueError, match="CUDA"):
        dd.BatchedDroneEnv(4, device="cpu")


def test_missing_library_fails_loudly(tmp_path):
    """No CPU fallback: with the .so gone, the product path raises ImportError."""
    code = (
        "import importlib, sys; sys.path.insert(0, %r)\n"
        "m = importlib.import_module('reinforcement-learning-101_b200')\n"
        "m.native.LIB_PATH = %r\n"
        "try:\n    m.native.lib()\nexcept ImportError as e:\n    print('RAISED', 'no CPU fallback' in str(e).replace('There is ', ''))\n"
    ) % (ROOT, str(tmp_path / "nope.so"))
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert "RAISED" in out.stdout, out.stderr


def test_policy_rollout_grid_covers_every_tile_once(lib):
    """Launch shape of dd_policy_rollout (host function): slot g of CTA b runs tile b + grid * g.  Every tile has exactly
    one slot; up to 3 tiles per SM the tiles are spread (never more than ceil(tiles / sms) on a CTA while SMs idle),
    above that packed four to a CTA (the measured optimum for BASELINE configs[3], DESIGN.md 4b)."""
    sms = 148
    for n in (1, 127, 128, 129, 1000, 4096, 148 * 128, 148 * 128 + 1, 32768, 50000, 148 * 3 * 128, 148 * 3 * 128 + 1, 60000, 65536,
              148 * 4 * 128, 148 * 4 * 128 + 1, 131072, 1 << 20):
        tiles = -(-n // 128)
        grid = lib.dd_policy_rollout_grid(n, sms)
        assert grid >= 1
        owners = {}
        for b in range(grid):
            for g in range(4):
                t = b + grid * g
                if t < tiles:
                    assert t not in owners
                    owners[t] = b
        assert len(owners) == tiles, (n, grid)
        per_cta = max(sum(1 for v in owners.values() if v == b) for b in range(min(grid, 200)))
        if tiles <= 3 * sms:
            assert grid == min(tiles, sms) and per_cta == -(-tiles // grid) <= 3
        else:
            assert grid == -(-tiles // 4) and per_cta == 4
    assert lib.dd_policy_rollout_grid(65536, sms) == 128 and lib.dd_policy_rollout_grid(32768, sms) == 148
    assert lib.dd_policy_rollout_grid(0, sms) == 0 and lib.dd_policy_rollout_grid(-5, sms) == 0


def test_the_product_never_imports_the_oracle():
    """oracle/ is test infrastructure: only tests/, __graft_entry__.smoke() and bench.py's CPU-baseline legs may touch it.
    Static check of every import statement of the package and of bench.py, plus a fresh interpreter that imports the
    package and looks at sys.modules."""
    import ast
    pkg_dir = os.path.join(ROOT, "reinforcement-learning-101_b200")

    def oracle_imports(path):
        tree = ast.parse(open(path).read(), path)
        parents = {}
        for node in ast.walk(tree):
            for ch in ast.iter_child_nodes(node):
                parents[ch] = node
        found = []
        for node in ast.walk(tree):
            mods = []
            if isinstance(node, ast.Import):
                mods = [a_.name for a_ in node.names]
            elif isinstance(node, ast.ImportFrom):
                mods = [node.module or ""]
            if any(m == "oracle" or m.startswith("oracle.") or m == "tests" or m.startswith("tests.") for m in mods):
                fn, cur = None, node
                while cur in parents:
                    cur = parents[cur]
                    if isinstance(cur, ast.FunctionDef):
                        fn = cur.name
                        break
                found.append(fn)
        return found

    for name in sorted(os.listdir(pkg_dir)):
        if name.endswith(".py"):
            assert oracle_imports(os.path.join(pkg_dir, name)) == [], name
    for name in sorted(os.listdir(os.path.join(pkg_dir, "csrc"))):
        includes = [l for l in open(os.path.join(pkg_dir, "csrc", name)).read().splitlines() if l.lstrip().startswith("#include")]
        assert not any("oracle" in l or "tests/" in l for l in includes), name        # (comments may cite the oracle)
    # bench.py: only inside the CPU-baseline legs (the reference arm and the cpu_baseline key)
    assert set(oracle_imports(os.path.join(ROOT, "bench.py"))) <= {"cpu_port_multiprocess", "c_oracle_threads", "run_reference"}
    code = ("import importlib, sys; sys.path.insert(0, %r); importlib.import_module('reinforcement-learning-101_b200'); "
            "import importlib as _i; m = _i.import_module('reinforcement-learning-101_b200'); "
            "[getattr(m, k) for k in ('BatchedDroneEnv', 'ShardedDroneEnv', 'policy_rollout', 'gae', 'curriculum_sweep', 'compat')]; "
            "bad = [k for k in sys.modules if k == 'oracle' or k.startswith('oracle.')]; print('BAD' if bad else 'CLEAN', bad)" % ROOT)
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert "CLEAN" in out.stdout, out.stdout + out.stderr


def test_shard_range_covers_all_ids():
    for total, ws in ((16, 1), (16, 8), (17, 4), (3, 8), (1 << 24, 8)):
        spans = [dd.shard_range(total, r, ws) for r in range(ws)]
        assert spans[0][0] == 0 and sum(n for _, n in spans) == total
        for (b0, n0), (b1, _) in zip(spans, spans[1:]):
            assert b0 + n0 == b1
    assert dd.shard_range(1 << 24, 3, 8) == (3 << 21, 1 << 21)
    with pytest.raises(ValueError):
        dd.shard_range(8, 8, 8)


def test_stats_dict_rates():
    w = torch.tensor([10, 3, 6, 1, int(-12.5 * nv.RETURN_FIXED_SCALE), 1500, 1600, 0])
    d = dd.stats_dict(w)
    assert d["landing_rate"] == 0.3 and d["mean_return"] == -1.25 and d["mean_length"] == 150.0
    assert d["episodes"] == 10 and d["env_steps"] == 1600 and "reserved" not in d
    assert dd.mean_std_from_moments(torch.tensor([4.0, 10.0, 30.0], dtype=torch.float64)) == \
        (2.5, pytest.approx(torch.tensor([1.0, 2.0, 3.0, 4.0]).std().item()))


_WORKER = r"""
import importlib, os, sys
sys.path.insert(0, %(root)r)
import torch, torch.distributed as dist
dd = importlib.import_module('reinforcement-learning-101_b200')
rank, local, ws = dd.init_from_env('gloo')
assert ws == 2 and dist.get_world_size() == 2
base, n = dd.shard_range(1001, rank, ws)
w = torch.tensor([n, rank + 1, 2, 3, -(rank + 1) * (1 << 20), 10 * n, 20 * n, 0])
dd.allreduce_stats(w)
m = torch.tensor([float(n), float(base), float(rank + 1) ** 2], dtype=torch.float64)
dd.allreduce_moments(m)
if rank == 0:
    d = dd.stats_dict(w)
    print('RESULT', d['episodes'], d['landed'], d['sum_return'], d['env_steps'], m.tolist())
dist.barrier()
dist.destroy_process_group()
"""


def test_gloo_world_size_2(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(_WORKER % {"root": ROOT})
    port = 29000 + os.getpid() % 2000
    out = subprocess.run(
        [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
         "--master-addr", "127.0.0.1", "--master-port", str(port), str(script)],
        capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = [l for l in out.stdout.splitlines() if l.startswith("RESULT")][0]
    assert line == "RESULT 1001 3 -3.0 20020 [1001.0, 501.0, 5.0]", line


def test_step_schedule_is_the_notebook_formula():
    """Actor_Critic_PPO.ipynb c19:L13-17 (300 -> 500) and README.md:55 (75 -> 250)."""
    import numpy as np
    s = dd.step_schedule(2000)
    x = np.linspace(0, 1, num=2000)
    assert np.array_equal(s, np.round(300 + 200 * x ** 0.65).astype(np.int32))
    assert s[0] == 300 and s[-1] == 500 and s.dtype == np.int32 and np.all(np.diff(s) >= 0)
    assert dd.step_schedule(8, 75, 250).tolist() == [75, 124, 153, 176, 197, 216, 233, 250]


def test_sharded_schedule_is_a_pure_function_of_offset_and_length():
    """ShardedDroneEnv.run: launch j steps shard j % S with trace row (j // S) % L; a piece is identified by
    (offset in the S*L period, length) -- the same key must always mean the same job list (graph cache), whatever
    sequence of run(k) calls led there, and consecutive pieces must tile the launch sequence without gaps."""
    sharded = importlib.import_module("reinforcement-learning-101_b200.sharded")
    for S, L in ((6, 16), (3, 4), (1, 5), (4, 1)):
        period = S * L
        seen = {}
        t = 0
        for k in (1, 5, 20, 20, 20, 7, 12, 1, 30, 2 * period + 3, 20, period, 19):
            flat = []
            for off, seg, jobs in sharded.schedule_pieces(t, k, S, L):
                assert 0 <= off < period and 1 <= seg <= period and len(jobs) == seg and off == (t + len(flat)) % period
                assert seen.setdefault((off, seg), jobs) == jobs                 # same key -> same jobs, always
                flat += jobs
            assert flat == [(j % S, (j // S) % L) for j in range(t, t + k)]      # exactly launches t .. t+k-1, in order
            t += k
        # every shard sees its trace rows in order, one row per visit
        visits = {}
        for j in range(t):
            s, row = j % S, (j // S) % L
            assert row == visits.get(s, 0) % L
            visits[s] = visits.get(s, 0) + 1
    assert list(sharded.schedule_pieces(5, 0, 6, 16)) == []


def test_packed_output_layout():
    """The per-step output block [obs | reward | flags] that step_host moves with one copy: 256-byte aligned parts,
    no overlap, sized for both dtypes and both observation strides."""
    envmod = importlib.import_module("reinforcement-learning-101_b200.env")
    for n in (0, 1, 255, 4096, 1 << 20):
        for stride in (15, 16):
            for dt, isz in ((torch.float32, 4), (torch.float64, 8)):
                o_obs, o_rew, o_flg, end = envmod._out_layout(n, stride, dt)
                assert o_obs == 0 and o_rew % 256 == 0 and o_flg % 256 == 0 and end % 256 == 0
                assert o_rew >= n * stride * isz and o_flg >= o_rew + n * isz and end >= o_flg + n and end >= 256
                blk = torch.zeros(end, dtype=torch.uint8)
                obs, rew, fl = envmod._carve(blk, (o_obs, o_rew, o_flg, end), n, stride, dt)
                assert obs.shape == (n, stride) and rew.shape == (n,) and fl.shape == (n,) and obs.dtype == dt
                obs.fill_(1); rew.fill_(2); fl.fill_(3)
                assert int(blk[o_rew:o_rew + n * isz].view(dt).sum().item()) == 2 * n and int(fl.sum().item()) == 3 * n

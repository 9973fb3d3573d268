"""dd_policy_rollout_sets without a GPU: every argument check of dd_policy_rollout and every DDParamSets check returns the
same code from it, before any CUDA call; the symbol is declared, exported and bound."""
import ctypes as C
import importlib
import os
import re

import pytest

from test_host_cpu import K5, SETS, SINGLE, _ARGUMENT_CASES, _env_call_args

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
dd = importlib.import_module("reinforcement-learning-101_b200")
nv = dd.native


@pytest.fixture(scope="module")
def lib():
    dd.build_native()
    return nv.lib()


def _call(L, a):
    return L.dd_policy_rollout_sets(a.s, a.ps, a.c, a.blob, a.consts, a.mode, a.temperature, 0, a.T, None, None, None, None,
                                    a.obs, None, a.shaped, None, a.n, None)


def _cases():
    """The cases of dd_policy_rollout (but a NULL DDParams, which this entry point does not take) and the DDParamSets cases:
    those of every _sets entry point and of no single-set one."""
    k5 = [(f, w) for e, f, w in _ARGUMENT_CASES if K5[0] in e and "p" not in f]
    ps = [(f, w) for e, f, w in _ARGUMENT_CASES if set(SETS) <= set(e) and not set(SINGLE) & set(e)]
    return k5 + ps


def test_argument_codes_are_those_of_k5_and_of_the_sets(lib):
    cases = _cases()
    faults = [f for f, _ in cases]
    for want in (dict(ps=None), dict(sets_count=0), dict(sets_count=65), dict(sets_flags=2), dict(sets_table=4104),
                 dict(sets_dtype=nv.F64), dict(state_dtype=nv.F64), dict(T=0), dict(mode=2), dict(blob=16392)):
        assert want in faults, want
    assert any(f.get("n") == 0 for f in faults)
    for fault, want in cases:
        assert _call(lib, _env_call_args(**fault)) == want, fault
    # n == 0 / T == 0 with a valid call otherwise: 0 without touching a device (there is none here)
    assert _call(lib, _env_call_args(T=0)) == 0
    assert _call(lib, _env_call_args(n=0, sets_table=None, sets_index=None)) == 0


def test_declared_exported_and_bound(lib):
    h = open(os.path.join(ROOT, "include", "drone_b200.h")).read()

    def params(name):
        m = re.search(rf"int\s+{name}\s*\((.*?)\);", h, re.S)
        return [re.sub(r"\s+", " ", p.strip()) for p in m.group(1).split(",")]

    single, sets = params("dd_policy_rollout"), params("dd_policy_rollout_sets")
    assert sets == [p.replace("const DDParams *p", "const DDParamSets *ps") for p in single]
    assert "dd_policy_rollout_sets" in nv.EXPORTS and hasattr(lib, "dd_policy_rollout_sets")
    f = lib.dd_policy_rollout_sets
    assert f.restype == C.c_int and len(f.argtypes) == len(lib.dd_policy_rollout.argtypes) == 19
    assert f.argtypes[1] == C.POINTER(nv.DDParamSets)
    assert f.argtypes[:1] + f.argtypes[2:] == lib.dd_policy_rollout.argtypes[:1] + lib.dd_policy_rollout.argtypes[2:]
    assert lib.dd_abi_version() == nv.ABI_VERSION == 6

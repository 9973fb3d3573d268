"""Loader + ctypes binding of ``libdrone_b200.so`` (the C ABI of ``include/drone_b200.h``).

There is NO fallback: if the CUDA library has not been built, importing this module raises.
Build it with ``python __graft_entry__.py build`` (or ``python -m``-style via
``build_native()`` below); the ``.so`` stays in-tree next to this file.
"""
from __future__ import annotations

import ctypes as C
import os
import shutil
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
# DRONE_B200_LIB selects another build of the sources (A/B timing of two versions in one process run)
LIB_PATH = os.environ.get("DRONE_B200_LIB") or os.path.join(_HERE, "libdrone_b200.so")
SOURCES = ("drone_kernels.cu", "ppo_kernels.cu", "policy_rollout.cu")
NVCC_FLAGS = (
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "--extended-lambda", "--expt-relaxed-constexpr", "--threads", "0", "-Xcompiler", "-fPIC", "-Xcompiler", "-ffp-contract=off", "-shared",
)
# The HOST twins of dd_reset / dd_step / dd_rollout (include/drone_b200_host.h): test infrastructure in its own
# library, built here so that it travels with the tree, loaded only by tests/ (never by this package).
HOST_TWIN_PATH = os.path.join(_HERE, "libdrone_b200_host.so")
HOST_TWIN_SOURCE = "host_twin.cpp"
HOST_TWIN_FLAGS = ("-O2", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared")

# ---- constants of include/drone_b200.h ------------------------------------------------------
ABI_VERSION = 6
DONE, LANDED, CRASHED, TRUNCATED = 0x01, 0x02, 0x04, 0x08
CAUSE_MASK, CAUSE_GROUND, CAUSE_FUEL, CAUSE_OOB = 0x30, 0x10, 0x20, 0x30
ACT_MAIN, ACT_LEFT, ACT_RIGHT, ACT_SKIP = 0x01, 0x02, 0x04, 0x80
F32, F64 = 0, 1
POLICY_TRACE, POLICY_RANDOM, POLICY_BANGBANG = 0, 1, 2
OBS_DIM = 15
STATS_SLOTS, STATS_WORDS = 64, 8
ENV_RECORD_DOUBLES = 32
SHAPING_PPO, SHAPING_PG = 0, 1
RETURN_FIXED_SCALE = 1048576.0
LAUNCH_PDL, LAUNCH_BLOCK_128, LAUNCH_BLOCK_512 = 0x01, 0x10, 0x20
OPERANDS_AUTO, OPERANDS_BF16, OPERANDS_FP16 = 0, 1, 2
OBS_NATIVE, OBS_F16, OBS_BF16 = 0, 1, 2
MAX_PARAM_SETS, PARAM_TABLE_BYTES, PARAM_SETS_RESAMPLE = 64, 32768, 0x01

_PARAM_FIELDS = (
    "width", "height", "gravity", "drag", "angular_drag", "drone_height", "main_thrust", "side_thrust",
    "max_fuel", "fuel_main", "fuel_side", "platform_w", "platform_h", "land_speed", "land_angle",
    "oob_margin", "ground_margin", "r_land", "r_crash", "r_fuel", "r_oob", "r_step",
    "shape_offset", "shape_div", "start_x", "start_y", "plat_default_x", "plat_default_y",
    "spawn_x_min", "spawn_x_count", "spawn_y_min", "spawn_y_count",
    "plat_x_min", "plat_x_count", "plat_y_min", "plat_y_count",
    "vel_norm", "angle_norm", "angvel_norm",
)


class DDParams(C.Structure):
    _fields_ = [(k, C.c_double) for k in _PARAM_FIELDS]


class DDState(C.Structure):
    _fields_ = [
        ("pos_vel", C.c_void_p), ("att_fuel", C.c_void_p), ("platform", C.c_void_p),
        ("steps", C.c_void_p), ("episode", C.c_void_p), ("flags", C.c_void_p),
        ("dtype", C.c_int32), ("reserved", C.c_int32), ("prev_dist", C.c_void_p),
    ]


class DDEnvConfig(C.Structure):
    _fields_ = [
        ("seed", C.c_uint64), ("env_id_base", C.c_uint64),
        ("max_steps", C.c_int32), ("auto_reset", C.c_int32),
        ("randomize_drone", C.c_int32), ("randomize_platform", C.c_int32),
        ("launch_flags", C.c_int32), ("shaping", C.c_int32),
        ("obs_format", C.c_int32), ("reserved2", C.c_int32),
    ]


class DDParamSets(C.Structure):
    """Per-env parameter sets of the _sets entry points: device table (dd_param_sets_build's bytes) + uint8 index [n]."""
    _fields_ = [("table", C.c_void_p), ("index", C.c_void_p), ("count", C.c_int32), ("dtype", C.c_int32),
                ("flags", C.c_int32), ("reserved", C.c_int32)]


class DDStepPlan(C.Structure):
    """Caller-owned storage of a resolved dd_step launch (dd_step_plan / dd_step_planned)."""
    _fields_ = [("opaque", C.c_uint64 * 128)]


class DDPolicy(C.Structure):
    """Device pointers to the fp32 parameters of the 15-128-128-64-3 LayerNorm MLP."""
    _fields_ = [(k, C.c_void_p) for k in (
        "w0", "b0", "g0", "be0", "w1", "b1", "g1", "be1", "w2", "b2", "g2", "be2", "w3", "b3")]


class DDPolicyConsts(C.Structure):
    """Host-side per-column parameters of the fused policy kernel (passed by value at launch)."""
    _fields_ = [("beta0", C.c_float * 128), ("beta1", C.c_float * 128), ("beta2", C.c_float * 64),
                ("w3", (C.c_float * 64) * 3), ("b3", C.c_float * 4),
                ("operands", C.c_int32), ("reserved", C.c_int32 * 3)]


def nvcc_path() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: cannot build libdrone_b200.so")


def build_native(force: bool = False, verbose: bool = False) -> str:
    """Compile every CUDA source for sm_100a into the in-tree shared library."""
    srcs = [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    deps = srcs + [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    deps.append(os.path.join(os.path.dirname(_HERE), "include", "drone_b200.h"))
    if not force and os.path.exists(LIB_PATH) and all(
            os.path.getmtime(LIB_PATH) >= os.path.getmtime(d) for d in deps):
        return LIB_PATH
    cmd = [nvcc_path(), *NVCC_FLAGS, "-o", LIB_PATH + ".tmp", *srcs]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
        print(" ".join(cmd))
    subprocess.check_call(cmd)
    os.replace(LIB_PATH + ".tmp", LIB_PATH)
    return LIB_PATH


def build_host_twin(force: bool = False) -> str:
    """g++ -ffp-contract=off csrc/host_twin.cpp -> libdrone_b200_host.so (the host instantiation of drone_core.cuh
    that tests/ check against the golden vectors on a machine without a GPU)."""
    src = os.path.join(CSRC, HOST_TWIN_SOURCE)
    deps = [src, os.path.join(CSRC, "drone_core.cuh"), os.path.join(os.path.dirname(_HERE), "include", "drone_b200.h"),
            os.path.join(os.path.dirname(_HERE), "include", "drone_b200_host.h")]
    if not force and os.path.exists(HOST_TWIN_PATH) and all(
            os.path.getmtime(HOST_TWIN_PATH) >= os.path.getmtime(d) for d in deps):
        return HOST_TWIN_PATH
    cxx = os.environ.get("CXX") or shutil.which("g++") or "g++"
    subprocess.check_call([cxx, *HOST_TWIN_FLAGS, "-o", HOST_TWIN_PATH + ".tmp", src])
    os.replace(HOST_TWIN_PATH + ".tmp", HOST_TWIN_PATH)
    return HOST_TWIN_PATH


class NativeError(RuntimeError):
    pass


_lib = None


def lib():
    """The loaded C-ABI library; raises (never falls back) when it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: the CUDA extension has not been built. "
            "Run `python __graft_entry__.py build` (needs nvcc). There is no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    vp, i32, i64, u32, u64 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint32, C.c_uint64
    PS, PP, PC = C.POINTER(DDState), C.POINTER(DDParams), C.POINTER(DDEnvConfig)
    L.dd_abi_version.restype = C.c_int
    L.dd_abi_version.argtypes = []
    L.dd_default_params.restype = None
    L.dd_default_params.argtypes = [PP]
    L.dd_error_string.restype = C.c_char_p
    L.dd_error_string.argtypes = [C.c_int]
    L.dd_reset.restype = C.c_int
    L.dd_reset.argtypes = [PS, PP, PC, vp, vp, i32, i64, vp]
    L.dd_step.restype = C.c_int
    L.dd_step.argtypes = [PS, PP, PC, vp, vp, i32, vp, vp, vp, vp, i64, vp]
    L.dd_step_plan.restype = C.c_int
    L.dd_step_plan.argtypes = [PS, PP, PC, vp, i32, vp, vp, vp, vp, i64, C.POINTER(DDStepPlan)]
    L.dd_step_planned.restype = C.c_int
    L.dd_step_planned.argtypes = [C.POINTER(DDStepPlan), vp, vp]
    L.dd_rollout.restype = C.c_int
    L.dd_rollout.argtypes = [PS, PP, PC, i32, vp, u32, i32, vp, vp, vp, i32, vp, i64, vp]
    L.dd_rollout_shaped.restype = C.c_int
    L.dd_rollout_shaped.argtypes = [PS, PP, PC, i32, vp, u32, i32, vp, vp, vp, i32, vp, vp, i64, vp]
    PSS = C.POINTER(DDParamSets)
    L.dd_param_sets_build.restype = C.c_int
    L.dd_param_sets_build.argtypes = [PP, i32, i32, vp]
    L.dd_reset_sets.restype = C.c_int
    L.dd_reset_sets.argtypes = [PS, PSS, PC, vp, vp, i32, i64, vp]
    L.dd_step_sets.restype = C.c_int
    L.dd_step_sets.argtypes = [PS, PSS, PC, vp, vp, i32, vp, vp, vp, vp, i64, vp]
    L.dd_step_plan_sets.restype = C.c_int
    L.dd_step_plan_sets.argtypes = [PS, PSS, PC, vp, i32, vp, vp, vp, vp, i64, C.POINTER(DDStepPlan)]
    L.dd_rollout_sets.restype = C.c_int
    L.dd_rollout_sets.argtypes = [PS, PSS, PC, i32, vp, u32, i32, vp, vp, vp, i32, vp, vp, i64, vp]
    L.dd_fill_random_actions.restype = C.c_int
    L.dd_fill_random_actions.argtypes = [vp, u64, u64, u32, i32, i64, vp]
    L.dd_pack_actions.restype = C.c_int
    L.dd_pack_actions.argtypes = [vp, vp, i64, vp]
    L.dd_stats_collapse.restype = C.c_int
    L.dd_stats_collapse.argtypes = [vp, vp, vp, i64, vp, vp]
    L.dd_moments.restype = C.c_int
    L.dd_moments.argtypes = [vp, i64, vp, vp]
    L.dd_normalize.restype = C.c_int
    L.dd_normalize.argtypes = [vp, vp, vp, C.c_double, i64, vp]
    L.dd_gae.restype = C.c_int
    L.dd_gae.argtypes = [vp, vp, vp, vp, vp, C.c_double, C.c_double, i32, i64, vp]
    L.dd_gae_moments.restype = C.c_int
    L.dd_gae_moments.argtypes = [vp, vp, vp, vp, vp, vp, C.c_double, C.c_double, i32, i64, vp]
    L.dd_policy_pack.restype = C.c_int
    L.dd_policy_pack.argtypes = [C.POINTER(DDPolicy), vp, C.POINTER(DDPolicyConsts), vp]
    L.dd_policy_pack_ex.restype = C.c_int
    L.dd_policy_pack_ex.argtypes = [C.POINTER(DDPolicy), i32, i32, vp, C.POINTER(DDPolicyConsts), vp]
    L.dd_policy_forward.restype = C.c_int
    L.dd_policy_forward.argtypes = [vp, C.POINTER(DDPolicyConsts), vp, vp, i64, vp]
    L.dd_discounted_returns.restype = C.c_int
    L.dd_discounted_returns.argtypes = [vp, vp, vp, C.c_double, i32, i64, vp]
    L.dd_gather_env.restype = C.c_int
    L.dd_gather_env.argtypes = [PS, vp, i32, vp, vp, i64, i64, vp, vp]
    L.dd_value_pack.restype = C.c_int
    L.dd_value_pack.argtypes = [C.POINTER(DDPolicy), vp, C.POINTER(DDPolicyConsts), vp]
    L.dd_value_forward.restype = C.c_int
    L.dd_value_forward.argtypes = [vp, C.POINTER(DDPolicyConsts), vp, vp, i64, vp]
    L.dd_policy_rollout.restype = C.c_int
    L.dd_policy_rollout.argtypes = [PS, PP, PC, vp, C.POINTER(DDPolicyConsts), i32, C.c_float, u32, i32, vp, vp, vp, vp, vp, vp, vp, vp, i64, vp]
    L.dd_policy_rollout_grid.restype = C.c_int
    L.dd_policy_rollout_grid.argtypes = [i64, i32]
    if L.dd_abi_version() != ABI_VERSION:
        raise NativeError(f"libdrone_b200.so ABI {L.dd_abi_version()} != binding {ABI_VERSION}; rebuild")
    _lib = L
    return L


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = lib().dd_error_string(rc).decode()
        raise NativeError(f"{what} failed: {msg} (code {rc})")


def default_params() -> DDParams:
    p = DDParams()
    lib().dd_default_params(C.byref(p))
    return p


def build_param_table(sets, dtype: int) -> bytes:
    """dd_param_sets_build: the DD_PARAM_TABLE_BYTES of 1..64 DDParams structs in DD_F32 / DD_F64 (host bytes)."""
    sets = list(sets)
    if not 1 <= len(sets) <= MAX_PARAM_SETS:
        raise ValueError(f"param_sets must hold 1 to {MAX_PARAM_SETS} DDParams structs")
    if not all(isinstance(p, DDParams) for p in sets):
        raise TypeError("param_sets must be DDParams structs")
    arr = (DDParams * len(sets))(*sets)
    out = C.create_string_buffer(PARAM_TABLE_BYTES)
    check(lib().dd_param_sets_build(arr, len(sets), int(dtype), out), "dd_param_sets_build")
    return out.raw


EXPORTS = (
    "dd_abi_version", "dd_default_params", "dd_error_string", "dd_reset", "dd_step", "dd_step_plan", "dd_step_planned",
    "dd_rollout", "dd_rollout_shaped",
    "dd_param_sets_build", "dd_reset_sets", "dd_step_sets", "dd_step_plan_sets", "dd_rollout_sets",
    "dd_fill_random_actions", "dd_pack_actions", "dd_stats_collapse", "dd_moments", "dd_normalize", "dd_gae", "dd_gae_moments",
    "dd_policy_pack", "dd_policy_pack_ex", "dd_policy_forward", "dd_policy_rollout", "dd_policy_rollout_grid", "dd_value_pack", "dd_value_forward", "dd_gather_env", "dd_discounted_returns",
)
HOST_TWIN_EXPORTS = ("dd_host_abi_version", "dd_reset_host", "dd_step_host", "dd_rollout_host", "dd_obs16_convert_host",
                     "dd_param_sets_build_host", "dd_reset_sets_host", "dd_step_sets_host", "dd_rollout_sets_host")

#!/usr/bin/env python
"""bench.py -- env-steps/sec of the batched delivery_drone simulator (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W]           # ours (CUDA, sm_100a): K timed steps
    python bench.py ... --dump-outputs DIR                         # + the last timed step's outputs as DIR/*.npy
    python bench.py --impl reference [--gpus N] --steps K ...      # the reference's CPU path (port)
    torchrun ... bench.py --gpus N ...                             # one rank per GPU, weak scaling

Workload (BASELINE.json configs[2]): 1,048,576 drone envs per GPU, auto-reset with Philox spawn
randomisation of drone and platform, 250-step truncation, synthetic random actions (p = 0.5 per
thruster) read from a pre-generated device trace.  One "step" = one DroneGame.step for every env
of one 1M-env shard = ONE launch of the fused step kernel.  The state of one shard (~56 MB, ~116 MB
with observations) would sit in the 126 MB L2, so the GPU holds SHARDS independent 1M-env shards
and consecutive steps rotate over them: every launch streams its state from HBM (working set
SHARDS x ~116 MB > L2).  All shards are real, distinct environments (own global env ids).

Printed JSON line (rank 0): value = env-steps/s over all ranks for the gym-surface step (obs +
reward + flags written, 146 algorithmic B/env-step); `variants` carries the step-only (86 B) and
T-steps-per-launch numbers; `e2e` = the same step through HOST buffers (pinned H2D of actions, D2H
of obs/reward/flags each step); `roofline` for the dominant kernel; `cpu_baseline` = the
reference-faithful Python port stepped by os.cpu_count() processes on this box.
"""
from __future__ import annotations

import argparse
import importlib
import json
import math
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "env-steps/sec"
UNIT = "env-steps/s"
ENVS_PER_GPU = 1 << 20
MAX_STEPS = 250
LEAD_IN = 32              # launches queued, untimed, ahead of the timed steps (~0.8 ms of GPU work at 1M envs per launch)
BYTES_STEP_ONLY = 86      # SURVEY.md 8d: read 44 + action 1, write 36 + reward 4 + flags 1
BYTES_GYM = 146           # + 60 B observation row
WORKLOAD = ("1M drone envs per GPU, auto-reset + spawn randomisation (drone+platform), max_steps 250, "
            "synthetic random actions from a device trace")


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ---------------------------------------------------------------------------------------------
# clocks sampling during the timed region (NVML in a thread; no subprocess, no GPU work)
# ---------------------------------------------------------------------------------------------
class ClockSampler:
    REASONS = {
        0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
        0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
        0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting",
    }

    def __init__(self, index: int, period_s: float = 0.01):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self.period, self._stop, self._thr, self.h = period_s, threading.Event(), None, None
        try:
            import pynvml
            self.nv = pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            if vis:
                try:
                    index = int(vis.split(",")[index])
                except ValueError:
                    pass
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception as e:          # NVML missing: report it, do not fail the bench
            self.err = repr(e)

    def _one(self):
        nv = self.nv
        self.samples.append(int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
        try:
            r = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
        except Exception:
            r = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
        for bit, name in self.REASONS.items():
            if r & bit and name != "gpu_idle":
                self.reasons.add(name)

    def _run(self):
        while not self._stop.is_set():
            try:
                self._one()
            except Exception:
                pass
            self._stop.wait(self.period)

    def start(self):
        if self.h is not None:
            self._stop.clear()
            self._thr = threading.Thread(target=self._run, daemon=True)
            self._thr.start()

    def stop(self):
        if self._thr is not None:
            self._stop.set()
            self._thr.join()
            self._thr = None

    def summary(self):
        if self.h is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "error": getattr(self, "err", "nvml unavailable")}
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


# ---------------------------------------------------------------------------------------------
# the CPU reference arm: reference-faithful Python port, one process per host core
# ---------------------------------------------------------------------------------------------
def cpu_port_multiprocess(ticks: int, warmup_ticks: int, procs: int | None = None, games: int = 6):
    """BASELINE.json configs[0]: 6 DroneGame instances per process, random actions, 250-step cap.
    Returns (env_steps_per_s aggregate, per-process mean, procs, seconds)."""
    import multiprocessing as mp
    from oracle.drone_port import cpu_rollout_worker
    procs = procs or os.cpu_count() or 1
    ctx = mp.get_context("fork")
    with ctx.Pool(procs) as pool:
        res = pool.map(cpu_rollout_worker, [(p, ticks, games, MAX_STEPS, warmup_ticks) for p in range(procs)])
    steps = sum(n for n, _ in res)
    slowest = max(s for _, s in res)
    per_proc = sum(n / s for n, s in res) / procs
    return steps / slowest, per_proc, procs, slowest


def c_oracle_threads(n: int, T: int, threads: int | None = None):
    """The C float64 restatement (oracle/drone_oracle.c) on all host cores: env-steps/s."""
    from concurrent.futures import ThreadPoolExecutor
    from oracle import c_oracle as co
    threads = threads or os.cpu_count() or 1
    b = co.OracleBatch(n, seed=0, randomize_drone=True, randomize_platform=True, max_steps=MAX_STEPS, auto_reset=True)
    b.reset()
    cuts = [n * i // threads for i in range(threads + 1)]
    t0 = time.perf_counter()
    with ThreadPoolExecutor(threads) as ex:     # ctypes releases the GIL inside the C call
        list(ex.map(lambda k: b.rollout(T, policy=co.POL_RANDOM, lo=cuts[k], hi=cuts[k + 1]), range(threads)))
    return n * T / (time.perf_counter() - t0), threads


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    K, W = args.steps, args.warmup
    # one "step" = `tps` ticks of (6 games x P processes); sized so K steps take ~10 s of CPU work
    rate_guess = 7000.0                                   # ticks/s/process of the Python port
    tps = max(1, int(math.ceil(10.0 * rate_guess / max(K, 1))))
    tps = min(tps, max(1, int(120.0 * rate_guess / max(K + W, 1))))   # never more than ~2 min in total
    agg, per_proc, procs, secs = cpu_port_multiprocess(K * tps, W * tps)
    sample = (f"{procs} processes x 6 PortDroneGame (reference-faithful Python port of DroneGame), random actions, "
              f"250-step cap, {K} steps x {tps} ticks x {6 * procs} envs = {K * tps * 6 * procs} env-steps")
    line = {
        "impl": "reference", "metric": METRIC, "value": agg, "unit": UNIT, "n_gpus": args.gpus, "steps": K, "warmup": W,
        "ms_per_step": secs / K * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "reference_sample": sample},
        "cpu_baseline": {"value": agg, "unit": UNIT, "cores": procs, "kind": "port", "sample": sample,
                         "per_process": per_proc},
        "e2e": {"value": agg, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


# ---------------------------------------------------------------------------------------------
# ours
# ---------------------------------------------------------------------------------------------
BYTES_GYM_F64 = 282       # the float64 (exact-parity) instantiation: read 84 + 1, write 68 + reward 8 + flags 1 + obs 120
FLOP_STEP = 2 * (15 * 128 + 128 * 128 + 128 * 64 + 64 * 3)              # SURVEY.md 8d: 53,376 per env-step (policy)
FLOP_ROW_CRITIC = 2 * (15 * 128 + 128 * 128 + 128 * 64 + 64 * 1)        # critic head is 64 -> 1


def _peaks_all():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    d = json.load(open(p)) if os.path.exists(p) else {}
    return {"hbm_gbs": float(d.get("hbm_gbs", 6650.0)), "hbm_src": "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in d else "fallback (B200_PROFILING.md 6.65 TB/s)",
            "bf16_sustained": float(d.get("bf16_tflops_sustained", 1400.0)), "bf16_burst": float(d.get("bf16_tflops", 1600.0)),
            "bf16_src": "measured (MEASURED_PEAKS.json bf16_tflops_sustained: kernels timed inside a long loop)" if "bf16_tflops_sustained" in d else "fallback (B200_PROFILING.md)"}


def _ncu_traffic(n: int):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of step_kernel<float,AUTO,OBS> from the COMMITTED
    ncu capture (the newest of profiles/r02_traffic_steady.json, r01_traffic_steady.json; ncu cannot run inside the
    bench) -- a constant read from that file, not measured in this run, and only valid for the launch size it was
    captured at."""
    for name in ("r02_traffic_steady.json", "r01_traffic_steady.json"):
        path = os.path.join(ROOT, "profiles", name)
        try:
            with open(path) as f:
                d = json.load(f)
            k = next(v for kk, v in d["kernels"].items() if "step_kernel<float, 1, 1, 1, 256>" in kk)
            if d["algorithmic_bytes_per_launch"]["step_kernel<float,AUTO,OBS>"] != BYTES_GYM * n:
                return None, f"profiles/{name} was captured at another launch size than {n} envs"
            return k["dram_bytes_per_launch"], f"constant from the committed capture profiles/{name} (ncu, steady state, --cache-control none); not measured in this run"
        except (OSError, KeyError, ValueError, StopIteration):
            continue
    return None, "no ncu capture committed"


def socket_shim_rate(dev, games: int = 6, seconds: float = 2.0):
    """Context number (SURVEY.md 8d): the reference's TCP/JSON protocol served from the batched env -- 6 games,
    one client stepping them round-robin with random actions, reset on done, like the notebooks do.  The
    reference documents 300-500 steps/s for its own server (SOCKET_API.md:373); measured 58.5 steps/s at its
    default --fps 60 and ~6.7e3 with the fps cap lifted (BASELINE.md section 2)."""
    import random
    compat = importlib.import_module("reinforcement-learning-101_b200.compat")
    pool = compat.DroneGamePool(games, device=dev, seed=0, randomize_drone=True, randomize_platform=True)
    srv = compat.DroneSocketServer(pool, host="127.0.0.1", port=0)
    srv.start(background=True)
    cli = compat.DroneGameClient(host="127.0.0.1", port=srv.port, timeout=10.0)
    rng = random.Random(0)
    lat = []
    try:
        for g in range(games):
            cli.reset(g)
        t_end = time.perf_counter() + seconds
        n = 0
        while time.perf_counter() < t_end:
            g = n % games
            t0 = time.perf_counter()
            _, _, done, _ = cli.step({"main_thrust": rng.getrandbits(1), "left_thrust": rng.getrandbits(1),
                                      "right_thrust": rng.getrandbits(1)}, g)
            lat.append(time.perf_counter() - t0)
            if done:
                cli.reset(g)
            n += 1
    finally:
        cli.close()
        srv.stop()
    lat.sort()
    return {"steps_per_s": len(lat) / sum(lat), "median_step_latency_ms": lat[len(lat) // 2] * 1e3,
            "p99_step_latency_ms": lat[int(len(lat) * 0.99)] * 1e3, "games": games, "steps": len(lat),
            "what": "compat.DroneSocketServer + DroneGameClient over 127.0.0.1 (the reference's wire protocol), one request per step"}


DUMP_ROWS = 1 << 19      # env rows written by --dump-outputs: 17 float32 + 1 float64 per row, 40 MB at most


def dump_outputs(out_dir: str, env) -> dict:
    """What the last timed step handed its caller, as DIR/<name>.npy: the observations, rewards and flags (DD_* bits,
    as numbers) of the shard that step advanced, in float32.  A shard of more than DUMP_ROWS envs is sampled at fixed,
    seeded rows; env_index.npy (float64) lists the rows written."""
    import numpy as np
    import torch
    env.join()
    s = (env.t - 1) % env.S
    sh = env.shards[s]
    n = sh.num_envs
    rows = np.arange(n) if n <= DUMP_ROWS else np.sort(np.random.default_rng(0).choice(n, DUMP_ROWS, replace=False))
    idx = torch.from_numpy(rows).to(sh.obs.device)
    arrays = {"obs": sh.obs[idx], "reward": sh.reward[idx], "flags": sh.step_flags[idx]}
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "env_index.npy"), rows.astype(np.float64))
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.float().cpu().numpy())
    return {"dir": out_dir, "shard": s, "launch": env.t - 1, "rows": len(rows), "of": n,
            "files": ["env_index.npy"] + [name + ".npy" for name in arrays]}


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    dd = importlib.import_module("reinforcement-learning-101_b200")

    # keep stdout to the one JSON line: NCCL prints its version banner to stdout at communicator creation when the
    # box sets NCCL_DEBUG -- send NCCL's log to stderr and, belt and braces, point fd 1 at stderr while NCCL initialises
    os.environ["NCCL_DEBUG_FILE"] = os.environ.get("NCCL_DEBUG_FILE") or "/dev/stderr"
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    try:
        rank, local, ws = dd.init_from_env("nccl")
        if ws != args.gpus and ws > 1:
            raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={ws}")
        torch.cuda.set_device(local)
        dev = torch.device("cuda", local)
        if ws > 1:                                             # first collective: the communicator exists after this
            warm = torch.zeros(1, device=dev)
            dist.all_reduce(warm)
            torch.cuda.synchronize(dev)
    finally:
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        os.close(saved_stdout)
    cpus = dd.bind_to_gpu_numa(local) if ws > 1 and not args.no_numa_bind else None   # host buffers next to the GPU
    K, W, S, n = args.steps, max(args.warmup, 3), args.shards, args.envs
    PK = _peaks_all()
    peak_gbs = PK["hbm_gbs"]
    launches = 0

    def barrier():
        if ws > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(ms: float) -> float:
        if ws == 1:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def timed(fn_warm, fn_run, sampler=None):
        """warm-up, barrier + sync, CUDA events around fn_run on the current stream, barrier + sync, max over ranks.
        `sampler` polls NVML from a thread exactly while the timed region runs."""
        fn_warm()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if sampler is not None:
            sampler.start()
        e0.record()
        fn_run()
        e1.record()
        torch.cuda.synchronize(dev)
        if sampler is not None:
            sampler.stop()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1))

    # ---- the product path: dd.ShardedDroneEnv (S independent 1M-env shards, parallel chains, CUDA graphs) ----
    def make_sharded(dtype, shards):
        env = dd.ShardedDroneEnv(shards, n, device=dev, chains=args.chains, trace_len=args.trace_len,
                                 use_graphs=not args.eager, env_id_base=rank * shards * n, launch_flags=args.launch_flags,
                                 seed=0, randomize_drone=True, randomize_platform=True, max_steps=MAX_STEPS,
                                 auto_reset=True, dtype=dtype)
        env.reset()
        env.random_trace()
        return env

    def time_steps(env, want_obs, sampler=None):
        """The K timed steps: one block env.run(K) (graph replays whatever K is), after the warm-up steps, a rehearsal that
        captures every graph a block can replay and an untimed lead-in: one run() of at least LEAD_IN launches, whole
        K-step blocks, so that the host has queued the timed block long before the GPU reaches it.  The events are
        recorded on the env's chain streams, after the lead-in and after the K steps: each chain's share of the K launches
        is timed from the end of its own lead-in to its own end, and the region is the longest of these spans.  So the
        launches are timed as they flow behind work in flight, and neither the host's launch latency, the fork and join
        of the chains, the refill of an idle GPU nor the phase offset between the chains enters it.  On a B200 at 1,000 W,
        one CUDA-event pair on the caller's stream around the block measured ~22 us per region above the steady per-step
        time, these spans ~10 us (the drain of the last launch).  Returns the milliseconds of the K steps (max over ranks)."""
        period = env.S * env.L

        def blocks(r):
            for _ in range(r):
                env.run(K, want_obs=want_obs)
            env.join()
        blocks(-(-W // K))                                      # the W warm-up steps
        blocks(period // math.gcd(K, period))                   # visits every (offset, length) piece of the schedule

        def measure():
            barrier()
            env.run(K * -(-max(LEAD_IN, env.C) // K), want_obs=want_obs)   # the lead-in (may capture: not timed)
            g0 = env.graphs_cached
            t0, t1 = ([torch.cuda.Event(enable_timing=True) for _ in env._chains] for _ in range(2))
            for ev, ch in zip(t0, env._chains):
                ev.record(ch)
            if sampler is not None:
                sampler.start()
            env.run(K, want_obs=want_obs)
            for ev, ch in zip(t1, env._chains):
                ev.record(ch)
            env.join()
            torch.cuda.synchronize(dev)
            if sampler is not None:
                sampler.stop()
            barrier()
            return max_over_ranks(max(a.elapsed_time(b) for a, b in zip(t0, t1))), env.graphs_cached != g0
        ms, captured = measure()
        if max_over_ranks(float(captured)) > 0:                 # a capture happened inside the timed region (any rank): redo
            ms, _ = measure()
        return ms

    sampler = ClockSampler(local, period_s=0.004)
    env = make_sharded(torch.float32, S)
    ms_gym = time_steps(env, True, sampler)
    launches += K
    dumped = dump_outputs(args.dump_outputs, env) if args.dump_outputs and rank == 0 else None
    ms_so = time_steps(env, False, None)
    launches += K
    launch_mode = (f"eager: one dd_step_planned call per step on {env.C} chain stream(s)" if args.eager else
                   f"CUDA graphs (product path ShardedDroneEnv.run): each K-step block is one piece of the {env.S * env.L}-launch "
                   f"schedule and replays one cached graph per chain; {env.C} parallel chain(s) over independent shards, joined to "
                   f"the timing stream once per timed region; {env.graphs_cached} pieces cached, {env.graph_replays} graph replays, "
                   f"{env.eager_launches} eager launches")
    launch_mode += f"; launch_flags={args.launch_flags:#x}"

    # host cost of one eager step through the public API (BatchedDroneEnv.step_raw -> dd_step_planned), GPU idle-free:
    # time the Python loop alone for a small env so the GPU never back-pressures the queue
    tiny = dd.BatchedDroneEnv(256, device=dev, seed=0, randomize_drone=True, randomize_platform=True, max_steps=MAX_STEPS,
                              auto_reset=True, dtype=torch.float32)
    tiny.reset()
    tact = tiny.random_actions(1)[0]
    for _ in range(200):
        tiny.step_raw(tact)
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    for _ in range(2000):
        tiny.step_raw(tact)
    host_us = (time.perf_counter() - t0) / 2000 * 1e6
    torch.cuda.synchronize(dev)
    launches += 2200
    # ... and the eager product path on the full-size shards: what a caller that cannot use graphs gets -- the same
    # schedule and chains, every launch a Python -> dd_step_planned call
    def eager_steps(k):
        env.run(k)
        env.join()
    Ke = max(K, 240)
    env.use_graphs = False
    ms_eager = timed(lambda: eager_steps(S), lambda: eager_steps(Ke))
    env.use_graphs = not args.eager
    launches += Ke + S

    # ---- the exact (float64) instantiation on the same workload: north_star's flag rule is met by this one ----
    f64 = None
    if not args.no_f64:
        S64 = max(2, min(S, 4))
        env64 = make_sharded(torch.float64, S64)
        ms64 = time_steps(env64, True, None)
        launches += K
        a64 = n * BYTES_GYM_F64 / (ms64 * 1e-3 / K) / 1e9
        f64 = {"value": n * K * ws / (ms64 * 1e-3), "ms_per_step": ms64 / K, "dtype": "f64",
               "algorithmic_bytes_per_env_step": BYTES_GYM_F64, "achieved_gbs": a64, "frac": a64 / peak_gbs,
               "shards_per_gpu": S64, "timed_region_ms": ms64,
               "what": "step_kernel<double,AUTO,OBS>: state, observations and rewards in float64, flags / counters bit-exact "
                       "against the oracle (tests/test_gpu_parity.py); FP64 pipe bound on B200, not HBM bound"}
        del env64
        torch.cuda.empty_cache()

    # ---- T-steps-per-launch rollout kernel (state in registers; Philox actions in-kernel) ----
    T_ROLL = 50
    reps = max(1, K // T_ROLL // S) * S
    env.join()
    shards = env.shards

    def run_rollouts(k):
        for j in range(k):
            shards[j % S].rollout(T_ROLL, "random")
    ms_roll = timed(lambda: run_rollouts(S), lambda: run_rollouts(reps))
    launches += reps

    def run_rollouts_bb(k):                                 # cfg 3 (ii): fixed policy main = vy > 1.5, computed in-kernel
        for j in range(k):
            shards[j % S].rollout(T_ROLL, "bangbang")
    ms_roll_bb = timed(lambda: run_rollouts_bb(S), lambda: run_rollouts_bb(reps))
    launches += reps

    # ---- K5: fused policy rollout, BASELINE configs[3]: 65,536 envs x 250 steps, policy MLP in-kernel ----
    k5, others = None, {}
    fix = os.path.join(ROOT, "tests", "golden", "policy_v1.npz")
    cfix_path = os.path.join(ROOT, "tests", "golden", "critic_v1.npz")
    if not args.no_policy and not (os.path.exists(fix) and os.path.exists(cfix_path)):
        k5 = {"skipped": "checkpoint fixtures tests/golden/policy_v1.npz / critic_v1.npz not found"}   # same on every rank
    elif not args.no_policy:
        d = np.load(fix)
        sd = {kk: torch.from_numpy(d[kk]) for kk in d.files if kk.startswith("network")}
        blob = dd.PolicyBlob(sd, device=dev)
        NP, TP = args.policy_envs, 250
        penv = dd.BatchedDroneEnv(NP, device=dev, seed=0, randomize_drone=True, randomize_platform=True,
                                  max_steps=MAX_STEPS, auto_reset=True, dtype=torch.float32, env_id_base=rank * NP)
        penv.reset()
        pbuf = dd.policy_rollout(penv, blob, TP, sample=True, want="arldo")      # allocates the rollout buffers
        reps_p = 40                                          # ~50 ms per timed region

        def run_policy(kk):
            for _ in range(kk):
                dd.policy_rollout(penv, blob, TP, sample=True, want="arldo", out=pbuf)      # t0: the env's running counter
        ms_pol = timed(lambda: run_policy(2), lambda: run_policy(reps_p))
        launches += reps_p + 2
        steps_s = NP * TP * reps_p * ws / (ms_pol * 1e-3)
        tf = steps_s / ws * FLOP_STEP / 1e12
        k5 = {"value": steps_s, "envs_per_gpu": NP, "steps_per_launch": TP, "ms_per_launch": ms_pol / reps_p, "launches_timed": reps_p,
              "mlp_tflops": tf, "flop_per_env_step": FLOP_STEP, "frac_of_sustained_bf16": tf / PK["bf16_sustained"],
              "buffers": "obs[T,N,15] f32, action u8, logp f32, reward f32, done u8 (70 B/env-step)",
              "policy": "drone_policy_v1 (27,651 params), Bernoulli sampling, 16-bit tcgen05 MMA operands / fp32 accumulate",
              "operands": getattr(blob, "operand_dtype", "bf16"),
              "stats": penv.stats(reduce=ws > 1)}
        others["fused_policy_rollout_K5"] = {"bound": "tensor", "achieved": tf, "peak": PK["bf16_sustained"], "unit": "TFLOP/s",
                                             "frac": tf / PK["bf16_sustained"], "frac_of_burst": tf / PK["bf16_burst"],
                                             "ms_per_launch": ms_pol / reps_p, "algorithmic": f"{FLOP_STEP} FLOP x {NP} envs x {TP} steps per launch"}
        # 65,536 envs are 512 tiles of 128 = 128 CTAs: 20 of the 148 SMs idle.  One tile set per SM for reference.
        NF = 148 * 512
        fenv = dd.BatchedDroneEnv(NF, device=dev, seed=0, randomize_drone=True, randomize_platform=True,
                                  max_steps=MAX_STEPS, auto_reset=True, dtype=torch.float32, env_id_base=rank * NF)
        fenv.reset()
        fbuf = dd.policy_rollout(fenv, blob, TP, sample=True, want="arldo")

        def run_policy_full(kk):
            for _ in range(kk):
                dd.policy_rollout(fenv, blob, TP, sample=True, want="arldo", out=fbuf)
        ms_full = timed(lambda: run_policy_full(1), lambda: run_policy_full(reps_p))
        launches += reps_p + 1
        k5["all_148_sms"] = {"envs_per_gpu": NF, "ms_per_launch": ms_full / reps_p,
                             "value": NF * TP * reps_p * ws / (ms_full * 1e-3),
                             "mlp_tflops": NF * TP * reps_p / (ms_full * 1e-3) * FLOP_STEP / 1e12}
        del fenv, fbuf
        # what follows the rollout in the PPO loop (Actor_Critic_PPO.ipynb, PHASE 2): critic values over the stored
        # states + bootstrap row, compute_gae, advantage normalisation -- all on the rollout buffers in HBM
        cfix = np.load(cfix_path)
        vblob = dd.ValueBlob({kk: torch.from_numpy(cfix[kk]) for kk in cfix.files if kk.startswith("network")}, device=dev)
        final_obs = penv.observe().clone()
        vals = dd.rollout_values(vblob, pbuf["obs"], final_obs)
        dones = (pbuf["done"] != 0).to(torch.uint8)
        adv = dd.gae(pbuf["reward"], vals, dones)
        nadv = torch.empty_like(adv)

        mom_f = torch.zeros(3, dtype=torch.float64, device=dev)

        def run_ppo_tail(kk):
            for _ in range(kk):
                dd.rollout_values(vblob, pbuf["obs"], final_obs)
                mom_f.zero_()
                dd.gae(pbuf["reward"], vals, dones, out=adv, moments=mom_f)        # scan + advantage moments in one pass
                dd.normalize_advantages(adv, reduce=ws > 1, out=nadv, moments=mom_f)
        ms_tail = timed(lambda: run_ppo_tail(1), lambda: run_ppo_tail(reps_p))
        launches += 5 * (reps_p + 1)
        # each kernel of the tail alone, against its own roofline.  Working sets: critic 983 MB of observations, GAE 213 MB
        # (> the 126 MB L2); moments / normalise rotate over four / two distinct 65 MB buffers so that no launch finds its
        # input in L2.
        ne = NP * TP
        rot = [pbuf["reward"], pbuf["logp"], adv, nadv]
        nrm_out = [torch.empty_like(adv), torch.empty_like(adv)]
        mom = torch.zeros(3, dtype=torch.float64, device=dev)
        mom1 = dd.advantage_moments(adv)

        # the timing loops call the C ABI directly with pre-extracted pointers (3-4 us of host time per launch), so that
        # the 15-40 us kernels are timed, not the Python wrappers' argument checks; every region is >= 30 ms.  Order =
        # pipeline order: the GAE scan is timed right after the tensor-heavy critic forward, i.e. at the SM clock the
        # power cap leaves then (stand-alone, at boost clock, the same launch takes 38 us instead of 42: profiles/README.md)
        lib = dd.native.lib()
        st = torch.cuda.current_stream(dev).cuda_stream
        p_rew, p_val, p_don, p_adv, p_mom = (pbuf["reward"].data_ptr(), vals.data_ptr(), dones.data_ptr(), adv.data_ptr(), mom_f.data_ptr())
        p_rot = [t_.data_ptr() for t_ in rot]
        p_out = [t_.data_ptr() for t_ in nrm_out]
        p_mom1, p_momacc = mom1.data_ptr(), mom.data_ptr()

        def t_values(kk):
            for _ in range(kk):
                dd.value_forward(vblob, pbuf["obs"], out=vals[:TP])
        def t_gae(kk):
            for _ in range(kk):
                lib.dd_gae_moments(p_rew, p_val, p_don, p_adv, None, p_mom, 0.99, 0.95, TP, NP, st)
        def t_mom(kk):
            for j in range(kk):
                lib.dd_moments(p_rot[j % 4], ne, p_momacc, st)
        def t_nrm(kk):
            for j in range(kk):
                lib.dd_normalize(p_rot[j % 2], p_out[j % 2], p_mom1, 1e-8, ne, st)
        n_g, n_m, n_n = 800, 2000, 1200
        ms_v = timed(lambda: t_values(1), lambda: t_values(reps_p)) / reps_p
        ms_g = timed(lambda: t_gae(4), lambda: t_gae(n_g)) / n_g
        ms_m = timed(lambda: t_mom(8), lambda: t_mom(n_m)) / n_m
        ms_n = timed(lambda: t_nrm(4), lambda: t_nrm(n_n)) / n_n
        launches += reps_p + n_g + n_m + n_n + 17
        vtf = ne * FLOP_ROW_CRITIC / (ms_v * 1e-3) / 1e12
        others["critic_value_forward"] = {"bound": "tensor", "achieved": vtf, "peak": PK["bf16_sustained"], "unit": "TFLOP/s",
                                          "frac": vtf / PK["bf16_sustained"], "ms_per_launch": ms_v, "rows": ne}
        for name, ms_, bytes_el, what in (
                ("gae_kernel", ms_g, 13.0 + 4.0 / TP, "read reward 4 + value 4 + done 1, write advantage 4 B per element (+ the bootstrap row); the advantage moments are accumulated in the same pass"),
                ("moments_kernel", ms_m, 4.0, "one read of a [T,N] buffer (stand-alone K4; the PPO tail gets its moments from the GAE pass)"),
                ("normalize_kernel", ms_n, 8.0, "read 4 + write 4 B per element")):
            ach = ne * bytes_el / (ms_ * 1e-3) / 1e9
            others[name] = {"bound": "hbm", "achieved": ach, "peak": peak_gbs, "unit": "GB/s", "frac": ach / peak_gbs,
                            "ms_per_launch": ms_, "elements": ne, "algorithmic_bytes_per_element": bytes_el, "what": what}
        # The figures above are taken in pipeline order, back to back, on a board that the 40-launch loops of the tensor
        # kernels have driven into its power cap (SM clock ~1.7-1.8 GHz).  For reference, the same two kernels again after
        # 0.4 s of idle, i.e. from the boost clock a PPO loop sees when its rollout follows a learning phase (not used for
        # any headline number; the clock-sensitive ones are K5 itself and the GAE scan, 443 threads per SM).
        torch.cuda.synchronize(dev); time.sleep(0.4)
        ms_g_idle = timed(lambda: t_gae(4), lambda: t_gae(n_g)) / n_g
        torch.cuda.synchronize(dev); time.sleep(0.4)
        ms_pol_idle = timed(lambda: run_policy(2), lambda: run_policy(20)) / 20
        launches += n_g + 4 + 22
        others["gae_kernel"].update({"ms_per_launch_after_idle": ms_g_idle, "frac_after_idle": ne * (13.0 + 4.0 / TP) / (ms_g_idle * 1e-3) / 1e9 / peak_gbs})
        others["fused_policy_rollout_K5"].update({"ms_per_launch_after_idle": ms_pol_idle,
                                                  "frac_after_idle": NP * TP * FLOP_STEP / (ms_pol_idle * 1e-3) / 1e12 / PK["bf16_sustained"],
                                                  "after_idle_what": "the same launch timed again (20 launches) after 0.4 s of idle: boost clock instead of the power-capped clock the preceding timing loops leave"})
        del rot, nrm_out
        # the same through HOST-side inputs / outputs, as one PPO iteration sees it: policy + critic weights come from
        # host state_dicts (packed and uploaded every iteration, like after an optimiser step), the rollout buffers
        # stay in HBM for the learner, the episode statistics and advantage moments go back to the host
        sd_host = {kk: v.clone() for kk, v in sd.items()}
        sdc_host = {kk: torch.from_numpy(cfix[kk]) for kk in cfix.files if kk.startswith("network")}
        t_it = []
        n_it = 3 + min(reps_p, 10)
        for it in range(n_it):
            barrier()
            t0 = time.perf_counter()
            b_it = dd.PolicyBlob(sd_host, device=dev)
            vb_it = dd.ValueBlob(sdc_host, device=dev)
            penv.reset_stats()
            dd.policy_rollout(penv, b_it, TP, sample=True, want="arldo", out=pbuf)
            dd.rollout_values(vb_it, pbuf["obs"], penv.observe())
            mom_f.zero_()
            dd.gae(pbuf["reward"], vals, dones, out=adv, moments=mom_f)
            dd.normalize_advantages(adv, reduce=ws > 1, out=nadv, moments=mom_f)
            st_it = penv.stats(reduce=ws > 1)                  # device -> host: synchronises
            t_it.append(time.perf_counter() - t0)
        launches += 9 * len(t_it)
        it_s = max_over_ranks(sum(t_it[3:]) / (n_it - 3) * 1e3) * 1e-3
        k5["ppo_iteration_e2e"] = {"what": "host state_dicts -> pack + upload (policy, critic) -> fused rollout -> critic values -> GAE -> "
                                           "advantage normalisation -> episode statistics back on the host; wall clock per iteration",
                                   "ms": it_s * 1e3, "env_steps_per_s": NP * TP * ws / it_s,
                                   "landing_rate": st_it["landing_rate"]}
        k5["ppo_data_path"] = {"what": "critic values [T+1,N] (tcgen05, persistent forward) + GAE + advantage normalisation on the rollout buffers",
                               "ms": ms_tail / reps_p, "samples_per_s": NP * TP * reps_p * ws / (ms_tail * 1e-3),
                               "rollout_plus_tail_ms": (ms_pol + ms_tail) / reps_p,
                               "kernels_ms": {"value_forward": ms_v, "gae": ms_g, "moments": ms_m, "normalize": ms_n}}

    # ---- BASELINE configs[4]: curriculum sweep 75 -> 250, 2M envs per GPU, stats all-reduced over ranks ----
    cur = None
    mgc = None
    if not args.no_curriculum:
        NC = args.curriculum_envs
        cenv = dd.BatchedDroneEnv(NC, device=dev, seed=0, randomize_drone=True, randomize_platform=True,
                                  auto_reset=False, dtype=torch.float32, env_id_base=rank * NC)
        caps = dd.step_schedule(8, 75, 250).tolist()
        dd.collect_episodes(cenv, caps[0], policy="bangbang", reduce=ws > 1)           # warm-up
        stages = []

        def run_sweep():
            stages[:] = dd.curriculum_sweep(cenv, caps, policy="bangbang", reduce=ws > 1)
        ms_cur = timed(lambda: None, run_sweep)
        launches += 2 * len(caps)
        cur = {"envs_total": NC * ws, "caps": caps, "ms_total": ms_cur,
               "env_steps_per_s": sum(s_["env_steps"] for s_ in stages) / (ms_cur * 1e-3),
               "policy": "bang-bang (main = vy > 1.5), one episode per env per stage, freeze after done",
               "stages": [{k_: s_[k_] for k_ in ("max_steps", "success_rate", "avg_reward", "avg_steps")} for s_ in stages]}
        # ---- N > 1: is the all-reduced result the sum of what every shard computes?  (SURVEY.md 8d cfg 5: "check
        # against single-GPU recomputation"; Actor_Critic_PPO.ipynb c21:L94-95,L105,L169 is what the numbers stand for) ----
        if ws > 1:
            mgc = multi_gpu_check(dd, dist, cenv, caps[2], rank, ws, NC, dev)
            launches += 8
        del cenv

    # ---- e2e: HOST buffers in, HOST buffers out, every step ----
    io = [shards[s].make_host_io() for s in range(min(S, 2))]
    host_trace = env.trace[:, 0].cpu().pin_memory()         # [L, N]: the caller's actions of shard 0, on the host
    Ke2 = max(3, min(K * 4, args.e2e_steps))
    e2e_modes = {}
    for mode in ("copy", "zero_copy"):
        def run_e2e(k):
            for j in range(k):                               # the caller's actions of this step: a row of pinned host memory
                shards[j % S].step_host(io[j % len(io)], mode=mode, actions=host_trace[j % env.L])
        ms_e2e = timed(lambda: run_e2e(3), lambda: run_e2e(Ke2))
        launches += Ke2 + 3
        e2e_modes[mode] = ms_e2e / Ke2
    # the same steps, two in flight: step j+1 (another shard, another pinned buffer, another stream) is enqueued before the
    # host waits for step j, so the device->host copy of one shard overlaps the host->device copy + kernel of the next.
    # Every step still takes its actions from pinned host memory and delivers obs / reward / flags to pinned host memory,
    # and the host waits for every step's results (event) before that buffer is reused.
    side = [torch.cuda.Stream(dev) for _ in io]

    def run_e2e_pipelined(k):
        cur = torch.cuda.current_stream(dev)
        for sd in side:
            sd.wait_stream(cur)
        pend = [None] * len(io)
        for j in range(k):
            b = j % len(io)
            if pend[b] is not None:
                pend[b].synchronize()                        # the host consumes the results of step j - 2 here
            with torch.cuda.stream(side[b]):
                pend[b] = shards[j % S].step_host(io[b], mode="copy", actions=host_trace[j % env.L], wait=False)
        for p_ in pend:
            if p_ is not None:
                p_.synchronize()
        for sd in side:
            cur.wait_stream(sd)
    ms_e2e = timed(lambda: run_e2e_pipelined(4), lambda: run_e2e_pipelined(Ke2))
    launches += Ke2 + 4
    e2e_modes["copy_2_in_flight"] = ms_e2e / Ke2
    h2d = n * 1
    d2h = n * (shards[0].obs_stride * 4 + 4 + 1)
    # the ceiling of this box for the same bytes: plain cudaMemcpyAsync of the packed block into pinned memory, all
    # ranks at once (profiles/pcie_ceiling.py is the standalone version)
    blk_d, blk_h = shards[0]._out_block, io[0]["block"]

    def run_copy(k):
        for _ in range(k):
            blk_h.copy_(blk_d, non_blocking=True)
    ms_ceil = timed(lambda: run_copy(3), lambda: run_copy(30)) / 30
    ceil_gbs = blk_d.numel() / (ms_ceil * 1e-3) / 1e9
    best_mode = min(e2e_modes, key=e2e_modes.get)
    ms_e2e_step = e2e_modes[best_mode]

    stats = env.stats(reduce=ws > 1)

    if rank == 0:
        value = n * K * ws / (ms_gym * 1e-3)
        per_launch_s = ms_gym * 1e-3 / K
        achieved = n * BYTES_GYM / per_launch_s / 1e9
        traffic, traffic_src = _ncu_traffic(n)
        so_per = ms_so * 1e-3 / K
        so_achieved = n * BYTES_STEP_ONLY / so_per / 1e9
        eg_ach = n * BYTES_GYM / (ms_eager * 1e-3 / Ke) / 1e9
        others["step_kernel_step_only"] = {"bound": "hbm", "achieved": so_achieved, "peak": peak_gbs, "unit": "GB/s",
                                           "frac": so_achieved / peak_gbs, "algorithmic_bytes_per_env_step": BYTES_STEP_ONLY}
        if f64 is not None:
            others["step_kernel_f64"] = {"bound": "hbm", "achieved": f64["achieved_gbs"], "peak": peak_gbs, "unit": "GB/s",
                                         "frac": f64["frac"], "algorithmic_bytes_per_env_step": BYTES_GYM_F64,
                                         "note": "limited by the FP64 pipe of B200, reported against HBM for comparison"}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": ws, "steps": K, "warmup": W,
            "ms_per_step": ms_gym / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "timed_region_ms": ms_gym, "steps_timed": K,
            "config": {"workload": WORKLOAD, "envs_per_gpu_per_step": n, "shards_per_gpu": S,
                       "l2": f"inputs larger than L2: steps rotate over {S} independent {n}-env shards "
                             f"({S} x ~{n * 116 >> 20} MiB state+outputs > 126 MB L2)",
                       "launch": launch_mode, "parallelism": f"env-sharded x{ws}, no per-step comms",
                       "timing": f"the K = {K} steps as one block behind an untimed lead-in, timed by CUDA events on "
                                 f"the chain streams: the longest span of a chain from the end of its lead-in to the end of its "
                                 f"share; ms_per_step = timed_region_ms / K; clocks sampled by NVML every 4 ms inside that region"},
            "roofline": {"bound": "hbm", "kernel": "step_kernel<float,AUTO,OBS>", "achieved": achieved, "peak": peak_gbs,
                         "unit": "GB/s", "frac": achieved / peak_gbs, "frac_of_nominal_8000_gbs": achieved / 8000.0,
                         "traffic": traffic, "traffic_unit": "bytes per launch",
                         "traffic_source": traffic_src, "algorithmic_bytes_per_launch": BYTES_GYM * n, "peak_source": PK["hbm_src"],
                         "algorithmic_bytes_per_env_step": BYTES_GYM, "env_steps_per_launch": n,
                         "others": others, "others_tensor_peak_source": PK["bf16_src"]},
            "variants": {
                "step_only": {"value": n * K * ws / (ms_so * 1e-3), "ms_per_step": so_per * 1e3,
                              "algorithmic_bytes_per_env_step": BYTES_STEP_ONLY, "achieved_gbs": so_achieved,
                              "frac": so_achieved / peak_gbs, "timed_region_ms": ms_so},
                "gym_step_f64": f64,
                "gym_step_eager_api": {"value": n * Ke * ws / (ms_eager * 1e-3), "ms_per_step": ms_eager / Ke, "achieved_gbs": eg_ach,
                                       "frac": eg_ach / peak_gbs, "steps": Ke, "host_us_per_step_raw_call": host_us,
                                       "what": "ShardedDroneEnv(use_graphs=False): BatchedDroneEnv.step_raw called from Python once per step "
                                               "(dd_step_planned) on the chain streams, no graph: the path of a caller that cannot capture"},
                "rollout_T50_fixed_policy_bangbang": {"value": n * T_ROLL * reps * ws / (ms_roll_bb * 1e-3),
                                                      "ms_per_launch": ms_roll_bb / reps, "steps_per_launch": T_ROLL},
                "rollout_T50_in_kernel_actions": {"value": n * T_ROLL * reps * ws / (ms_roll * 1e-3),
                                                  "ms_per_launch": ms_roll / reps, "steps_per_launch": T_ROLL},
                "fused_policy_rollout": k5,
                "curriculum_sweep": cur,
            },
            "e2e": {"value": n * ws / (ms_e2e_step * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "steps": Ke2, "ms_per_step": ms_e2e_step,
                    "api": {"copy": "BatchedDroneEnv.step_host(mode='copy'): one step at a time, the host waits for each",
                            "zero_copy": "BatchedDroneEnv.step_host(mode='zero_copy'): the kernel writes straight into pinned host memory",
                            "copy_2_in_flight": "BatchedDroneEnv.step_host(mode='copy', wait=False) on two streams over independent shards: "
                                                "two steps in flight, the host waits for every step's event"}[best_mode]
                           + " (pinned host actions in; obs, reward, flags out in pinned host memory, every step)",
                    "modes_ms_per_step": e2e_modes,
                    "pcie_gbs": (h2d + d2h) / (ms_e2e_step * 1e-3) / 1e9,
                    "pcie_ceiling_gbs": ceil_gbs, "frac_of_pcie_ceiling": (d2h / (ms_e2e_step * 1e-3) / 1e9) / ceil_gbs,
                    "pcie_ceiling_what": f"cudaMemcpyAsync device->pinned host of the same {blk_d.numel()} B block, {ws} rank(s) concurrently, max over ranks",
                    "bound": "PCIe: 65 B per env-step device->host (obs 60 + reward 4 + flags 1)",
                    "rank0_cpu_affinity": None if cpus is None else f"{len(cpus)} CPUs local to the GPU (NVML)"},
            "gpu_launches": launches,
            "clocks": sampler.summary(),
            "episode_stats": stats,
        }
        if mgc is not None:
            line["multi_gpu_check"] = mgc
        if dumped is not None:
            line["dumped_outputs"] = dumped
        if ws == 1 and not args.no_socket:
            try:
                line["socket_shim"] = socket_shim_rate(dev)
            except Exception as exc:                       # context only: never fail the bench line over it
                line["socket_shim"] = {"error": repr(exc)}
        if ws == 1 and not args.no_cpu_baseline:
            ticks = args.cpu_ticks
            agg, per_proc, procs, secs = cpu_port_multiprocess(ticks, 200)
            c_rate, c_thr = c_oracle_threads(1 << 16, 250)
            line["cpu_baseline"] = {
                "value": agg, "unit": UNIT, "cores": procs, "kind": "port",
                "sample": f"{procs} processes x 6 PortDroneGame x {ticks} ticks (random actions, 250-step cap), {secs:.1f} s",
                "per_process": per_proc,
                "c_oracle": {"value": c_rate, "threads": c_thr, "sample": "65,536 envs x 250 steps, float64 C restatement"},
            }
        print(json.dumps(line), flush=True)
    if ws > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def multi_gpu_check(dd, dist, cenv, cap, rank, ws, NC, dev):
    """On-hardware check of the two collectives (every rank computes it; returns the same dict everywhere).
    (1) episode statistics: every rank plays one curriculum stage on its own env ids AND on its right neighbour's
        (env_id_base = ((rank + 1) % ws) * NC -- trajectories are keyed by the global env id, so another GPU must get the
        same 8 words); the per-rank words are all-gathered and the all-reduced block must equal their sum, and each
        rank's neighbour recomputation must equal what the neighbour itself reported.
    (2) advantage moments: normalize_advantages(reduce=True) on per-rank buffers must equal normalising the
        concatenation of all ranks' buffers on one GPU."""
    import torch

    def fresh_stage(base):
        """One curriculum stage on a FRESH env (episode counters at 0, so the Philox spawn of env id g is the same
        whichever GPU plays it): returns (stats dict, the 8 device words)."""
        e = dd.BatchedDroneEnv(NC, device=dev, seed=0, randomize_drone=True, randomize_platform=True,
                               auto_reset=False, dtype=torch.float32, env_id_base=base)
        st = dd.collect_episodes(e, cap, policy="bangbang", reduce=False)
        return st, e.stats_tensor().clone()
    own, w_own = fresh_stage(rank * NC)
    w_red = dd.allreduce_stats(w_own.clone())
    gathered = [torch.zeros_like(w_own) for _ in range(ws)]
    dist.all_gather(gathered, w_own)
    G = torch.stack(gathered)
    nb = (rank + 1) % ws
    _, w_nb = fresh_stage(nb * NC)
    ok_sum = bool(torch.equal(G.sum(0), w_red))
    ok_nb = bool(torch.equal(w_nb, G[nb]))
    # moments: a deterministic per-rank buffer (the shaped rewards of a short rollout would do; a hash is enough here)
    m = 1 << 18
    idx = torch.arange(m, device=dev, dtype=torch.float32)
    x = torch.sin(idx * 0.37 + rank) * (3.0 + rank) + 0.1 * rank
    y_red = dd.normalize_advantages(x, reduce=True)
    xs = [torch.zeros_like(x) for _ in range(ws)]
    dist.all_gather(xs, x)
    y_all = dd.normalize_advantages(torch.cat(xs), reduce=False)
    err = float((y_all[rank * m:(rank + 1) * m] - y_red).abs().max())
    flags = torch.tensor([int(ok_sum), int(ok_nb), int(err < 1e-6)], device=dev, dtype=torch.int32)
    dist.all_reduce(flags, op=dist.ReduceOp.MIN)
    errt = torch.tensor([err], device=dev, dtype=torch.float64)
    dist.all_reduce(errt, op=dist.ReduceOp.MAX)
    ok = bool(flags.min().item() == 1)
    return {"status": "ok" if ok else "FAILED", "stats_allreduce_equals_sum_of_gathered": bool(flags[0].item()),
            "neighbour_shard_recomputed_on_another_gpu_matches": bool(flags[1].item()),
            "normalize_reduce_vs_single_buffer_max_abs_err": float(errt.item()),
            "stage_max_steps": int(cap), "envs_per_rank": NC, "episodes_all_ranks": int(w_red[0].item()),
            "landed_all_ranks": int(w_red[1].item()), "own_success_rate_rank0": own["success_rate"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=int(os.environ.get("WORLD_SIZE", "1")))
    ap.add_argument("--steps", type=int, default=12000, help="timed steps (of the gym step, the step-only and the float64 variants)")
    ap.add_argument("--warmup", type=int, default=600)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--envs", type=int, default=ENVS_PER_GPU, help="envs per shard (= per step launch)")
    ap.add_argument("--shards", type=int, default=6, help="independent shards per GPU that steps rotate over")
    ap.add_argument("--chains", type=int, default=2, help="parallel launch chains in the CUDA graph (shard s -> chain s %% chains)")
    ap.add_argument("--e2e-steps", type=int, default=100)
    ap.add_argument("--trace-len", type=int, default=16, help="rows of the device action trace per shard (schedule period = shards x this)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/*.npy")
    ap.add_argument("--eager", action="store_true", help="no CUDA graphs: one Python -> C-ABI launch per step (A/B)")
    ap.add_argument("--no-f64", action="store_true", help="skip the float64 (exact-parity) instantiation variant")
    ap.add_argument("--cpu-ticks", type=int, default=250000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-numa-bind", action="store_true", help="do not pin each rank to its GPU's local CPUs (N > 1)")
    ap.add_argument("--no-socket", action="store_true", help="skip the socket-shim context measurement")
    ap.add_argument("--no-policy", action="store_true", help="skip the fused policy rollout variant (K5)")
    ap.add_argument("--no-curriculum", action="store_true", help="skip the curriculum sweep variant (cfg 5)")
    ap.add_argument("--curriculum-envs", type=int, default=1 << 21, help="envs per GPU in the curriculum sweep")
    ap.add_argument("--policy-envs", type=int, default=65536, help="envs per GPU for the K5 variant (BASELINE configs[3])")
    ap.add_argument("--launch-flags", type=lambda v: int(v, 0), default=0x01,
                    help="DD_LAUNCH_* bits (include/drone_b200.h): 0x01 PDL, 0x10 CTA 128, 0x20 CTA 512")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())

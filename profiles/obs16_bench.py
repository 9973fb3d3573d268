"""Throughput of the env kernels with 16-bit observation outputs (BatchedDroneEnv(obs_dtype=...)) against float32 ones.

  * the product path, timed like bench.py's gym step: ShardedDroneEnv.run with 6 shards x 1,048,576 envs, 2 chains, a
    random trace; exactly K timed steps behind an untimed lead-in, CUDA events on the chain streams, the longest chain
    span reported; K = 20 and K = 1,000; the formats alternate over --rounds rounds;
  * step_host (host in / host out) in 'copy' and 'zero_copy' modes, with the PCIe bytes per env-step;
  * dd_rollout with T = 50 and obs_tn written.

Usage: python profiles/obs16_bench.py [--out FILE]   (needs a CUDA device; prints one JSON document)
"""
import argparse
import importlib
import json
import math
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
dd = importlib.import_module("reinforcement-learning-101_b200")

PEAK_GBS = 6543.0          # measured HBM bandwidth of one B200 (DESIGN.md section 7)
FMTS = {"float32": torch.float32, "float16": torch.float16, "bfloat16": torch.bfloat16}
# algorithmic HBM bytes per env-step of the gym step (DESIGN.md section 3): step-only 86 B + the observation row,
# 15 x 4 B (float32) or 15 x 2 B (16-bit)
BYTES_GYM = {"float32": 146, "float16": 116, "bfloat16": 116}
MAX_STEPS, LEAD_IN = 250, 32


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        name, pl, clk = [s.strip() for s in out.split(",")]
        return {"gpu": name, "power_limit": pl, "max_sm_clock": clk}
    except Exception as e:                                   # the numbers stay valid; the card is then unnamed
        return {"gpu": torch.cuda.get_device_name(0), "query_error": str(e)}


def sharded_ms(env, K, W):
    """bench.py's time_steps for one rank: milliseconds of K gym steps."""
    period = env.S * env.L

    def blocks(r):
        for _ in range(r):
            env.run(K)
        env.join()
    blocks(-(-W // K))
    blocks(period // math.gcd(K, period))

    def measure():
        env.run(K * -(-max(LEAD_IN, env.C) // K))
        g0 = env.graphs_cached
        t0, t1 = ([torch.cuda.Event(enable_timing=True) for _ in env._chains] for _ in range(2))
        for ev, ch in zip(t0, env._chains):
            ev.record(ch)
        env.run(K)
        for ev, ch in zip(t1, env._chains):
            ev.record(ch)
        env.join()
        torch.cuda.synchronize()
        return max(a.elapsed_time(b) for a, b in zip(t0, t1)), env.graphs_cached != g0
    ms, captured = measure()
    if captured:
        ms, _ = measure()
    return ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--envs", type=int, default=1 << 20)
    ap.add_argument("--shards", type=int, default=6)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=200)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("obs16_bench.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    n, S = args.envs, args.shards
    res = {"device": gpu_info(), "envs_per_shard": n, "shards": S, "chains": 2, "peak_gbs": PEAK_GBS, "sharded": {}, "step_host": {},
           "rollout": {}}

    # ---- product path ----
    envs = {f: dd.ShardedDroneEnv(S, n, device=dev, chains=2, trace_len=16, seed=0, randomize_drone=True,
                                  randomize_platform=True, max_steps=MAX_STEPS, auto_reset=True, obs_dtype=dt)
            for f, dt in FMTS.items()}
    for e in envs.values():
        e.reset(); e.random_trace()
    for K in (20, 1000):
        runs = {f: [] for f in FMTS}
        for _ in range(args.rounds):
            for f, e in envs.items():
                runs[f].append(sharded_ms(e, K, args.warmup))
        for f, ms in runs.items():
            best = min(ms)
            rate = n * K / (best * 1e-3)
            res["sharded"][f"{f}_K{K}"] = {
                "obs_dtype": f, "K": K, "ms_runs": ms, "env_steps_per_s": rate, "us_per_1M_env_step": best * 1e3 / K * (1 << 20) / n,
                "bytes_per_env_step": BYTES_GYM[f], "achieved_gbs": rate * BYTES_GYM[f] / 1e9,
                "frac_of_peak": rate * BYTES_GYM[f] / 1e9 / PEAK_GBS,
                "frac_of_peak_at_146B": rate * 146 / 1e9 / PEAK_GBS}
    # the float32 and 16-bit envs ran the same launches (unless a timed block had to be repeated): then their
    # observations agree after the conversion
    res["outputs_checked"] = len({e.t for e in envs.values()}) == 1
    for f in ("float16", "bfloat16") if res["outputs_checked"] else ():
        for s in range(S):
            a, b = envs["float32"].shards[s], envs[f].shards[s]
            assert torch.equal(a.obs.to(FMTS[f]).view(torch.int16), b.obs.view(torch.int16)), (f, s)
            assert torch.equal(a.pos_vel, b.pos_vel) and torch.equal(a.steps, b.steps)
    del envs
    torch.cuda.empty_cache()

    # ---- step_host ----
    steps = 100
    for f, dt in FMTS.items():
        e = dd.BatchedDroneEnv(n, device=dev, seed=0, randomize_drone=True, max_steps=MAX_STEPS, obs_dtype=dt)
        e.reset()
        io = e.make_host_io()
        io["actions"].copy_(e.random_actions(1)[0].cpu())
        osz = torch.empty((), dtype=dt).element_size()
        for mode in ("copy", "zero_copy"):
            for _ in range(10):
                e.step_host(io, mode=mode)
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record()
            for _ in range(steps):
                e.step_host(io, mode=mode)
            t1.record(); torch.cuda.synchronize()
            ms = t0.elapsed_time(t1) / steps
            d2h = 15 * osz + 4 + 1
            res["step_host"][f"{f}_{mode}"] = {"obs_dtype": f, "mode": mode, "ms_per_step": ms, "env_steps_per_s": n / (ms * 1e-3),
                                               "pcie_h2d_bytes_per_env_step": 1, "pcie_d2h_bytes_per_env_step": d2h,
                                               "pcie_gbs": n * (1 + d2h) / (ms * 1e-3) / 1e9}
        del e, io
    torch.cuda.empty_cache()

    # ---- dd_rollout, T = 50, obs_tn written ----
    T = 50
    for f, dt in FMTS.items():
        e = dd.BatchedDroneEnv(n, device=dev, seed=0, randomize_drone=True, max_steps=MAX_STEPS, obs_dtype=dt)
        e.reset(want_obs=False)
        buf = torch.empty(T, n, 15, device=dev, dtype=dt)
        for _ in range(3):
            e.rollout(T, "random", obs_out=buf)
        ms = []
        for _ in range(5):
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record(); e.rollout(T, "random", obs_out=buf); t1.record(); torch.cuda.synchronize()
            ms.append(t0.elapsed_time(t1))
        best = min(ms)
        res["rollout"][f] = {"obs_dtype": f, "T": T, "ms_runs": ms, "env_steps_per_s": n * T / (best * 1e-3),
                             "obs_bytes_per_env_step": 15 * buf.element_size()}
        del e, buf
    txt = json.dumps(res, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(txt + "\n")


if __name__ == "__main__":
    main()

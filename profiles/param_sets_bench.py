"""Throughput of the per-env parameter-set kernels (BatchedDroneEnv(param_sets=...), DESIGN.md section 4e).

  * the product path, timed like bench.py's gym step: ShardedDroneEnv.run with 6 shards x 1,048,576 envs, 2 chains, a
    random trace; exactly K timed steps behind an untimed lead-in, CUDA events on the chain streams, the longest chain
    span reported; K = 20 and K = 1,000; the variants alternate over --rounds rounds.  Variants: the default kernel
    (immediates), the generic uniform kernel (defaults with one count moved by 1e-7: constants from the argument block),
    per-env sets with 1 / 4 / 16 / 64 randomly assigned sets and 16 sets in contiguous 256-env blocks, 16 sets with
    resampling, float64 default and float64 with 16 sets, and step-only (no observation) default and 16 sets;
  * dd_rollout with T = 50 and random actions, default against 16 sets.

Usage: python profiles/param_sets_bench.py [--out FILE]   (needs a CUDA device; prints one JSON document)
"""
import argparse
import importlib
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))
dd = importlib.import_module("reinforcement-learning-101_b200")
nv = dd.native
from obs16_bench import PEAK_GBS, gpu_info, sharded_ms     # noqa: E402  (same timing as the obs16 record)

# algorithmic HBM bytes per env-step (DESIGN.md section 3): gym step 146 B, step-only 86 B; + 1 B index per env-step
BYTES = {True: 146, False: 86}
MAX_STEPS = 250


def _sets(count):
    """``count`` sets around config.py's defaults: gravity, thrust, drag, tank, landing tolerance, platform and spawn
    ranges moved per set (domain randomisation)."""
    out = []
    for j in range(count):
        p = nv.default_params()
        f = j / max(count - 1, 1)
        p.gravity = 0.25 + 0.1 * f; p.main_thrust = 0.55 + 0.1 * f; p.drag = 0.985 + 0.01 * f
        p.max_fuel = 800.0 + 400.0 * f; p.land_speed = 2.5 + 1.0 * f; p.platform_w = 80.0 + 40.0 * f
        p.spawn_y_min = 50.0 + 40.0 * f
        out.append(p)
    return out


def _generic_defaults():
    p = nv.default_params()
    p.spawn_x_count = 601.0000001                        # (uint32) 601 as before, but not the default bytes
    return p


def variants(n, S):
    def idx_random(count, seed=0):
        g = torch.Generator().manual_seed(seed)
        return torch.randint(0, count, (S, n), generator=g, dtype=torch.int32).to(torch.uint8)

    def idx_blocks(count, block=256):
        i = (torch.arange(S * n) // block) % count
        return i.to(torch.uint8).view(S, n)
    return {
        "default": dict(),
        "generic_uniform": dict(params=_generic_defaults()),
        "sets1": dict(sets=_sets(1), index=idx_random(1)),
        "sets4": dict(sets=_sets(4), index=idx_random(4)),
        "sets16": dict(sets=_sets(16), index=idx_random(16)),
        "sets64": dict(sets=_sets(64), index=idx_random(64)),
        "sets16_blocks256": dict(sets=_sets(16), index=idx_blocks(16)),
        "sets16_resample": dict(sets=_sets(16), index=idx_random(16), resample=True),
        "f64_default": dict(dtype=torch.float64),
        "f64_sets16": dict(dtype=torch.float64, sets=_sets(16), index=idx_random(16)),
        "steponly_default": dict(obs=False),
        "steponly_sets16": dict(obs=False, sets=_sets(16), index=idx_random(16)),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--envs", type=int, default=1 << 20)
    ap.add_argument("--shards", type=int, default=6)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=200)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("param_sets_bench.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    n, S = args.envs, args.shards
    res = {"device": gpu_info(), "envs_per_shard": n, "shards": S, "chains": 2, "peak_gbs": PEAK_GBS, "sharded": {},
           "rollout": {}}

    V = variants(n, S)
    envs, want_obs = {}, {}
    for name, v in V.items():
        e = dd.ShardedDroneEnv(S, n, device=dev, chains=2, trace_len=16, seed=0, randomize_drone=True,
                               randomize_platform=True, max_steps=MAX_STEPS, auto_reset=True,
                               dtype=v.get("dtype", torch.float32), params=v.get("params"))
        if "sets" in v:
            e.set_param_sets(v["sets"], v["index"].to(dev), v.get("resample", False))
        e.reset(); e.random_trace()
        envs[name], want_obs[name] = e, v.get("obs", True)
    for K in (20, 1000):
        runs = {k: [] for k in envs}
        for _ in range(args.rounds):
            for k, e in envs.items():
                if want_obs[k]:
                    runs[k].append(sharded_ms(e, K, args.warmup))
                else:                                          # the same timing with run(want_obs=False)
                    run = e.run
                    e.run = lambda k_, run=run: run(k_, want_obs=False)
                    try:
                        runs[k].append(sharded_ms(e, K, args.warmup))
                    finally:
                        del e.run
        base = {True: min(runs["default"]), False: min(runs["steponly_default"])}
        for k, ms in runs.items():
            best = min(ms)
            rate = n * K / (best * 1e-3)                       # a timed block is K launches of one n-env shard each
            sets = "sets" in V[k]
            b_alg = BYTES[want_obs[k]] + (1 if sets else 0)
            res["sharded"][f"{k}_K{K}"] = {
                "variant": k, "K": K, "ms_runs": ms, "env_steps_per_s": rate,
                "rate_vs_default": base[want_obs[k]] / best if V[k].get("dtype") != torch.float64 else None,
                "bytes_per_env_step_f32_layout": b_alg,
                "frac_of_peak_at_f32_bytes": rate * b_alg / 1e9 / PEAK_GBS}
        res["sharded"][f"f64_sets16_K{K}"]["rate_vs_f64_default"] = min(runs["f64_default"]) / min(runs["f64_sets16"])
    del envs
    torch.cuda.empty_cache()

    # ---- dd_rollout, T = 50, random actions, statistics only ----
    T = 50
    for name, sets in (("default", None), ("sets16", _sets(16))):
        e = dd.BatchedDroneEnv(n, device=dev, seed=0, randomize_drone=True, max_steps=MAX_STEPS)
        if sets is not None:
            e.set_param_sets(sets, torch.randint(0, 16, (n,), dtype=torch.int32).to(torch.uint8))
        e.reset(want_obs=False)
        for _ in range(3):
            e.rollout(T, "random")
        ms = []
        for _ in range(5):
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record(); e.rollout(T, "random"); t1.record(); torch.cuda.synchronize()
            ms.append(t0.elapsed_time(t1))
        res["rollout"][name] = {"T": T, "ms_runs": ms, "env_steps_per_s": n * T / (min(ms) * 1e-3)}
        del e
    res["rollout"]["sets16"]["rate_vs_default"] = min(res["rollout"]["default"]["ms_runs"]) / min(res["rollout"]["sets16"]["ms_runs"])
    txt = json.dumps(res, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(txt + "\n")


if __name__ == "__main__":
    main()

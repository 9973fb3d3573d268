"""Cost of episode statistics per parameter set (DD_PARAM_SETS_STATS_BY_SET, DESIGN.md section 4e): each row times one
workload with 16 randomly assigned sets twice, with the plain totals block and with per-set blocks, the two alternating
over --rounds rounds in the same process; the best round of each counts.

  * K1 on the product path, timed like bench.py's gym step (profiles/obs16_bench.py sharded_ms): ShardedDroneEnv.run
    with 6 shards x 1,048,576 envs, 2 chains, a random trace, K = 1,000 steps; without and with resampling;
  * dd_rollout, T = 50, random actions, statistics only; without and with resampling;
  * K5 on cfg 4 (65,536 envs x 250 steps, FAST, want="arldo", tests/golden/policy_v1.npz); without and with resampling.

Usage: python profiles/stats_by_set_bench.py [--out FILE]   (needs a CUDA device; prints one JSON document)
"""
import argparse
import importlib
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))
dd = importlib.import_module("reinforcement-learning-101_b200")
nv = dd.native
from obs16_bench import gpu_info, sharded_ms             # noqa: E402
from param_sets_bench import _sets                       # noqa: E402  (the sets of the parameter-set record)

COUNT, MAX_STEPS = 16, 250


def _index(n, seed=0):
    g = torch.Generator().manual_seed(seed)
    return torch.randint(0, COUNT, (n,), generator=g, dtype=torch.int32).to(torch.uint8)


def _timed(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def _row(ms, steps_per_call):
    best = {k: min(v) for k, v in ms.items()}
    return {"ms_runs": ms, "ms_best": best, "env_steps_per_s": {k: steps_per_call / (b * 1e-3) for k, b in best.items()},
            "by_set_rate_vs_plain": best["plain"] / best["by_set"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--envs", type=int, default=1 << 20)
    ap.add_argument("--shards", type=int, default=6)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=200)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("stats_by_set_bench.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    res = {"device": gpu_info(), "sets": COUNT, "rounds": args.rounds, "rows": {}}
    n, S = args.envs, args.shards

    # ---- K1 on the product path ----
    K = 1000
    for resample in (False, True):
        envs = {}
        for mode in ("plain", "by_set"):
            e = dd.ShardedDroneEnv(S, n, device=dev, chains=2, trace_len=16, seed=0, randomize_drone=True,
                                   randomize_platform=True, max_steps=MAX_STEPS, auto_reset=True)
            e.set_param_sets(_sets(COUNT), _index(S * n).view(S, n).to(dev), resample, stats_by_set=mode == "by_set")
            e.reset(); e.random_trace()
            envs[mode] = e
        ms = {k: [] for k in envs}
        for _ in range(args.rounds):
            for k, e in envs.items():
                ms[k].append(sharded_ms(e, K, args.warmup))
        row = _row(ms, n * K)                              # a timed block: K launches of one n-env shard each
        row["totals_equal"] = bool(torch.equal(envs["plain"].stats_tensor(), envs["by_set"].stats_tensor()))
        res["rows"][f"k1_sharded_{S}x{n}_K{K}" + ("_resample" if resample else "")] = row
        del envs
        torch.cuda.empty_cache()

    # ---- dd_rollout, T = 50 ----
    T = 50
    for resample in (False, True):
        envs = {}
        for mode in ("plain", "by_set"):
            e = dd.BatchedDroneEnv(n, device=dev, seed=0, randomize_drone=True, max_steps=MAX_STEPS)
            e.set_param_sets(_sets(COUNT), _index(n), resample, stats_by_set=mode == "by_set")
            e.reset(want_obs=False)
            for _ in range(3):
                e.rollout(T, "random")
            envs[mode] = e
        ms = {k: [] for k in envs}
        for _ in range(args.rounds):
            for k, e in envs.items():
                ms[k].append(_timed(lambda e=e: e.rollout(T, "random"), 5))
        res["rows"][f"rollout_{n}_T{T}" + ("_resample" if resample else "")] = _row(ms, n * T)
        del envs
        torch.cuda.empty_cache()

    # ---- K5, cfg 4 ----
    n5, T5 = 65536, 250
    d = np.load(os.path.join(ROOT, "tests", "golden", "policy_v1.npz"))
    blob = dd.PolicyBlob({k: torch.from_numpy(d[k]) for k in d.files if k.startswith("network")}, device=dev)
    res["k5_operands"] = blob.operand_dtype
    for resample in (False, True):
        envs, bufs = {}, {}
        for mode in ("plain", "by_set"):
            e = dd.BatchedDroneEnv(n5, device=dev, seed=0, randomize_drone=True, randomize_platform=True,
                                   max_steps=MAX_STEPS, auto_reset=True)
            e.set_param_sets(_sets(COUNT), _index(n5), resample, stats_by_set=mode == "by_set")
            e.reset(want_obs=False)
            bufs[mode] = dd.policy_rollout(e, blob, T5, want="arldo")
            envs[mode] = e
        for k in envs:
            for _ in range(5):
                dd.policy_rollout(envs[k], blob, T5, want="arldo", out=bufs[k])
        ms = {k: [] for k in envs}
        for _ in range(args.rounds):
            for k, e in envs.items():
                ms[k].append(_timed(lambda e=e, k=k: dd.policy_rollout(e, blob, T5, want="arldo", out=bufs[k]), 20))
        res["rows"][f"k5_cfg4_{n5}x{T5}" + ("_resample" if resample else "")] = _row(ms, n5 * T5)
        del envs, bufs
        torch.cuda.empty_cache()

    txt = json.dumps(res, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(txt + "\n")


if __name__ == "__main__":
    main()

"""Throughput of the fused policy rollout (K5) under per-env parameter sets (dd_policy_rollout_sets, DESIGN.md sections 4b
and 4e) against the single-set kernels.

cfg 4 (BASELINE configs[3]): 65,536 envs x 250 steps of the PPO collection call -- the FAST instantiation,
want="arldo", Bernoulli sampling, the fp16 operands dd_policy_pack picks for tests/golden/policy_v1.npz -- and 75,776
envs (592 tiles: four tiles on each of the 148 SMs).  Each timing is CUDA events around --reps back-to-back launches
after --warmup untimed ones; the variants alternate over --rounds rounds and the best round counts.  Variants: the default
kernel (config.py's parameters as immediates), the generic kernel (one non-default DDParams: constants from the argument
block), per-env sets with 1 / 4 / 16 / 64 randomly assigned sets, 16 sets with resampling at every auto-reset, and
threshold actions (want="ard") with the generic kernel and with 16 sets.

Usage: python profiles/policy_sets_bench.py [--out FILE]   (needs a CUDA device; prints one JSON document)
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
from obs16_bench import gpu_info                           # noqa: E402
from param_sets_bench import _generic_defaults, _sets      # noqa: E402  (the same sets as the env-kernel record)

T = 250


def variants(n):
    def idx(count, seed=0):
        g = torch.Generator().manual_seed(seed)
        return torch.randint(0, count, (n,), generator=g, dtype=torch.int32).to(torch.uint8)
    return {
        "default": dict(),
        "generic": dict(params=_generic_defaults()),
        "sets1": dict(sets=_sets(1), index=idx(1)),
        "sets4": dict(sets=_sets(4), index=idx(4)),
        "sets16": dict(sets=_sets(16), index=idx(16)),
        "sets64": dict(sets=_sets(64), index=idx(64)),
        "sets16_resample": dict(sets=_sets(16), index=idx(16), resample=True),
        "threshold_generic": dict(params=_generic_defaults(), threshold=True),
        "threshold_sets16": dict(sets=_sets(16), index=idx(16), threshold=True),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--sizes", default="65536,75776")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("policy_sets_bench.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    d = np.load(os.path.join(ROOT, "tests", "golden", "policy_v1.npz"))
    blob = dd.PolicyBlob({k: torch.from_numpy(d[k]) for k in d.files if k.startswith("network")}, device=dev)
    res = {"device": gpu_info(), "T": T, "operands": blob.operand_dtype, "reps": args.reps, "rounds": args.rounds, "sizes": {}}
    for n in (int(s) for s in args.sizes.split(",")):
        V = variants(n)
        envs, bufs = {}, {}
        for name, v in V.items():
            e = dd.BatchedDroneEnv(n, device=dev, seed=0, randomize_drone=True, randomize_platform=True, max_steps=250,
                                   auto_reset=True, dtype=torch.float32, params=v.get("params"))
            if "sets" in v:
                e.set_param_sets(v["sets"], v["index"].to(dev), v.get("resample", False))
            e.reset(want_obs=False)
            want = "ard" if v.get("threshold") else "arldo"
            bufs[name] = dd.policy_rollout(e, blob, T, sample=not v.get("threshold"), want=want)
            envs[name] = e
        run = lambda k: dd.policy_rollout(envs[k], blob, T, sample=not V[k].get("threshold"),
                                          want="ard" if V[k].get("threshold") else "arldo", out=bufs[k])
        for k in envs:
            for _ in range(args.warmup):
                run(k)
        torch.cuda.synchronize()
        ms = {k: [] for k in envs}
        for _ in range(args.rounds):
            for k in envs:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(args.reps):
                    run(k)
                e1.record()
                torch.cuda.synchronize()
                ms[k].append(e0.elapsed_time(e1) / args.reps)
        best = {k: min(v) for k, v in ms.items()}
        out = {}
        for k in envs:
            ref = "threshold_generic" if V[k].get("threshold") else "generic"
            out[k] = {"ms_per_launch_runs": ms[k], "ms_per_launch": best[k], "env_steps_per_s": n * T / (best[k] * 1e-3),
                      "rate_vs_generic": best[ref] / best[k], "rate_vs_default": best["default"] / best[k],
                      "episodes": envs[k].stats()["episodes"]}
        res["sizes"][str(n)] = out
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

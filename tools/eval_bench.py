#!/usr/bin/env python
"""Throughput of policy evaluation (ses_evaluate) on the GPU, with the training K1 on the same policy beside it.

  cartpole_mlp  the converged CartPole mu of tests/golden/bench_state_gen30.npz, M = 2^16 and 2^20 episodes
  train_k1      ses_rollout of that mu's population (sigma of the same state, E = 5, P * E ~ 2^16 episodes): the training figure
  mountaincar_gru  a random GRU policy (every episode runs the 200-step TimeLimit), M = 2^16

CUDA events around `--reps` calls (default 100: a window of 0.1 s or more) after `--warmup` calls of the same shape; the
working set (weights and a few MB of results) stays in L2, as it does in use.  Prints one JSON line with the card's name and
power limit read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from simple_es_b200.engine import RolloutEngine  # noqa: E402


def timed(fn, warmup, reps):
    for _ in range(warmup):
        out = fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        out = fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / 1e3 / reps, out


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
    name, _, limit = q.partition(",")
    return name.strip() or torch.cuda.get_device_name(0), limit.strip()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--reps", type=int, default=100)
    args = ap.parse_args()
    st = np.load(os.path.join(ROOT, "tests", "golden", "bench_state_gen30.npz"))
    mu = torch.from_numpy(st["mu"]).cuda()
    name, limit = card()
    res = {"card": name, "power_limit": limit, "warmup": args.warmup, "reps": args.reps, "runs": []}

    eng = RolloutEngine("CartPole-v1", 4, 2, False, False, 500, 5, 2, 2, 1, 1, seed=0)
    for M in (1 << 16, 1 << 20):
        t, (ret, lng) = timed(lambda: eng.evaluate(mu, M, round=0), args.warmup, args.reps)
        steps = int(lng.sum())
        res["runs"].append({"name": "cartpole_mlp_eval", "episodes": M, "seconds": t, "episodes_per_s": M / t,
                            "env_steps_per_s": steps / t, "mean_return": float(ret.mean()), "mean_length": steps / M})

    P, E = 13108, 5                                              # P * E = 65540 episodes, the openai_es layout
    tr = RolloutEngine("CartPole-v1", 4, 2, False, False, 500, E, P, P, 1, 1, seed=0)
    fit = torch.zeros(P, dtype=torch.float64, device="cuda")
    steps_t = torch.zeros(P, dtype=torch.int64, device="cuda")
    sigma = float(st["sigma"])
    t, _ = timed(lambda: tr.rollout(int(st["generation"]), sigma, mu[None], fitness=fit, steps=steps_t), args.warmup, args.reps)
    steps = int(steps_t.sum())
    res["runs"].append({"name": "cartpole_mlp_train_k1", "episodes": P * E, "sigma": sigma, "seconds": t,
                        "episodes_per_s": P * E / t, "env_steps_per_s": steps / t, "mean_length": steps / (P * E)})

    g = RolloutEngine("MountainCar-v0", 2, 3, True, False, 200, 5, 2, 2, 1, 1, seed=0)
    w = torch.from_numpy(np.random.default_rng(0).normal(0, 0.5, g.D).astype(np.float32)).cuda()
    M = 1 << 16
    t, (ret, lng) = timed(lambda: g.evaluate(w, M, round=0), args.warmup, args.reps)
    steps = int(lng.sum())
    res["runs"].append({"name": "mountaincar_gru_eval", "episodes": M, "seconds": t, "episodes_per_s": M / t,
                        "env_steps_per_s": steps / t, "mean_return": float(ret.mean()), "mean_length": steps / M})
    print(json.dumps(res))


if __name__ == "__main__":
    main()

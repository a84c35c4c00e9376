#!/usr/bin/env python
"""Throughput of policy evaluation (ses_evaluate) on the GPU, with the training K1 on the same policy beside it.

  cartpole_mlp  the converged CartPole mu of tests/golden/bench_state_gen30.npz, M = 2^16 and 2^20 episodes
  train_k1      ses_rollout of that mu's population (sigma of the same state, E = 5, P * E ~ 2^16 episodes): the training figure
  mountaincar_gru  a random GRU policy (every episode runs the 200-step TimeLimit), M = 2^16

CUDA events around `--reps` calls (default 100: a window of 0.1 s or more) after `--warmup` calls of the same shape; the
working set (weights and a few MB of results) stays in L2, as it does in use.  Prints one JSON line with the card's name and
power limit read in the same run.

--record K instead times recording (ses_record, RolloutEngine.record: every step's state, action and return) against plain
evaluation of the same K episodes, for the converged CartPole mu and the random MountainCar GRU policy.  A record call
includes what a user pays for it: allocating and NaN-filling its output tensors; `record_kernel_seconds` is ses_record alone
into buffers allocated once.  `bytes_per_step` is what the kernel writes per env step (state, actions, return);
`kernel_written_GB_per_s` is those bytes over the kernel-only time.
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
from simple_es_b200.engine import RolloutEngine, _ptr  # noqa: E402


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


def record_vs_evaluate(res, name, eng, w, K, warmup, reps):
    t_eval, (ret, lng) = timed(lambda: eng.evaluate(w, K, round=0), warmup, reps)
    t_rec, rec = timed(lambda: eng.record(w, K, round=0), warmup, reps)
    assert torch.equal(rec[4], lng)                              # the same episodes
    bufs = [_ptr(t) for t in rec]
    t_kern, _ = timed(lambda: eng._check(eng.lib.ses_record(eng._h, 0, _ptr(w), 1, K, None, *bufs, eng._stream())), warmup, reps)
    steps = int(lng.sum())
    per_step = 8 * eng.state_dim + 4 * eng.n_agents + 8
    res["runs"].append({"name": name, "episodes": K, "env_steps": steps, "mean_length": steps / K,
                        "evaluate_seconds": t_eval, "record_seconds": t_rec, "record_kernel_seconds": t_kern,
                        "record_over_evaluate": t_rec / t_eval, "record_kernel_over_evaluate": t_kern / t_eval,
                        "evaluate_env_steps_per_s": steps / t_eval, "record_env_steps_per_s": steps / t_rec,
                        "bytes_per_step": per_step, "kernel_written_GB_per_s": steps * per_step / t_kern / 1e9,
                        "allocated_GB": sum(t.numel() * t.element_size() for t in rec) / 1e9})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--reps", type=int, default=100)
    ap.add_argument("--record", type=int, default=0, metavar="K", help="time recording against evaluation of K episodes")
    args = ap.parse_args()
    st = np.load(os.path.join(ROOT, "tests", "golden", "bench_state_gen30.npz"))
    mu = torch.from_numpy(st["mu"]).cuda()
    name, limit = card()
    res = {"card": name, "power_limit": limit, "warmup": args.warmup, "reps": args.reps, "runs": []}
    if args.record:
        eng = RolloutEngine("CartPole-v1", 4, 2, False, False, 500, 5, 2, 2, 1, 1, seed=0)
        record_vs_evaluate(res, "cartpole_mlp", eng, mu, args.record, args.warmup, args.reps)
        g = RolloutEngine("MountainCar-v0", 2, 3, True, False, 200, 5, 2, 2, 1, 1, seed=0)
        w = torch.from_numpy(np.random.default_rng(0).normal(0, 0.5, g.D).astype(np.float32)).cuda()
        record_vs_evaluate(res, "mountaincar_gru", g, w, args.record, args.warmup, args.reps)
        print(json.dumps(res))
        return

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

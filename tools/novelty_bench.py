#!/usr/bin/env python
"""Cost of novelty search with reward (nsr_es) on the GPU.  Prints JSON lines, each with the card's name and power limit read
in the same run; --out DIR also writes them to DIR/novelty_bench.jsonl.

  novelty     ses_novelty alone at P in {16384, 65536} x A in {1e2, 1e3, 1e4}, k = 10, state_dim 2 (MountainCar) and 4
              (CartPole), on random behaviours; `fp64_gflops` counts P * A * state_dim * 3 operations (difference, square,
              add) over the kernel time -- the algorithmic work, not the instructions issued.
  k1          ses_rollout with and without the final-state output: the converged CartPole population of
              tests/golden/bench_state_gen30.npz (P = 65536) and a MountainCar generation-0 population (P = 16384).
  generation  one nsr_es generation (k = 10, w = 0.5) against one openai_es generation on the same two workloads, each from
              the same state, timed with CUDA events around step(); the archive holds `archive` rows before the timed steps.
  learning    (--learning G) conf/mountaincar_nsr.yaml against the same hyper-parameters with openai_es, for 3 seeds: best
              fitness and the mean return of mu over 100 evaluation episodes every 10 generations.

Kernel and step times are means over --reps calls after --warmup calls of the same shape.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch
import yaml

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from simple_es_b200.engine import RolloutEngine  # noqa: E402
from simple_es_b200.strategies import STRATEGIES  # noqa: E402


def timed(fn, warmup, reps):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / 1e3 / reps


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
    name, _, limit = q.partition(",")
    return name.strip() or torch.cuda.get_device_name(0), limit.strip()


def novelty_kernel(args, emit):
    for env, obs, act, sd in (("MountainCar-v0", 2, 3, 2), ("CartPole-v1", 4, 2, 4)):
        eng = RolloutEngine(env, obs, act, False, False, None, 5, 65536, 65536, 1, 1)
        g = torch.Generator(device="cuda").manual_seed(0)
        for P in (16384, 65536):
            bc = torch.randn((P, sd), dtype=torch.float64, device="cuda", generator=g)
            for A in (100, 1000, 10000):
                archive = torch.randn((A, sd), dtype=torch.float64, device="cuda", generator=g)
                out = torch.empty(P, dtype=torch.float64, device="cuda")
                reps = max(5, min(args.reps, int(2e10 / (P * A * sd))))
                t = timed(lambda: eng.novelty(bc, archive, A, 10, out=out), args.warmup, reps)
                emit({"kind": "novelty", "env": env, "state_dim": sd, "P": P, "A": A, "k": 10, "reps": reps,
                      "kernel_seconds": t, "fp64_gflops": 3.0 * P * A * sd / t / 1e9})
        eng.close()


def _cfg(conf, name, P, **strategy):
    cfg = yaml.load(open(os.path.join(ROOT, "conf", conf)), Loader=yaml.FullLoader)
    s = dict(cfg["strategy"], name=name, offspring_num=P, **strategy)
    if name != "nsr_es":
        s.pop("novelty_weight", None)
        s.pop("novelty_k", None)
    else:
        s.setdefault("novelty_weight", 0.5)
        s.setdefault("novelty_k", 10)
    return s, cfg


def _make(conf, name, P, seed=0, **strategy):
    s, cfg = _cfg(conf, name, P, **strategy)
    return STRATEGIES[name](s, cfg["env"], cfg["network"], 5, seed, 0, dict(cfg["engine"]))


def _load_fixture(s):
    z = np.load(os.path.join(ROOT, "tests", "golden", "bench_state_gen30.npz"))
    s.parents.copy_(torch.from_numpy(z["mu"]).view_as(s.parents))
    s.m.copy_(torch.from_numpy(z["m"]))
    s.v.copy_(torch.from_numpy(z["v"]))
    s.sigma = s.curr_sigma = float(z["sigma"])
    s.t = int(z["t"])
    s.generation = 30


WORKLOADS = [("cartpole_converged", "cartpole_openai.yaml", 65536, True), ("mountaincar_gen0", "mountaincar_nsr.yaml", 16384, False)]


def k1_and_generation(args, emit):
    for label, conf, P, fixture in WORKLOADS:
        times = {}
        for name in ("openai_es", "nsr_es"):
            s = _make(conf, name, P)
            if fixture:
                _load_fixture(s)
            if name == "nsr_es":                                  # an archive of args.archive rows
                for _ in range(args.archive):
                    s._reserve(s.n_archive + 1)
                    s.archive[s.n_archive].copy_(torch.randn(s.archive.shape[1], dtype=torch.float64))
                    s.n_archive += 1
            # the same generation every time: the state is restored before each step; nsr_es's archive grows by one row per
            # step (reported as nsr_es_archive_rows_at_end)
            gen0, sig0, t0 = s.generation, s.sigma, s.t
            par0, m0, v0 = s.parents.clone(), s.m.clone(), s.v.clone()

            def reset():
                s.generation, s.sigma, s.curr_sigma, s.t = gen0, sig0, sig0, t0
                s.parents.copy_(par0); s.m.copy_(m0); s.v.copy_(v0)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            total = 0.0
            for i in range(args.warmup + args.gen_reps):
                reset()
                torch.cuda.synchronize()
                a.record()
                s.step()
                b.record()
                torch.cuda.synchronize()
                if i >= args.warmup:
                    total += a.elapsed_time(b) / 1e3
            times[name] = total / args.gen_reps
            if name == "nsr_es":
                e = s.engine
                reset()
                parents = s.parents
                t_final = timed(lambda: e.rollout(gen0, sig0, parents, fitness=s.fitness, steps=s.steps), args.warmup, args.reps)
                e.set_final_states(None)
                t_plain = timed(lambda: e.rollout(gen0, sig0, parents, fitness=s.fitness, steps=s.steps), args.warmup, args.reps)
                e.set_final_states(s.final_states)
                torch.cuda.synchronize()
                steps = int(s.steps.sum().item())
                emit({"kind": "k1", "workload": label, "P": P, "env_steps": steps, "k1_seconds_final_states": t_final,
                      "k1_seconds_plain": t_plain, "final_states_overhead": t_final / t_plain - 1.0})
                archive_rows = s.n_archive
            s.engine.close()
        emit({"kind": "generation", "workload": label, "P": P, "openai_es_seconds": times["openai_es"],
              "nsr_es_seconds": times["nsr_es"], "nsr_es_over_openai_es": times["nsr_es"] / times["openai_es"],
              "nsr_es_archive_rows_at_end": archive_rows})


def learning(args, emit):
    for seed in (0, 1, 2):
        for name in ("openai_es", "nsr_es"):
            s = _make("mountaincar_nsr.yaml", name, 16384, seed=seed)
            best, curve = -1e9, []
            for g in range(args.learning):
                s.step()
                b = float(s.best_reward().item())
                best = max(best, b)
                if (g + 1) % 10 == 0:
                    ret, _ = s.engine.evaluate(s.elite_flat(), 100, round=g)
                    curve.append([g + 1, b, float(ret.mean().item())])
            emit({"kind": "learning", "config": "mountaincar_nsr.yaml", "strategy": name, "seed": seed, "generations": args.learning,
                  "best_fitness": best, "curve_gen_best_evalmean": curve})
            s.engine.close()


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--gen-reps", type=int, default=10)
    ap.add_argument("--archive", type=int, default=1000, help="archive rows before the timed nsr_es generations")
    ap.add_argument("--learning", type=int, default=0, help="generations of the learning comparison (0: skip)")
    ap.add_argument("--skip", default="", help="comma list of novelty,generation to skip")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("novelty_bench.py needs a CUDA device")
    name, limit = card()
    out = open(os.path.join(args.out, "novelty_bench.jsonl"), "a") if args.out else None

    def emit(rec):
        rec = dict(rec, gpu=name, power_limit=limit)
        line = json.dumps(rec)
        print(line, flush=True)
        if out:
            out.write(line + "\n")
            out.flush()
    skip = set(args.skip.split(","))
    if "novelty" not in skip:
        novelty_kernel(args, emit)
    if "generation" not in skip:
        k1_and_generation(args, emit)
    if args.learning > 0:
        learning(args, emit)


if __name__ == "__main__":
    main()

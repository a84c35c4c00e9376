#!/usr/bin/env python
"""Cost and learning of MAP-Elites (map_elites) on the GPU.  Prints JSON lines, each with the card's name and power limit read
in the same run; --out DIR also writes them to DIR/map_elites_bench.jsonl.

  kernels     ses_map_insert and ses_map_select (CUDA events around each call) at the shapes of tests/test_gpu_map_elites.py:
              CartPole MLP P = 65536 with 32 x 32 and 2^20 cells, MountainCar P = 16384, CartPole-GRU P = 4097 (D = 6562),
              simple_spread N = 3 with a 4-dimensional descriptor.  Random behaviours and fitness; the archive is the one
              the warm-up calls filled.
  generation  one map_elites generation against one openai_es generation on CartPole P = 65536 and CartPole-GRU P = 4097, each
              timed with CUDA events around step() after --warmup steps.  map_elites' K1 reads P distinct parent rows.
  learning    (--learning G) conf/mountaincar_map_elites.yaml against openai_es and nsr_es at their shipped settings on 3 seeds:
              coverage, the best elite's mean return over 100 eval_es-style evaluation episodes, and whether any elite (every
              one evaluated) reaches the flag (an episode shorter than 200 steps).
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
from simple_es_b200.engine import RolloutEngine, map_spec  # noqa: E402
from simple_es_b200.strategies import STRATEGIES  # noqa: E402

KERNEL_CASES = {
    "cartpole-65536-32x32": ("CartPole-v1", False, 1, 65536, [0, 2], [-2.4, -0.2095], [2.4, 0.2095], [32, 32]),
    "cartpole-65536-2^20": ("CartPole-v1", False, 1, 65536, [0, 1, 2, 3], [-2.4, -3, -0.2095, -3], [2.4, 3, 0.2095, 3], [32] * 4),
    "mountaincar-16384": ("MountainCar-v0", False, 1, 16384, [0, 1], [-1.2, -0.07], [0.6, 0.07], [32, 32]),
    "cartpole-gru-4097": ("CartPole-v1", True, 1, 4097, [2, 0], [-0.2095, -2.4], [0.2095, 2.4], [40, 25]),
    "spread3-4d": ("simple_spread", False, 3, 16384, [0, 1, 6, 7], [-1.5, -1.5, -1, -1], [1.5, 1.5, 1, 1], [8, 8, 6, 6]),
}


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


def kernels(args, emit):
    for case, (env, gru, N, P, dims, low, high, cells) in KERNEL_CASES.items():
        obs, act = {"CartPole-v1": (4, 2), "MountainCar-v0": (2, 3), "simple_spread": (18, 5)}[env]
        eng = RolloutEngine(env, obs, act, gru, False, None, 1, P, 1, 0, P, seed=1, n_agents=N)
        sd, D, dev = eng.state_dim, eng.D, eng.device
        n_cells = int(np.prod(cells))
        spec = map_spec(dims, low, high, cells)
        g = torch.Generator(device=dev).manual_seed(0)
        lo, hi = torch.tensor(low, dtype=torch.float64, device=dev), torch.tensor(high, dtype=torch.float64, device=dev)
        bc = torch.rand((P, sd), dtype=torch.float64, device=dev, generator=g)
        bc[:, dims] = lo + bc[:, dims] * (hi - lo)
        fit = torch.randn(P, dtype=torch.float64, device=dev, generator=g)
        order = eng.rank_desc(fit, full_key=True)
        parents = torch.randn((P, D), dtype=torch.float32, device=dev, generator=g)
        F = torch.full((n_cells,), float("nan"), dtype=torch.float64, device=dev)
        B = torch.zeros((n_cells, sd), dtype=torch.float64, device=dev)
        born = torch.zeros((n_cells, 2), dtype=torch.int32, device=dev)
        W = torch.zeros((n_cells, D), dtype=torch.float32, device=dev)
        seed_row, stats = torch.zeros(D, dtype=torch.float32, device=dev), torch.zeros(4, dtype=torch.float64, device=dev)
        out = torch.empty((P, D), dtype=torch.float32, device=dev)
        t_ins = timed(lambda: eng.map_insert(0, 0.1, parents, order, fit, bc, spec, F, B, born, W), args.warmup, args.reps)
        t_sel = timed(lambda: eng.map_select(1, spec, F, W, seed_row, stats, out), args.warmup, args.reps)
        emit({"kind": "kernels", "case": case, "P": P, "D": D, "n_cells": n_cells, "occupied": int(stats[0].item()),
              "insert_ms": t_ins * 1e3, "select_ms": t_sel * 1e3})
        eng.close()
        del W, out, parents
        torch.cuda.empty_cache()


def _cfg(conf):
    return yaml.load(open(os.path.join(ROOT, "conf", conf)), Loader=yaml.FullLoader)


def generation(args, emit):
    for name, gru, P in (("mlp", False, 65536), ("gru", True, 4097)):
        res = {}
        for strat, conf in (("openai_es", "cartpole_openai.yaml"), ("map_elites", "cartpole_map_elites.yaml")):
            cfg = _cfg(conf)
            cfg["strategy"]["offspring_num"] = P
            cfg["network"]["gru"] = gru
            s = STRATEGIES[strat](cfg["strategy"], cfg["env"], cfg["network"], 5, 0, 0, dict(cfg["engine"] or {}))
            res[strat] = timed(s.step, args.warmup, args.reps)
            del s
            torch.cuda.empty_cache()
        emit({"kind": "generation", "workload": "CartPole-%s" % name, "P": P, "openai_es_ms": res["openai_es"] * 1e3,
              "map_elites_ms": res["map_elites"] * 1e3, "ratio": res["map_elites"] / res["openai_es"]})


def learning(args, emit):
    from simple_es_b200.loop import B200Loop
    runs = [("map_elites", "mountaincar_map_elites.yaml"), ("nsr_es", "mountaincar_nsr.yaml"), ("openai_es", None)]
    for seed in (0, 1, 2):
        for strat, conf in runs:
            if conf is None:                        # openai_es with the nsr_es config's shared hyper-parameters (w = 0 is openai_es)
                cfg = _cfg("mountaincar_nsr.yaml")
                cfg["strategy"] = {k: v for k, v in cfg["strategy"].items() if k not in ("novelty_weight", "novelty_k")}
                cfg["strategy"]["name"] = "openai_es"
            else:
                cfg = _cfg(conf)
            loop = B200Loop(cfg, args.learning, 1, 5, save_model_period=0, seed=seed, quiet=True)
            loop.run()
            s = loop.strategy
            row = {"kind": "learning", "strategy": strat, "seed": seed, "generations": args.learning, "P": s.P,
                   "best_fitness_last": loop.history[-1][1], "best_fitness_max": max(h[1] for h in loop.history)}
            ret, lng = s.engine.evaluate(s.elite_flat(), 100, round=0)
            row["elite_eval_mean"] = float(ret.mean())
            if strat == "map_elites":
                n_occ, n_cells, best, qd = s.archive_stats()
                a = s.archive()
                r_all, l_all = s.engine.evaluate(a["weights"].cuda(), 100, round=0)
                means = r_all.mean(dim=1)
                row.update(coverage=n_occ / n_cells, occupied=n_occ, qd_score=qd, archive_best=best,
                           best_elite_eval_mean=float(means.max()), elites_reaching_flag=int((l_all < 200).any(dim=1).sum()))
            else:
                row["reaches_flag"] = bool((lng < 200).any())
            emit(row)
            del loop, s
            torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--learning", type=int, default=0, metavar="G", help="also run G learning generations per strategy and seed")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    name, limit = card()
    lines = []

    def emit(d):
        d = dict(d, gpu=name, power_limit=limit)
        print(json.dumps(d), flush=True)
        lines.append(d)
    kernels(args, emit)
    generation(args, emit)
    if args.learning:
        learning(args, emit)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "map_elites_bench.jsonl"), "w") as fh:
            for d in lines:
                fh.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()

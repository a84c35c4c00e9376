#!/usr/bin/env python
"""Cost and learning of separable CMA-ES (sep_cma_es) on the GPU.  Prints JSON lines, each with the card's name and power
limit read in the same run; --out DIR also writes them to DIR/cma_bench.jsonl.

  kernels     ses_cma_sample and ses_cma_update (CUDA events around each call), and the kernels inside them from
              torch.profiler: k_cma_sample, k_cma_weights, k_grad_partial<true> (both tables) next to k_grad_partial<false>
              (openai_es's one table), k_cma_final.  CartPole MLP at P = 65536 and CartPole-GRU at P = 4097.
  generation  one sep_cma_es generation against one openai_es generation on the same two workloads, each timed with CUDA
              events around step() from its generation-0 state (restored before every step; the same init_sigma 0.5, so both
              roll out populations of the same spread around the zero policy).
  learning    (--learning G) conf/cartpole_sep_cma.yaml and conf/pendulum_sep_cma.yaml against openai_es with the shipped
              openai_es hyper-parameters (conf/cartpole_openai.yaml, conf/pendulum.yaml) at the same population, 3 seeds:
              best fitness and the mean return of the saved policy over 100 evaluation episodes every 10 generations.

Kernel and step times are means over --reps calls after --warmup calls of the same shape.
"""
import argparse
import json
import os
import subprocess
import sys

import torch
import yaml

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from simple_es_b200.engine import RolloutEngine, sep_cma_constants  # noqa: E402
from simple_es_b200.strategies import STRATEGIES  # noqa: E402

WORKLOADS = [("mlp", False, 65536), ("gru", True, 4097)]


def timed(fn, warmup, reps, before=None):
    """Mean seconds of fn() over reps calls; before() (untimed) runs ahead of every call."""
    for _ in range(warmup):
        if before:
            before()
        fn()
    torch.cuda.synchronize()
    total = 0.0
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(reps):
        if before:
            before()
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        total += a.elapsed_time(b) / 1e3
    return total / reps


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
    name, _, limit = q.partition(",")
    return name.strip() or torch.cuda.get_device_name(0), limit.strip()


def kernels(args, emit):
    from torch.profiler import ProfilerActivity, profile
    for net, gru, P in WORKLOADS:
        eng = RolloutEngine("CartPole-v1", 4, 2, gru, False, 500, 5, P, P, 0, 1, seed=1)
        D = eng.D
        k = sep_cma_constants(D, P, P // 2)
        g = torch.Generator(device="cuda").manual_seed(0)
        mean = torch.randn(D, dtype=torch.float64, device="cuda", generator=g) * 0.3
        c = torch.rand(D, dtype=torch.float64, device="cuda", generator=g) + 0.5
        ps, pc = torch.zeros_like(mean), torch.zeros_like(mean)
        sigma = torch.full((1,), 0.5, dtype=torch.float64, device="cuda")
        out = torch.empty((P, D), dtype=torch.float32, device="cuda")
        order = torch.randperm(P, device="cuda", generator=g).to(torch.int32)
        w = torch.from_numpy(k["weights"]).cuda()
        s = torch.empty(P, dtype=torch.float64, device="cuda")
        parent = torch.empty(D, dtype=torch.float32, device="cuda")
        state = [t.clone() for t in (mean, c, ps, pc, sigma)]

        def restore():
            for t, t0 in zip((mean, c, ps, pc, sigma), state):
                t.copy_(t0)

        def update():
            eng.cma_update(0, order, k, w, s, mean, c, ps, pc, sigma, parent)

        t_sample = timed(lambda: eng.cma_sample(0, mean, c, sigma, out=out), args.warmup, args.reps)
        t_update = timed(update, args.warmup, args.reps, before=restore)
        shaped = torch.randn(P, dtype=torch.float64, device="cuda", generator=g)
        mu32, m32, v32 = (torch.zeros(D, dtype=torch.float32, device="cuda") for _ in range(3))
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(args.reps):
                eng.cma_sample(0, mean, c, sigma, out=out)
                restore()
                update()
                eng.update_openai(0, 0.5, 0.1, 1, shaped, mu32, m32, v32)
            torch.cuda.synchronize()
        per = {}
        for ev in prof.key_averages():
            for short in ("k_cma_sample", "k_cma_weights", "k_cma_final", "k_grad_partial<true>", "k_grad_partial<false>",
                          "k_grad_final_adam"):
                if short in ev.key:
                    per[short] = ev.device_time / 1e6            # mean per call, microseconds -> seconds
        emit({"bench": "kernels", "net": net, "P": P, "D": D, "mu": P // 2, "cma_sample_s": t_sample, "cma_update_s": t_update,
              "kernel_mean_s": per})
        eng.close()


def _strategy(name, gru, P, seed=0):
    conf = "cartpole_sep_cma.yaml" if name == "sep_cma_es" else "cartpole_openai.yaml"
    cfg = yaml.load(open(os.path.join(ROOT, "conf", conf)), Loader=yaml.FullLoader)
    strat = dict(cfg["strategy"], offspring_num=P, init_sigma=0.5)
    net = dict(cfg["network"], gru=gru)
    return STRATEGIES[name](strat, cfg["env"], net, 5, seed, 0, dict(cfg["engine"]))


def generation(args, emit):
    for net, gru, P in WORKLOADS:
        row = {"bench": "generation", "net": net, "P": P}
        for name in ("sep_cma_es", "openai_es"):
            s = _strategy(name, gru, P)
            st = s.state()
            row[name + "_s"] = timed(s.step, args.warmup, args.reps, before=lambda: s.load_state(st))
        row["ratio"] = row["sep_cma_es_s"] / row["openai_es_s"]
        emit(row)


def learning(args, emit):
    from simple_es_b200.loop import B200Loop
    pairs = {"CartPole-v1": ("cartpole_sep_cma.yaml", "cartpole_openai.yaml"), "Pendulum-v0": ("pendulum_sep_cma.yaml", "pendulum.yaml")}
    for env, confs in pairs.items():
        P = yaml.load(open(os.path.join(ROOT, "conf", confs[0])), Loader=yaml.FullLoader)["strategy"]["offspring_num"]
        for conf in confs:
            for seed in (0, 1, 2):
                cfg = yaml.load(open(os.path.join(ROOT, "conf", conf)), Loader=yaml.FullLoader)
                cfg["strategy"]["offspring_num"] = P
                cfg["engine"]["eval_every"] = 10
                loop = B200Loop(cfg, args.learning, 1, 5, save_model_period=0, seed=seed, quiet=True)
                hist = loop.run()
                emit({"bench": "learning", "env": env, "strategy": cfg["strategy"]["name"], "conf": conf, "P": P, "seed": seed,
                      "best_fitness": [round(h[1], 3) for h in hist[9::10]],
                      "eval_mean_return": [round(e[2], 3) for e in loop.eval_history], "final_sigma": hist[-1][2]})


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--learning", type=int, default=0, metavar="G", help="generations of the learning comparison (0: skip)")
    ap.add_argument("--out", default=None, help="directory for cma_bench.jsonl")
    args = ap.parse_args()
    name, limit = card()
    lines = []

    def emit(row):
        row = dict(row, gpu=name, power_limit=limit)
        print(json.dumps(row), flush=True)
        lines.append(row)
    kernels(args, emit)
    generation(args, emit)
    if args.learning:
        learning(args, emit)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "cma_bench.jsonl"), "w") as fh:
            fh.writelines(json.dumps(r) + "\n" for r in lines)


if __name__ == "__main__":
    main()

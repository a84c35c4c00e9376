#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 population-rollout engine.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json metric: "env-steps/sec/GPU, CartPole-v1 pop=65536 ...; ES generations/sec"):
CartPole-v1, 32-hidden MLP policy (D = 226), openai_es (centered ranks + Adam), population 65536
sharded over N GPUs (strong scaling), eval_ep_num 5, max_step 500, seed 0, mu = 0 at generation 0
(conf/cartpole_openai.yaml).  A "step" is one ES generation: K1 rollout of the rank's slice ->
fitness all-gather (N > 1) -> K2 rank/shape -> K3 gradient + Adam.  `value` counts env steps that were
actually simulated (sum of episode lengths), not P*E*500.

Prints ONE JSON line on rank 0 (see DESIGN.md section 8 for every key).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# The benchmark may run from a read-only tree and leaves the tree as it found it: no bytecode caches written there.
sys.dont_write_bytecode = True
# One OpenMP thread per process (what torchrun sets for N > 1 anyway): the CPU legs run one forked worker per
# core, and torch's intra-op pool inside each of them only oversubscribes the box (measured here: 116 k -> 180 k
# env-steps/s for the reference path on 8 cores).  The GPU arm does no CPU compute.
os.environ.setdefault("OMP_NUM_THREADS", "1")
os.environ.setdefault("MKL_NUM_THREADS", "1")

P_DEFAULT = 65536
E_DEFAULT = 5
D = 226
FLOP_PER_STEP = 418          # SURVEY.md section 8d: 192 FMA + 34 bias adds per env step (CartPole MLP)
FMA_LANE_OPS_PER_STEP = 640  # executed on the FP32 FMA pipe per env step: fc1 128 + fc2 64 + 32 tanh x 14 (DESIGN.md 5.1)
K1_DRAM_BYTES_PER_LAUNCH = 166912       # dram__bytes_read.sum + dram__bytes_write.sum of K1 in profiles/r02_k1_conv.txt (one converged launch, P = 65536)
K1_PROFILE = "profiles/r02_k1_conv.txt"
GRU_WAVEFRONTS_PER_OFFSPRING_STEP = 288   # see run_extra_config: algorithmic shared-memory wavefronts of the CartPole-GRU kernel
K1_SYMBOL = "ses::k_rollout_slots<ses::CartpoleMlpEnvT<7>, 8, 4, false, false>"   # the kernel ses_rollout launches for this workload
STRATEGY = dict(name="openai_es", init_sigma=0.2, sigma_decay=0.9999, learning_rate=0.1)


# ----------------------------------------------------------------------------------------------
# clocks (B200_PROFILING.md "clocks DURING the timed region")
# ----------------------------------------------------------------------------------------------
class ClockSampler:
    """Samples SM clock + throttle reasons every ~5 ms through NVML (nvidia_ml_py) while the timed
    region runs; the same fields as the recipe's nvidia-smi clocks line."""
    BITS = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40,
            "hw_power_brake_slowdown": 0x80}

    def __init__(self, gpu_index=0):
        self.gpu = gpu_index
        self.sm, self.reasons, self.power = [], set(), []
        self.max_mhz = None
        self._stop = threading.Event()
        self.thread = None
        self.err = None

    def _phys_index(self):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            try:
                return int(vis.split(",")[self.gpu])
            except Exception:
                return self.gpu
        return self.gpu

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self._phys_index())
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception as exc:
            self.err = "nvml unavailable: %s" % (exc,)
            return
        self.thread = threading.Thread(target=self._run, daemon=True)
        self.thread.start()

    def _sample(self):
        nv = self.nv
        self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
        try:
            r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
        except Exception:
            r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
        for name, bit in self.BITS.items():
            if r & bit:
                self.reasons.add(name)
        try:
            self.power.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
        except Exception:
            pass

    def _run(self):
        while not self._stop.is_set():
            try:
                self._sample()
            except Exception as exc:
                self.err = str(exc)
                return
            time.sleep(0.005)

    def stop(self):
        if self.thread is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [self.err or "no sampler"]}
        try:
            self._sample()
        except Exception:
            pass
        self._stop.set()
        self.thread.join(timeout=1)
        sm = sorted(self.sm)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(sm), "power_w_max": max(self.power) if self.power else None}


# ----------------------------------------------------------------------------------------------
# CPU legs (oracle; allowed importers of oracle/: tests, smoke, and these two functions)
# ----------------------------------------------------------------------------------------------
STATE_FIXTURE = os.path.join(ROOT, "tests", "golden", "bench_state_gen30.npz")
CALIBRATION = ("calibration (profiles/r02_reference_calibration.json, tools/calibrate_reference.py, dev container, 8 cores, same 365-offspring "
               "sample): the UNMODIFIED reference ESLoop + openai_es + GymEnvModel + RolloutWorker runs 93.7 k env-steps/s where this "
               "port runs 131 k -- the port is 1.40x faster than the reference's own code (it ships flat weight vectors instead of "
               "deep-copied, pickled nn.Modules), so ratios against it are conservative")
REGIME = ("population drawn around the generation-30 state of this very workload (tests/golden/bench_state_gen30.npz, "
          "tools/make_bench_fixture.py): episodes of ~500 steps, the regime the GPU arm's timed generations run in")
CPU_SEC_PER_OFFSPRING = 0.21   # 5 episodes x 500 steps x ~85 us per reference policy-forward + env step on one core


def bench_state():
    """The trained openai_es state the CPU legs start from (a committed fixture; not an oracle import)."""
    import numpy as np
    z = np.load(STATE_FIXTURE)
    return {"mu": z["mu"], "m": z["m"], "v": z["v"], "sigma": float(z["sigma"]), "t": int(z["t"])}


def cpu_reference_generation(n_offspring, cores, gen_seed, eval_ep_num=E_DEFAULT, state=None):
    """One generation of the reference's CPU path (port: oracle/pyref.py -- torch-CPU policy per
    offspring, Python CartPole, a fresh mp.Pool(cores), strategy.evaluate) on a population sample of
    n_offspring drawn around `state` (None: the all-zero generation-0 network).  Returns (env_steps, seconds)."""
    import numpy as np
    import torch
    from oracle import pyref
    torch.set_num_threads(1)
    np.random.seed(gen_seed)
    init = np.random.RandomState(0).uniform(-0.05, 0.05, size=(eval_ep_num, 4))
    env = pyref.CartPoleShim(max_step=500, init_states=init)
    cfg = dict(STRATEGY, offspring_num=n_offspring)
    t0 = time.perf_counter()
    rec = pyref.es_loop_port(env, (4, 2, False), cfg, 1, cores, eval_ep_num, seed=gen_seed, state=state)
    return rec[0]["env_steps"], time.perf_counter() - t0


def cpu_baseline_block(cores):
    """Bounded CPU baseline reported beside the GPU number (rank 0, N = 1)."""
    n = max(64, min(P_DEFAULT, 96 * cores))            # 10-20 s of CPU work on the box's cores
    steps, dt = cpu_reference_generation(n, cores, 12345, state=bench_state())
    out = {"value": steps / dt, "unit": "env-steps/s", "cores": cores, "kind": "port",
           "sample": "1 generation of the reference CPU path (oracle/pyref.py port: torch-CPU policy, Python CartPole, "
                     "mp.Pool(%d), evaluate) on %d offspring x %d episodes = %d env steps in %.1f s; %s"
                     % (cores, n, E_DEFAULT, steps, dt, REGIME)}
    try:  # a much stronger CPU number for context: the C bit-twin on every host thread, same regime
        import numpy as np
        from oracle import twin
        st = bench_state()
        n2 = 512 * cores
        t0 = time.perf_counter()
        _, ts = twin.population_cartpole(st["mu"][None], sigma=st["sigma"], seed=0, gen=30, group=P_DEFAULT, n_head=1,
                                         n=n2, E=E_DEFAULT, nthreads=cores)
        dt2 = time.perf_counter() - t0
        out["c_twin"] = {"value": float(ts.sum()) / dt2, "unit": "env-steps/s", "cores": cores,
                         "sample": "%d offspring of generation 30 x %d episodes = %d env steps, oracle/ses_twin.c, %d pthreads"
                                   % (n2, E_DEFAULT, int(ts.sum()), cores)}
    except Exception as exc:  # pragma: no cover
        out["c_twin"] = {"error": str(exc)}
    return out


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path, timed on the host cores."""
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return 0
    cores = os.cpu_count() or 1
    # per-step sample: the whole run (K timed + W warm-up steps) should take about two minutes on this box
    per_step_s = 120.0 / max(1, args.steps + args.warmup)
    n = int(max(2 * cores, min(64 * cores, per_step_s * cores / CPU_SEC_PER_OFFSPRING)))
    state = bench_state()
    for w in range(args.warmup):
        cpu_reference_generation(n, cores, 100 + w, state=state)
    tot_steps, tot_t = 0, 0.0
    for k in range(args.steps):
        s, dt = cpu_reference_generation(n, cores, 1000 + k, state=state)
        tot_steps += s; tot_t += dt
    v = tot_steps / tot_t
    sample = ("each step = 1 generation of the reference CPU path (oracle/pyref.py port, mp.Pool(%d)) on %d offspring x %d "
              "episodes (bounded sample of the 65536 population); %s; %s" % (cores, n, E_DEFAULT, REGIME, CALIBRATION))
    line = {
        "impl": "reference", "metric": "env-steps/sec", "value": v, "unit": "env-steps/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot_t / max(1, args.steps),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32 policy / f64 physics",
        "data": "synthetic", "config": workload_config(args, 1),
        "cpu_baseline": {"value": v, "unit": "env-steps/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


def workload_config(args, world):
    return {"workload": "CartPole-v1 MLP(4-32-2, D=226) openai_es pop=%d eval_ep_num=%d max_step=500 "
                        "(BASELINE configs[2]; conf/cartpole_openai.yaml)" % (args.pop, E_DEFAULT),
            "population": args.pop, "eval_ep_num": E_DEFAULT, "strategy": STRATEGY,
            "regime": REGIME_TEXT[args.regime],
            "parallelism": "pop-shard x%d (%s)" % (world, args.shard if world > 1 else "single"), "fitness_exchange": (args.exchange if world > 1 else "local"),
            "init_states": "shared [E] table (reference mp.Pool semantics)",
            "l2": "flushed between timed generations (256 MiB write); the hot path itself reads 904 B of parameters per generation"}


REGIME_TEXT = {
    "converged": "converged (SURVEY 8d): K real consecutive ES generations continuing the committed generation-30 state of this very "
                 "run (tests/golden/bench_state_gen30.npz: mu, Adam m/v, t, sigma), nearly every episode 500 steps -- the regime the "
                 "reference arm and cpu_baseline are timed in",
    "from_scratch": "from scratch: real consecutive ES generations W..W+K-1 of a run started at mu = 0 (a converging mixture of "
                    "episode lengths)",
    "gen0": "generation 0 (SURVEY 8d): mu = 0, sigma = sigma0, ragged episode lengths of ~10-20 steps with a few 500-step stragglers; "
            "every timed step is a generation-0 population with fresh noise",
}

# BASELINE.json configs other than the headline one, each as (key, YAML, overrides, steps the config is timed for)
EXTRA_CONFIGS = [
    ("c1_cartpole_simple_evolution_as_shipped", "conf/cartpole.yaml", {}, "BASELINE configs[0]: conf/cartpole.yaml as shipped (P = 97)"),
    ("c2_cartpole_pomdp_gru_pop4096", "conf/cartpole_pomdp_gru.yaml", {}, "BASELINE configs[1]: CartPole POMDP + GRU, simple_evolution, P = 4097"),
    ("c2_converged_gru_pop4096", "conf/cartpole_pomdp_gru.yaml", {"env.pomdp": False, "strategy.init_sigma": 0.02, "init": "gru_balancing"},
     "configs[1]'s kernel in the converged regime: the same GRU policy / population started from a hand-built balancing parent on the fully "
     "observed pole (every episode 500 steps); the POMDP mask only zeroes two observations, the arithmetic per step is identical"),
    ("c4_simple_spread_n3_pop16384", "conf/simplespread.yaml", {"network.num_state": 18, "engine.n_agents": 3},
     "BASELINE configs[3]: simple_spread, 3 agents, shared MLP, openai_es, P = 16384 (env steps = world steps)"),
    ("c4_simple_spread_n2_pop16384", "conf/simplespread.yaml", {}, "the reference's own N = 2 form of configs[3] (pettingzoo_wrapper.py:9)"),
    ("c5_cartpole_simple_genetic_pop1m", "conf/cartpole_genetic.yaml", {}, "BASELINE configs[4]: CartPole simple_genetic, P = 2^20"),
]


def gru_balancing_parent():
    """A GRU policy that balances the fully observed pole: fc1 unit 0 is a bang-bang feature, the n gate carries it, z ~ 0."""
    import numpy as np
    mu = np.zeros(6562, np.float32)
    mu[0:128].reshape(32, 4)[0] = [0.0, 0.5, 10.0, 3.0]
    mu[160:160 + 3072].reshape(96, 32)[64, 0] = 3.0
    mu[160 + 6144:160 + 6144 + 96][32:64] = -10.0
    w2 = mu[160 + 6144 + 192:160 + 6144 + 192 + 64].reshape(2, 32)
    w2[1, 0] = 5.0; w2[0, 0] = -5.0
    return mu


def converged_state():
    """The committed generation-30 state as a strategy resume dict (strategies._Base.load_state)."""
    import torch
    st = bench_state()
    return {"strategy": "openai_es", "generation": 30, "sigma": st["sigma"], "curr_sigma": st["sigma"], "population": P_DEFAULT,
            "parents": torch.from_numpy(st["mu"].copy()).reshape(1, -1), "m": torch.from_numpy(st["m"].copy()),
            "v": torch.from_numpy(st["v"].copy()), "t": st["t"]}


def bits_checksum(t):
    """Position-weighted wrap-around checksum of a tensor's BITS (int64): equal on two ranks iff (for all practical
    purposes) the tensors are bit-identical."""
    import torch
    b = t.detach().contiguous().view(torch.uint8).to(torch.int64)
    w = torch.arange(1, b.numel() + 1, dtype=torch.int64, device=b.device) * 2654435761
    return (b * w).sum()


# ----------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------
def make_loop(args, local, gens):
    from simple_es_b200.loop import B200Loop
    config = {"env": {"name": "CartPole-v1", "max_step": 500, "pomdp": False},
              "network": {"name": "gym_model", "num_state": 4, "num_action": 2, "discrete_action": True, "gru": False},
              "strategy": dict(STRATEGY, offspring_num=args.pop),
              "engine": {"name": "b200", "fitness_exchange": args.exchange, "shard": args.shard}}
    return B200Loop(config, gens, 1, E_DEFAULT, log=False, save_model_period=0, seed=0, device=local, quiet=True)


def reset_to_regime(s, regime, rep=0):
    """Put an OpenAIES strategy at the start of `regime` (rep: which generation-0 repetition)."""
    if regime == "converged":
        if s.P == P_DEFAULT:
            s.load_state(converged_state())
        else:                                        # another population size: the same parameters, Adam state and sigma
            st = converged_state(); st["population"] = s.P
            s.load_state(st)
    else:
        s.parents.zero_(); s.m.zero_(); s.v.zero_()
        s.t = 0
        s.sigma = s.curr_sigma = float(STRATEGY["init_sigma"])
        s.generation = rep


def timed_generations(s, steps, flush, barrier, gen0=False, keep_prev_mu=None):
    """`steps` openai_es generations of strategy `s`, each bracketed by CUDA events on the launching stream with one more
    event after K1 (the dominant kernel is timed alone); the L2 flush sits outside the events.  gen0: every step is a
    generation-0 population (state reset between steps, outside the events).  Returns (gen_ms, k1_ms, env_steps, wall_s)."""
    import torch
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(steps)]
    e = s.engine
    before = int(s.total_env_steps.item())
    barrier()
    wall0 = time.perf_counter()
    for k in range(steps):
        if gen0:
            reset_to_regime(s, "gen0", rep=1000 + k)
        if keep_prev_mu is not None:
            keep_prev_mu.copy_(s.parents)            # 904 B device copy: the population of the last generation can be re-derived
        flush.fill_(k & 0xFF)                        # L2 flush, outside the timed events
        ev[k][0].record()
        s.fitness = s._fit[s.generation & 1]
        e.rollout(s.generation, s.sigma, s.parents, fitness=s.fitness, steps=s.steps)
        ev[k][1].record()
        s.exchange_fitness()
        e.rank_desc(s.fitness, shaped=True, order=s.order, shaped_out=s.shaped)
        s.t += 1
        e.update_openai(s.generation, s.sigma, s.lr, s.t, s.shaped, s.parents.view(-1), s.m, s.v)
        s.last_sigma = s.sigma
        s.sigma *= s.decay; s.curr_sigma = s.sigma; s.generation += 1
        ev[k][2].record()
    barrier()
    wall = time.perf_counter() - wall0
    gen_ms = sum(ev[k][0].elapsed_time(ev[k][2]) for k in range(steps))
    k1_ms = sum(ev[k][0].elapsed_time(ev[k][1]) for k in range(steps))
    return gen_ms, k1_ms, int(s.total_env_steps.item()) - before, wall


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, per_offspring, per_parameter):
    """--dump-outputs: what the last timed generation handed its caller, as <out_dir>/<name>.npy (float32 arrays stay
    float32, everything else becomes float64; integer ids below 2^53 are exact).  If the per-offspring arrays would take
    the files past DUMP_LIMIT_BYTES, a fixed, seeded sample of offspring is written instead and its ids go to
    offspring_ids.npy."""
    import numpy as np

    def host(t):
        a = t.detach().cpu().numpy()
        return a if a.dtype == np.float32 else a.astype(np.float64)
    off = {k: host(t) for k, t in per_offspring.items()}
    par = {k: host(t) for k, t in per_parameter.items()}
    n = len(next(iter(off.values())))
    room = DUMP_LIMIT_BYTES - sum(a.nbytes for a in par.values())
    row = sum(a.itemsize for a in off.values())
    if n * row > room:
        keep = room // (row + 8)
        ids = np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
        off = {k: a[ids] for k, a in off.items()}
        off["offspring_ids"] = ids.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, a in dict(off, **par).items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def reduce_over_ranks(dev, world, gen_ms, k1_ms, n_steps):
    """max over ranks of the times, sum over ranks of the env steps (device-timed numbers, never wall clock)."""
    import torch
    import torch.distributed as dist
    t = torch.tensor([gen_ms, k1_ms], dtype=torch.float64, device=dev)
    tsum = t.clone()
    n = torch.tensor([n_steps], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        dist.all_reduce(n, op=dist.ReduceOp.SUM)
    return float(t[0]), float(t[1]), float(tsum[1]) / world, int(n[0])


def regime_block(gen_ms, k1_ms, total_steps, steps, pop):
    return {"ms_per_generation": gen_ms / steps, "k1_ms_per_generation": k1_ms / steps, "generations_per_sec": steps / (gen_ms * 1e-3),
            "env_steps_per_sec": total_steps / (gen_ms * 1e-3), "env_steps": total_steps, "steps": steps,
            "mean_episode_len": total_steps / float(steps * pop * E_DEFAULT)}


def run_extra_config(key, path, overrides, note, local, world, steps, warmup, flush, barrier, args):
    """One of the other BASELINE configs through the public API (B200Loop.strategy.step()), device-timed."""
    import torch
    import yaml
    from simple_es_b200.loop import B200Loop
    with open(os.path.join(ROOT, path)) as fh:
        cfg = yaml.load(fh, Loader=yaml.FullLoader)
    init = None
    for k, v in overrides.items():
        if k == "init":
            init = v
            continue
        a, b = k.split(".")
        cfg[a][b] = v
    cfg["engine"] = dict(cfg.get("engine") or {}, fitness_exchange=args.exchange, shard=args.shard)
    loop = B200Loop(cfg, steps + warmup, 1, E_DEFAULT, log=False, save_model_period=0, seed=0, device=local, quiet=True)
    s = loop.strategy
    if init == "gru_balancing":
        s.load_elite(gru_balancing_parent())
    for _ in range(warmup):
        s.step()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(steps)]
    before = int(s.total_env_steps.item())
    barrier()
    for k in range(steps):
        flush.fill_(k & 0xFF)
        ev[k][0].record(); s.step(); ev[k][1].record()
    barrier()
    ms = sum(a.elapsed_time(b) for a, b in ev)
    n = int(s.total_env_steps.item()) - before
    best = float(s.best_reward().item())
    ms, _, _, n = reduce_over_ranks(s.engine.device, world, ms, 0.0, n)
    out = {"config": note, "yaml": path, "overrides": overrides, "strategy": cfg["strategy"]["name"], "population": s.P, "D": s.D,
           "steps": steps, "warmup": warmup, "ms_per_generation": ms / steps, "generations_per_sec": steps / (ms * 1e-3),
           "env_steps_per_sec": n / (ms * 1e-3), "env_steps": n, "mean_episode_len": n / float(steps * s.P * E_DEFAULT),
           "best_reward_last_gen": best, "n_gpus": world, "regime": "generations %d..%d of a run started from %s" % (warmup, warmup + steps - 1, "mu = 0" if init is None else init)}
    if key == "c2_converged_gru_pop4096" and world == 1:
        # The GRU rollout kernel is bound by the shared-memory crossbar (one wavefront per cycle per SM), not by the FMA pipe
        # (DESIGN 5.2, profiles/r02_gru_variants_ncu.txt).  Algorithmic wavefronts per offspring-step (E = 5 episodes in lockstep):
        # two weight tables x 16 conflict-free LDS.128 x 4 wavefronts + 80 broadcast LDS.128 x 2 = 288 (the n-gate table lives in
        # registers); ncu counts 365 with the staging stores and the logit reads.  One offspring-step = E env steps.
        sms = torch.cuda.get_device_properties(s.engine.device).multi_processor_count
        mhz = 1965.0                                                    # B200 max SM clock (B200_PROFILING.md); NVML's value if it answers
        try:
            import pynvml
            pynvml.nvmlInit()
            mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(pynvml.nvmlDeviceGetHandleByIndex(local), pynvml.NVML_CLOCK_SM))
        except Exception:
            pass
        peak = sms * mhz * 1e6 / 1e9
        achieved = GRU_WAVEFRONTS_PER_OFFSPRING_STEP * (n / float(E_DEFAULT)) / (ms * 1e-3) / 1e9
        out["roofline"] = {"bound": "shared_memory", "kernel": "ses::k_rollout_cartpole_gru<5, 4, false, true, 1>", "achieved": achieved, "peak": peak,
                           "unit": "Gwavefronts/s", "frac": achieved / peak,
                           "algorithmic": "%d shared-memory wavefronts per offspring-step x %d offspring-steps / %.3f ms of whole generations (K1 is 97 %% of them)"
                                          % (GRU_WAVEFRONTS_PER_OFFSPRING_STEP, n // E_DEFAULT, ms),
                           "peak_source": "%d SMs x 1 wavefront per cycle x %.0f MHz (the max SM clock; ncu of the kernel alone: 62 %% of the wavefront peak, "
                                          "profiles/r02_gru_variants_ncu.txt)" % (sms, mhz)}
    if s.exchange == "peer":
        s.engine.peer_check()
    del loop, s
    torch.cuda.synchronize()
    return out


def run_b200(args):
    import torch
    import torch.distributed as dist
    from simple_es_b200 import dist as sdist

    rank, world = sdist.init_from_env()
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- headline: K timed generations in the chosen regime (default: converged)
    loop = make_loop(args, local, args.steps + args.warmup)
    s = loop.strategy
    eng = s.engine
    reset_to_regime(s, args.regime)
    for w in range(args.warmup):
        if args.regime == "gen0":
            reset_to_regime(s, "gen0", rep=900 + w)
        s.step()
    barrier()
    launches_before = eng.launches
    prev_mu = torch.empty_like(s.parents)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    gen_ms_l, k1_ms_l, local_steps, wall = timed_generations(s, args.steps, flush, barrier, gen0=args.regime == "gen0", keep_prev_mu=prev_mu)
    clocks = sampler.stop() if rank == 0 else None
    launches = eng.launches - launches_before
    best = float(s.best_reward().item())
    gen_ms, k1_ms, k1_mean_ms, total_steps = reduce_over_ranks(dev, world, gen_ms_l, k1_ms_l, local_steps)
    k1_rank_ms = {"max": k1_ms / args.steps, "mean": k1_mean_ms / args.steps}
    if s.exchange == "peer":
        eng.peer_check()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"fitness": s.fitness, "rank_order": s.order, "shaped_fitness": s.shaped},
                     {"mu": s.parents[0], "adam_m": s.m, "adam_v": s.v})

    # ---------------- N > 1: every rank must hold the same bits, and a sample of the last generation must equal a 1-GPU rollout
    rank_consistency = None
    if world > 1:
        sums = torch.stack([bits_checksum(x) for x in (s.parents, s.m, s.v, s.order, s.fitness, s.shaped)])
        allsums = [torch.empty_like(sums) for _ in range(world)]
        dist.all_gather(allsums, sums)
        identical = all(bool(torch.equal(a, allsums[0])) for a in allsums)
        sample_equal, n_sample = None, min(512, args.pop)
        if rank == 0:
            from simple_es_b200.engine import RolloutEngine
            chk = RolloutEngine("CartPole-v1", 4, 2, False, False, 500, E_DEFAULT, args.pop, args.pop, 1, 1, seed=0, device=local,
                                id_begin=0, id_end=n_sample)
            fit1, _ = chk.rollout(s.generation - 1, s.last_sigma, prev_mu)
            torch.cuda.synchronize()
            sample_equal = bool(torch.equal(fit1[:n_sample], s.fitness[:n_sample]))
            chk.close()
        barrier()
        rank_consistency = {"identical": identical, "sample_equal": sample_equal,
                            "checked": "bit checksums of mu, Adam m, Adam v, rank order, fitness[P] and shaped fitness[P] after the last timed "
                                       "generation, all-gathered from %d ranks; fitness of offspring 0..%d of that generation recomputed on rank 0 "
                                       "alone by a single-GPU engine (same mu, sigma, seed, generation) and compared bit for bit with the exchanged vector"
                                       % (world, n_sample - 1)}

    # ---------------- the other regimes of the headline workload (SURVEY 8d: generation-0 and converged reported separately)
    regimes = {args.regime: regime_block(gen_ms, k1_ms, total_steps, args.steps, args.pop)}
    if not args.no_regimes:
        k_other = args.steps
        for reg in ("converged", "gen0", "from_scratch"):
            if reg in regimes:
                continue
            reset_to_regime(s, reg)
            for w in range(3):
                if reg == "gen0":
                    reset_to_regime(s, "gen0", rep=900 + w)
                s.step()
            if reg == "from_scratch":
                for _ in range(max(0, args.warmup - 3)):
                    s.step()
            g, k1, n, _ = timed_generations(s, k_other, flush, barrier, gen0=reg == "gen0")
            g, k1, _, n = reduce_over_ranks(dev, world, g, k1, n)
            regimes[reg] = regime_block(g, k1, n, k_other, args.pop)
        if s.exchange == "peer":
            eng.peer_check()
    n_local = eng.n_local
    del loop, s, eng
    torch.cuda.synchronize()

    # ---------------- e2e: THE SAME generations with HOST buffers, copies inside the timed region (wall clock, max over ranks)
    e2e = None
    P = args.pop
    if world == 1:
        # the reference-facing C-ABI call: ses_generation_openai_host (H2D mu/m/v, K1-K3, D2H fitness[P] + mu/m/v + steps)
        import numpy as np
        from simple_es_b200.engine import RolloutEngine
        eng2 = RolloutEngine("CartPole-v1", 4, 2, False, False, 500, E_DEFAULT, P, P, 1, 1, seed=0, device=local)
        pin = lambda n_, dt: torch.empty(n_, dtype=dt).pin_memory().numpy()
        mu, m, v = pin(D, torch.float32), pin(D, torch.float32), pin(D, torch.float32)
        fit = pin(P, torch.float64)
        reps = []
        for rep in range(2):                          # two passes over the same generations; the better one is reported
            if args.regime == "converged":
                st = bench_state()
                mu[:] = st["mu"]; m[:] = st["m"]; v[:] = st["v"]
                sigma, t, g0 = st["sigma"], st["t"], 30
            else:
                mu[:] = 0; m[:] = 0; v[:] = 0
                sigma, t, g0 = STRATEGY["init_sigma"], 0, 0

            def host_gen(g, sigma, t):
                return eng2.generation_openai_host(g, sigma, STRATEGY["learning_rate"], t, mu, m, v, fit)
            for w in range(args.warmup):
                if args.regime == "gen0":
                    mu[:] = 0; m[:] = 0; v[:] = 0
                    host_gen(900 + w, STRATEGY["init_sigma"], 1)
                else:
                    t += 1; host_gen(g0, sigma, t); sigma *= STRATEGY["sigma_decay"]; g0 += 1
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            tot = 0
            for k in range(args.steps):
                if args.regime == "gen0":
                    mu[:] = 0; m[:] = 0; v[:] = 0
                    tot += host_gen(1000 + k, STRATEGY["init_sigma"], 1)
                else:
                    t += 1; tot += host_gen(g0, sigma, t); sigma *= STRATEGY["sigma_decay"]; g0 += 1
            torch.cuda.synchronize()
            reps.append((time.perf_counter() - t0, tot))
        dt, tot = min(reps)
        e2e = {"value": tot / dt, "unit": "env-steps/s", "h2d_bytes_per_step": 3 * D * 4, "d2h_bytes_per_step": P * 8 + 3 * D * 4 + 8,
               "api": "ses_generation_openai_host (C ABI, pinned host buffers, synchronous)", "n_gpus": 1, "env_steps": tot,
               "generations_per_sec": args.steps / dt, "same_generations_as_value": tot == total_steps,
               "note": "the generations `value` was measured on, replayed through the host-buffer call (the engine is deterministic: "
                       "env_steps equals the device-timed run's); wall clock around K synchronous calls, L2 not flushed in between"}
        eng2.close()
    else:
        # N ranks: a fresh strategy replays the same generations; every rank stages mu/m/v from pinned host memory, runs its
        # shard of the generation through the public strategy API, and reads the full fitness vector + mu/m/v back to the host
        loop2 = make_loop(args, local, args.steps + args.warmup)
        s2 = loop2.strategy
        reset_to_regime(s2, args.regime)
        pinned = lambda n_, dt: torch.empty(n_, dtype=dt).pin_memory()
        mu_h, m_h, v_h, fit_h = pinned(D, torch.float32), pinned(D, torch.float32), pinned(D, torch.float32), pinned(P, torch.float64)

        def host_step():
            s2.parents[0].copy_(mu_h, non_blocking=True); s2.m.copy_(m_h, non_blocking=True); s2.v.copy_(v_h, non_blocking=True)
            s2.step()
            fit_h.copy_(s2.fitness, non_blocking=True)
            mu_h.copy_(s2.parents[0], non_blocking=True); m_h.copy_(s2.m, non_blocking=True); v_h.copy_(s2.v, non_blocking=True)
            torch.cuda.synchronize()
        mu_h.copy_(s2.parents[0]); m_h.copy_(s2.m); v_h.copy_(s2.v)
        torch.cuda.synchronize()
        for w in range(args.warmup):
            if args.regime == "gen0":
                reset_to_regime(s2, "gen0", rep=900 + w); mu_h.zero_(); m_h.zero_(); v_h.zero_()
            host_step()
        steps0 = int(s2.total_env_steps.item())
        barrier()
        t0 = time.perf_counter()
        for k in range(args.steps):
            if args.regime == "gen0":
                reset_to_regime(s2, "gen0", rep=1000 + k); mu_h.zero_(); m_h.zero_(); v_h.zero_()
            host_step()
        barrier()
        dt = time.perf_counter() - t0
        tt = torch.tensor([dt], dtype=torch.float64, device=dev)
        nn = torch.tensor([int(s2.total_env_steps.item()) - steps0], dtype=torch.int64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dist.all_reduce(nn, op=dist.ReduceOp.SUM)
        if s2.exchange == "peer":
            s2.engine.peer_check()
        e2e = {"value": int(nn[0]) / float(tt[0]), "unit": "env-steps/s", "h2d_bytes_per_step": 3 * D * 4,
               "d2h_bytes_per_step": P * 8 + 3 * D * 4,
               "api": "B200Loop.strategy.step() per rank with pinned host staging of mu/m/v (H2D) and fitness[P] + mu/m/v (D2H), "
                      "synchronous; bytes are per rank", "n_gpus": world, "env_steps": int(nn[0]),
               "generations_per_sec": args.steps / float(tt[0]), "same_generations_as_value": int(nn[0]) == total_steps,
               "note": "a fresh strategy replays the generations `value` was measured on (same state, same warm-up); wall clock, max over ranks"}
        del loop2, s2
        torch.cuda.synchronize()

    # ---------------- the other BASELINE configs (N = 1: all of them; N > 1: the 8-GPU scaling config)
    extra = None
    if not args.no_extra:
        extra = {}
        for key, path, overrides, note in EXTRA_CONFIGS:
            if world > 1 and not key.startswith("c5"):
                continue
            try:
                extra[key] = run_extra_config(key, path, overrides, note, local, world, args.extra_steps, 3, flush, barrier, args)
            except Exception as exc:  # pragma: no cover
                extra[key] = {"error": "%s: %s" % (type(exc).__name__, exc)}
            barrier()

    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return 0
    peak_tf = measure_fp32_peak(local)
    achieved_tf = local_steps * FLOP_PER_STEP / (k1_ms_l * 1e-3) / 1e12 if k1_ms_l > 0 else 0.0
    value = total_steps / (gen_ms * 1e-3)
    line = {
        "metric": "env-steps/sec", "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": gen_ms / args.steps, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32 policy / f64 physics", "data": "synthetic",
        "config": workload_config(args, world),
        "per_gpu": value / world, "generations_per_sec": args.steps / (gen_ms * 1e-3), "env_steps": total_steps,
        "best_reward_last_gen": best, "wall_s": wall, "k1_ms_per_generation_over_ranks": k1_rank_ms,
        "regimes": regimes,
        "roofline": {"bound": "fp32_pipe", "kernel": K1_SYMBOL, "achieved": achieved_tf, "peak": peak_tf,
                     "unit": "TFLOP/s", "frac": achieved_tf / peak_tf if peak_tf else None, "traffic": K1_DRAM_BYTES_PER_LAUNCH,
                     "traffic_source": "dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full` capture of K1 (%s); "
                                       "algorithmic bytes per launch: 904 B of parameters + 16 B per offspring of results" % K1_PROFILE,
                     "peak_source": "measured live: dependent-free FFMA microbenchmark on this GPU (MEASURED_PEAKS.json has only HBM and bf16-tensor peaks)",
                     "algorithmic": "%d FP32 FLOP per env step (SURVEY 8d) x %d env steps of rank 0 / %.3f ms in K1 on rank 0" % (FLOP_PER_STEP, local_steps, k1_ms_l),
                     "frac_ceiling": FLOP_PER_STEP / float(2 * FMA_LANE_OPS_PER_STEP),
                     "frac_ceiling_note": "the 418 algorithmic FLOP exclude the 32 float32 tanh per env step, each 14 FMA-pipe operations in the bit-reproducible "
                                          "contract: 640 executed FMA-pipe lane operations (1280 FLOP-equivalents) per env step, so `frac` cannot exceed 418 / 1280 = 0.33; "
                                          "`fma_pipe_frac` is the executed share and compares with ncu's sm__pipe_fmaheavy_cycles_active",
                     "k1_share_of_step": k1_ms / gen_ms if gen_ms else None,
                     "fma_pipe_frac": (local_steps * FMA_LANE_OPS_PER_STEP * 2 / (k1_ms_l * 1e-3) / 1e12 / peak_tf) if (peak_tf and k1_ms_l > 0) else None,
                     "fma_pipe_note": "share of the FP32 FMA pipe K1 keeps busy: 640 FMA-pipe lane operations per env step (the 418 algorithmic "
                                      "FLOP count no tanh; an accurate float32 tanh costs 14 FMA-pipe operations) x 2 FLOP / measured FFMA peak"},
        "clocks": clocks, "e2e": e2e, "gpu_launches": launches,
    }
    if rank_consistency is not None:
        line["rank_consistency"] = rank_consistency
    if extra is not None:
        line["extra_configs"] = extra
    line["roofline"]["hbm_check"] = hbm_check(n_local, k1_ms_l / args.steps if args.steps else 0.0)
    if world == 1 and not args.no_cpu:
        try:
            line["cpu_baseline"] = cpu_baseline_block(os.cpu_count() or 1)
        except Exception as exc:  # pragma: no cover
            line["cpu_baseline"] = {"error": str(exc)}
    print(json.dumps(line))
    if rank_consistency is not None and not (rank_consistency["identical"] and rank_consistency["sample_equal"]):
        sys.stderr.write("bench.py: ranks disagree after the timed generations: %r\n" % (rank_consistency,))
        return 3
    return 0


def hbm_check(n_local, k1_ms_per_launch):
    """Why `roofline.bound` is not "hbm": K1's ALGORITHMIC bytes per launch (904 B of parameters read + 16 B of results
    written per offspring, DESIGN.md section 3) over its measured duration, against the measured HBM peak of
    MEASURED_PEAKS.json (driver-written; fallback 6650 GB/s per B200_PROFILING.md)."""
    try:
        alg = D * 4 + 16 * int(n_local)
        peak, src = 6650.0, "of fallback (B200_PROFILING.md)"
        path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(path):
            with open(path) as f:
                peak, src = float(json.load(f)["hbm_gbs"]), "of measured (MEASURED_PEAKS.json hbm_gbs)"
        gbs = alg / (k1_ms_per_launch * 1e-3) / 1e9 if k1_ms_per_launch > 0 else 0.0
        return {"algorithmic_bytes_per_launch": alg, "achieved_gbs": gbs, "peak_gbs": peak, "peak_source": src,
                "frac": gbs / peak, "note": "K1 is five orders of magnitude below the HBM roofline and uses no tensor-core "
                "shaped work (per-offspring weights: GEMV only); the FP32 pipe is the bound that applies"}
    except Exception as exc:  # pragma: no cover
        return {"error": str(exc)}


def measure_fp32_peak(device):
    """FFMA microbenchmark (library test hook) -> TFLOP/s; None if the hook is missing."""
    try:
        import ctypes as C
        from simple_es_b200 import _lib
        lib = _lib.load()
        out = C.c_double(0.0)
        _lib.check(lib.ses_measure_fp32_peak(int(device), C.byref(out)))
        return out.value
    except Exception:
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100,
                    help="timed generations of the headline workload (and of each of its other regimes)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--pop", type=int, default=P_DEFAULT)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--regime", default="converged", choices=["converged", "from_scratch", "gen0"],
                    help="policy regime of the headline `value` (SURVEY 8d); the other two are reported under `regimes`")
    ap.add_argument("--no-regimes", action="store_true", help="skip the other regimes of the headline workload")
    ap.add_argument("--no-extra", action="store_true", help="skip the other BASELINE configs (`extra_configs`)")
    ap.add_argument("--extra-steps", type=int, default=10, help="timed generations per extra config")
    ap.add_argument("--exchange", default=os.environ.get("SES_FITNESS_EXCHANGE", "peer"), choices=["peer", "nccl"],
                    help="N > 1: fitness exchange fused into K1 over NVLink peer memory (default) or an NCCL all-gather")
    ap.add_argument("--shard", default="cyclic", choices=["cyclic", "contiguous"],
                    help="N > 1: block-cyclic (default) or contiguous offspring-id ranges per rank")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed generations, write what the last one computed (fitness, rank order, shaped fitness, "
                         "mu, Adam m and v) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3
    if args.impl == "reference":
        return run_reference(args)
    return run_b200(args)


if __name__ == "__main__":
    sys.exit(main())

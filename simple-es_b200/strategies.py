"""Device-resident strategy state for the offspring strategies: the reference's three, and three opt-in additions: nsr_es
(novelty search with reward), sep_cma_es (separable CMA-ES) and map_elites (MAP-Elites).

Each class keeps what the reference strategy keeps (learning_strategies/evolution/offspring_strategies.py)
-- mu / elite table, sigma, Adam moments -- as a few small CUDA tensors, and never materialises the
population: offspring i of generation g is (parent(i), sigma, Philox(seed, g, i)).  `step()` is one
generation: K1 rollout of this rank's slice, fitness exchange, K2 rank, K3 update -- the GPU form of
``results = p.map(RolloutWorker, ...); strategy.evaluate(results)`` (loop.py:66-84).
"""
import math

import torch

from . import dist as sdist
from .engine import ENV_SPECS, RolloutEngine, cyclic_block, map_spec, owned_ids, population_layout, sep_cma_constants, shard_bounds


class _Base:
    name = None

    def __init__(self, strategy_cfg, env_cfg, network_cfg, eval_ep_num, seed, device, engine_cfg):
        rank, ws = sdist.world()
        self.cfg = strategy_cfg
        self.engine_cfg = engine_cfg
        self.sigma = float(strategy_cfg["init_sigma"])           # sigma the CURRENT population was drawn with
        self.curr_sigma = self.sigma                              # what the reference reports (post-decay)
        self.decay = float(strategy_cfg["sigma_decay"])
        self.n = int(strategy_cfg["offspring_num"])
        self.k = int(strategy_cfg.get("elite_num", 1))
        self.P, group, n_head, n_par = population_layout(self.name, self.n, self.k)
        self.lo, self.hi = shard_bounds(self.P, rank, ws)
        # engine.shard: "cyclic" (default with several ranks: blocks of <= 256 consecutive ids dealt round robin, so that
        # ranks stay balanced when neighbouring offspring behave alike -- simple_genetic keeps each elite's offspring
        # together) or "contiguous" (one id range per rank)
        mode = engine_cfg.get("shard", "cyclic") if ws > 1 else "contiguous"
        if mode not in ("cyclic", "contiguous"):
            raise ValueError("engine.shard must be 'cyclic' or 'contiguous'")
        self.shard = (rank, ws, cyclic_block(self.P, ws)) if mode == "cyclic" else None
        name = env_cfg["name"]
        self.engine = RolloutEngine(
            name, int(network_cfg["num_state"]), int(network_cfg["num_action"]), bool(network_cfg["gru"]),
            bool(env_cfg.get("pomdp", False)), env_cfg.get("max_step"), eval_ep_num, self.P, group, n_head, n_par,
            seed=seed, init_mode=engine_cfg.get("init_states", "shared"), n_agents=int(engine_cfg.get("n_agents", 2)),
            id_begin=0 if self.shard else self.lo, id_end=None if self.shard else self.hi, device=device,
            antithetic=bool(engine_cfg.get("antithetic", False)), shard=self.shard,
            discrete_action=bool(network_cfg.get("discrete_action", True)))
        self.D = self.engine.D
        # what a resumed run must share with the run that wrote the state (state() / load_state())
        self._run_key = {"env": name, "seed": int(seed) & 0xFFFFFFFF, "eval_ep_num": int(eval_ep_num),
                         "init_states": engine_cfg.get("init_states", "shared"), "antithetic": bool(engine_cfg.get("antithetic", False)),
                         "max_step": self.engine.max_step, "gru": bool(network_cfg["gru"]), "pomdp": bool(env_cfg.get("pomdp", False))}
        dev = self.engine.device
        self.parents = torch.zeros(n_par, self.D, dtype=torch.float32, device=dev)   # network.zero_init() (loop.py:31)
        # fitness exchange: "peer" = K1 stores fitness into every rank's buffer over NVLink + flag barrier (default);
        # "nccl" = all-gather after K1 (baseline).  Two buffers, alternating by generation parity (peer mode).
        self.exchange = engine_cfg.get("fitness_exchange", "peer") if ws > 1 else "local"
        if self.exchange == "peer":
            import torch.distributed as tdist

            def gather(b):
                out = [None] * ws
                tdist.all_gather_object(out, b)
                return out
            self._fit = self.engine.peer_setup(rank, ws, gather)
            tdist.barrier()
        elif self.exchange in ("nccl", "local"):
            self._fit = [torch.zeros(self.P, dtype=torch.float64, device=dev)] * 2
        else:
            raise ValueError("engine.fitness_exchange must be 'peer' or 'nccl'")
        if self.shard and self.exchange == "nccl":
            mask = torch.ones(self.P, dtype=torch.bool)
            mask[torch.from_numpy(owned_ids(self.P, *self.shard))] = False
            self._not_mine = mask.to(dev)
        self.fitness = self._fit[0]
        self.steps = torch.zeros(self.P, dtype=torch.int64, device=dev)
        self.order = torch.empty(self.P, dtype=torch.int32, device=dev)
        self.generation = 0
        self.total_env_steps = torch.zeros(1, dtype=torch.int64, device=dev)     # accumulated by K1 itself
        self.engine.set_step_counter(self.total_env_steps)
        # CUDA-event phase marks of a generation (start / after K1 + exchange / end).  B200Loop reads them after its one
        # host sync per generation to fill the reference's `rollout_t` / `eval_t` fields (loop.py:70-91) with device times
        # instead of adding host syncs between the phases.
        self.timing = False
        self._ev = None

    def _mark(self, i):
        if self.timing:
            if self._ev is None:
                self._ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            self._ev[i].record(torch.cuda.current_stream(self.engine.device))

    def phase_times(self):
        """(rollout seconds, evaluate seconds) of the last step(); call after the stream has been synchronised
        (B200Loop does so by reading best_reward).  None unless `timing` was on during that step."""
        if not self.timing or self._ev is None:
            return None
        return self._ev[0].elapsed_time(self._ev[1]) * 1e-3, self._ev[1].elapsed_time(self._ev[2]) * 1e-3

    def _rollout_and_exchange(self):
        """K1 on this rank's slice, then the full fitness vector on every rank."""
        e = self.engine
        self._mark(0)
        self.fitness = self._fit[self.generation & 1]
        e.rollout(self.generation, self.sigma, self.parents, fitness=self.fitness, steps=self.steps)
        self.exchange_fitness()
        self._mark(1)

    def exchange_fitness(self):
        """After K1: make the full fitness vector visible on every rank."""
        if self.exchange == "peer":
            self.engine.peer_barrier()                 # the values were stored into every peer's buffer by K1 itself
        elif self.exchange == "nccl":
            if self.shard:
                sdist.exchange_fitness_masked(self.fitness, self._not_mine)
            else:
                sdist.exchange_fitness(self.fitness, self.lo, self.hi)

    def _final_state_output(self):
        """Have K1 store every episode's final state (nsr_es, map_elites): final_states [P, E, state_dim] and the behaviours
        bc [P, state_dim] that _behaviors() computes from them."""
        e, dev = self.engine, self.engine.device
        self.final_states = torch.zeros((self.P, e.E, e.state_dim), dtype=torch.float64, device=dev)
        e.set_final_states(self.final_states)
        self.bc = torch.empty((self.P, e.state_dim), dtype=torch.float64, device=dev)
        if self.shard and not hasattr(self, "_not_mine"):
            mask = torch.ones(self.P, dtype=torch.bool)
            mask[torch.from_numpy(owned_ids(self.P, *self.shard))] = False
            self._not_mine = mask.to(dev)

    def _behaviors(self):
        """After K1: every rank's final states on every rank, exactly, then bc := their means over episodes."""
        if sdist.world()[1] > 1:                       # every rank gets every row, exactly; then all compute the same
            if self.shard:
                sdist.exchange_fitness_masked(self.final_states, self._not_mine)
            else:
                sdist.exchange_fitness(self.final_states, self.lo, self.hi)
        self.engine.behavior(self.final_states, out=self.bc)

    def _rollout_and_rank(self, shaped=False):
        self._rollout_and_exchange()
        return self.engine.rank_desc(self.fitness, shaped=shaped, order=self.order)

    # ------------------------------------------------------------------ resume (SURVEY.md section 8f rank 1)
    def state(self):
        """Everything needed to continue this run bit for bit: the reference cannot resume (it only saves the elite's
        state_dict, loop.py:101-104); populations are functions of (parents, sigma, seed, generation) here."""
        st = {"strategy": self.name, "generation": self.generation, "sigma": self.sigma, "curr_sigma": self.curr_sigma,
              "parents": self.parents.detach().cpu().clone(), "population": self.P, "run_key": dict(self._run_key),
              "total_env_steps": int(self.total_env_steps.item())}
        for k in ("m", "v"):
            if hasattr(self, k):
                st[k] = getattr(self, k).detach().cpu().clone()
        if hasattr(self, "t"):
            st["t"] = self.t
        return st

    def load_state(self, st):
        if st.get("strategy") != self.name or tuple(st["parents"].shape) != tuple(self.parents.shape):
            raise ValueError("resume state is for strategy %r with parents %s; this run is %r with parents %s"
                             % (st.get("strategy"), tuple(st["parents"].shape), self.name, tuple(self.parents.shape)))
        if int(st.get("population", self.P)) != self.P:
            raise ValueError("resume state is for a population of %d, this run has %d" % (int(st["population"]), self.P))
        # populations are functions of (parents, sigma, seed, generation) and fitness of (env, E, initial states): a resumed
        # run continues the old one bit for bit only if all of these are the same (ADVICE r1)
        theirs = st.get("run_key")
        if theirs is not None:
            diff = {k: (theirs.get(k), v) for k, v in self._run_key.items() if theirs.get(k) != v}
            if diff:
                raise ValueError("resume state was written by a different run: " +
                                 ", ".join("%s was %r, now %r" % (k, a, b) for k, (a, b) in sorted(diff.items())))
        if "total_env_steps" in st:
            self.total_env_steps.fill_(int(st["total_env_steps"]))
        self.generation = int(st["generation"])
        self.sigma, self.curr_sigma = float(st["sigma"]), float(st["curr_sigma"])
        self.parents.copy_(st["parents"])
        for k in ("m", "v"):
            if hasattr(self, k):
                getattr(self, k).copy_(st[k])
        if hasattr(self, "t"):
            self.t = int(st["t"])

    def load_elite(self, flat):
        """Start from a saved policy (a reference-format checkpoint): every parent row := flat."""
        flat = torch.as_tensor(flat, dtype=torch.float32).reshape(-1)
        if flat.numel() != self.D:
            raise ValueError("checkpoint has %d parameters, the configured network has %d" % (flat.numel(), self.D))
        self.parents.copy_(flat.to(self.parents.device).expand_as(self.parents))

    def best_reward(self):
        """max(rewards) (offspring_strategies.py:113,235,381) -- a 0-d device tensor."""
        return self.fitness[self.order[0].long()]

    def elite_flat(self):
        raise NotImplementedError

    def step(self):
        raise NotImplementedError


class OpenAIES(_Base):
    """offspring_strategies.py:270-434 + optimizers.py:30-57."""
    name = "openai_es"

    def __init__(self, *a, **kw):
        super().__init__(*a, **kw)
        self.lr = float(self.cfg["learning_rate"])
        dev = self.engine.device
        self.m = torch.zeros(self.D, dtype=torch.float32, device=dev)
        self.v = torch.zeros(self.D, dtype=torch.float32, device=dev)
        self.t = 0
        self.shaped = torch.empty(self.P, dtype=torch.float64, device=dev)
        # engine.optimizer: "adam" (the reference's only optimizer, optimizers.py:30-57) or, opt-in, "sgd" with
        # engine.momentum (the SGD of the OpenAI file optimizers.py names as its source; uses v only)
        self.optimizer = self.engine_cfg.get("optimizer", "adam")
        if self.optimizer not in ("adam", "sgd"):
            raise ValueError("engine.optimizer must be 'adam' or 'sgd'")
        self.momentum = float(self.engine_cfg.get("momentum", 0.9))

    def step(self):
        self._rollout_and_exchange()
        self.engine.rank_desc(self.fitness, shaped=True, order=self.order, shaped_out=self.shaped)
        self._update()

    def _update(self):
        """K3 from self.shaped, then the sigma decay and the next generation."""
        e = self.engine
        self.t += 1
        if self.optimizer == "sgd":
            e.update_openai_sgd(self.generation, self.sigma, self.lr, self.shaped, self.parents.view(-1), self.v, self.momentum)
        else:
            e.update_openai(self.generation, self.sigma, self.lr, self.t, self.shaped, self.parents.view(-1), self.m, self.v)
        self.sigma *= self.decay                                  # :418, after update_factor used the old sigma
        self.curr_sigma = self.sigma
        self.generation += 1
        self._mark(2)

    def elite_flat(self):
        return self.parents[0]                                    # get_elite_model() is mu_model (:330-331)


class SimpleEvolution(_Base):
    """offspring_strategies.py:137-267 (quirk Q2: the stored elite is the mean)."""
    name = "simple_evolution"

    def step(self):
        e = self.engine
        self._rollout_and_rank()
        new_mu = e.elite_mean(self.generation, self.sigma, self.parents, self.order, self.k)
        self.parents[0].copy_(new_mu)
        self.sigma *= self.decay                                  # :251, BEFORE regenerating
        self.curr_sigma = self.sigma
        self.generation += 1
        self._mark(2)

    def elite_flat(self):
        return self.parents[0]                                    # elite_models[0] was overwritten by the mean (Q2)


class SimpleGenetic(_Base):
    """offspring_strategies.py:11-134."""
    name = "simple_genetic"

    def step(self):
        e = self.engine
        self._rollout_and_rank()
        elites = e.materialize(self.generation, self.sigma, self.parents, self.order[:self.k].contiguous())
        self.parents.copy_(elites)
        # the next population is regenerated with the CURRENT sigma, then sigma decays (:117-124):
        # population g+1 was drawn with the sigma reported after generation g-1.
        self.sigma = self.curr_sigma
        self.curr_sigma = self.curr_sigma * self.decay
        self.generation += 1
        self._mark(2)

    def elite_flat(self):
        return self.parents[0]                                    # elite_models[0] (:64-65)


def _novelty_params(cfg):
    """(novelty_weight, novelty_k) of an nsr_es strategy section, validated."""
    allowed = {"name", "init_sigma", "sigma_decay", "learning_rate", "offspring_num", "novelty_weight", "novelty_k"}
    unknown = sorted(set(cfg) - allowed)
    if unknown:
        raise ValueError("strategy nsr_es: unknown key(s) %s (allowed: %s)" % (", ".join(unknown), ", ".join(sorted(allowed))))
    w, k = cfg.get("novelty_weight", 0.5), cfg.get("novelty_k", 10)
    if isinstance(w, bool) or not isinstance(w, (int, float)) or not 0.0 <= float(w) <= 1.0:
        raise ValueError("strategy nsr_es: novelty_weight must be a number in [0, 1] (got %r)" % (w,))
    if isinstance(k, bool) or not isinstance(k, int) or not 1 <= k <= 32:
        raise ValueError("strategy nsr_es: novelty_k must be an integer in [1, 32] (got %r)" % (k,))
    return float(w), int(k)


class NoveltyES(OpenAIES):
    """openai_es plus novelty (NSR-ES, Conti et al. 2018; opt-in, the reference has no such strategy).  The same population,
    update and sigma decay as openai_es, but K3 follows (1 - w) * the centered ranks of fitness + w * the centered ranks of
    novelty.  An offspring's behaviour is the mean of its episodes' final states; its novelty is the mean distance to the k
    nearest behaviours in the archive, which holds mu's behaviour of every generation so far (DESIGN.md section 4.10).
    w = 0 trains exactly as openai_es."""
    name = "nsr_es"

    def __init__(self, strategy_cfg, *a, **kw):
        self.novelty_weight, self.novelty_k = _novelty_params(strategy_cfg)
        super().__init__(strategy_cfg, *a, **kw)
        e, dev = self.engine, self.engine.device
        self._run_key.update(novelty_k=self.novelty_k, novelty_weight=self.novelty_weight)
        self._final_state_output()
        self.novelty = torch.empty(self.P, dtype=torch.float64, device=dev)
        self.novelty_order = torch.empty(self.P, dtype=torch.int32, device=dev)
        self.shaped_f = torch.empty(self.P, dtype=torch.float64, device=dev)
        self.shaped_n = torch.empty(self.P, dtype=torch.float64, device=dev)
        self.archive = torch.empty((16, e.state_dim), dtype=torch.float64, device=dev)   # grows by doubling
        self.n_archive = 0

    def _reserve(self, n):
        if n > self.archive.shape[0]:
            grown = torch.empty((max(16, 1 << (n - 1).bit_length()), self.archive.shape[1]), dtype=torch.float64,
                                device=self.archive.device)
            grown[:self.n_archive].copy_(self.archive[:self.n_archive])
            self.archive = grown

    def step(self):
        e = self.engine
        self._rollout_and_exchange()                   # K1 also stores every episode's final state (set_final_states)
        self._behaviors()
        self._reserve(self.n_archive + 1)
        self.archive[self.n_archive].copy_(self.bc[0])   # mu's behaviour joins the archive before novelty is measured
        self.n_archive += 1
        e.novelty(self.bc, self.archive, self.n_archive, self.novelty_k, out=self.novelty)
        e.rank_desc(self.fitness, shaped=True, order=self.order, shaped_out=self.shaped_f)
        e.rank_desc(self.novelty, shaped=True, order=self.novelty_order, shaped_out=self.shaped_n, full_key=True)
        e.blend_shaped(self.shaped_f, self.shaped_n, self.novelty_weight, out=self.shaped)
        self._update()

    def state(self):
        st = super().state()
        st["archive"] = self.archive[:self.n_archive].detach().cpu().clone()
        return st

    def load_state(self, st):
        super().load_state(st)
        a = st["archive"]
        if a.dim() != 2 or a.shape[1] != self.archive.shape[1]:
            raise ValueError("resume state has an archive of shape %s, this run needs [n, %d]" % (tuple(a.shape), self.archive.shape[1]))
        self.n_archive = 0
        self._reserve(a.shape[0])
        self.archive[:a.shape[0]].copy_(a)
        self.n_archive = int(a.shape[0])


def _cma_params(cfg):
    """(offspring_num, elite_num, init_sigma) of a sep_cma_es strategy section, validated."""
    allowed = {"name", "init_sigma", "offspring_num", "elite_num"}
    unknown = sorted(set(cfg) - allowed)
    if unknown:
        raise ValueError("strategy sep_cma_es: unknown key(s) %s (allowed: %s)" % (", ".join(unknown), ", ".join(sorted(allowed))))
    sigma, lam = cfg.get("init_sigma"), cfg.get("offspring_num")
    if isinstance(sigma, bool) or not isinstance(sigma, (int, float)) or not float(sigma) > 0.0 or sigma == float("inf"):
        raise ValueError("strategy sep_cma_es: init_sigma must be a finite number > 0 (got %r)" % (sigma,))
    if isinstance(lam, bool) or not isinstance(lam, int) or lam < 2:
        raise ValueError("strategy sep_cma_es: offspring_num must be an integer >= 2 (got %r)" % (lam,))
    mu = cfg.get("elite_num", lam // 2)
    if isinstance(mu, bool) or not isinstance(mu, int) or not 1 <= mu <= lam:
        raise ValueError("strategy sep_cma_es: elite_num must be an integer in [1, offspring_num = %d] (got %r)" % (lam, mu))
    return lam, mu, float(sigma)


class SepCMAES(_Base):
    """Separable CMA-ES (Ros & Hansen 2008; opt-in, the reference has no such strategy): every offspring is drawn from
    N(m, sigma^2 diag(c)), and the mu best recombine into the new mean, the evolution paths, the diagonal c and sigma.  The
    state (m, c, p_sigma, p_c, sigma) is float64 and lives on the device; the samples are the w_override table K1 rolls out
    (DESIGN.md section 4.11)."""
    name = "sep_cma_es"

    def __init__(self, strategy_cfg, env_cfg, network_cfg, eval_ep_num, seed, device, engine_cfg):
        lam, mu, sigma = _cma_params(strategy_cfg)
        if engine_cfg.get("antithetic", False):
            raise ValueError("sep_cma_es does not support engine.antithetic: mirrored samples bias its step-size adaptation")
        super().__init__(dict(strategy_cfg, sigma_decay=1.0, elite_num=mu), env_cfg, network_cfg, eval_ep_num, seed, device, engine_cfg)
        dev = self.engine.device
        self.mu = mu
        self.consts = sep_cma_constants(self.D, self.P, mu)
        self._run_key.update(elite_num=mu)
        self.weights = torch.from_numpy(self.consts["weights"]).to(dev)
        self.mean = torch.zeros(self.D, dtype=torch.float64, device=dev)
        self.c = torch.ones(self.D, dtype=torch.float64, device=dev)
        self.p_sigma = torch.zeros(self.D, dtype=torch.float64, device=dev)
        self.p_c = torch.zeros(self.D, dtype=torch.float64, device=dev)
        self.sigma_dev = torch.full((1,), sigma, dtype=torch.float64, device=dev)
        self.s = torch.empty(self.P, dtype=torch.float64, device=dev)
        self.samples = torch.empty((self.engine.n_local, self.D), dtype=torch.float32, device=dev)

    @property
    def curr_sigma(self):
        """sigma of the next generation: the device value (B200Loop reads it after its one sync per generation)."""
        return float(self.sigma_dev.item()) if hasattr(self, "sigma_dev") else self.sigma

    @curr_sigma.setter
    def curr_sigma(self, value):
        if hasattr(self, "sigma_dev"):
            self.sigma_dev.fill_(float(value))

    def step(self):
        e = self.engine
        self._mark(0)
        e.cma_sample(self.generation, self.mean, self.c, self.sigma_dev, out=self.samples)
        self.fitness = self._fit[self.generation & 1]
        e.rollout(self.generation, 0.0, self.parents, fitness=self.fitness, steps=self.steps, w_override=self.samples)
        self.exchange_fitness()
        self._mark(1)
        e.rank_desc(self.fitness, order=self.order)
        e.cma_update(self.generation, self.order, self.consts, self.weights, self.s, self.mean, self.c, self.p_sigma, self.p_c,
                     self.sigma_dev, self.parents[0])
        self.generation += 1
        self._mark(2)

    def elite_flat(self):
        return self.parents[0]                                    # (float)m, written by every update

    def load_elite(self, flat):
        """Start from a saved policy: m := flat, c := 1, both paths := 0 (sigma stays init_sigma)."""
        super().load_elite(flat)
        self.mean.copy_(self.parents[0].double())
        self.c.fill_(1.0)
        self.p_sigma.zero_()
        self.p_c.zero_()

    def state(self):
        st = super().state()
        for k in ("mean", "c", "p_sigma", "p_c", "sigma_dev"):
            st[k] = getattr(self, k).detach().cpu().clone()
        return st

    def load_state(self, st):
        super().load_state(st)
        for k in ("mean", "c", "p_sigma", "p_c", "sigma_dev"):
            if tuple(st[k].shape) != tuple(getattr(self, k).shape):
                raise ValueError("resume state has %s of shape %s, this run needs %s" % (k, tuple(st[k].shape), tuple(getattr(self, k).shape)))
            getattr(self, k).copy_(st[k])


MAP_MAX_CELLS = 1 << 20
MAP_MAX_WEIGHT_BYTES = 1 << 32


def _map_state_dim(env_cfg, engine_cfg):
    name = env_cfg["name"]
    if name not in ENV_SPECS:
        raise ValueError("env %r is not supported by the B200 engine" % (name,))
    sd = ENV_SPECS[name][2]
    return 4 * int(engine_cfg.get("n_agents", 2)) if sd is None else sd


def _map_params(cfg, state_dim, D):
    """(offspring_num, dims, low, high, cells) of a map_elites strategy section, validated against the final-state size
    state_dim and the parameter count D (DESIGN.md section 4.12)."""
    allowed = {"name", "init_sigma", "sigma_decay", "offspring_num", "behavior_dims", "behavior_low", "behavior_high", "behavior_cells"}
    unknown = sorted(set(cfg) - allowed)
    if unknown:
        raise ValueError("strategy map_elites: unknown key(s) %s (allowed: %s)" % (", ".join(unknown), ", ".join(sorted(allowed))))
    missing = sorted(k for k in allowed - {"name"} if k not in cfg)
    if missing:
        raise ValueError("strategy map_elites: missing key(s) %s" % ", ".join(missing))

    def num(x):
        return not isinstance(x, bool) and isinstance(x, (int, float))

    def intg(x):
        return not isinstance(x, bool) and isinstance(x, int)
    n = cfg["offspring_num"]
    if not intg(n) or n < 2:
        raise ValueError("strategy map_elites: offspring_num must be an integer >= 2 (got %r)" % (n,))
    for k in ("init_sigma", "sigma_decay"):
        if not num(cfg[k]) or not math.isfinite(cfg[k]):
            raise ValueError("strategy map_elites: %s must be a finite number (got %r)" % (k, cfg[k]))
    dims, low, high, cells = (cfg[k] for k in ("behavior_dims", "behavior_low", "behavior_high", "behavior_cells"))
    for k, v in (("behavior_dims", dims), ("behavior_low", low), ("behavior_high", high), ("behavior_cells", cells)):
        if not isinstance(v, (list, tuple)) or not 1 <= len(v) <= 4:
            raise ValueError("strategy map_elites: %s must be a list of 1 to 4 entries (got %r)" % (k, v))
    if not len(dims) == len(low) == len(high) == len(cells):
        raise ValueError("strategy map_elites: behavior_dims, behavior_low, behavior_high and behavior_cells must have one entry per "
                         "descriptor dimension (got %d, %d, %d, %d)" % (len(dims), len(low), len(high), len(cells)))
    if not all(intg(d) and 0 <= d < state_dim for d in dims):
        raise ValueError("strategy map_elites: behavior_dims must be indices into the final state [0, %d) (got %r)" % (state_dim, dims))
    if len(set(dims)) != len(dims):
        raise ValueError("strategy map_elites: behavior_dims must be distinct (got %r)" % (dims,))
    for j, (lo, hi) in enumerate(zip(low, high)):
        if not (num(lo) and num(hi) and math.isfinite(lo) and math.isfinite(hi)):
            raise ValueError("strategy map_elites: behavior_low / behavior_high must be finite numbers (dimension %d: %r, %r)" % (j, lo, hi))
        if not float(hi) - float(lo) > 0.0:
            raise ValueError("strategy map_elites: behavior_low must be below behavior_high (dimension %d: %r, %r)" % (j, lo, hi))
    if not all(intg(c) and c >= 1 for c in cells):
        raise ValueError("strategy map_elites: behavior_cells must be integers >= 1 (got %r)" % (cells,))
    n_cells = math.prod(cells)
    if n_cells > MAP_MAX_CELLS:
        raise ValueError("strategy map_elites: %s = %d cells exceed 2^20 = %d" % (" x ".join(map(str, cells)), n_cells, MAP_MAX_CELLS))
    if n_cells * D * 4 > MAP_MAX_WEIGHT_BYTES:
        raise ValueError("strategy map_elites: %d cells x %d parameters x 4 bytes = %d bytes of elite weights exceed 4 GiB = %d"
                         % (n_cells, D, n_cells * D * 4, MAP_MAX_WEIGHT_BYTES))
    return int(n), [int(d) for d in dims], [float(x) for x in low], [float(x) for x in high], [int(c) for c in cells]


class MapElites(_Base):
    """MAP-Elites (Mouret & Clune 2015; opt-in, the reference has no such strategy): an archive of one elite per cell of a grid
    over final-state coordinates.  Every generation, parent row i is the elite of an occupied cell drawn by Philox, offspring i
    is that row + sigma * noise, and the best-ranked offspring of each cell replaces the cell's elite if its fitness is higher.
    The archive (fitness F, behaviour B, birth and weights W of every cell) lives on the device (DESIGN.md section 4.12)."""
    name = "map_elites"

    def __init__(self, strategy_cfg, env_cfg, network_cfg, eval_ep_num, seed, device, engine_cfg):
        from .checkpoint import param_shapes
        D = sum(math.prod(shape) for _, shape in param_shapes(int(network_cfg["num_state"]), int(network_cfg["num_action"]),
                                                             bool(network_cfg["gru"])))
        _, self.dims, self.low, self.high, self.cells = _map_params(strategy_cfg, _map_state_dim(env_cfg, engine_cfg), D)
        if engine_cfg.get("antithetic", False):
            raise ValueError("map_elites does not support engine.antithetic: with one parent row per offspring there are no pairs to mirror")
        super().__init__(strategy_cfg, env_cfg, network_cfg, eval_ep_num, seed, device, engine_cfg)
        e, dev = self.engine, self.engine.device
        self._run_key.update(behavior_dims=list(self.dims), behavior_low=list(self.low), behavior_high=list(self.high),
                             behavior_cells=list(self.cells))
        self._final_state_output()
        self.spec = map_spec(self.dims, self.low, self.high, self.cells)
        self.n_cells = math.prod(self.cells)
        self.F = torch.full((self.n_cells,), float("nan"), dtype=torch.float64, device=dev)
        self.B = torch.full((self.n_cells, e.state_dim), float("nan"), dtype=torch.float64, device=dev)
        self.born = torch.full((self.n_cells, 2), -1, dtype=torch.int32, device=dev)
        self.W = torch.zeros((self.n_cells, self.D), dtype=torch.float32, device=dev)
        self.seed_row = torch.zeros(self.D, dtype=torch.float32, device=dev)     # network.zero_init(), or engine.init_from
        self.stats = torch.zeros(4, dtype=torch.float64, device=dev)
        self._select()

    def _select(self):
        self.engine.map_select(self.generation, self.spec, self.F, self.W, self.seed_row, self.stats, self.parents)

    def step(self):
        e = self.engine
        self._rollout_and_exchange()                   # K1 also stores every episode's final state (set_final_states)
        self._behaviors()
        e.rank_desc(self.fitness, order=self.order)
        e.map_insert(self.generation, self.sigma, self.parents, self.order, self.fitness, self.bc, self.spec, self.F, self.B, self.born, self.W)
        self.sigma *= self.decay
        self.curr_sigma = self.sigma
        self.generation += 1
        self._select()                                 # the parent table of the next generation, and the archive's statistics
        self._mark(2)

    def archive_stats(self):
        """(occupied cells, n_cells, best fitness, QD score) after the last insertion; reads 4 doubles from the device."""
        n_occ, _, best, qd = self.stats.tolist()
        return int(n_occ), self.n_cells, best, qd

    def elite_flat(self):
        c = int(self.stats[1].item())
        return self.W[c] if c >= 0 else self.seed_row

    def load_elite(self, flat):
        """Start from a saved policy: the seed row S := flat (every parent row while the archive is empty)."""
        flat = torch.as_tensor(flat, dtype=torch.float32).reshape(-1)
        if flat.numel() != self.D:
            raise ValueError("checkpoint has %d parameters, the configured network has %d" % (flat.numel(), self.D))
        self.seed_row.copy_(flat.to(self.seed_row.device))
        self._select()

    def archive(self):
        """The occupied cells as CPU tensors: cells [n] i64 ascending, fitness [n] f64, behavior [n, state_dim] f64,
        weights [n, D] f32, born [n, 2] i64 (generation, offspring id)."""
        cells = torch.nonzero(~torch.isnan(self.F)).reshape(-1)
        return {"cells": cells.cpu(), "fitness": self.F[cells].cpu(), "behavior": self.B[cells].cpu(), "weights": self.W[cells].cpu(),
                "born": self.born[cells].to(torch.int64).cpu()}

    def state(self):
        st = super().state()
        st["archive"] = self.archive()
        st["seed_row"] = self.seed_row.detach().cpu().clone()
        return st

    def load_state(self, st):
        super().load_state(st)
        a = st["archive"]
        n = a["cells"].numel()
        if a["weights"].shape != (n, self.D) or a["behavior"].shape != (n, self.B.shape[1]) or n and int(a["cells"].max()) >= self.n_cells:
            raise ValueError("resume state's archive does not fit this run (%d cells of %d parameters)" % (self.n_cells, self.D))
        cells = a["cells"].to(self.F.device)
        self.F.fill_(float("nan"))
        self.B.fill_(float("nan"))
        self.born.fill_(-1)
        self.W.zero_()
        self.F[cells] = a["fitness"].to(self.F.device)
        self.B[cells] = a["behavior"].to(self.B.device)
        self.born[cells] = a["born"].to(self.born.device, torch.int32)
        self.W[cells] = a["weights"].to(self.W.device)
        self.seed_row.copy_(st["seed_row"])
        self._select()


STRATEGIES = {c.name: c for c in (OpenAIES, SimpleEvolution, SimpleGenetic, NoveltyES, SepCMAES, MapElites)}

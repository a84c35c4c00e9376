"""RolloutEngine: torch-tensor front end of the C ABI (include/ses_b200.h).

torch is plumbing only: it owns device memory and the CUDA stream; every computation is one of the
library's own sm_100a kernels.  Replaces, inside one generation of the reference loop
(learning_strategies/evolution/loop.py:61-84):
  * ``p.map(RolloutWorker, arguments)``           -> :meth:`RolloutEngine.rollout`
  * ``np.flip(np.argsort(rewards))`` + shaping     -> :meth:`RolloutEngine.rank_desc`
  * the strategy updates of ``evaluate``          -> :meth:`update_openai`, :meth:`elite_mean`,
                                                     :meth:`materialize`
"""
import ctypes as C
import math
import os

import numpy as np
import torch

from . import _lib

# env.name -> (SES_ENV_*, episode cap, state_dim, (num_state, num_action)); the cap is gym's TimeLimit
# (max_episode_steps of the registered id) or simple_spread_v2's default max_cycles
ENV_SPECS = {
    "CartPole-v1": (0, 500, 4, (4, 2)),
    "CartPole-v0": (0, 200, 4, (4, 2)),          # same physics, TimeLimit 200
    "simple_spread": (1, 25, None, None),
    "MountainCar-v0": (2, 200, 2, (2, 3)),
    "Acrobot-v1": (3, 500, 4, (6, 3)),
    "Pendulum-v0": (4, 200, 2, (3, 1)),          # continuous action: the policy's tanh head (discrete_action: False)
}
CONTINUOUS_ENVS = ("Pendulum-v0",)
ENV_IDS = {k: v[0] for k, v in ENV_SPECS.items()}


def population_layout(strategy, offspring_num, elite_num=None):
    """(P, group, n_head, n_parents) of a strategy (offspring_strategies.py:48-61,165-176,299-328)."""
    n = int(offspring_num)
    if strategy == "simple_evolution":
        return n + 1, n + 1, 2, 1            # [mu, elite0 (== mu), n-1 perturbed]
    if strategy in ("openai_es", "nsr_es"):
        return n, n, 1, 1                    # [mu, n-1 perturbed]
    if strategy == "simple_genetic":
        k = int(elite_num)
        g = n // k
        if g < 1:
            raise ValueError("simple_genetic needs offspring_num >= elite_num")
        return k * g, g, 1, k                # per elite: [elite, g-1 perturbed]
    raise ValueError("unknown strategy %r" % (strategy,))


def shard_bounds(P, rank, world):
    """Contiguous offspring-id range of `rank` (SURVEY.md section 8e); remainder to the low ranks."""
    base, rem = divmod(P, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def cyclic_block(P, world):
    """Block size of the block-cyclic sharding: small enough that every rank gets >= 8 blocks, at most 256 ids."""
    return max(1, min(256, int(P) // (8 * int(world))))


def owned_ids(P, rank, world, block):
    """Global offspring ids of `rank` under block-cyclic sharding, in local (work-queue) order -- the host-side mirror
    of `Shard::local_to_id` (csrc/ses_common.cuh)."""
    blocks = np.arange(rank, (P + block - 1) // block, world, dtype=np.int64)
    ids = (blocks[:, None] * block + np.arange(block, dtype=np.int64)[None, :]).reshape(-1)
    return ids[ids < P]


def _ptr(t):
    if t is None:
        return None
    return C.c_void_p(t.data_ptr())


class _DeviceArray:
    """Wraps library-owned device memory for torch.as_tensor (CUDA array interface, no copy)."""

    def __init__(self, ptr, n, typestr):
        self.__cuda_array_interface__ = {"shape": (int(n),), "typestr": typestr, "data": (int(ptr), False), "version": 2}


class RolloutEngine:
    """One engine instance == one ses_handle == one GPU's slice of the population."""

    def __init__(self, env_name, obs_dim, act_dim, gru, pomdp, max_step, eval_ep_num, population, group, n_head,
                 n_parents, seed=0, init_mode="shared", n_agents=2, id_begin=0, id_end=None, device=0, antithetic=False,
                 shard=None, discrete_action=True, test_build=None):
        """`shard` = (rank, world, block): block-cyclic slice instead of the contiguous [id_begin, id_end)."""
        if env_name not in ENV_IDS:
            raise ValueError(
                "env %r is not supported by the B200 engine (%s; Box2D, PyBullet and "
                "Unity environments stay on the reference CPU path)" % (env_name, ", ".join(sorted(ENV_IDS))))
        if bool(discrete_action) == (env_name in CONTINUOUS_ENVS):
            raise ValueError("%s runs with discrete_action: %s (networks/neural_network.py:29-33); the continuous-action head is "
                             "implemented for %s" % (env_name, env_name not in CONTINUOUS_ENVS, ", ".join(CONTINUOUS_ENVS)))
        if not torch.cuda.is_available():
            raise RuntimeError("simple-es_b200: no CUDA device; the engine has no CPU fallback")
        # test_build: libses_b200_tests.so -- test hooks and the alternative kernels behind SES_K1_VARIANT & co (tests / tools only;
        # SES_B200_TEST_BUILD=1 makes it the default of a process)
        if test_build is None:
            test_build = os.environ.get("SES_B200_TEST_BUILD", "0") not in ("", "0")
        self.test_build = bool(test_build)
        self.lib = _lib.load(tests=self.test_build)
        self.device = torch.device("cuda", device)
        self.P = int(population)
        self.id_begin = int(id_begin)
        self.id_end = self.P if id_end is None else int(id_end)
        self.shard = None if shard is None else tuple(int(x) for x in shard)
        if self.shard is not None and (self.id_begin, self.id_end) != (0, self.P):
            raise ValueError("a block-cyclic shard covers the whole population: leave id_begin / id_end at their defaults")
        self._n_local = int(owned_ids(self.P, *self.shard).size) if self.shard is not None else self.id_end - self.id_begin
        self.E = int(eval_ep_num)
        self.env_name = env_name
        self.n_agents = int(n_agents) if env_name == "simple_spread" else 1
        ms = 0 if max_step in (None, "None") else int(max_step)
        _, cap, sdim, dims = ENV_SPECS[env_name]
        if dims is not None and (int(obs_dim), int(act_dim)) != dims:
            raise ValueError("%s needs num_state=%d, num_action=%d (got %d, %d)" % ((env_name,) + dims + (obs_dim, act_dim)))
        self.max_step = min(ms, cap) if ms > 0 else cap
        self.state_dim = 4 * self.n_agents if sdim is None else sdim
        self.D = self.lib.ses_param_count(obs_dim, act_dim, int(bool(gru)))
        self.cfg = _lib.ses_config(
            env=ENV_IDS[env_name], obs_dim=obs_dim, act_dim=act_dim, gru=int(bool(gru)), pomdp=int(bool(pomdp)),
            n_agents=self.n_agents, max_step=self.max_step, eval_ep_num=self.E, population=self.P, group=int(group),
            n_head=int(n_head), n_parents=int(n_parents), seed=int(seed) & 0xFFFFFFFF,
            init_mode={"shared": 0, "fresh": 1}[init_mode], id_begin=self.id_begin, id_end=self.id_end, device=device,
            antithetic=int(bool(antithetic)), shard_block=self.shard[2] if self.shard else 0,
            shard_rank=self.shard[0] if self.shard else 0, shard_world=self.shard[1] if self.shard else 0,
            continuous_action=int(not discrete_action))
        h = C.c_void_p()
        self._check(self.lib.ses_create(C.byref(self.cfg), C.byref(h)))
        self._h = h
        # integer-key fast path of K2: CartPole fitness*E is an integer < 2^key_bits
        # (CartPole: +1 per step; MountainCar / Acrobot: -1 or 0 per step => |fitness * E| <= E * max_step)
        if env_name != "simple_spread" and env_name not in CONTINUOUS_ENVS:
            self.key_bits = int(self.E * self.max_step).bit_length()
            self.key_scale = float(self.E)
        else:
            self.key_bits, self.key_scale = 0, 1.0

    def _check(self, rc):
        _lib.check(rc, self.lib)

    def _hooks(self):
        if not self.test_build:
            raise RuntimeError("test hooks live in libses_b200_tests.so: construct the engine with test_build=True")
        return self.lib

    def close(self):
        if getattr(self, "_h", None):
            self.lib.ses_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------------------ helpers
    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _chk(self, t, dtype, numel=None, name="tensor"):
        if t is None:
            return None
        if not (t.is_cuda and t.dtype == dtype and t.is_contiguous()):
            raise ValueError("%s must be a contiguous CUDA tensor of dtype %s" % (name, dtype))
        if numel is not None and t.numel() != numel:
            raise ValueError("%s has %d elements, expected %d" % (name, t.numel(), numel))
        return t

    @property
    def n_local(self):
        return self._n_local

    @property
    def launches(self):
        return int(self.lib.ses_launch_count(self._h))

    def set_step_counter(self, counter):
        """`counter`: 0-d / 1-element int64 CUDA tensor; every rollout() adds the env steps it simulated."""
        self._chk(counter, torch.int64, 1, "counter")
        self._step_counter = counter            # keep alive
        self._check(self.lib.ses_set_step_counter(self._h, _ptr(counter)))

    def set_final_states(self, final_states):
        """`final_states`: [P, E, state_dim] float64 CUDA tensor, or None (off).  While set, every rollout() also stores the
        state after each episode's last step in the rows of the ids this engine owns (DESIGN.md section 4.10)."""
        self._chk(final_states, torch.float64, self.P * self.E * self.state_dim, "final_states")
        self._final_states = final_states       # keep alive
        self._check(self.lib.ses_set_final_states(self._h, _ptr(final_states)))

    # ------------------------------------------------------------------------------ novelty search (nsr_es)
    def behavior(self, final_states, out=None):
        """Behaviour characterisations [n, state_dim] f64: the mean over episodes of final_states [n, E, state_dim]."""
        self._chk(final_states, torch.float64, name="final_states")
        n = final_states.numel() // (self.E * self.state_dim)
        if final_states.numel() != n * self.E * self.state_dim:
            raise ValueError("final_states has %d elements, not a multiple of E * state_dim = %d"
                             % (final_states.numel(), self.E * self.state_dim))
        if out is None:
            out = torch.empty((n, self.state_dim), dtype=torch.float64, device=self.device)
        self._chk(out, torch.float64, n * self.state_dim, "out")
        self._check(self.lib.ses_behavior(self._h, _ptr(final_states), n, _ptr(out), self._stream()))
        return out

    def novelty(self, bc, archive, n_archive, k, out=None):
        """novelty [n] f64: mean distance from each row of bc [n, state_dim] to its min(k, n_archive) nearest rows of
        archive[:n_archive] (archive: [>= n_archive, state_dim] f64)."""
        self._chk(bc, torch.float64, name="bc")
        self._chk(archive, torch.float64, name="archive")
        n = bc.numel() // self.state_dim
        if bc.numel() != n * self.state_dim:
            raise ValueError("bc has %d elements, not a multiple of state_dim = %d" % (bc.numel(), self.state_dim))
        if archive.numel() < int(n_archive) * self.state_dim:
            raise ValueError("archive has %d elements, fewer than n_archive * state_dim = %d"
                             % (archive.numel(), int(n_archive) * self.state_dim))
        if out is None:
            out = torch.empty(n, dtype=torch.float64, device=self.device)
        self._chk(out, torch.float64, n, "out")
        self._check(self.lib.ses_novelty(self._h, _ptr(bc), n, _ptr(archive), int(n_archive), int(k), _ptr(out), self._stream()))
        return out

    def blend_shaped(self, shaped_f, shaped_n, w, out=None):
        """(1 - w) shaped_f + w shaped_n, float64, each operation separately rounded."""
        self._chk(shaped_f, torch.float64, name="shaped_f")
        n = shaped_f.numel()
        self._chk(shaped_n, torch.float64, n, "shaped_n")
        if out is None:
            out = torch.empty(n, dtype=torch.float64, device=self.device)
        self._chk(out, torch.float64, n, "out")
        self._check(self.lib.ses_blend_shaped(self._h, _ptr(shaped_f), _ptr(shaped_n), n, float(w), _ptr(out), self._stream()))
        return out

    # ------------------------------------------------------------------------------ K1
    def rollout(self, generation, sigma, parents, fitness=None, steps=None, w_override=None, init_states=None,
                n_trace=0):
        """Roll out this engine's slice.  Returns (fitness[P] f64, steps[P] i64[, trace, trace_actions]);
        only [id_begin, id_end) is written."""
        dev = self.device
        parents = self._chk(parents, torch.float32, name="parents")
        w_override = self._chk(w_override, torch.float32, self.n_local * self.D, "w_override")
        init_states = self._chk(init_states, torch.float64, self.E * self.state_dim, "init_states")
        if fitness is None:
            fitness = torch.zeros(self.P, dtype=torch.float64, device=dev)
        if steps is None:
            steps = torch.zeros(self.P, dtype=torch.int64, device=dev)
        self._chk(fitness, torch.float64, self.P, "fitness")
        self._chk(steps, torch.int64, self.P, "steps")
        trace = actions = None
        if n_trace > 0:
            n_trace = min(n_trace, self.n_local)
            trace = torch.full((n_trace, 200, self.state_dim), float("nan"), dtype=torch.float64, device=dev)
            actions = torch.full((n_trace, 200, self.n_agents), -1, dtype=torch.int32, device=dev)
        self._check(self.lib.ses_rollout(self._h, int(generation), float(sigma), _ptr(parents), _ptr(w_override),
                                        _ptr(init_states), _ptr(fitness), _ptr(steps), _ptr(trace), _ptr(actions),
                                        int(n_trace), self._stream()))
        if n_trace > 0:
            return fitness, steps, trace, actions
        return fitness, steps

    # ------------------------------------------------------------------------------ policy evaluation
    def evaluate(self, policies, n_episodes, round=0, init_states=None):
        """Run every policy ([D] or [n_pol, D] f32, used as given: no noise) for n_episodes episodes of this engine's env.
        Episode m starts from the same state for every policy: drawn from the env's reset distribution keyed by
        (seed, round, m), or init_states[m] ([n_episodes, state_dim] f64).  Returns (returns [n_pol, n_episodes] f64,
        lengths [n_pol, n_episodes] i32), CUDA tensors on this engine's stream (DESIGN.md section 4.9)."""
        if not torch.is_tensor(policies) or policies.dim() not in (1, 2) or policies.shape[-1] != self.D:
            raise ValueError("policies has shape %s, expected [%d] or [n_pol, %d] (D of this env / network)"
                             % (tuple(getattr(policies, "shape", ())), self.D, self.D))
        if not (policies.is_cuda and policies.dtype == torch.float32):
            raise ValueError("policies must be a float32 CUDA tensor")
        policies = policies.reshape(-1, self.D).contiguous()
        n_pol, M = policies.shape[0], int(n_episodes)
        if M < 1:
            raise ValueError("n_episodes must be >= 1 (got %d)" % M)
        init_states = self._chk(init_states, torch.float64, M * self.state_dim, "init_states")
        returns = torch.empty((n_pol, M), dtype=torch.float64, device=self.device)
        lengths = torch.empty((n_pol, M), dtype=torch.int32, device=self.device)
        self._check(self.lib.ses_evaluate(self._h, int(round) & 0xFFFFFFFF, _ptr(policies), n_pol, M, _ptr(init_states),
                                          _ptr(returns), _ptr(lengths), self._stream()))
        return returns, lengths

    def record(self, policies, n_episodes, round=0, init_states=None):
        """Record, step by step, episodes 0 .. n_episodes-1 of what `evaluate` runs with the same round / init_states (episode m
        does not depend on the episode count).  Returns, as CUDA tensors on this engine's stream, with K = n_episodes and
        T = max_step (DESIGN.md section 4.9):
          initial [K, state_dim] f64            the initial states, laid out as init_states rows
          states  [n_pol, K, T, state_dim] f64  the state after step t + 1 (gym envs: env.unwrapped.state; simple_spread:
                                                agent positions, then agent velocities)
          actions [n_pol, K, T, n_agents] i32   the action of step t + 1; float32 for continuous-action envs
          returns [n_pol, K, T] f64             the return after step t + 1: returns[j, m, lengths[j, m] - 1] is evaluate's
          lengths [n_pol, K] i32
        Steps past an episode's end hold NaN (actions: -1, or NaN for float32 actions)."""
        if not torch.is_tensor(policies) or policies.dim() not in (1, 2) or policies.shape[-1] != self.D:
            raise ValueError("policies has shape %s, expected [%d] or [n_pol, %d] (D of this env / network)"
                             % (tuple(getattr(policies, "shape", ())), self.D, self.D))
        if not (policies.is_cuda and policies.dtype == torch.float32):
            raise ValueError("policies must be a float32 CUDA tensor")
        policies = policies.reshape(-1, self.D).contiguous()
        n_pol, K, T = policies.shape[0], int(n_episodes), self.max_step
        if K < 1:
            raise ValueError("n_episodes must be >= 1 (got %d)" % K)
        init_states = self._chk(init_states, torch.float64, K * self.state_dim, "init_states")
        dev, nan = self.device, float("nan")
        initial = torch.full((K, self.state_dim), nan, dtype=torch.float64, device=dev)
        states = torch.full((n_pol, K, T, self.state_dim), nan, dtype=torch.float64, device=dev)
        actions = torch.full((n_pol, K, T, self.n_agents), -1, dtype=torch.int32, device=dev)
        returns = torch.full((n_pol, K, T), nan, dtype=torch.float64, device=dev)
        lengths = torch.full((n_pol, K), -1, dtype=torch.int32, device=dev)
        self._check(self.lib.ses_record(self._h, int(round) & 0xFFFFFFFF, _ptr(policies), n_pol, K, _ptr(init_states),
                                        _ptr(initial), _ptr(states), _ptr(actions), _ptr(returns), _ptr(lengths), self._stream()))
        if self.env_name in CONTINUOUS_ENVS:
            actions = actions.view(torch.float32)
        return initial, states, actions, returns, lengths

    # ------------------------------------------------------------------------------ K2
    def rank_desc(self, fitness, shaped=False, order=None, shaped_out=None, full_key=False):
        """order[r] = offspring with rank r (0 = best; ties by descending index); optional centered ranks."""
        n = fitness.numel()
        self._chk(fitness, torch.float64, name="fitness")
        if order is None:
            order = torch.empty(n, dtype=torch.int32, device=self.device)
        if shaped and shaped_out is None:
            shaped_out = torch.empty(n, dtype=torch.float64, device=self.device)
        kb, ks = (0, 1.0) if full_key else (self.key_bits, self.key_scale)
        self._check(self.lib.ses_rank_desc(self._h, _ptr(fitness), n, kb, ks, _ptr(order),
                                          _ptr(shaped_out) if shaped else None, self._stream()))
        return (order, shaped_out) if shaped else order

    # ------------------------------------------------------------------------------ K3
    @staticmethod
    def adam_a(lr, t, beta1=0.99, beta2=0.999):
        """optimizers.py:43-47 (float64)."""
        return lr * math.sqrt(1 - beta2 ** t) / (1 - beta1 ** t)

    def update_openai(self, generation, sigma, lr, t, shaped, mu, m, v, eps_override=None, grad_out=None,
                      beta1=0.99, beta2=0.999, eps=1e-8):
        """In-place openai_es step on (mu, m, v); `t` is Adam's step count AFTER the increment."""
        for name, x in (("mu", mu), ("m", m), ("v", v)):
            self._chk(x, torch.float32, self.D, name)
        self._chk(shaped, torch.float64, self.P, "shaped")
        eps_override = self._chk(eps_override, torch.float32, self.P * self.D, "eps_override")
        uf = -1.0 * (lr / (self.P * sigma))              # offspring_strategies.py:406-408
        self._check(self.lib.ses_update_openai(self._h, int(generation), _ptr(shaped), _ptr(eps_override), uf,
                                              self.adam_a(lr, t, beta1, beta2), beta1, beta2, eps, _ptr(mu), _ptr(m),
                                              _ptr(v), _ptr(grad_out), self._stream()))

    def update_openai_sgd(self, generation, sigma, lr, shaped, mu, v, momentum=0.9, eps_override=None, grad_out=None):
        """In-place openai_es step on (mu, v) with SGD + momentum instead of Adam (engine.optimizer: sgd; the reference
        ships Adam only -- this is the SGD of the OpenAI file optimizers.py names as its source)."""
        for name, x in (("mu", mu), ("v", v)):
            self._chk(x, torch.float32, self.D, name)
        self._chk(shaped, torch.float64, self.P, "shaped")
        eps_override = self._chk(eps_override, torch.float32, self.P * self.D, "eps_override")
        uf = -1.0 * (lr / (self.P * sigma))              # offspring_strategies.py:406-408
        self._check(self.lib.ses_update_openai_sgd(self._h, int(generation), _ptr(shaped), _ptr(eps_override), uf, float(lr),
                                                  float(momentum), _ptr(mu), _ptr(v), _ptr(grad_out), self._stream()))

    def materialize(self, generation, sigma, parents, ids, w_override=None, out=None):
        ids = self._chk(ids, torch.int32, name="ids")
        n = ids.numel()
        if out is None:
            out = torch.empty((n, self.D), dtype=torch.float32, device=self.device)
        self._check(self.lib.ses_materialize(self._h, int(generation), float(sigma), _ptr(parents), _ptr(w_override),
                                            _ptr(ids), n, _ptr(out), self._stream()))
        return out

    def elite_mean(self, generation, sigma, parents, order, k, w_override=None, out=None):
        if out is None:
            out = torch.empty(self.D, dtype=torch.float32, device=self.device)
        self._check(self.lib.ses_update_elite_mean(self._h, int(generation), float(sigma), _ptr(parents),
                                                  _ptr(w_override), _ptr(order), int(k), _ptr(out), self._stream()))
        return out

    # ------------------------------------------------------------------------------ peer fitness exchange
    def peer_setup(self, rank, world, all_gather_bytes):
        """Map every rank's exchange buffer over NVLink.  `all_gather_bytes(b) -> [bytes per rank]` is any host
        channel (torch.distributed.all_gather_object).  Returns the two [P] float64 exchange tensors (double
        buffered by generation parity) that rollout() must be given as `fitness`."""
        mine = C.create_string_buffer(64)
        self._check(self.lib.ses_peer_export(self._h, mine))
        handles = all_gather_bytes(mine.raw)
        assert len(handles) == world and all(len(b) == 64 for b in handles)
        blob = C.create_string_buffer(b"".join(handles), 64 * world)
        self._check(self.lib.ses_peer_attach(self._h, blob, int(rank), int(world)))
        bufs = []
        for parity in (0, 1):
            ptr = C.c_void_p()
            self._check(self.lib.ses_peer_fitness_ptr(self._h, parity, C.byref(ptr)))
            bufs.append(torch.as_tensor(_DeviceArray(ptr.value, self.P, "<f8"), device=self.device))
        return bufs

    def peer_barrier(self):
        self._check(self.lib.ses_peer_barrier(self._h, self._stream()))

    def peer_check(self):
        self._check(self.lib.ses_peer_check(self._h))

    # ------------------------------------------------------------------------------ host-buffer generation
    def generation_openai_host(self, generation, sigma, lr, t, mu, m, v, fitness):
        """Whole openai_es generation on HOST numpy buffers (pinned recommended); updates mu/m/v/fitness in
        place and returns the number of env steps simulated.  Synchronous."""
        total = np.zeros(1, dtype=np.int64)
        for a, dt in ((mu, np.float32), (m, np.float32), (v, np.float32), (fitness, np.float64)):
            assert isinstance(a, np.ndarray) and a.dtype == dt and a.flags.c_contiguous
        self._check(self.lib.ses_generation_openai_host(
            self._h, int(generation), float(sigma), float(lr), int(t), C.c_void_p(mu.ctypes.data),
            C.c_void_p(m.ctypes.data), C.c_void_p(v.ctypes.data), C.c_void_p(fitness.ctypes.data),
            C.c_void_p(total.ctypes.data), self._stream()))
        return int(total[0])

    def generation_evolution_host(self, generation, sigma, elite_num, mu, fitness):
        """Whole simple_evolution generation on HOST numpy buffers: mu [D] float32 in / out (the elite mean), fitness [P]
        float64 out; returns the env steps simulated.  Synchronous; the caller decays sigma afterwards."""
        return self._elite_host(self.lib.ses_generation_evolution_host, (int(generation), float(sigma), int(elite_num)), mu, self.D, fitness)

    def generation_genetic_host(self, generation, sigma, elites, fitness):
        """Whole simple_genetic generation on HOST numpy buffers: elites [n_parents][D] float32 in / out (the weights of the
        n_parents best offspring), fitness [P] float64 out; returns the env steps simulated.  Synchronous."""
        return self._elite_host(self.lib.ses_generation_genetic_host, (int(generation), float(sigma)), elites,
                                int(self.cfg.n_parents) * self.D, fitness)

    def _elite_host(self, fn, head, parents, numel, fitness):
        total = np.zeros(1, dtype=np.int64)
        assert isinstance(parents, np.ndarray) and parents.dtype == np.float32 and parents.flags.c_contiguous and parents.size == numel
        assert isinstance(fitness, np.ndarray) and fitness.dtype == np.float64 and fitness.flags.c_contiguous and fitness.size == self.P
        self._check(fn(self._h, *head, C.c_void_p(parents.ctypes.data), C.c_void_p(fitness.ctypes.data),
                      C.c_void_p(total.ctypes.data), self._stream()))
        return int(total[0])

    # ------------------------------------------------------------------------------ test hooks
    def test_math(self, kind, x):
        kinds = {"tanh": 0, "sigmoid": 1, "ln": 2, "sin2pi": 3, "cos2pi": 4, "sin64": 5, "cos64": 6, "tanh_fast": 7,
                 "sin64_full": 8, "cos64_full": 9}
        out = torch.empty_like(x)
        self._check(self._hooks().ses_test_math(kinds[kind], _ptr(x), _ptr(out), x.numel(), self._stream()))
        return out

    def test_tanh_fast_exhaustive(self, lo=0.0, hi=10.0):
        """Number of float32 inputs in [lo, hi] (and their negatives) where K1's fast-path tanh != the contract's."""
        bad = C.c_uint64(0)
        self._check(self._hooks().ses_test_tanh_fast_exhaustive(float(lo), float(hi), C.byref(bad)))
        return int(bad.value)

    def test_tanh_x2_exhaustive(self, newton, lo=0.0, hi=10.0):
        """The same for the packed (FFMA2) tanh of K1's hidden-unit pairs; newton=False is K1 variant 2."""
        bad = C.c_uint64(0)
        self._check(self._hooks().ses_test_tanh_x2_exhaustive(int(bool(newton)), float(lo), float(hi), C.byref(bad)))
        return int(bad.value)

    def test_div_total_mass(self, n=1 << 33):
        """Mismatches between K1's multiply+2fma division by total_mass (1.1) and IEEE division on n random doubles."""
        bad = C.c_uint64(0)
        self._check(self._hooks().ses_test_div_total_mass(int(n), C.byref(bad)))
        return int(bad.value)

    def test_ddiv_fast(self, n=1 << 30):
        """Mismatches between K1 variant 6's branch-free double division and IEEE division on n random in-range operand pairs."""
        bad = C.c_uint64(0)
        self._check(self._hooks().ses_test_ddiv_fast(int(n), C.byref(bad)))
        return int(bad.value)

    def test_k1_geometry(self):
        """Launch geometry of the last slot-kernel rollout (test build): dict of grid, lanes, tail_start, sparse_rank, sparse_quota,
        ctas_per_sm, resident_warps."""
        out = (C.c_int32 * 8)()
        self._check(self._hooks().ses_test_k1_geometry(self._h, out))
        return dict(zip(("grid", "lanes", "tail_start", "sparse_rank", "sparse_quota", "ctas_per_sm", "resident_warps", "reserved"), list(out)))

    def test_normals(self, generation, idx):
        out = torch.empty(self.D, dtype=torch.float32, device=self.device)
        self._check(self._hooks().ses_test_normals(self._h, int(generation), int(idx), _ptr(out), self._stream()))
        return out

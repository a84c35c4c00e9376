"""K1 for MountainCar-v0, Acrobot-v1, Pendulum-v0, simple_spread below E = 5 and the generic GRU kernel at the sizes the shipped
configs run (P = 16384) and past one round of resident warps, bit for bit against the C twin (oracle/twin.py).  What only a
multi-round launch exercises: a warp taking a second offspring into a slot it already used (the per-episode returns of
SlotSmem<..., true>, summed in episode order when the slot retires), the queue of whole offspring of the envs without episode
units (lanes_used = E floor(32 / E), no queue B), the generic GRU kernel's next-offspring loop (gate tables reloaded into
shared memory the warp has used), the evaluation kernels past one round, and the episode bound for Pendulum.  The populations
are ragged, so that slots retire and refill at different times, and they reach the envs' rare branches (MountainCar's
left-wall reset and its goal, Acrobot's angle wrap and velocity clips, Pendulum's speed clip and the negative fmod of its
angle normalisation).  Slot-kernel shapes are derived from the occupancy the test build reports and each asserts, through
the geometry hook, that it still runs the path it was chosen for.  Every twin vector is computed once per module."""
import multiprocessing as mp
import os
import sys
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))

import eval_reference as ref  # noqa: E402

NT = os.cpu_count() or 1
# env -> (obs, act, D of the MLP, time limit)
CLASSIC = {"MountainCar-v0": (2, 3, 195, 200), "Acrobot-v1": (6, 3, 323, 500), "Pendulum-v0": (3, 1, 161, 200)}


def _cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _host(*ts):
    return tuple(t.cpu().numpy() for t in ts)


def _engine(env, P, E, gru=False, n_agents=2, max_step=None, **kw):
    from simple_es_b200.engine import RolloutEngine
    obs, act = (6 * n_agents, 5) if env == "simple_spread" else CLASSIC[env][:2]
    args = dict(seed=7, init_mode="shared", n_agents=n_agents, discrete_action=env != "Pendulum-v0")
    args.update(kw)
    return RolloutEngine(env, obs, act, gru, False, max_step, E, P, P, 1, 1, **args)


def _lanes(E):
    """launch_slots: lanes of a warp that take episodes for an env without episode units."""
    return 32 if E >= 32 else E * (32 // E)


def pumping_parent():
    """A MountainCar policy that pushes in the direction of the velocity: fc1 unit 0 reads the velocity, fc2 turns its sign
    into action 2 (right) or 0 (left).  Perturbed at sigma 0.7, about two thirds of the episodes reach the flag, at varying
    times, and the rest are truncated at 200 steps."""
    mu = np.zeros(195, np.float32)
    mu[:64].reshape(32, 2)[0] = [0.0, 100.0]
    w2 = mu[96:192].reshape(3, 32)
    w2[2, 0] = 5.0
    w2[0, 0] = -5.0
    return mu


# env -> (parent, sigma): MountainCar from the pumping parent; Acrobot and Pendulum from a random parent at sigma 2 (Acrobot:
# ragged lengths, with a fifth of the episodes ending before 500 steps; Pendulum spins: the speed clip and the negative angle)
POPULATIONS = {"MountainCar-v0": (pumping_parent()[None], 0.7),
               "Acrobot-v1": (np.random.default_rng(4).normal(0, 0.5, (1, 323)).astype(np.float32), 2.0),
               "Pendulum-v0": (np.random.default_rng(6).normal(0, 0.5, (1, 161)).astype(np.float32), 2.0)}
GEN = 2


def _assert_ragged(env, E, tf, ts, label):
    cap = CLASSIC[env][3]
    if env == "Pendulum-v0":                     # never terminates: the check is the float64 episode-order sum of every slot
        assert np.all(ts == cap * E) and len(np.unique(tf)) > 0.95 * tf.size, label
        return "all %d steps, %d distinct returns" % (cap * E, len(np.unique(tf)))
    distinct = len(np.unique(ts))
    short = float((ts < cap * E).mean())
    assert distinct >= 50 and short >= 0.05, (label, distinct, short)
    return "%d distinct step totals, %.1f %% of the offspring with an episode shorter than %d steps" % (distinct, 100 * short, cap)


# ------------------------------------------------------------------------------------- 1. classic-control slot kernel across rounds
@pytest.fixture(scope="module")
def occupancy():
    """Resident warps of the slot kernel instance of (env, E): one small launch of the test build, read off the geometry hook."""
    cache = {}

    def get(env, E):
        if (env, E) not in cache:
            eng = _engine(env, 64, E, test_build=True)
            mu, sigma = POPULATIONS[env]
            eng.rollout(GEN, sigma, _cuda(mu))
            torch.cuda.synchronize()
            cache[env, E] = eng.test_k1_geometry()["resident_warps"]
            eng.close()
        return cache[env, E]
    return get


# shape -> (E, init_mode, rounds: "below" one round, "past" one round, or at least this many rounds)
SLOT_SHAPES = {"E5_below_R": (5, "shared", "below"), "E5_past_R": (5, "shared", "past"), "E5_3_rounds": (5, "fresh", 3.0),
               "E1": (1, "shared", 2.5), "E2": (2, "fresh", 2.5), "E3": (3, "shared", 2.5), "E4": (4, "shared", 2.5),
               "E7": (7, "fresh", 2.5), "E17": (17, "shared", 2.5), "E32": (32, "fresh", 2.5)}


def _slot_shape(shape, R):
    E, _, rounds = SLOT_SHAPES[shape]
    if rounds == "below":
        return R // E                            # n_ep <= R: one round
    if rounds == "past":
        return R // E + 1                        # R < n_ep <= 2 R
    return -(-int(rounds * R) // E) + 1          # n_ep > rounds x R


@pytest.mark.parametrize("shape", list(SLOT_SHAPES))
@pytest.mark.parametrize("env", list(CLASSIC))
def test_classic_slot_kernel_rounds_equal_the_twin(twin, occupancy, env, shape):
    """MLP policies on the slot kernel (32 / 16 / 8 slots at E = 1 / 2-3 / >= 4) just below and just past one round, at three
    rounds, and at 2.5 rounds for E = 1, 2, 3, 4, 7 (28 lanes), 17 (17 lanes) and 32 (one offspring fills a warp); at E = 2 and
    4 a warp's offspring fill its slots exactly.  The test build reports the path, then the test build and the product build
    must each give the twin's fitness and steps."""
    E, init_mode, rounds = SLOT_SHAPES[shape]
    rw = occupancy(env, E)
    R = rw * _lanes(E)                           # one round, in episodes
    P = _slot_shape(shape, R)
    n_ep = P * E
    mu, sigma = POPULATIONS[env]
    tf, ts = twin.population_classic(env, mu, sigma=sigma, seed=7, gen=GEN, group=P, n_head=1, n=P, E=E,
                                     init_mode=0 if init_mode == "shared" else 1, nthreads=NT)
    rag = _assert_ragged(env, E, tf, ts, shape)

    t = _engine(env, P, E, init_mode=init_mode, test_build=True)
    fit, steps = _host(*t.rollout(GEN, sigma, _cuda(mu)))
    g = t.test_k1_geometry()
    t.close()
    print("\n%s %s: P = %d, E = %d, %s, episodes = %d = %.2f rounds of R = %d; %s; geometry %s"
          % (env, shape, P, E, init_mode, n_ep, n_ep / R, R, rag, g))
    assert g["resident_warps"] == rw and g["lanes"] == _lanes(E)
    assert g["tail_start"] == n_ep and g["sparse_rank"] < 0            # whole offspring from queue A only, no sparse warps
    if rounds == "below":
        path = n_ep <= R
    elif rounds == "past":
        path = R < n_ep <= 2 * R
    else:
        path = n_ep > rounds * R
    assert path, "shape %s no longer runs the path it was chosen for: n_ep = %d, R = %d" % (shape, n_ep, R)
    assert np.array_equal(steps, ts) and np.array_equal(fit, tf)

    eng = _engine(env, P, E, init_mode=init_mode)
    fit, steps = _host(*eng.rollout(GEN, sigma, _cuda(mu)))
    eng.close()
    assert np.array_equal(steps, ts)
    assert np.array_equal(fit, tf)


# ------------------------------------------------------------------------------------- 2. simple_spread below E = 5
def _mpe_windows(twin, mu, N, P, E, gru=False, **kw):
    """population_mpe over every offspring, in id windows on host threads (the twin's ctypes calls release the GIL)."""
    step = max(256, -(-P // (4 * NT)))
    windows = [(lo, min(P, lo + step)) for lo in range(0, P, step)]
    with ThreadPoolExecutor(NT) as ex:
        parts = list(ex.map(lambda w: twin.population_mpe(mu, N=N, gru=gru, group=P, n_head=1, id0=w[0], n=w[1] - w[0], E=E, **kw),
                            windows))
    return np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts])


@pytest.mark.parametrize("E", [2, 4])
@pytest.mark.parametrize("N", [2, 3])
def test_spread_8_slot_instances_every_offspring(twin, N, E):
    """simple_spread at P = 16384 (conf/simplespread.yaml) with E = 2 and 4: the 8-slot, 4-warp instances, which the
    full-size config test (E = 5, 6 slots) does not run; every offspring's float64 team return."""
    P = 16384
    Dn = 6 * N * 32 + 32 + 165
    mu = np.random.default_rng(N).normal(0, 0.3, (1, Dn)).astype(np.float32)
    tf, ts = _mpe_windows(twin, mu, N, P, E, sigma=0.2, seed=4, gen=2, init_mode=1)
    assert np.all(ts == 25 * E) and len(np.unique(tf)) > 0.99 * P
    t = _engine("simple_spread", P, E, n_agents=N, seed=4, init_mode="fresh", test_build=True)
    fit, steps = _host(*t.rollout(2, 0.2, _cuda(mu)))
    g = t.test_k1_geometry()
    t.close()
    R = g["resident_warps"] * _lanes(E)
    print("\nsimple_spread N = %d, E = %d: P = %d, episodes = %d = %.2f rounds of R = %d; geometry %s" % (N, E, P, P * E, P * E / R, R, g))
    assert g["lanes"] == _lanes(E) and g["tail_start"] == P * E and g["sparse_rank"] < 0
    assert np.array_equal(steps, ts) and np.array_equal(fit, tf)
    eng = _engine("simple_spread", P, E, n_agents=N, seed=4, init_mode="fresh")
    fit, steps = _host(*eng.rollout(2, 0.2, _cuda(mu)))
    assert np.array_equal(steps, ts) and np.array_equal(fit, tf)


# ------------------------------------------------------------------------------------- 3. the generic GRU kernel past one round
def gru_pumping_parent():
    """pumping_parent with the recurrent policy: fc1 unit 0 reads the velocity, the n gate of hidden unit 0 carries it (z ~ 0,
    so h = n), fc2 turns its sign into a push.  At sigma 0.3 the episodes reach the flag after 100 to 200 steps."""
    mu = np.zeros(6531, np.float32)
    mu[0:64].reshape(32, 2)[0] = [0.0, 100.0]
    mu[96:96 + 3072].reshape(96, 32)[64, 0] = 3.0          # W_ih, n gate row of unit 0, fc1 unit 0
    mu[6240:6240 + 96][32:64] = -10.0                       # b_ih of the z gate
    w2 = mu[6432:6432 + 96].reshape(3, 32)
    w2[2, 0] = 5.0
    w2[0, 0] = -5.0
    return mu


def _residency_bound():
    """Warps the device can hold at most: no launch of a one-warp-per-offspring kernel with more offspring than this can give
    every warp a single offspring."""
    pr = torch.cuda.get_device_properties(0)
    return getattr(pr, "max_threads_per_multi_processor", 2048) // 32 * pr.multi_processor_count


# case -> (env, N, EC of GruGenConfig)
GRU_ENVS = {"mountaincar": ("MountainCar-v0", 1, 5), "acrobot": ("Acrobot-v1", 1, 5), "pendulum": ("Pendulum-v0", 1, 5),
            "spread2": ("simple_spread", 2, 3), "spread3": ("simple_spread", 3, 2)}
# (case, E, init_mode, antithetic, max_step): E = 5 and EC + 1 (a partial last lockstep chunk); Acrobot keeps its 500-step limit
# (the instance with local memory, and random policies end episodes only late); Pendulum is cut at 60 steps for the twin's sake
GRU_CASES = [("mountaincar", 5, "fresh", False, None), ("mountaincar", 6, "shared", True, None),
             ("acrobot", 5, "shared", False, None), ("acrobot", 6, "fresh", False, None),
             ("pendulum", 5, "fresh", True, 60), ("pendulum", 6, "shared", False, 60),
             ("spread2", 5, "fresh", False, None), ("spread2", 4, "shared", True, None),
             ("spread3", 5, "shared", False, None), ("spread3", 3, "fresh", False, None)]


@pytest.mark.parametrize("case,E,init_mode,antithetic,max_step", GRU_CASES,
                         ids=["%s-E%d-%s%s" % (c[0], c[1], c[2], "-anti" if c[3] else "") for c in GRU_CASES])
def test_gru_generic_past_one_round_every_offspring(twin, case, E, init_mode, antithetic, max_step):
    """More offspring than the device can hold warps: some warp takes a second offspring (the work-counter loop), reloads the
    gate tables, and must start its sums afresh.  Every offspring's fitness and steps equal the twin's."""
    env, N, EC = GRU_ENVS[case]
    bound = _residency_bound()
    P = bound + 1031
    eng = _engine(env, P, E, gru=True, n_agents=N, max_step=max_step, seed=5, init_mode=init_mode, antithetic=antithetic)
    if env == "MountainCar-v0":
        mu, sigma = gru_pumping_parent()[None], 0.3
    else:
        mu = np.random.default_rng(1).normal(0, 0.3, (1, eng.D)).astype(np.float32)
        sigma = 1.0 if env != "simple_spread" else 0.5
    fit, steps = _host(*eng.rollout(3, sigma, _cuda(mu)))
    eng.close()
    kw = dict(sigma=sigma, seed=5, gen=3, init_mode=0 if init_mode == "shared" else 1)
    twin.set_antithetic(antithetic)
    try:
        if env == "simple_spread":
            tf, ts = _mpe_windows(twin, mu, N, P, E, gru=True, **kw)
        else:
            tf, ts = twin.population_classic(env, mu, gru=True, group=P, n_head=1, n=P, E=E, max_step=max_step, nthreads=NT, **kw)
    finally:
        twin.set_antithetic(False)
    print("\nGRU %s E = %d (EC = %d), %s%s, max_step %s: P = %d > residency bound %d; %d distinct step totals, %d distinct fitness values"
          % (case, E, EC, init_mode, ", antithetic" if antithetic else "", max_step, P, bound, len(np.unique(ts)), len(np.unique(tf))))
    assert P > bound and (E == 5 or E % EC != 0)
    if env in ("MountainCar-v0", "Acrobot-v1"):
        assert len(np.unique(ts)) >= 20
    else:
        assert len(np.unique(tf)) > 0.95 * P
    assert np.array_equal(steps, ts)
    assert np.array_equal(fit, tf)


# ------------------------------------------------------------------------------------- 4. evaluation past one round
def _eval_window(args):
    """Episodes [lo, hi) of every policy: the twin's single-episode rollouts under the evaluation keying (a pool worker)."""
    env, gru, W, lo, hi, seed, rnd, max_step = args
    from oracle import twin as tw
    tw.build()
    init = np.stack([ref.eval_init(tw, env, seed, rnd, m) for m in range(lo, hi)])
    return ref.evaluate(tw, env, W, hi - lo, gru=gru, max_step=max_step, init_states=init)


# (env, gru, chunk of episodes per virtual offspring, policies, max_step)
EVAL_CASES = {"mountaincar_mlp": ("MountainCar-v0", False, 32, 3, None), "acrobot_gru": ("Acrobot-v1", True, 5, 2, None)}


@pytest.mark.parametrize("case", list(EVAL_CASES))
def test_evaluate_past_one_round_every_episode(twin, case):
    """ses_evaluate with more (policy, chunk) virtual offspring than the device can hold warps and a partial last chunk: every
    episode's return and length equal the twin's (tests/eval_reference.py); on windows of up to 32 episodes (the most one
    ses_rollout takes) -- the first, the chunk boundaries around the middle and the partial end -- the returns added in episode
    order and divided by the window's length equal ses_rollout's fitness in verification mode (DESIGN 4.9 bit rule)."""
    env, gru, chunk, n_pol, max_step = EVAL_CASES[case]
    bound = _residency_bound()
    M = chunk * (bound // n_pol + 1) + chunk // 2 + 1
    assert n_pol * -(-M // chunk) > bound and M % chunk
    eng = _engine(env, n_pol, 1, gru=gru, max_step=max_step, seed=11)
    rng = np.random.default_rng(3)
    if env == "MountainCar-v0":                  # ragged episodes: perturbed pumping parents, some reach the flag
        W = (pumping_parent()[None] + rng.normal(0, 0.7, (n_pol, eng.D))).astype(np.float32)
    else:                                        # random GRU policies at scale 1: some episodes end before 500 steps
        W = rng.normal(0, 1.0, (n_pol, eng.D)).astype(np.float32)
    Wd = _cuda(W)
    ret, lng = _host(*eng.evaluate(Wd, M, round=6))

    step = -(-M // (8 * NT))
    jobs = [(env, gru, W, lo, min(M, lo + step), 11, 6, max_step) for lo in range(0, M, step)]
    pool = mp.get_context("spawn").Pool(min(NT, 32))
    try:
        parts = pool.map(_eval_window, jobs)
    finally:
        pool.close()
        pool.join()
    tr = np.concatenate([p[0] for p in parts], axis=1)
    tl = np.concatenate([p[1] for p in parts], axis=1)
    cap = max_step or ref.CAPS[env]
    print("\nevaluate %s: %d policies x %d episodes = %d chunks of %d > residency bound %d; %d distinct lengths, %.1f %% truncated"
          % (case, n_pol, M, n_pol * -(-M // chunk), chunk, bound, len(np.unique(tl)), 100 * float((tl == cap).mean())))
    assert len(np.unique(tl)) >= 20 and (tl < cap).mean() > 0.05
    assert np.array_equal(lng, tl)
    assert np.array_equal(ret.view(np.int64), tr.view(np.int64))

    mid = (M // 2) // chunk * chunk
    for lo, hi in [(0, 32), (mid - 16, mid + 16), (M - (M % 32 or 32), M)]:
        E = hi - lo
        init = np.stack([ref.eval_init(twin, env, 11, 6, m) for m in range(lo, hi)])
        v = _engine(env, n_pol, E, gru=gru, max_step=max_step)
        fit, steps = _host(*v.rollout(0, 0.0, Wd[:1], w_override=Wd, init_states=_cuda(init).reshape(-1)))
        v.close()
        for j in range(n_pol):
            total = 0.0
            for m in range(lo, hi):
                total = total + ret[j, m]
            assert total / E == fit[j] and int(lng[j, lo:hi].sum()) == steps[j], (lo, hi, j)


# ------------------------------------------------------------------------------------- 5. the episode bound without episode units
def test_pendulum_rollout_at_the_episode_bound(twin):
    """P = 2^25 offspring x E = 32 = 2^30 episodes of Pendulum (the most ses_create accepts), 2 steps each, a fresh initial
    state per episode, so that every offspring's return depends on its id.  tail_start = n_ep = 2^30: queue A only.  The twin
    checks the first and last ids and every id whose first episode index crosses a multiple of 2^24."""
    P, E, sigma, gen = 1 << 25, 32, 0.5, 3
    mu = np.random.default_rng(8).normal(0, 0.5, (1, 161)).astype(np.float32)
    eng = _engine("Pendulum-v0", P, E, max_step=2, seed=0, init_mode="fresh")
    fit_d = torch.full((P,), float("nan"), dtype=torch.float64, device="cuda")
    steps_d = torch.full((P,), -1, dtype=torch.int64, device="cuda")
    eng.rollout(gen, sigma, _cuda(mu), fitness=fit_d, steps=steps_d)
    assert bool(torch.all(steps_d == 2 * E)) and bool(torch.all(torch.isfinite(fit_d)))
    eng.close()
    windows = [(0, 4096), (P - 4096, P)] + [(i - 256, i + 256) for i in (k << 19 for k in range(1, 64))]
    for lo, hi in windows:
        tf, ts = twin.population_classic("Pendulum-v0", mu, sigma=sigma, seed=0, gen=gen, group=P, n_head=1, id0=lo, n=hi - lo, E=E,
                                         max_step=2, init_mode=1, nthreads=NT)
        assert len(np.unique(tf)) == hi - lo, (lo, hi)
        assert np.array_equal(steps_d[lo:hi].cpu().numpy(), ts) and np.array_equal(fit_d[lo:hi].cpu().numpy(), tf), (lo, hi)

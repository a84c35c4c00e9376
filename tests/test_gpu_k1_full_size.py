"""K1 at the sizes the benchmark and the BASELINE configurations run, bit for bit against the C twin (oracle/twin.py on every
host thread).  The launch scheduler (queue A of whole offspring, queue B of exact requests for the last two rounds' worth of
episodes, sparse warps, the mean-length feedback that decides whether a launch gets a queue B) only runs in full above a
few hundred thousand episodes on a B200, and DESIGN 5.1 promises that none of it changes a result bit.  The launch shapes
are derived from the occupancy the device reports, and each asserts (through the test build's geometry hook) that it
still exercises the path it was chosen for.  Every twin vector is computed once per module."""
import multiprocessing as mp
import os

import numpy as np
import pytest

import bench

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

D = 226
DG = 6562
E = 5
P_HEAD = bench.P_DEFAULT                  # 65536: the benchmark's population
NT = os.cpu_count() or 1


def _cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _engine(P, E=E, **kw):
    from simple_es_b200.engine import RolloutEngine
    args = dict(env_name="CartPole-v1", obs_dim=4, act_dim=2, gru=False, pomdp=False, max_step=500, eval_ep_num=E,
                population=P, group=P, n_head=1, n_parents=1, seed=0, init_mode="shared")
    args.update(kw)
    return RolloutEngine(**args)


def _host(*ts):
    return tuple(t.cpu().numpy() for t in ts)           # a synchronising copy: the launch and its step-count copy are done


def _tail_start(n_ep, E, resident_warps, tail=True):
    """ses_abi.cu launch_slots: the first episode of queue B (queue A hands out [0, tail_start) in whole offspring)."""
    R = resident_warps * 32
    if n_ep <= R:
        return 0                                        # a single round: exact requests from the start
    t = 2 * R if tail else 0
    return (n_ep - t) // E * E if n_ep > t else 0


@pytest.fixture(scope="module")
def state():
    return bench.bench_state()


@pytest.fixture(scope="module")
def geometry(state):
    """The slot kernel's occupancy on this device: one converged launch of the test build at the headline size."""
    eng = _engine(P_HEAD, test_build=True)
    eng.rollout(30, state["sigma"], _cuda(state["mu"][None]))
    torch.cuda.synchronize()
    g = eng.test_k1_geometry()
    eng.close()
    assert g["lanes"] == 32 and g["resident_warps"] == g["ctas_per_sm"] * torch.cuda.get_device_properties(0).multi_processor_count * 4
    print("\nK1 geometry at P = %d, E = %d: %s, R = %d episodes" % (P_HEAD, E, g, g["resident_warps"] * 32))
    return g


@pytest.fixture(scope="module")
def conv30(twin, state):
    """The twin's generation-30 vector of the benchmark's converged population (P = 65536, E = 5, seed 0)."""
    return twin.population_cartpole(state["mu"][None], sigma=state["sigma"], seed=0, gen=30, group=P_HEAD, n_head=1, n=P_HEAD,
                                    E=E, nthreads=NT)


@pytest.fixture(scope="module")
def gen0(twin):
    """A generation-0 population at the headline size: mu = 0, sigma = 0.2, ragged episodes of ~17 steps."""
    return twin.population_cartpole(np.zeros((1, D), np.float32), sigma=0.2, seed=0, gen=0, group=P_HEAD, n_head=1, n=P_HEAD,
                                    E=E, nthreads=NT)


# ------------------------------------------------------------------------------------- 1. launch shapes from the device
SHAPES = ["one_round", "past_one_round", "below_2R", "past_2R_queue_a_0", "past_2R_queue_a_1", "headline",
          "E1", "E3", "E7", "E32"]


def _shape(name, R):
    """(P, E) of a shape, from the round size R = resident warps x 32 episodes."""
    return {"one_round": (R // 5, 5), "past_one_round": (R // 5 + 1, 5), "below_2R": (2 * R // 5, 5),
            "past_2R_queue_a_0": (2 * R // 5 + 1, 5), "past_2R_queue_a_1": (2 * R // 5 + 2, 5), "headline": (P_HEAD, 5),
            "E1": (-(-21 * R // 10), 1), "E3": (-(-21 * R // 30), 3), "E7": (-(-21 * R // 70), 7), "E32": (-(-21 * R // 320), 32)}[name]


@pytest.mark.parametrize("shape", SHAPES)
def test_k1_launch_shapes_equal_the_twin(twin, state, geometry, conv30, shape):
    """Converged populations (every episode 500 steps) at the round and tail boundaries of the device's own occupancy, and
    at E = 1, 3, 7, 32 (32, 16, 8, 8 slots per warp; at E = 32 one offspring fills a warp) with queue A non-empty.  The test
    build reports the path; the product build, which bench.py runs, must give the twin's fitness and steps."""
    R = geometry["resident_warps"] * 32
    P, Ek = _shape(shape, R)
    n_ep = P * Ek
    mu, sigma = state["mu"][None], state["sigma"]
    if shape == "headline":
        tf, ts = conv30
    else:
        tf, ts = twin.population_cartpole(mu, sigma=sigma, seed=0, gen=30, group=P, n_head=1, n=P, E=Ek, nthreads=NT)
    assert (ts == 500 * Ek).mean() > 0.95                                        # converged: nearly every episode is truncated

    t = _engine(P, Ek, test_build=True)
    fit, steps = _host(*t.rollout(30, sigma, _cuda(mu)))
    g = t.test_k1_geometry()
    t.close()
    print("\n%s: P = %d, E = %d, episodes = %d, geometry %s" % (shape, P, Ek, n_ep, g))
    Rk = g["resident_warps"] * 32
    assert g["lanes"] == 32 and g["sparse_rank"] < 0
    assert g["tail_start"] == _tail_start(n_ep, Ek, g["resident_warps"])
    if Ek == 5:
        assert g["resident_warps"] == geometry["resident_warps"]                 # the kernel whose occupancy chose P
    path = {"one_round": n_ep <= Rk, "past_one_round": Rk < n_ep <= 2 * Rk, "below_2R": Rk < n_ep <= 2 * Rk,
            "past_2R_queue_a_0": n_ep > 2 * Rk and g["tail_start"] == 0,
            "past_2R_queue_a_1": n_ep > 2 * Rk and g["tail_start"] == Ek}.get(shape, g["tail_start"] > 0)
    assert path, "shape %s no longer runs the path it was chosen for: %s" % (shape, g)
    assert np.array_equal(steps, ts) and np.array_equal(fit, tf)                 # the test build's kernel: same bits

    eng = _engine(P, Ek)
    fit, steps = _host(*eng.rollout(30, sigma, _cuda(mu)))
    assert np.array_equal(steps, ts)
    assert np.array_equal(fit, tf)
    if shape == "headline":                                                      # a second generation: the launch after a
        fit, steps = _host(*eng.rollout(31, sigma, _cuda(mu)))                   # converged one (feedback says "long")
        tf, ts = twin.population_cartpole(mu, sigma=sigma, seed=0, gen=31, group=P, n_head=1, n=P, E=E, nthreads=NT)
        assert np.array_equal(steps, ts) and np.array_equal(fit, tf)
    eng.close()


# ------------------------------------------------------------------------------------- 2. feedback transitions
def test_k1_feedback_regime_changes(state, geometry, conv30, gen0):
    """One handle at P = 65536: converged, converged, generation 0 (the stale mean says "long": a tail), generation 0,
    converged (the stale mean says "ragged": no tail).  Every launch equals the twin; the hook shows which decision each
    launch took.  Each launch is synchronised before the next so that the previous mean is known to the launcher."""
    zero = np.zeros((1, D), np.float32)
    pops = {"converged": (30, state["sigma"], state["mu"][None], conv30), "gen0": (0, 0.2, zero, gen0)}
    assert conv30[1].mean() / E >= 0.25 * 500 and gen0[1].mean() / E < 0.25 * 500
    eng = _engine(P_HEAD, test_build=True)
    for i, (label, tail) in enumerate([("converged", True), ("converged", True), ("gen0", True), ("gen0", False), ("converged", False)]):
        gen, sigma, mu, (tf, ts) = pops[label]
        fit, steps = _host(*eng.rollout(gen, sigma, _cuda(mu)))
        torch.cuda.synchronize()
        g = eng.test_k1_geometry()
        assert g["sparse_rank"] < 0 and g["tail_start"] == _tail_start(P_HEAD * E, E, g["resident_warps"], tail), (i, label, g)
        assert np.array_equal(steps, ts), (i, label)
        assert np.array_equal(fit, tf), (i, label)
    eng.close()


# ------------------------------------------------------------------------------------- 3. the benchmarked generation
def test_benchmarked_generations_equal_the_twin_composition(twin, state, conv30):
    """bench.py's loop (openai_es, P = 65536, E = 5, seed 0) from the committed generation-30 state, two generations: fitness,
    order, shaped fitness, mu and the Adam moments equal population_cartpole -> rank_desc -> centered_rank -> grad_openai
    -> adam, with sigma decayed by 0.9999 in between.  These are the arrays bench.py --dump-outputs writes."""
    from types import SimpleNamespace
    loop = bench.make_loop(SimpleNamespace(pop=P_HEAD, exchange="peer", shard="cyclic"), 0, 2)
    s = loop.strategy
    s.load_state(bench.converged_state())
    lr = float(bench.STRATEGY["learning_rate"])
    mu, m, v, sigma, t = state["mu"].copy(), state["m"].copy(), state["v"].copy(), state["sigma"], state["t"]
    for gen in (30, 31):
        s.step()
        tf, ts = conv30 if gen == 30 else twin.population_cartpole(mu[None], sigma=sigma, seed=0, gen=gen, group=P_HEAD, n_head=1,
                                                                      n=P_HEAD, E=E, nthreads=NT)
        assert np.array_equal(s.steps.cpu().numpy(), ts) and np.array_equal(s.fitness.cpu().numpy(), tf), gen
        order = twin.rank_desc(tf)
        assert np.array_equal(s.order.cpu().numpy(), order), gen
        shaped = twin.centered_rank(order)
        assert np.array_equal(s.shaped.cpu().numpy(), shaped), gen
        g = twin.grad_openai(shaped, D, 0, gen, P_HEAD, 1, -(lr / (P_HEAD * sigma)))
        mu, m, v = twin.adam(mu, m, v, g, s.engine.adam_a(lr, t + 1))
        t += 1
        assert np.array_equal(s.parents.cpu().numpy()[0], mu), gen
        assert np.array_equal(s.m.cpu().numpy(), m) and np.array_equal(s.v.cpu().numpy(), v), gen
        sigma *= float(bench.STRATEGY["sigma_decay"])
        assert s.sigma == sigma and s.t == t


# ------------------------------------------------------------------------------------- 4. multi-GPU shares on one GPU
@pytest.mark.parametrize("N", [2, 4, 8])
def test_cyclic_shard_shares_equal_the_twin(state, conv30, N):
    """The converged headline population cut into N block-cyclic shares (engine.shard: cyclic), each rolled out by its own
    handle into one vector: N = 2 runs queue A + B per rank, N = 4 a launch between one and two rounds, N = 8 sparse warps.
    The vector equals the single-handle vector and the twin; the test build reports the path of every share."""
    from simple_es_b200.engine import cyclic_block
    mu, sigma = _cuda(state["mu"][None]), state["sigma"]
    single = _host(*_engine(P_HEAD).rollout(30, sigma, mu))
    B = cyclic_block(P_HEAD, N)
    for test_build in (False, True):
        fit = torch.full((P_HEAD,), float("nan"), dtype=torch.float64, device="cuda")
        steps = torch.full((P_HEAD,), -1, dtype=torch.int64, device="cuda")
        for r in range(N):
            eng = _engine(P_HEAD, shard=(r, N, B), test_build=test_build)
            eng.rollout(30, sigma, mu, fitness=fit, steps=steps)
            if test_build:
                torch.cuda.synchronize()
                g = eng.test_k1_geometry()
                n_ep = eng.n_local * E
                R = g["resident_warps"] * 32
                want = {2: n_ep > 2 * R and g["tail_start"] > 0 and g["sparse_rank"] < 0,
                        4: R < n_ep <= 2 * R and g["tail_start"] == 0 and g["sparse_rank"] < 0,
                        8: n_ep < R and g["sparse_rank"] >= 0 and g["tail_start"] == 0}[N]
                assert want, (N, r, eng.n_local, g)
                if g["sparse_rank"] < 0:
                    assert g["tail_start"] == _tail_start(n_ep, E, g["resident_warps"]), (N, r, g)
            eng.close()
        fit, steps = _host(fit, steps)
        assert np.array_equal(steps, single[1]) and np.array_equal(fit, single[0]), (N, test_build)
        assert np.array_equal(steps, conv30[1]) and np.array_equal(fit, conv30[0]), (N, test_build)


# ------------------------------------------------------------------------------------- 5. the other BASELINE configurations
@pytest.mark.parametrize("regime", ["pomdp_random", "balancing"])
def test_full_size_gru_config_every_offspring(twin, regime):
    """BASELINE config 1 (CartPole + GRU, simple_evolution, P = 4097) in both regimes bench.py times: POMDP from a random mu,
    and the hand-built balancing parent on the fully observed pole with sigma = 0.02 (500-step episodes)."""
    P = 4097
    if regime == "pomdp_random":
        mu, sigma, pomdp, gen = np.random.default_rng(5).normal(0, 0.3, (1, DG)).astype(np.float32), 0.5, True, 3
    else:
        mu, sigma, pomdp, gen = bench.gru_balancing_parent()[None], 0.02, False, 1
    eng = _engine(P, gru=True, pomdp=pomdp, n_head=2, seed=2)
    fit, steps = _host(*eng.rollout(gen, sigma, _cuda(mu)))
    tf, ts = twin.population_cartpole(mu, gru=True, pomdp=pomdp, sigma=sigma, seed=2, gen=gen, group=P, n_head=2, n=P, E=E,
                                      nthreads=NT)
    assert np.array_equal(steps, ts) and np.array_equal(fit, tf)
    if regime == "balancing":
        assert (ts == 500 * E).mean() > 0.9


@pytest.mark.parametrize("N", [2, 3])
def test_full_size_spread_config_every_offspring(twin, N):
    """BASELINE config 3: simple_spread, shared MLP, openai_es, P = 16384, every offspring's float64 return."""
    P = 16384
    Dn = 6 * N * 32 + 32 + 165
    mu = np.random.default_rng(N).normal(0, 0.3, (1, Dn)).astype(np.float32)
    eng = _engine(P, env_name="simple_spread", obs_dim=6 * N, act_dim=5, n_agents=N, max_step="None", seed=4, init_mode="fresh")
    fit, steps = _host(*eng.rollout(2, 0.2, _cuda(mu)))
    tf, ts = twin.population_mpe(mu, N=N, sigma=0.2, seed=4, gen=2, group=P, n_head=1, n=P, E=E, init_mode=1)
    assert np.array_equal(steps, ts) and np.array_equal(fit, tf)


def _genetic(parents, sigma, gen):
    P, k = 1 << 20, 16
    eng = _engine(P, group=P // k, n_parents=k, seed=1)
    return eng, _host(*eng.rollout(gen, sigma, _cuda(parents)))


def test_full_size_genetic_config_random_elites_every_offspring(twin):
    """BASELINE config 4 (simple_genetic, 16 elites, P = 2^20) from random elites: short episodes, every offspring."""
    parents = np.random.default_rng(0).normal(0, 1, (16, D)).astype(np.float32)
    _, (fit, steps) = _genetic(parents, 1.0, 2)
    tf, ts = twin.population_cartpole(parents, sigma=1.0, seed=1, gen=2, group=1 << 16, n_head=1, n=1 << 20, E=E, nthreads=NT)
    assert np.array_equal(steps, ts) and np.array_equal(fit, tf)


def test_full_size_genetic_config_long_episodes_windows(twin, state):
    """Config 4 with 16 perturbed copies of the generation-30 mu as elites: the whole 2^20 launch runs (its geometry is the
    one under test), the twin checks contiguous id windows at the start, around every elite-group boundary and at the end;
    every offspring's fitness is its step count / E."""
    P, k, grp = 1 << 20, 16, 1 << 16
    parents = (state["mu"][None] + np.random.default_rng(3).normal(0, 0.01, (k, D))).astype(np.float32)
    _, (fit, steps) = _genetic(parents, state["sigma"], 4)
    assert np.array_equal(fit, steps / E) and steps.min() >= E
    windows = [(0, 4096)] + [(j * grp - 2048, j * grp + 2048) for j in range(1, k)] + [(P - 4096, P)]
    for lo, hi in windows:
        tf, ts = twin.population_cartpole(parents, sigma=state["sigma"], seed=1, gen=4, group=grp, n_head=1, id0=lo, n=hi - lo,
                                          E=E, nthreads=NT)
        assert np.array_equal(steps[lo:hi], ts) and np.array_equal(fit[lo:hi], tf), (lo, hi)
        assert (ts == 500 * E).mean() > 0.9, (lo, hi)


# ------------------------------------------------------------------------------------- 6. the episode bound
def test_rollout_at_the_episode_bound(twin):
    """P = 2^25 offspring x E = 32 = 2^30 episodes, the most ses_create accepts: the twin checks the first and last ids and
    every id whose first episode index i * 32 crosses a multiple of 2^24 (where 32-bit index arithmetic in the work queue or
    ep_acc would wrap or change sign); every offspring's fitness is its step count / E."""
    P, Ek, sigma, gen = 1 << 25, 32, 0.02, 3
    zero = np.zeros((1, D), np.float32)
    eng = _engine(P, Ek)
    fit_d = torch.full((P,), float("nan"), dtype=torch.float64, device="cuda")
    steps_d = torch.full((P,), -1, dtype=torch.int64, device="cuda")
    eng.rollout(gen, sigma, _cuda(zero), fitness=fit_d, steps=steps_d)
    assert int(steps_d.min()) >= Ek and torch.equal(fit_d, steps_d.double() / Ek)
    eng.close()
    windows = [(0, 4096), (P - 4096, P)] + [(i - 256, i + 256) for i in (k << 19 for k in range(1, 64))]
    for lo, hi in windows:
        tf, ts = twin.population_cartpole(zero, sigma=sigma, seed=0, gen=gen, group=P, n_head=1, id0=lo, n=hi - lo, E=Ek, nthreads=NT)
        assert np.array_equal(steps_d[lo:hi].cpu().numpy(), ts) and np.array_equal(fit_d[lo:hi].cpu().numpy(), tf), (lo, hi)


# ------------------------------------------------------------------------------------- 7. Philox offspring vs the reference's own algorithm
def test_philox_offspring_match_the_reference_rollout(twin, state):
    """256 seeded offspring of the converged headline launch, their weights from the engine's materialiser, the shared
    initial-state table from the twin, rolled out by oracle/pyref.py (the reference's torch policy and CartPole in Python
    floats with libm sin / cos): K1's returns must equal the reference's, up to near-tie action flips (<= 2 of 256)."""
    from oracle import pyref
    ids = np.sort(np.random.default_rng(30).choice(P_HEAD, 256, replace=False)).astype(np.int32)
    mu, sigma = _cuda(state["mu"][None]), state["sigma"]
    eng = _engine(P_HEAD)
    fit, _ = _host(*eng.rollout(30, sigma, mu))
    W = eng.materialize(30, sigma, mu, _cuda(ids)).cpu().numpy()
    assert np.array_equal(W, twin.materialize(state["mu"][None], sigma, 0, 30, P_HEAD, 1, ids))
    init = np.stack([twin.cartpole_init(0, 0, 30, 0, e) for e in range(E)])
    env = pyref.CartPoleShim(max_step=500, init_states=init)
    pool = mp.get_context("spawn").Pool(min(NT, 32))
    try:
        res = pool.map(pyref.rollout_worker, [(env, w, (4, 2, False), E) for w in W])
    finally:
        pool.close()
        pool.join()
    ref = np.array([r for r, _ in res])
    same = int((ref == fit[ids]).sum())
    print("\nPhilox offspring equal to the reference rollout: %d of %d" % (same, ids.size))
    assert same >= 254

"""Host logic of nsr_es without a device: the strategy section's validation, its population layout, the exchange of
final states ([P, E, state_dim]) between world-size-2 gloo ranks through the generalised fitness exchange, and the references
the full-size GPU tests use: the vectorised novelty against the loop, the twin's population final states against its
single-episode traces."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import novelty_reference as nref  # noqa: E402
from simple_es_b200.engine import population_layout  # noqa: E402
from simple_es_b200.strategies import STRATEGIES, NoveltyES, _novelty_params  # noqa: E402

BASE = {"name": "nsr_es", "init_sigma": 0.5, "sigma_decay": 0.999, "learning_rate": 0.05, "offspring_num": 1024}


def test_nsr_es_is_registered_with_the_openai_layout():
    assert STRATEGIES["nsr_es"] is NoveltyES
    for n in (2, 1024, 65536, 4097):
        assert population_layout("nsr_es", n) == population_layout("openai_es", n) == (n, n, 1, 1)


def test_nsr_es_defaults():
    assert _novelty_params(BASE) == (0.5, 10)
    assert _novelty_params(dict(BASE, novelty_weight=0, novelty_k=1)) == (0.0, 1)
    assert _novelty_params(dict(BASE, novelty_weight=1, novelty_k=32)) == (1.0, 32)
    assert _novelty_params(dict(BASE, novelty_weight=0.25)) == (0.25, 10)


@pytest.mark.parametrize("w", [-0.01, 1.01, float("nan"), "0.5", True, None, float("inf")])
def test_nsr_es_rejects_bad_weight(w):
    with pytest.raises(ValueError, match="novelty_weight"):
        _novelty_params(dict(BASE, novelty_weight=w))


@pytest.mark.parametrize("k", [0, 33, -1, 10.0, 2.5, "10", True, None])
def test_nsr_es_rejects_bad_k(k):
    with pytest.raises(ValueError, match="novelty_k"):
        _novelty_params(dict(BASE, novelty_k=k))


@pytest.mark.parametrize("key", ["elite_num", "novelty", "novelty_weigth", "archive_size"])
def test_nsr_es_rejects_unknown_keys(key):
    with pytest.raises(ValueError, match="unknown key"):
        _novelty_params(dict(BASE, **{key: 1}))


def _worker(rank, world, port, P, cyclic, q):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    from simple_es_b200 import dist as sdist
    from simple_es_b200.engine import cyclic_block, owned_ids, shard_bounds
    sdist.init_from_env(backend="gloo")
    full = np.random.RandomState(3).normal(0, 1, (P, 5, 4))                  # what an unsharded rollout would store
    full[::7] = -0.0
    fs = torch.full((P, 5, 4), float("nan"), dtype=torch.float64)           # stale garbage outside this rank's rows
    if cyclic:
        mine = owned_ids(P, rank, world, cyclic_block(P, world))
        fs[torch.from_numpy(mine)] = torch.from_numpy(full[mine])
        mask = torch.ones(P, dtype=torch.bool)
        mask[torch.from_numpy(mine)] = False
        sdist.exchange_fitness_masked(fs, mask)
    else:
        lo, hi = shard_bounds(P, rank, world)
        fs[lo:hi] = torch.from_numpy(full[lo:hi])
        sdist.exchange_fitness(fs, lo, hi)
    # equal values everywhere; a -0.0 may come back as +0.0 from the summing exchanges (distances cannot tell them apart)
    q.put((rank, bool(np.array_equal(fs.numpy(), full)), fs.numpy().tobytes()))
    dist.destroy_process_group()


@pytest.mark.parametrize("P,cyclic", [(64, False), (97, False), (97, True), (4096, True)])
def test_final_states_exchange_world2_gloo(P, cyclic):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29000 + (os.getpid() + P + 7 * cyclic) % 300
    procs = [ctx.Process(target=_worker, args=(r, 2, port, P, cyclic, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=120) for _ in procs)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    (_, ok0, b0), (_, ok1, b1) = res
    assert ok0 and ok1
    assert b0 == b1                                                          # bit-identical on every rank


def _novelty_case(rng, n, A, sd):
    """Behaviours and an archive with the value families the kernel must get right: rows near archive rows, exact duplicates
    (distance 0), integer lattice points (ties at every place), magnitudes from 1e-160 to 1e160 (squares that underflow to
    subnormals or 0 and overflow to inf) and rows whose every distance is inf."""
    arch = rng.normal(0, 1, (A, sd))
    arch[A // 4:A // 2] = rng.integers(-2, 3, (A // 2 - A // 4, sd))
    arch[A // 2:A // 2 + A // 8] = arch[:A // 8]
    wide = rng.uniform(-160, 160, (A // 8, sd))
    arch[A - A // 8:] = np.sign(rng.normal(size=wide.shape)) * 10.0 ** wide
    arch = arch[rng.permutation(A)]
    bc = rng.normal(0, 1, (n, sd))
    fam = rng.integers(0, 6, n)
    src = arch[rng.integers(0, A, n)]
    bc[fam == 0] = src[fam == 0] + rng.normal(0, 1e-9, (int((fam == 0).sum()), sd))
    bc[fam == 1] = src[fam == 1]
    bc[fam == 2] = rng.integers(-2, 3, (int((fam == 2).sum()), sd))
    w = rng.uniform(-160, 160, (int((fam == 3).sum()), sd))
    bc[fam == 3] = np.sign(rng.normal(size=w.shape)) * 10.0 ** w
    bc[fam == 4] = 1e200
    return bc, arch


def test_novelty_table_equals_the_loop():
    """nref.novelty_table (chunked, vectorised, one distance pass for every archive prefix and k) gives nref.novelty's bits
    for every prefix and k, chunk boundaries included; the cases reach 0, subnormal and inf distances."""
    rng = np.random.default_rng(0)
    for sd in (2, 4, 8, 12):
        bc, arch = _novelty_case(rng, 300, 70, sd)
        sizes, ks = [1, 2, 3, 16, 17, 32, 33, 70], [1, 2, 3, 4, 5, 8, 9, 16, 17, 32]
        tab = nref.novelty_table(bc, arch, sizes, ks, chunk=97, threads=3)
        for a in sizes:
            for k in ks:
                want = nref.novelty(bc, arch[:a], k)
                assert np.array_equal(tab[a, k].view(np.int64), want.view(np.int64)), (sd, a, k)
        v = tab[70, 32]
        assert np.isinf(v).any() and np.isfinite(v).any() and (tab[70, 1] == 0).any()


def _population(twin, env, gru, ids_n, final):
    rng = np.random.default_rng(1)
    if env.startswith("CartPole"):
        D = twin.param_count(4, 2, gru)
        mu = rng.normal(0, 0.3, (1, D)).astype(np.float32)
        return mu, twin.population_cartpole(mu, gru=gru, sigma=0.5, seed=3, gen=2, group=1000, n_head=1, n=ids_n, E=3, nthreads=4,
                                            final=final)
    if env == "simple_spread":
        N = 3 if gru else 2
        D = twin.param_count(6 * N, 5, gru) if gru else 6 * N * 32 + 32 + 165
        mu = rng.normal(0, 0.3, (1, D)).astype(np.float32)
        return mu, twin.population_mpe(mu, N=N, gru=gru, sigma=0.2, seed=3, gen=2, group=1000, n_head=1, n=ids_n, E=3, init_mode=1,
                                       final=final)
    obs, act, _, _ = twin.classic_dims(env)
    D = twin.param_count(obs, act, gru)
    mu = rng.normal(0, 0.5, (1, D)).astype(np.float32)
    return mu, twin.population_classic(env, mu, gru=gru, sigma=2.0, seed=3, gen=2, group=1000, n_head=1, n=ids_n, E=3, nthreads=4,
                                       max_step=60 if gru else None, final=final)


@pytest.mark.parametrize("gru", [False, True])
@pytest.mark.parametrize("env", ["CartPole-v1", "MountainCar-v0", "Acrobot-v1", "Pendulum-v0", "simple_spread"])
def test_twin_population_final_states_equal_the_traces(env, gru):
    """tw_population_* with a final-state buffer: fitness and steps as without it, and every row equal to the last trace row
    of the twin's single-episode rollout (nref.final_states) of the same offspring and episode."""
    from oracle import twin
    twin.build()
    n = 24
    mu, (fit, steps, fs) = _population(twin, env, gru, n, True)
    _, (fit0, steps0) = _population(twin, env, gru, n, False)
    assert np.array_equal(fit, fit0) and np.array_equal(steps, steps0)
    sigma = 0.5 if env.startswith("CartPole") else 0.2 if env == "simple_spread" else 2.0
    if gru and env in twin.CLASSIC_ENVS:          # the population ran at max_step 60: traces cut at the same step
        want = _classic_final_states(twin, env, mu, n, sigma)
    else:
        kw = dict(n_agents=3 if gru else 2, init_mode=1) if env == "simple_spread" else {}
        want = nref.final_states(twin, env, mu, np.arange(n), 3, sigma, 3, 2, 1000, 1, gru=gru, **kw)
    assert fs.shape == want.shape and np.array_equal(fs.view(np.int64), want.view(np.int64))


def _classic_final_states(twin, env, mu, n, sigma):
    W = twin.materialize(mu, sigma, 3, 2, 1000, 1, np.arange(n))
    rows = []
    for i in range(n):
        per = []
        for e in range(3):
            st = twin.classic_init(env, 3, 0, 2, i, e)
            _, k, tr, _ = twin.rollout_classic(env, W[i], E=1, max_step=60, init=np.asarray(st)[None], trace_steps=60, gru=True)
            per.append(tr[int(k) - 1])
        rows.append(per)
    return np.asarray(rows)

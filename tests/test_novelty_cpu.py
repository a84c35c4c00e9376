"""Host logic of nsr_es without a device: the strategy section's validation, its population layout, and the exchange of
final states ([P, E, state_dim]) between world-size-2 gloo ranks through the generalised fitness exchange."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

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

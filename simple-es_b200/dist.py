"""Population sharding across ranks (one process per GPU).

The population shards block-cyclically (engine.owned_ids; default) or by contiguous offspring-id ranges
(engine.shard_bounds); the only exchange of
a generation is the fitness vector (P float64 = 512 kB at P = 65536).  Every rank then ranks and
updates redundantly from identical inputs and identical Philox seeds, so parameters never travel.
Replaces the reference's only "distribution": multiprocessing.Pool.map over pickled
(env, offspring, eval_ep_num) tasks (learning_strategies/evolution/loop.py:66-78).
"""
import os

import torch
import torch.distributed as dist


def world():
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def init_from_env(backend=None):
    """Initialise torch.distributed from torchrun's env (RANK / WORLD_SIZE / MASTER_*) if present."""
    if "RANK" in os.environ and "WORLD_SIZE" in os.environ and int(os.environ["WORLD_SIZE"]) > 1:
        if not dist.is_initialized():
            if backend is None:
                backend = "nccl" if torch.cuda.is_available() else "gloo"
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            os.environ.setdefault("MASTER_PORT", "29500")
            dist.init_process_group(backend=backend)
    return world()


def exchange_fitness(fitness, lo, hi):
    """Make the full fitness vector [P] (or any [P, ...] tensor, e.g. nsr_es's final states) available on every rank;
    `fitness[lo:hi]` holds this rank's slice on entry.  Equal shards: one all_gather (NCCL over NVLink).  Ragged shards
    (simple_evolution's P = n + 1): all_reduce(SUM) of the zero-padded vector, which is exact
    because x + 0.0 == x."""
    rank, ws = world()
    if ws == 1:
        return fitness
    P = fitness.shape[0]
    if P % ws == 0:
        dist.all_gather_into_tensor(fitness, fitness[lo:hi].clone())
    else:
        fitness[:lo].zero_()
        fitness[hi:].zero_()
        dist.all_reduce(fitness, op=dist.ReduceOp.SUM)
    return fitness


def exchange_fitness_masked(fitness, not_mine):
    """The same for a non-contiguous (block-cyclic) slice: `not_mine` is a bool mask [P] of the rows other ranks own.
    all_reduce(SUM) of the tensor with those rows zeroed -- exact, every entry has exactly one non-zero contributor."""
    rank, ws = world()
    if ws == 1:
        return fitness
    fitness.masked_fill_(not_mine.view((-1,) + (1,) * (fitness.dim() - 1)), 0.0)
    dist.all_reduce(fitness, op=dist.ReduceOp.SUM)
    return fitness


def sum_scalar(t):
    rank, ws = world()
    if ws > 1:
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return t

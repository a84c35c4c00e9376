"""Novelty search with reward (nsr_es, DESIGN.md section 4.10) on the B200.

* The final-state instances of K1 at full size against the twin (tests/novelty_reference.py), with fitness and steps
  unchanged, for every env x {MLP, GRU} family.
* nsr_es with novelty_weight 0 trains exactly as openai_es; with 0.5 its shaped vector and update equal a host restatement
  built from the GPU's own final states; a resumed run continues bit for bit, archive included; two ranks equal one GPU.
"""
import os
import sys

import numpy as np
import pytest
import yaml

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, ROOT)

import k23_reference as k23  # noqa: E402
import novelty_reference as nref  # noqa: E402
from test_gpu_evaluate import engine  # noqa: E402


def same_bits(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and np.array_equal(a.view(np.uint8), b.view(np.uint8))


# (env, gru, n_agents, population)
FULL = [("CartPole-v1", False, 1, 65536), ("CartPole-v1", True, 1, 4096),
        ("simple_spread", False, 2, 16384), ("simple_spread", False, 3, 16384),
        ("simple_spread", True, 2, 4096), ("simple_spread", True, 3, 4096),
        ("MountainCar-v0", False, 1, 16384), ("MountainCar-v0", True, 1, 4096),
        ("Acrobot-v1", False, 1, 16384), ("Acrobot-v1", True, 1, 4096),
        ("Pendulum-v0", False, 1, 16384), ("Pendulum-v0", True, 1, 4096)]


@pytest.mark.parametrize("env,gru,N,P", FULL, ids=lambda x: str(x))
def test_gpu_final_states_equal_twin(twin, env, gru, N, P):
    """Fitness and steps equal the plain instance's; the final states of a sample of ids (both ends of the population and a
    random draw) equal the twin's; every row is written.  CartPole MLP runs the converged generation-30 population."""
    E, seed = 5, 11
    eng = engine(env, gru, False, N, seed=seed, population=P, eval_ep_num=E)
    if env == "CartPole-v1" and not gru:
        import bench
        st = bench.bench_state()
        mu, gen, sigma = st["mu"][None].astype(np.float32), 30, st["sigma"]
    else:
        mu, gen, sigma = np.random.default_rng(4).normal(0, 0.5, (1, eng.D)).astype(np.float32), 3, 0.3
    parents = torch.from_numpy(mu).cuda()
    fit0, steps0 = (t.cpu().numpy() for t in eng.rollout(gen, sigma, parents))
    fs = torch.full((P, E, eng.state_dim), float("nan"), dtype=torch.float64, device="cuda")
    eng.set_final_states(fs)
    fit, steps = (t.cpu().numpy() for t in eng.rollout(gen, sigma, parents))
    eng.set_final_states(None)
    got = fs.cpu().numpy()
    assert same_bits(fit, fit0) and same_bits(steps, steps0)
    assert not np.isnan(got).any()
    ids = np.unique(np.concatenate([np.arange(48), np.arange(P - 48, P), np.random.default_rng(P).choice(P, 96, replace=False)]))
    want = nref.final_states(twin, env, mu, ids, E, sigma, seed, gen, P, 1, gru=gru, n_agents=N)
    assert same_bits(got[ids], want)


def _strategy(name, P=4096, w=0.5, k=10, seed=5, conf="mountaincar_nsr.yaml", engine_cfg=None):
    from simple_es_b200.strategies import STRATEGIES
    cfg = yaml.load(open(os.path.join(ROOT, "conf", conf)), Loader=yaml.FullLoader)
    strat = dict(cfg["strategy"], name=name, offspring_num=P)
    if name == "nsr_es":
        strat.update(novelty_weight=w, novelty_k=k)
    else:
        strat.pop("novelty_weight", None)
        strat.pop("novelty_k", None)
    return STRATEGIES[name](strat, cfg["env"], cfg["network"], 5, seed, 0, dict(cfg["engine"], **(engine_cfg or {})))


def _snap(s):
    torch.cuda.synchronize()
    return [s.parents.cpu().numpy().copy(), s.m.cpu().numpy().copy(), s.v.cpu().numpy().copy(), s.fitness.cpu().numpy().copy()]


@pytest.mark.parametrize("conf", ["mountaincar_nsr.yaml", "cartpole_openai.yaml"])
def test_gpu_nsr_w0_trains_as_openai_es(conf):
    """novelty_weight 0: mu, m, v and fitness equal openai_es's, bit for bit, over 10 generations."""
    a, b = _strategy("nsr_es", w=0.0, conf=conf), _strategy("openai_es", conf=conf)
    for g in range(10):
        a.step(); b.step()
        for x, y, name in zip(_snap(a), _snap(b), ("mu", "m", "v", "fitness")):
            assert same_bits(x, y), (g, name)
    assert a.n_archive == 10


def centered(x):
    """K2's centered ranks (DESIGN.md section 4.5) in numpy, bit for bit: ranks by numpy's stable sort (ties by descending
    index), (n-1-r)/(n-1) - 0.5 divided by the closed-form std."""
    order = k23.rank_ref(x)
    n = x.size
    stdv = np.sqrt(np.float64(n + 1) / (12.0 * np.float64(n - 1)))
    out = np.empty(n)
    r = np.arange(n, dtype=np.float64)
    out[order] = ((np.float64(n - 1) - r) / np.float64(n - 1) - 0.5) / stdv
    return out


@pytest.mark.parametrize("conf,P", [("mountaincar_nsr.yaml", 4096), ("cartpole_openai.yaml", 3000)])
def test_gpu_nsr_equals_host_restatement(conf, P):
    """novelty_weight 0.5, 5 generations: from the GPU's own final states, numpy rebuilds the behaviours, the archive, the
    novelty, both centered-rank shapings and the blend; the shaped vector is the GPU's bit for bit, and ses_update_openai fed
    the host vector from the pre-step state gives the GPU's mu, m and v."""
    s = _strategy("nsr_es", P=P, w=0.5, k=3, conf=conf)
    ref = _strategy("openai_es", P=P, conf=conf)                 # a second handle: K3 alone, on the host's vector
    archive = []
    for g in range(5):
        mu0, m0, v0, _ = _snap(s)
        t0, sigma0 = s.t, s.sigma
        s.step()
        torch.cuda.synchronize()
        fs = s.final_states.cpu().numpy()
        bc = nref.behavior(fs)
        assert same_bits(s.bc.cpu().numpy(), bc), g
        archive.append(bc[0])
        nov = nref.novelty(bc, np.asarray(archive), 3)
        assert same_bits(s.novelty.cpu().numpy(), nov), g
        fit = s.fitness.cpu().numpy()
        shaped = nref.blend(centered(fit), centered(nov), 0.5)
        assert same_bits(s.shaped.cpu().numpy(), shaped), g
        mu, m, v = (torch.from_numpy(a).cuda() for a in (mu0[0], m0, v0))
        ref.engine.update_openai(g, sigma0, s.lr, t0 + 1, torch.from_numpy(shaped).cuda(), mu, m, v)
        torch.cuda.synchronize()
        assert same_bits(s.parents[0].cpu().numpy(), mu.cpu().numpy()), g
        assert same_bits(s.m.cpu().numpy(), m.cpu().numpy()) and same_bits(s.v.cpu().numpy(), v.cpu().numpy()), g
    assert same_bits(s.archive[:5].cpu().numpy(), np.asarray(archive))


def test_gpu_nsr_resume_continues_bit_for_bit():
    """13 generations, state(), a new run load_state()s it, 7 more == 20 uninterrupted: mu, m, v, fitness and the archive,
    which outgrows its first allocation of 16 rows after the resume.  A run with another novelty_k or novelty_weight is
    refused."""
    whole = _strategy("nsr_es")
    for _ in range(20):
        whole.step()
    first = _strategy("nsr_es")
    for _ in range(13):
        first.step()
    st = first.state()
    second = _strategy("nsr_es")
    second.load_state(st)
    for _ in range(7):
        second.step()
    for x, y, name in zip(_snap(second), _snap(whole), ("mu", "m", "v", "fitness")):
        assert same_bits(x, y), name
    assert second.n_archive == whole.n_archive == 20
    assert same_bits(second.archive[:20].cpu().numpy(), whole.archive[:20].cpu().numpy())
    with pytest.raises(ValueError, match="novelty_k"):
        _strategy("nsr_es", k=4).load_state(st)
    with pytest.raises(ValueError, match="novelty_weight"):
        _strategy("nsr_es", w=0.25).load_state(st)


def _worker(rank, world, port, exchange, shard, q):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    from simple_es_b200 import dist as sdist
    sdist.init_from_env()
    torch.cuda.set_device(rank)
    from simple_es_b200.strategies import STRATEGIES
    cfg = yaml.load(open(os.path.join(ROOT, "conf", "mountaincar_nsr.yaml")), Loader=yaml.FullLoader)
    strat = dict(cfg["strategy"], offspring_num=3001)
    s = STRATEGIES["nsr_es"](strat, cfg["env"], cfg["network"], 5, 3, rank, dict(cfg["engine"], fitness_exchange=exchange, shard=shard))
    for _ in range(4):
        s.step()
    torch.cuda.synchronize()
    q.put((rank, s.parents.cpu().numpy(), s.fitness.cpu().numpy(), s.archive[:s.n_archive].cpu().numpy(), s.final_states.cpu().numpy()))
    import torch.distributed as dist
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("exchange,shard", [("nccl", "cyclic"), ("nccl", "contiguous"), ("peer", "cyclic"), ("peer", "contiguous")])
def test_gpu_nsr_two_ranks_equal_single_gpu(exchange, shard):
    import torch.multiprocessing as mp
    from simple_es_b200.strategies import STRATEGIES
    cfg = yaml.load(open(os.path.join(ROOT, "conf", "mountaincar_nsr.yaml")), Loader=yaml.FullLoader)
    one = STRATEGIES["nsr_es"](dict(cfg["strategy"], offspring_num=3001), cfg["env"], cfg["network"], 5, 3, 0, dict(cfg["engine"]))
    for _ in range(4):
        one.step()
    want = (one.parents.cpu().numpy(), one.fitness.cpu().numpy(), one.archive[:one.n_archive].cpu().numpy(), one.final_states.cpu().numpy())
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29900 + os.getpid() % 90
    procs = [ctx.Process(target=_worker, args=(r, 2, port, exchange, shard, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted((q.get(timeout=600) for _ in procs), key=lambda r: r[0])
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    for rank, *got in res:
        for name, g, w in zip(("mu", "fitness", "archive"), got[:3], want[:3]):
            assert same_bits(g, w), (rank, name)
        assert np.array_equal(got[3], want[3]), rank            # equal values (a summing exchange may turn -0.0 into +0.0)

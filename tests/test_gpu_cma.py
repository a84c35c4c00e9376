"""sep_cma_es (DESIGN.md section 4.11) on the B200.

* The kernels at full size against tests/cma_reference.py: CartPole MLP at P = 65536 and CartPole-GRU at P = 4097 (D = 6562).
* Ten B200Loop generations, each one's device state equal to the numpy step from the previous GPU state; the same seed twice
  gives the same bits; a resume from resume_ep_5.pt continues bit for bit; the saved ep_<n>.pt loads in eval_es.py; two ranks
  (peer and nccl, block-cyclic and contiguous shards) equal one GPU.
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

import cma_reference as cref  # noqa: E402
import k23_reference as k23  # noqa: E402


def same_bits(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and np.array_equal(a.view(np.uint8), b.view(np.uint8))


def _t(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.mark.parametrize("gru,P", [(False, 65536), (True, 4097)], ids=["mlp-65536", "gru-4097"])
def test_gpu_cma_kernels_full_size(twin, gru, P):
    """Samples of every offspring, the weight scatter and two updates (h_sigma = 0, then 1) bit for bit, sigma within 2 ulp."""
    from simple_es_b200.engine import RolloutEngine, sep_cma_constants, sep_cma_threshold
    seed = 21
    eng = RolloutEngine("CartPole-v1", 4, 2, gru, False, 500, 1, P, P, 0, 1, seed=seed)
    D, mu = eng.D, P // 2
    k = sep_cma_constants(D, P, mu)
    rng = np.random.default_rng(P)
    mean, c, ps, pc = rng.normal(0, 0.3, D), rng.uniform(0.2, 3.0, D), 3000.0 * rng.normal(0, 1, D), rng.normal(0, 0.5, D)
    sigma = np.array([0.4])
    hs = []
    for gen in (0, 60):
        z = cref.normals(twin, seed, gen, range(P), D)
        x = eng.cma_sample(gen, _t(mean), _t(c), _t(sigma))
        assert same_bits(x.cpu().numpy(), cref.sample(mean, c, sigma[0], z)), gen
        order = rng.permutation(P).astype(np.int32)
        dev = [_t(a) for a in (mean, c, ps, pc, sigma)]
        s = torch.full((P,), float("nan"), dtype=torch.float64, device="cuda")
        parent = torch.empty(D, dtype=torch.float32, device="cuda")
        eng.cma_update(gen, _t(order), k, _t(k["weights"]), s, *dev, parent)
        s_ref = cref.weights(order, k["weights"], mu, P)
        assert same_bits(s.cpu().numpy(), s_ref), gen
        t1, t2 = cref.tables(s_ref, z)
        ref = cref.update(t1, t2, k, sep_cma_threshold(k, gen), mean, c, ps, pc, sigma[0])
        got = [t.cpu().numpy() for t in dev]
        for name, g, w in zip(("mean", "c", "p_sigma", "p_c"), got[:4], ref[:4]):
            assert same_bits(g, w), (gen, name)
        assert same_bits(parent.cpu().numpy(), ref[5]), gen
        assert cref.ulps(got[4][0], ref[4]) <= 2, (gen, got[4][0], ref[4])
        hs.append(ref[6])
        mean, c, ps, pc, sigma = got[0], got[1], 1e-6 * got[2], got[3], got[4]
    assert hs == [False, True]
    eng.close()


def _cfg(conf="cartpole_sep_cma.yaml", **strategy):
    cfg = yaml.load(open(os.path.join(ROOT, "conf", conf)), Loader=yaml.FullLoader)
    cfg["strategy"].update(strategy)
    return cfg


def _state(s):
    torch.cuda.synchronize()
    return [t.cpu().numpy().copy() for t in (s.mean, s.c, s.p_sigma, s.p_c, s.sigma_dev, s.parents[0], s.fitness)]


@pytest.mark.parametrize("conf", ["cartpole_sep_cma.yaml", "pendulum_sep_cma.yaml"])
def test_gpu_cma_loop_generations_equal_numpy(twin, conf):
    """Ten one-generation B200Loop runs: each generation's samples, order, weights and state equal the numpy step from the
    previous GPU state (sigma within 2 ulp, and the next generation continues from the GPU's own sigma)."""
    from simple_es_b200.engine import sep_cma_threshold
    from simple_es_b200.loop import B200Loop
    loop = B200Loop(_cfg(conf), 1, 1, 3, save_model_period=0, seed=9, quiet=True)
    s = loop.strategy
    P, D, k = s.P, s.D, s.consts
    prev = _state(s)
    for g in range(10):
        loop.run()
        now = _state(s)
        mean, c, ps, pc, sigma = prev[:5]
        z = cref.normals(twin, 9, g, range(P), D)
        assert same_bits(s.samples.cpu().numpy(), cref.sample(mean, c, sigma[0], z)), g
        fit = now[6]
        order = s.order.cpu().numpy()
        assert np.array_equal(order, k23.rank_ref(fit)), g
        s_ref = cref.weights(order, k["weights"], s.mu, P)
        assert same_bits(s.s.cpu().numpy(), s_ref), g
        ref = cref.update(*cref.tables(s_ref, z), k, sep_cma_threshold(k, g), mean, c, ps, pc, sigma[0])
        for name, a, b in zip(("mean", "c", "p_sigma", "p_c"), now[:4], ref[:4]):
            assert same_bits(a, b), (g, name)
        assert same_bits(now[5], ref[5]), g
        assert cref.ulps(now[4][0], ref[4]) <= 2, g
        assert loop.history[-1][2] == float(now[4][0])            # the loop reports the device sigma
        prev = now
    assert s.generation == 10


def test_gpu_cma_same_seed_twice_is_identical():
    from simple_es_b200.loop import B200Loop
    runs = []
    for _ in range(2):
        loop = B200Loop(_cfg(), 6, 1, 3, save_model_period=0, seed=3, quiet=True)
        loop.run()
        runs.append(_state(loop.strategy))
    for a, b in zip(*runs):
        assert same_bits(a, b)


def test_gpu_cma_resume_and_eval_es(tmp_path, capsys):
    """10 generations == 5, resume_ep_5.pt, 5 more: the whole state bit for bit.  The run's ep_10.pt loads in eval_es.py and
    evaluates as the policy elite_flat() returns.  A run with another elite_num refuses the resume state."""
    from simple_es_b200.loop import B200Loop
    whole_cfg = _cfg()
    whole_cfg["engine"]["save_state"] = True
    whole = B200Loop(whole_cfg, 10, 1, 3, save_model_period=5, seed=8, quiet=True, save_dir=str(tmp_path / "whole"))
    whole.run()
    b_cfg = _cfg()
    b_cfg["engine"]["resume"] = str(tmp_path / "whole" / "saved_models" / "resume_ep_5.pt")
    b = B200Loop(b_cfg, 5, 1, 3, save_model_period=0, seed=8, quiet=True)
    assert b.strategy.generation == 5
    b.run()
    for x, y in zip(_state(b.strategy), _state(whole.strategy)):
        assert same_bits(x, y)
    assert [h[1:3] for h in b.history] == [h[1:3] for h in whole.history[5:]]
    wrong = _cfg(elite_num=100)
    wrong["engine"]["resume"] = b_cfg["engine"]["resume"]
    with pytest.raises(ValueError, match="elite_num"):
        B200Loop(wrong, 1, 1, 3, save_model_period=0, seed=8, quiet=True)

    import eval_es
    ckpt = str(tmp_path / "whole" / "saved_models" / "ep_10.pt")
    cfg_path = str(tmp_path / "cfg.yaml")
    with open(cfg_path, "w") as fh:
        yaml.dump(_cfg(), fh)
    ret, lng = eval_es.main(["--cfg-path", cfg_path, "--ckpt-path", ckpt, "--episodes", "20", "--seed", "8"])
    want_r, want_l = whole.strategy.engine.evaluate(whole.strategy.elite_flat(), 20, round=0)
    # eval_es keys its episodes by --seed; the training engine has the same seed
    assert np.array_equal(ret, want_r.cpu().numpy()) and np.array_equal(lng, want_l.cpu().numpy())


def _worker(rank, world, port, exchange, shard, q):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    from simple_es_b200 import dist as sdist
    sdist.init_from_env()
    torch.cuda.set_device(rank)
    from simple_es_b200.strategies import STRATEGIES
    cfg = _cfg(offspring_num=3001)
    s = STRATEGIES["sep_cma_es"](cfg["strategy"], cfg["env"], cfg["network"], 3, 3, rank, dict(cfg["engine"], fitness_exchange=exchange, shard=shard))
    for _ in range(4):
        s.step()
    q.put((rank, _state(s)))
    import torch.distributed as dist
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("exchange,shard", [("nccl", "cyclic"), ("nccl", "contiguous"), ("peer", "cyclic"), ("peer", "contiguous")])
def test_gpu_cma_two_ranks_equal_single_gpu(exchange, shard):
    import torch.multiprocessing as mp
    from simple_es_b200.strategies import STRATEGIES
    cfg = _cfg(offspring_num=3001)
    one = STRATEGIES["sep_cma_es"](cfg["strategy"], cfg["env"], cfg["network"], 3, 3, 0, dict(cfg["engine"]))
    for _ in range(4):
        one.step()
    want = _state(one)
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
    for rank, got in res:
        for i, (g, w) in enumerate(zip(got, want)):
            assert same_bits(g, w), (rank, i)

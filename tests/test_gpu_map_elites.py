"""map_elites (DESIGN.md section 4.12) on the B200.

* ses_map_insert / ses_map_select at full size against tests/map_elites_reference.py, bit for bit: CartPole MLP at P = 65536
  with 32 x 32 cells and with 2^20 cells, MountainCar at P = 16384, CartPole-GRU at P = 4097 (D = 6562), simple_spread N = 3
  with a 4-dimensional descriptor.  Each case prints its shapes and the counts it compared.
* Ten B200Loop generations, each generation's archive and parent table equal to the numpy step from the previous GPU state; the
  same seed twice gives the same bits; a resume from resume_ep_5.pt continues bit for bit; ep_10.pt and archive_ep_10.pt
  evaluate in eval_es.py; two ranks (peer and nccl, cyclic and contiguous shards) equal one GPU.
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
import map_elites_reference as mref  # noqa: E402


def same_bits(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and np.array_equal(a.view(np.uint8), b.view(np.uint8))


def _t(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _np(a):
    torch.cuda.synchronize()
    return {k: v.cpu().numpy().copy() for k, v in a.items()}


# (env, gru, N, P, dims, low, high, cells)
FULL = {
    "cartpole-65536-32x32": ("CartPole-v1", False, 1, 65536, [0, 2], [-2.4, -0.2095], [2.4, 0.2095], [32, 32]),
    "cartpole-65536-2^20": ("CartPole-v1", False, 1, 65536, [0, 1, 2, 3], [-2.4, -3, -0.2095, -3], [2.4, 3, 0.2095, 3], [32, 32, 32, 32]),
    "mountaincar-16384": ("MountainCar-v0", False, 1, 16384, [0, 1], [-1.2, -0.07], [0.6, 0.07], [32, 32]),
    "cartpole-gru-4097": ("CartPole-v1", True, 1, 4097, [2, 0], [-0.2095, -2.4], [0.2095, 2.4], [40, 25]),
    "spread3-4d": ("simple_spread", False, 3, 16384, [0, 1, 6, 7], [-1.5, -1.5, -1, -1], [1.5, 1.5, 1, 1], [8, 8, 6, 6]),
}


@pytest.mark.parametrize("case", list(FULL))
def test_gpu_map_kernels_full_size(twin, case):
    """Two insertions (the second onto the first's archive, with ties, NaNs and out-of-range behaviour) and the selections
    after each, against numpy."""
    from simple_es_b200.engine import RolloutEngine
    env, gru, N, P, dims, low, high, cells = FULL[case]
    seed, sigma = 17, 0.3
    obs, act = {"CartPole-v1": (4, 2), "MountainCar-v0": (2, 3), "simple_spread": (18, 5)}[env]
    eng = RolloutEngine(env, obs, act, gru, False, None, 1, P, 1, 0, P, seed=seed, n_agents=N)
    spec = mref.Spec(dims, low, high, cells)
    sd, D = eng.state_dim, eng.D
    rng = np.random.default_rng(P + len(dims))
    a = mref.empty(spec, sd, D)
    dev = {k: _t(v) for k, v in a.items()}
    seed_row = rng.normal(0, 1, D).astype(np.float32)
    stats = torch.zeros(4, dtype=torch.float64, device="cuda")
    parents_out = torch.empty((P, D), dtype=torch.float32, device="cuda")
    for gen in (0, 1):
        parents = rng.normal(0, 1, (P, D)).astype(np.float32)
        span = np.array(high) - np.array(low)
        bc = rng.uniform(-0.1, 1.1, (P, sd)) * 1.0
        bc[:, dims] = np.array(low) + bc[:, dims] * span
        bc[rng.random(P) < 0.01, dims[0]] = np.nan
        bc[rng.random(P) < 0.01, dims[-1]] = np.inf
        fit = np.round(rng.normal(0, 20, P), 0)              # many ties
        fit[rng.random(P) < 0.01] = np.nan
        order = k23.rank_ref(fit)
        eng.map_insert(gen, sigma, _t(parents), _t(order.astype(np.int32)), _t(fit), _t(bc), spec.ctype(), dev["F"], dev["B"],
                       dev["born"], dev["W"])
        a, entered = mref.insert(a, spec, order, fit, bc, gen, lambda ids: twin.materialize(parents, sigma, seed, gen, 1, 0, ids))
        got = _np(dev)
        for k in ("F", "B", "born", "W"):
            assert same_bits(got[k], a[k]), (case, gen, k)
        eng.map_select(gen + 1, spec.ctype(), dev["F"], dev["W"], _t(seed_row), stats, parents_out)
        st = stats.cpu().numpy()
        n_occ, best, bf, qd = mref.stats(a["F"])
        assert st[0] == n_occ and st[1] == best and same_bits(st[2:], np.array([bf, qd])), (case, gen)
        want = mref.select(twin, a, P, gen + 1, seed, seed_row)
        assert same_bits(parents_out.cpu().numpy(), want), (case, gen)
        print(f"{case}: P={P} D={D} n_cells={spec.n_cells} gen {gen}: {len(entered)} entered, {n_occ} occupied, "
              f"{P} parent rows x {D} compared")
    eng.close()


def _cfg(conf="cartpole_map_elites.yaml", **strategy):
    cfg = yaml.load(open(os.path.join(ROOT, "conf", conf)), Loader=yaml.FullLoader)
    cfg["strategy"].update(strategy)
    return cfg


def _state(s):
    torch.cuda.synchronize()
    return {"F": s.F.cpu().numpy().copy(), "B": s.B.cpu().numpy().copy(), "born": s.born.cpu().numpy().copy(),
            "W": s.W.cpu().numpy().copy(), "parents": s.parents.cpu().numpy().copy(), "stats": s.stats.cpu().numpy().copy(),
            "fitness": s.fitness.cpu().numpy().copy()}


@pytest.mark.parametrize("conf,n", [("cartpole_map_elites.yaml", 4096), ("mountaincar_map_elites.yaml", 4096)])
def test_gpu_map_loop_generations_equal_numpy(twin, conf, n):
    """Ten one-generation B200Loop runs: each one's order, archive, statistics and next parent table equal the numpy step from
    the previous GPU state."""
    from simple_es_b200.loop import B200Loop
    seed = 9
    loop = B200Loop(_cfg(conf, offspring_num=n), 1, 1, 3, save_model_period=0, seed=seed, quiet=True)
    s = loop.strategy
    spec = mref.Spec(s.dims, s.low, s.high, s.cells)
    prev = _state(s)
    assert same_bits(prev["parents"], np.zeros_like(prev["parents"]))
    filled = []
    for g in range(10):
        sigma = s.sigma
        loop.run()
        now = _state(s)
        fit, bc, order = now["fitness"], s.bc.cpu().numpy(), s.order.cpu().numpy()
        assert np.array_equal(order, k23.rank_ref(fit)), g
        a, _ = mref.insert({k: prev[k] for k in ("F", "B", "born", "W")}, spec, order, fit, bc, g,
                           lambda ids: twin.materialize(prev["parents"], sigma, seed, g, 1, 0, ids))
        for k in ("F", "B", "born", "W"):
            assert same_bits(now[k], a[k]), (g, k)
        n_occ, best, bf, qd = mref.stats(a["F"])
        assert now["stats"][0] == n_occ and now["stats"][1] == best and same_bits(now["stats"][2:], np.array([bf, qd])), g
        assert same_bits(now["parents"], mref.select(twin, a, s.P, g + 1, seed, np.zeros(s.D, np.float32))), g
        filled.append(n_occ)
        prev = now
    assert s.generation == 10 and filled[-1] > 1
    print(f"{conf}: P={s.P} cells filled per generation {filled}")


def test_gpu_map_same_seed_twice_is_identical():
    from simple_es_b200.loop import B200Loop
    runs = []
    for _ in range(2):
        loop = B200Loop(_cfg(), 6, 1, 3, save_model_period=0, seed=3, quiet=True)
        loop.run()
        runs.append(_state(loop.strategy))
    for k in runs[0]:
        assert same_bits(runs[0][k], runs[1][k]), k


def test_gpu_map_resume_and_eval_es(tmp_path):
    """10 generations == 5, resume_ep_5.pt, 5 more; a run with another descriptor refuses the state.  ep_10.pt evaluates as
    elite_flat(), and archive_ep_10.pt evaluates every elite as the engine does."""
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
    x, y = _state(b.strategy), _state(whole.strategy)
    for k in x:
        assert same_bits(x[k], y[k]), k
    assert [h[1:3] for h in b.history] == [h[1:3] for h in whole.history[5:]]
    wrong = _cfg(behavior_cells=[16, 16])
    wrong["engine"]["resume"] = b_cfg["engine"]["resume"]
    with pytest.raises(ValueError, match="behavior_cells"):
        B200Loop(wrong, 1, 1, 3, save_model_period=0, seed=8, quiet=True)

    import eval_es
    saved = tmp_path / "whole" / "saved_models"
    arch = torch.load(str(saved / "archive_ep_10.pt"))
    s = whole.strategy
    occ = np.flatnonzero(~np.isnan(y["F"]))
    assert np.array_equal(arch["cells"].numpy(), occ) and same_bits(arch["weights"].numpy(), y["W"][occ])
    assert np.array_equal(arch["coords"].numpy(), np.stack(np.unravel_index(occ, s.cells), 1))
    assert np.array_equal(arch["born_id"].numpy(), y["born"][occ, 1]) and same_bits(arch["fitness"].numpy(), y["F"][occ])
    cfg_path = str(tmp_path / "cfg.yaml")
    with open(cfg_path, "w") as fh:
        yaml.dump(_cfg(), fh)
    ret, lng = eval_es.main(["--cfg-path", cfg_path, "--ckpt-path", str(saved / "ep_10.pt"), "--episodes", "20", "--seed", "8"])
    want_r, want_l = s.engine.evaluate(s.elite_flat(), 20, round=0)
    assert np.array_equal(ret, want_r.cpu().numpy()) and np.array_equal(lng, want_l.cpu().numpy())
    assert same_bits(s.elite_flat().cpu().numpy(), y["W"][int(y["stats"][1])])
    out = str(tmp_path / "archive_returns.npz")
    ret, lng = eval_es.main(["--cfg-path", cfg_path, "--archive", str(saved / "archive_ep_10.pt"), "--episodes", "7", "--seed", "8",
                             "--out", out])
    want_r, want_l = s.engine.evaluate(torch.from_numpy(y["W"][occ]).cuda(), 7, round=0)
    assert ret.shape == (occ.size, 7) and np.array_equal(ret, want_r.cpu().numpy()) and np.array_equal(lng, want_l.cpu().numpy())
    z = np.load(out)
    assert np.array_equal(z["cells"], occ) and np.array_equal(z["returns"], ret)


def _worker(rank, world, port, exchange, shard, q):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    from simple_es_b200 import dist as sdist
    sdist.init_from_env()
    torch.cuda.set_device(rank)
    from simple_es_b200.strategies import STRATEGIES
    cfg = _cfg(offspring_num=3001)
    s = STRATEGIES["map_elites"](cfg["strategy"], cfg["env"], cfg["network"], 3, 3, rank, dict(cfg["engine"], fitness_exchange=exchange, shard=shard))
    for _ in range(4):
        s.step()
    q.put((rank, _state(s)))
    import torch.distributed as dist
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("exchange,shard", [("nccl", "cyclic"), ("nccl", "contiguous"), ("peer", "cyclic"), ("peer", "contiguous")])
def test_gpu_map_two_ranks_equal_single_gpu(exchange, shard):
    import torch.multiprocessing as mp
    from simple_es_b200.strategies import STRATEGIES
    cfg = _cfg(offspring_num=3001)
    one = STRATEGIES["map_elites"](cfg["strategy"], cfg["env"], cfg["network"], 3, 3, 0, dict(cfg["engine"]))
    for _ in range(4):
        one.step()
    want = _state(one)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29800 + os.getpid() % 90
    procs = [ctx.Process(target=_worker, args=(r, 2, port, exchange, shard, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted((q.get(timeout=600) for _ in procs), key=lambda r: r[0])
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    for rank, got in res:
        for k in want:
            assert same_bits(got[k], want[k]), (rank, k)

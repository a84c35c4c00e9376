"""Policy evaluation (ses_evaluate, DESIGN.md section 4.9) through the product library on the B200: the twin's episodes under
the evaluation keying, the bit rule against ses_rollout in verification mode, invariances at large sizes, the loop's
engine.eval_every across a resume, and eval_es.py on a checkpoint of a training run."""
import os
import subprocess
import sys

import numpy as np
import pytest
import yaml

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))

import eval_reference as ref  # noqa: E402

CONFIGS = [("CartPole-v1", False, False, 1), ("CartPole-v1", False, True, 1), ("CartPole-v0", False, False, 1),
           ("CartPole-v1", True, True, 1), ("MountainCar-v0", False, False, 1), ("MountainCar-v0", True, False, 1),
           ("Acrobot-v1", False, False, 1), ("Acrobot-v1", True, False, 1), ("Pendulum-v0", False, False, 1),
           ("Pendulum-v0", True, False, 1), ("simple_spread", False, False, 2), ("simple_spread", True, False, 2),
           ("simple_spread", False, False, 3), ("simple_spread", True, False, 3)]


def engine(env, gru=False, pomdp=False, n_agents=2, seed=11, population=64, group=None, **kw):
    from simple_es_b200.engine import RolloutEngine
    obs, act = ref.dims(env, n_agents)
    return RolloutEngine(env, obs, act, gru, pomdp, None, kw.pop("eval_ep_num", 5), population, group or population,
                         kw.pop("n_head", 1), kw.pop("n_parents", 1), seed=seed, n_agents=n_agents,
                         discrete_action=env != "Pendulum-v0", **kw)


def policies(eng, n, seed):
    W = np.random.default_rng(seed).normal(0, 0.5, (n, eng.D)).astype(np.float32)
    if eng.D == 226:
        mu = np.zeros(226, np.float32)                        # balances the pole: 500-step episodes next to short ones
        w1 = mu[:128].reshape(32, 4); w2 = mu[160:224].reshape(2, 32)
        w1[0] = [0.0, 0.5, 10.0, 3.0]; w2[1, 0] = 5.0; w2[0, 0] = -5.0
        W[0] = mu
    return W


def _ids(c):
    return "%s-%s%s-N%d" % (c[0], "gru" if c[1] else "mlp", "-pomdp" if c[2] else "", c[3])


@pytest.mark.parametrize("cfg", CONFIGS, ids=_ids)
def test_gpu_evaluate_equals_twin(twin, cfg):
    """Every episode of a small call, and a sample of the episodes of a large one, bit for bit."""
    env, gru, pomdp, N = cfg
    eng = engine(env, gru, pomdp, N)
    W = policies(eng, 3, 1)
    Wd = torch.from_numpy(W).cuda()
    ret, lng = (t.cpu().numpy() for t in eng.evaluate(Wd, 70, round=6))
    tr, tl = ref.evaluate(twin, env, W, 70, seed=11, rnd=6, gru=gru, pomdp=pomdp, n_agents=N)
    assert np.array_equal(lng, tl) and np.array_equal(ret.view(np.int64), tr.view(np.int64))
    M = 1 << 16 if not gru else 1 << 13
    big_r, big_l = (t.cpu().numpy() for t in eng.evaluate(Wd, M, round=6))
    assert np.array_equal(big_r[:, :70], ret) and np.array_equal(big_l[:, :70], lng)      # episode m does not depend on M
    ms = np.random.default_rng(2).choice(M, 24, replace=False)
    init = np.stack([ref.eval_init(twin, env, 11, 6, int(m), N) for m in ms])
    sr, sl = ref.evaluate(twin, env, W, len(ms), gru=gru, pomdp=pomdp, n_agents=N, init_states=init)
    assert np.array_equal(big_l[:, ms], sl) and np.array_equal(big_r[:, ms], sr)


GOLDEN = {"rollout_cartpole_mlp": ("CartPole-v1", False, False), "rollout_cartpole_gru_pomdp": ("CartPole-v1", True, True),
          "rollout_mountaincar": ("MountainCar-v0", False, False), "rollout_mountaincar_gru": ("MountainCar-v0", True, False),
          "rollout_acrobot": ("Acrobot-v1", False, False), "rollout_acrobot_gru": ("Acrobot-v1", True, False),
          "rollout_pendulum": ("Pendulum-v0", False, False), "rollout_pendulum_gru": ("Pendulum-v0", True, False),
          "rollout_spread_n2": ("simple_spread", False, False), "rollout_spread_n2_gru": ("simple_spread", True, False),
          "rollout_spread_n3": ("simple_spread", False, False), "rollout_spread_n3_gru": ("simple_spread", True, False)}


@pytest.mark.parametrize("name", list(GOLDEN))
def test_gpu_evaluate_bit_rule_against_verification_rollout(golden, name):
    env, gru, pomdp = GOLDEN[name]
    g = golden(name)
    N = int(g["N"]) if "N" in g.files else 2
    W, init, E = g["W"], g["init"], int(g["E"])
    n = W.shape[0]
    eng = engine(env, gru, pomdp, N, population=n, eval_ep_num=E)
    Wd, Id = torch.from_numpy(W).cuda(), torch.from_numpy(init).cuda().reshape(-1)
    fit, steps = (t.cpu().numpy() for t in eng.rollout(0, 0.0, Wd[:1], w_override=Wd, init_states=Id))
    ret, lng = (t.cpu().numpy() for t in eng.evaluate(Wd, E, init_states=Id))
    for j in range(n):
        total = 0.0
        for e in range(E):
            total = total + ret[j, e]
        assert total / E == fit[j] and int(lng[j].sum()) == steps[j]
    np.testing.assert_allclose(fit, g["fitness"], rtol=1e-12 if env == "simple_spread" else 1e-4)


@pytest.mark.parametrize("env,gru", [("CartPole-v1", False), ("CartPole-v1", True), ("Acrobot-v1", True), ("simple_spread", False)])
def test_gpu_evaluate_invariances(twin, env, gru):
    M = 1 << 16 if not gru else 1 << 12
    eng = engine(env, gru)
    W = torch.from_numpy(policies(eng, 3, 4)).cuda()
    r1, l1 = eng.evaluate(W[1], M, round=9)
    r3, l3 = eng.evaluate(W[[2, 1, 0]], M, round=9)
    assert torch.equal(r3[1], r1[0]) and torch.equal(l3[1], l1[0])                       # other policies, any order
    r40, l40 = eng.evaluate(W[[2, 1, 0]], 40, round=9)
    assert torch.equal(r40, r3[:, :40]) and torch.equal(l40, l3[:, :40])
    # another round, other initial states: those of the evaluation keying at round 10 (a random Acrobot policy may well
    # return -500 from every one of them, so the returns alone need not differ)
    rb, lb = eng.evaluate(W[1], M, round=10)
    i9, i10 = (np.stack([ref.eval_init(twin, env, 11, r, m) for m in range(16)]) for r in (9, 10))
    assert not np.array_equal(i9, i10)
    re, le = eng.evaluate(W[1], 16, init_states=torch.from_numpy(i10).cuda().reshape(-1))
    assert torch.equal(re, rb[:, :16]) and torch.equal(le, lb[:, :16])
    # the handle's strategy layout, antithetic sampling, shard and initial-state mode play no part
    for other in (engine(env, gru, population=120, group=30, n_parents=4, antithetic=True, init_mode="fresh"),
                  engine(env, gru, population=256, group=256, n_head=2, id_begin=64, id_end=200),
                  engine(env, gru, population=512, shard=(3, 4, 16), eval_ep_num=3)):
        ro, lo = other.evaluate(W[[2, 1, 0]], M, round=9)
        assert torch.equal(ro, r3) and torch.equal(lo, l3)


def _cfg(name, **strategy):
    cfg = yaml.load(open(os.path.join(ROOT, "conf", name)), Loader=yaml.FullLoader)
    cfg["strategy"].update(strategy)
    return cfg


def test_gpu_loop_eval_every_survives_a_resume(tmp_path, capsys):
    """eval_every: 2 over 4 generations == 2 generations, stop, resume, 2 more: the same eval numbers and history."""
    from simple_es_b200.loop import B200Loop

    def cfg(**eng):
        c = _cfg("cartpole_openai.yaml", offspring_num=512)
        c["engine"].update(eval_every=2, eval_episodes=300, **eng)
        return c
    full = B200Loop(cfg(), 4, 1, 3, save_model_period=0, seed=7)
    full.run()
    out = capsys.readouterr().out
    assert out.count("  eval: 300 episodes, mean ") == 2
    a = B200Loop(cfg(save_state=True), 2, 1, 3, save_model_period=2, seed=7, quiet=True, save_dir=str(tmp_path / "a"))
    a.run()
    b = B200Loop(cfg(resume=str(tmp_path / "a" / "saved_models" / "resume_ep_2.pt")), 2, 1, 3, save_model_period=0, seed=7, quiet=True)
    b.run()
    assert [e[:7] for e in a.eval_history + b.eval_history] == [e[:7] for e in full.eval_history]
    assert [e[0] for e in full.eval_history] == [2, 4]
    assert [h[:3] for h in a.history + b.history] == [h[:3] for h in full.history]
    # the entry is the saved policy's: the engine's own evaluation of elite_flat() keyed by the generation
    ret, lng = full.strategy.engine.evaluate(full.strategy.elite_flat(), 300, round=4)
    assert full.eval_history[-1][2] == float(ret[0].cpu().mean()) and full.eval_history[-1][6] == float(lng[0].double().cpu().mean())


def test_gpu_eval_es_on_a_training_checkpoint(tmp_path):
    from simple_es_b200.engine import RolloutEngine
    from simple_es_b200.loop import B200Loop
    c = _cfg("cartpole_openai.yaml", offspring_num=1024)
    B200Loop(c, 4, 1, 5, save_model_period=2, seed=3, quiet=True, save_dir=str(tmp_path / "run")).run()
    ck = [str(tmp_path / "run" / "saved_models" / f) for f in ("ep_2.pt", "ep_4.pt")]
    cfg_path = tmp_path / "c.yaml"
    cfg_path.write_text(yaml.safe_dump(c))
    out = subprocess.run([sys.executable, os.path.join(ROOT, "eval_es.py"), "--cfg-path", str(cfg_path), "--ckpt-path", *ck,
                          "--episodes", "1000", "--seed", "5", "--round", "1", "--out", str(tmp_path / "r.npz")],
                         capture_output=True, text=True, cwd=ROOT, check=True).stdout.splitlines()
    z = np.load(tmp_path / "r.npz")
    assert z["returns"].shape == (2, 1000) and z["lengths"].dtype == np.int32 and list(z["ckpt_paths"]) == ck
    from simple_es_b200 import checkpoint
    eng = RolloutEngine("CartPole-v1", 4, 2, False, False, 500, 1, 2, 2, 1, 1, seed=5)
    W = torch.stack([checkpoint.state_dict_to_flat(torch.load(p), 4, 2, False) for p in ck]).cuda()
    ret, _ = eng.evaluate(W, 1000, round=1)
    assert np.array_equal(z["returns"], ret.cpu().numpy())
    for line, p, r in zip(out, ck, ret.cpu().numpy()):
        assert line.startswith(f"{p}: 1000 episodes, mean {r.mean():.2f}, ")

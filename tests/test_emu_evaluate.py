"""Policy evaluation (ses_evaluate, DESIGN.md section 4.9) on the SIMT emulator of tests/simt_emu: the evaluation instances
of the K1 kernels against the twin's single-episode rollouts under the evaluation keying (tests/eval_reference.py), the bit
rule that ties them to ses_rollout in verification mode, invariances and argument checks."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))

import eval_reference as ref  # noqa: E402


@pytest.fixture(scope="module")
def emu():
    from simt_emu import emu_engine
    emu_engine.load()
    return emu_engine.EmuEngine


def _p(a):
    return None if a is None else C.c_void_p(a.ctypes.data)


def evaluate(eng, policies, M, rnd=0, init_states=None):
    W = np.ascontiguousarray(policies, dtype=np.float32).reshape(-1, eng.D)
    ret = np.full((W.shape[0], M), np.nan)
    lng = np.full((W.shape[0], M), -1, dtype=np.int32)
    init = None if init_states is None else np.ascontiguousarray(init_states, dtype=np.float64)
    eng._check(eng.lib.ses_evaluate(eng._h, int(rnd), _p(W), W.shape[0], int(M), _p(init), _p(ret), _p(lng), None))
    return ret, lng


def balancing_policy():
    """CartPole MLP that balances the pole (bang-bang on theta + theta_dot): 500-step episodes."""
    mu = np.zeros(226, np.float32)
    w1 = mu[:128].reshape(32, 4); w2 = mu[160:224].reshape(2, 32)
    w1[0] = [0.0, 0.5, 10.0, 3.0]; w2[1, 0] = 5.0; w2[0, 0] = -5.0
    return mu


# (env, gru, pomdp, n_agents)
CONFIGS = [("CartPole-v1", False, False, 1), ("CartPole-v1", False, True, 1), ("CartPole-v0", False, False, 1),
           ("CartPole-v1", True, True, 1), ("CartPole-v1", True, False, 1),
           ("MountainCar-v0", False, False, 1), ("MountainCar-v0", True, False, 1),
           ("Acrobot-v1", False, False, 1), ("Acrobot-v1", True, False, 1),
           ("Pendulum-v0", False, False, 1), ("Pendulum-v0", True, False, 1),
           ("simple_spread", False, False, 2), ("simple_spread", True, False, 2),
           ("simple_spread", False, False, 3), ("simple_spread", True, False, 3)]


def make(emu, env, gru=False, pomdp=False, n_agents=2, seed=7, **kw):
    obs, act = ref.dims(env, n_agents)
    kw.setdefault("population", 16)
    kw.setdefault("group", kw["population"])
    return emu(env_name=env, obs_dim=obs, act_dim=act, gru=gru, pomdp=pomdp, n_agents=n_agents, max_step=None, seed=seed, **kw)


def policies(eng, n, seed=0, scale=0.5):
    W = np.random.default_rng(seed).normal(0, scale, (n, eng.D)).astype(np.float32)
    if eng.D == 226 and n > 1:
        W[1] = balancing_policy()                       # long episodes next to short ones
    return W


def _ids(c):
    return "%s-%s%s-N%d" % (c[0], "gru" if c[1] else "mlp", "-pomdp" if c[2] else "", c[3])


@pytest.mark.parametrize("cfg", CONFIGS, ids=_ids)
@pytest.mark.parametrize("n_pol,M", [(1, 1), (3, 33), (1, 31), (3, 70)])
def test_emu_evaluate_equals_twin(emu, twin, cfg, n_pol, M):
    env, gru, pomdp, N = cfg
    if gru and M > 33:
        M = 12                                           # GRU chunks are 5 (or 3, 2) episodes wide: 12 leaves a partial one too
    eng = make(emu, env, gru, pomdp, N)
    W = policies(eng, n_pol, seed=M)
    ret, lng = evaluate(eng, W, M, rnd=3)
    tr, tl = ref.evaluate(twin, env, W, M, seed=7, rnd=3, gru=gru, pomdp=pomdp, n_agents=N)
    assert np.array_equal(lng, tl)
    assert np.array_equal(ret.view(np.int64), tr.view(np.int64))        # bit for bit


GOLDEN = {"rollout_cartpole_mlp": ("CartPole-v1", False, False), "rollout_cartpole_gru_pomdp": ("CartPole-v1", True, True),
          "rollout_mountaincar": ("MountainCar-v0", False, False), "rollout_mountaincar_gru": ("MountainCar-v0", True, False),
          "rollout_acrobot": ("Acrobot-v1", False, False), "rollout_acrobot_gru": ("Acrobot-v1", True, False),
          "rollout_pendulum": ("Pendulum-v0", False, False), "rollout_pendulum_gru": ("Pendulum-v0", True, False),
          "rollout_spread_n2": ("simple_spread", False, False), "rollout_spread_n2_gru": ("simple_spread", True, False),
          "rollout_spread_n3": ("simple_spread", False, False), "rollout_spread_n3_gru": ("simple_spread", True, False)}


@pytest.mark.parametrize("name", list(GOLDEN))
def test_emu_evaluate_bit_rule_against_verification_rollout(emu, golden, name):
    """Returns added in episode order and divided by E are ses_rollout's verification-mode fitness, bit for bit; the lengths
    add up to its steps; and the fitness is within the golden tolerance of the reference's own."""
    env, gru, pomdp = GOLDEN[name]
    g = golden(name)
    N = int(g["N"]) if "N" in g.files else 1
    n = min(12, g["W"].shape[0])
    W, init, E = g["W"][:n], g["init"], int(g["E"])
    eng = make(emu, env, gru, pomdp, N if env == "simple_spread" else 2, population=n, eval_ep_num=E)
    assert eng.D == W.shape[1]
    fit, steps = eng.rollout(0, 0.0, None, w_override=W, init_states=init)
    ret, lng = evaluate(eng, W, E, init_states=init)
    for j in range(n):
        total = 0.0
        for e in range(E):
            total = total + ret[j, e]
        assert total / E == fit[j] and int(lng[j].sum()) == steps[j]
    np.testing.assert_allclose(fit, g["fitness"][:n], rtol=1e-12 if env == "simple_spread" else 1e-4)


def test_emu_evaluate_invariances(emu, twin):
    eng = make(emu, "CartPole-v1")
    W = policies(eng, 3, seed=5)
    r1, l1 = evaluate(eng, W[:1], 100, rnd=4)
    r3, l3 = evaluate(eng, W[[2, 0, 1]], 100, rnd=4)
    assert np.array_equal(r3[1], r1[0]) and np.array_equal(l3[1], l1[0])          # other policies, any order
    r40, l40 = evaluate(eng, W[[2, 0, 1]], 40, rnd=4)
    assert np.array_equal(r40, r3[:, :40]) and np.array_equal(l40, l3[:, :40])     # episode m does not depend on M
    rb, lb = evaluate(eng, W[:1], 100, rnd=5)
    assert not np.array_equal(lb, l1)                                                 # another round, other initial states
    s4, s5 = ref.eval_init(twin, "CartPole-v1", 7, 4, 0), ref.eval_init(twin, "CartPole-v1", 7, 5, 0)
    assert not np.array_equal(s4, s5)
    tr, tl = ref.evaluate(twin, "CartPole-v1", W[:1], 100, seed=7, rnd=5)
    assert np.array_equal(rb, tr) and np.array_equal(lb, tl)


@pytest.mark.parametrize("env,gru", [("CartPole-v1", False), ("CartPole-v1", True), ("MountainCar-v0", True), ("simple_spread", False)])
def test_emu_evaluate_ignores_strategy_antithetic_and_shard(emu, env, gru):
    base = make(emu, env, gru, population=16)
    W = policies(base, 2, seed=9)
    M = 9
    want = evaluate(base, W, M, rnd=1)
    others = [make(emu, env, gru, population=12, group=4, n_head=1, n_parents=3, antithetic=True),
              make(emu, env, gru, population=16, group=16, n_head=2, id_begin=4, id_end=9, init_mode="fresh"),
              make(emu, env, gru, population=64, group=64, shard=(1, 4, 4), eval_ep_num=3)]
    for eng in others:
        got = evaluate(eng, W, M, rnd=1)
        assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])


def test_emu_evaluate_rejects_bad_arguments(emu):
    eng = make(emu, "CartPole-v1")
    lib, h = eng.lib, eng._h
    W = np.zeros((2, eng.D), np.float32)
    ret = np.zeros((2, 4)); lng = np.zeros((2, 4), np.int32)

    def err(*args):
        assert lib.ses_evaluate(*args) != 0
        return lib.ses_last_error().decode()
    assert "null handle" in err(None, 0, _p(W), 2, 4, None, _p(ret), _p(lng), None)
    assert "required" in err(h, 0, None, 2, 4, None, _p(ret), _p(lng), None)
    assert "required" in err(h, 0, _p(W), 2, 4, None, None, _p(lng), None)
    assert "required" in err(h, 0, _p(W), 2, 4, None, _p(ret), None, None)
    assert ">= 1" in err(h, 0, _p(W), 0, 4, None, _p(ret), _p(lng), None)
    assert ">= 1" in err(h, 0, _p(W), 2, -3, None, _p(ret), _p(lng), None)
    assert "2^30" in err(h, 0, _p(W), 1 << 16, 1 << 16, None, _p(ret), _p(lng), None)
    assert "2^30" in err(h, 0, _p(W), 2, 0x7FFFFFFF, None, _p(ret), _p(lng), None)

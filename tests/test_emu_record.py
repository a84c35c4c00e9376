"""Episode recording (ses_record, DESIGN.md section 4.9) on the SIMT emulator of tests/simt_emu: the recording instances of
the K1 kernels against the twin's single-episode rollouts and traces (tests/record_reference.py) for every env x {MLP, GRU},
at episode counts around the kernels' chunk widths, the bit rule that ties them to ses_evaluate, invariances and argument
checks."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))

import eval_reference as ref  # noqa: E402
import record_reference  # noqa: E402
from test_emu_evaluate import CONFIGS, _ids, evaluate, make, policies  # noqa: E402


@pytest.fixture(scope="module")
def emu():
    from simt_emu import emu_engine
    emu_engine.load()
    return emu_engine.EmuEngine


def _p(a):
    return None if a is None else C.c_void_p(a.ctypes.data)


def record(eng, policies, K, rnd=0, init_states=None):
    """(initial, states, actions, returns, lengths) of ses_record, pre-filled with NaN / -1 as RolloutEngine.record does."""
    W = np.ascontiguousarray(policies, dtype=np.float32).reshape(-1, eng.D)
    n, T, sd = W.shape[0], eng.max_step, eng.state_dim
    out = (np.full((K, sd), np.nan), np.full((n, K, T, sd), np.nan), np.full((n, K, T, eng.n_agents), -1, dtype=np.int32),
           np.full((n, K, T), np.nan), np.full((n, K), -1, dtype=np.int32))
    init = None if init_states is None else np.ascontiguousarray(init_states, dtype=np.float64)
    eng._check(eng.lib.ses_record(eng._h, int(rnd), _p(W), n, int(K), _p(init), *(_p(a) for a in out), None))
    return out


def same_bits(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and np.array_equal(a.view(np.uint8), b.view(np.uint8))


def chunk(env, gru, N):
    """Episodes per virtual offspring: a warp of the slot kernel, the lockstep width of the GRU kernels."""
    if not gru:
        return 32
    if env.startswith("CartPole"):
        return 5
    return 3 if (env, N) == ("simple_spread", 2) else 2 if env == "simple_spread" else 5


@pytest.mark.parametrize("cfg", CONFIGS, ids=_ids)
def test_emu_record_equals_twin(emu, twin, cfg):
    """K in {1, c - 1, c, c + 1, 2c + 3} for chunk width c: every array bit for bit, NaN / -1 past each episode's end."""
    env, gru, pomdp, N = cfg
    c = chunk(env, gru, N)
    eng = make(emu, env, gru, pomdp, N)
    W = policies(eng, 2, seed=8)                     # CartPole MLP: a random policy next to one that balances for 500 steps
    want = record_reference.record(twin, env, W, 2 * c + 3, seed=7, rnd=2, gru=gru, pomdp=pomdp, n_agents=N)   # episode m: not K's
    for K in sorted({1, c - 1, c, c + 1, 2 * c + 3} - {0}):
        got = record(eng, W, K, rnd=2)
        initial, states, actions, returns, lengths = want
        for name, g, w in zip(("initial", "states", "actions", "returns", "lengths"), got,
                              (initial[:K], states[:, :K], actions[:, :K], returns[:, :K], lengths[:, :K])):
            assert same_bits(g, w), (K, name)


@pytest.mark.parametrize("cfg", CONFIGS, ids=_ids)
def test_emu_record_bit_rule_against_evaluate(emu, twin, cfg):
    """returns[j][m][lengths - 1] is ses_evaluate's return of the same episode in a call of more episodes, drawn or given."""
    env, gru, pomdp, N = cfg
    c = chunk(env, gru, N)
    K, M = c + 2, 2 * c + 5
    eng = make(emu, env, gru, pomdp, N)
    W = policies(eng, 3, seed=4)
    table = np.stack([ref.eval_init(twin, env, 7, 9, m, N) for m in range(M)])       # another round's states, given
    for rnd, init in ((5, None), (0, table)):
        ret, lng = evaluate(eng, W, M, rnd=rnd, init_states=init)
        initial, states, actions, returns, lengths = record(eng, W, K, rnd=rnd, init_states=None if init is None else init[:K])
        assert np.array_equal(lengths, lng[:, :K])
        last = np.take_along_axis(returns, (lengths - 1)[..., None].astype(np.int64), axis=2)[..., 0]
        assert same_bits(last, ret[:, :K])
        if init is not None:
            assert same_bits(initial, init[:K])
        else:
            assert same_bits(initial, np.stack([ref.eval_init(twin, env, 7, rnd, m, N) for m in range(K)]))


@pytest.mark.parametrize("env,gru", [("CartPole-v1", False), ("CartPole-v1", True), ("MountainCar-v0", True), ("simple_spread", False)])
def test_emu_record_rows_do_not_depend_on_the_other_policies(emu, env, gru):
    eng = make(emu, env, gru)
    W = policies(eng, 3, seed=6)
    K = 37 if not gru else 7
    one = record(eng, W[1:2], K, rnd=1)
    three = record(eng, W[[2, 1, 0]], K, rnd=1)
    assert same_bits(three[0], one[0])                                                # initial: common to every policy
    for a, b in zip(one[1:], three[1:]):
        assert same_bits(b[1:2], a)
    # a handle of another strategy layout, shard and initial-state mode records the same
    other = make(emu, env, gru, population=64, group=64, shard=(1, 4, 4), eval_ep_num=3, init_mode="fresh")
    for a, b in zip(record(other, W[[2, 1, 0]], K, rnd=1), three):
        assert same_bits(a, b)


def test_emu_record_rejects_bad_arguments(emu):
    eng = make(emu, "CartPole-v1")
    lib, h = eng.lib, eng._h
    W = np.zeros((2, eng.D), np.float32)
    bufs = [np.zeros((4, 4)), np.zeros((2, 4, 500, 4)), np.zeros((2, 4, 500, 1), np.int32), np.zeros((2, 4, 500)),
            np.zeros((2, 4), np.int32)]

    def err(h, W, n_pol, K, bufs):
        assert lib.ses_record(h, 0, _p(W), n_pol, K, None, *(_p(b) for b in bufs), None) != 0
        return lib.ses_last_error().decode()
    assert "null handle" in err(None, W, 2, 4, bufs)
    assert "required" in err(h, None, 2, 4, bufs)
    for i in range(len(bufs)):
        assert "required" in err(h, W, 2, 4, bufs[:i] + [None] + bufs[i + 1:])
    assert ">= 1" in err(h, W, 0, 4, bufs)
    assert ">= 1" in err(h, W, 2, 0, bufs)
    assert ">= 1" in err(h, W, 2, -3, bufs)
    assert "2^30" in err(h, W, 1 << 16, 1 << 16, bufs)
    assert "2^30" in err(h, W, 2, 0x7FFFFFFF, bufs)
    assert np.all(bufs[4] == 0) and np.all(bufs[1] == 0)                              # nothing was launched

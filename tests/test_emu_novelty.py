"""Novelty search with reward (nsr_es, DESIGN.md section 4.10) on the SIMT emulator of tests/simt_emu.

* The final-state instances of the K1 kernels against the twin's single-episode rollouts under the training keying
  (tests/novelty_reference.py) for every env x {MLP, GRU}, with shared / fresh initial states, antithetic sampling, a
  block-cyclic shard, and launches that take sparse warps and the queue B tail; fitness and steps equal the plain
  instance's bit for bit.
* ses_behavior / ses_novelty / ses_blend_shaped against numpy restatements, bit for bit, and their argument checks.
"""
import ctypes as C
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))

import k23_reference as k23  # noqa: E402
import novelty_reference as nref  # noqa: E402
from test_emu_evaluate import CONFIGS, _ids, make  # noqa: E402


@pytest.fixture(scope="module")
def emu():
    from simt_emu import emu_engine
    emu_engine.load()
    return emu_engine.EmuEngine


def _p(a):
    return None if a is None else C.c_void_p(a.ctypes.data)


def same_bits(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and np.array_equal(a.view(np.uint8), b.view(np.uint8))


def rollout_final(eng, gen, sigma, parents):
    """(fitness, steps, final_states [P][E][state_dim] NaN where not written) of one rollout with the output on, then the
    output switched off again."""
    fs = np.full((eng.P, eng.E, eng.state_dim), np.nan)
    eng._check(eng.lib.ses_set_final_states(eng._h, _p(fs)))
    fit, steps = eng.rollout(gen, sigma, parents)
    eng._check(eng.lib.ses_set_final_states(eng._h, None))
    return fit, steps, fs


def parents_for(eng, seed=3, scale=0.5):
    return np.random.default_rng(seed).normal(0, scale, (1, eng.D)).astype(np.float32)


def check_final(emu, twin, env, gru=False, pomdp=False, N=2, E=3, P=16, gen=2, sigma=0.5, init_mode="shared", antithetic=False,
                shard=None, seed=7):
    eng = make(emu, env, gru, pomdp, N, seed=seed, population=P, eval_ep_num=E, init_mode=init_mode, antithetic=antithetic,
               shard=shard)
    mu = parents_for(eng)
    fit0, steps0 = eng.rollout(gen, sigma, mu)
    fit, steps, fs = rollout_final(eng, gen, sigma, mu)
    geometry = eng.test_k1_geometry() if not gru else None
    assert same_bits(fit, fit0) and same_bits(steps, steps0), "the final-state instance changed fitness or steps"
    from simple_es_b200.engine import owned_ids
    ids = owned_ids(P, *shard) if shard else np.arange(P)
    want = nref.final_states(twin, env, mu, ids, E, sigma, seed, gen, P, 1, gru=gru, pomdp=pomdp, n_agents=N,
                             init_mode={"shared": 0, "fresh": 1}[init_mode], antithetic=antithetic)
    assert same_bits(fs[ids], want)
    others = np.setdiff1d(np.arange(P), ids)
    assert np.isnan(fs[others]).all(), "rows of ids the handle does not own were written"
    eng.close()
    return geometry


@pytest.mark.parametrize("cfg", CONFIGS, ids=_ids)
def test_emu_final_states_equal_twin(emu, twin, cfg):
    env, gru, pomdp, N = cfg
    check_final(emu, twin, env, gru, pomdp, N)


@pytest.mark.parametrize("env,gru,N", [("CartPole-v1", False, 1), ("CartPole-v1", True, 1), ("Acrobot-v1", False, 1),
                                       ("MountainCar-v0", True, 1), ("simple_spread", False, 3)])
@pytest.mark.parametrize("mode", ["fresh", "antithetic", "shard"])
def test_emu_final_states_keying_and_shards(emu, twin, env, gru, N, mode):
    """Fresh initial states, antithetic pairs, and rank 1 of a 3-way block-cyclic shard (rows at global ids, the others
    untouched)."""
    kw = {"fresh": {"init_mode": "fresh"}, "antithetic": {"antithetic": True}, "shard": {"shard": (1, 3, 2)}}[mode]
    check_final(emu, twin, env, gru, False, N, E=2, P=14, gen=5, **kw)


@pytest.mark.parametrize("P,E,path", [(60, 5, "sparse"), (250, 5, "tail"), (40, 1, "single")])
def test_emu_final_states_launch_paths(emu, twin, P, E, path, monkeypatch):
    """CartPole MLP launches that take sparse warps (and with them the 2 / 4-lane straggler phase), queue A followed by the
    queue B tail, and a single exact round with E = 1: the lane that ends each episode stores its row."""
    monkeypatch.setenv("SES_SIMT_EMU_SMS", "2")
    monkeypatch.setenv("SES_SIMT_EMU_CTAS_PER_SM", "2")
    monkeypatch.setenv("SES_K1_TAIL", "2" if path == "tail" else "0")     # 2 rounds of queue B, or none
    g = check_final(emu, twin, "CartPole-v1", E=E, P=P, gen=0, sigma=0.3)
    n_ep = P * E
    if path == "sparse":
        assert g["sparse_rank"] >= 0, g
    elif path == "tail":
        assert 0 < g["tail_start"] < n_ep and g["sparse_rank"] < 0, g
    else:
        assert g["tail_start"] == 0 and g["sparse_rank"] < 0, g


def test_emu_final_states_refuse_traces(emu):
    eng = make(emu, "CartPole-v1", population=8, eval_ep_num=2)
    fs = np.zeros((8, 2, 4))
    eng._check(eng.lib.ses_set_final_states(eng._h, _p(fs)))
    with pytest.raises(RuntimeError, match="final states"):
        eng.rollout(0, 0.1, parents_for(eng), n_trace=1)
    assert eng.lib.ses_set_final_states(None, _p(fs)) != 0
    eng._check(eng.lib.ses_set_final_states(eng._h, None))
    eng.rollout(0, 0.1, parents_for(eng), n_trace=1)


# ------------------------------------------------------------------------------------- behaviour, novelty, blend
def behavior(eng, fs):
    n = fs.shape[0]
    out = np.full((n, eng.state_dim), np.nan)
    eng._check(eng.lib.ses_behavior(eng._h, _p(np.ascontiguousarray(fs)), n, _p(out), None))
    return out


def novelty(eng, bc, archive, k):
    bc, archive = np.ascontiguousarray(bc, dtype=np.float64), np.ascontiguousarray(archive, dtype=np.float64)
    out = np.full(bc.shape[0], np.nan)
    eng._check(eng.lib.ses_novelty(eng._h, _p(bc), bc.shape[0], _p(archive), archive.shape[0], int(k), _p(out), None))
    return out


def blend(eng, a, b, w):
    out = np.full(a.size, np.nan)
    eng._check(eng.lib.ses_blend_shaped(eng._h, _p(np.ascontiguousarray(a)), _p(np.ascontiguousarray(b)), a.size, float(w), _p(out), None))
    return out


@pytest.mark.parametrize("env,N,E", [("MountainCar-v0", 1, 5), ("CartPole-v1", 1, 1), ("simple_spread", 3, 7)])
def test_emu_behavior_equals_numpy(emu, env, N, E):
    eng = make(emu, env, n_agents=N, population=300, eval_ep_num=E)
    rng = np.random.default_rng(1)
    fs = rng.normal(0, 1, (300, E, eng.state_dim)) * np.exp(rng.uniform(-20, 20, (300, E, eng.state_dim)))
    fs[:, 0, 0] = -0.0                                   # a sum that starts at -0.0
    for n in (1, 65, 300):
        assert same_bits(behavior(eng, fs[:n]), nref.behavior(fs[:n]))


@pytest.mark.parametrize("k", [1, 2, 3, 10, 17, 32])
@pytest.mark.parametrize("A_rel", [-1, 0, 1])
def test_emu_novelty_archive_around_k(emu, k, A_rel):
    """|A| = k - 1, k, k + 1 (|A| >= 1), n not a multiple of the block."""
    eng = make(emu, "CartPole-v1", population=200)
    rng = np.random.default_rng(k)
    A = max(1, k + A_rel)
    bc, archive = rng.normal(0, 1, (131, 4)), rng.normal(0, 1, (A, 4))
    assert same_bits(novelty(eng, bc, archive, k), nref.novelty(bc, archive, k))


@pytest.mark.parametrize("A", [255, 256, 257, 600])
@pytest.mark.parametrize("env,N", [("MountainCar-v0", 1), ("Acrobot-v1", 1), ("simple_spread", 2), ("simple_spread", 3)])
def test_emu_novelty_across_tiles(emu, A, env, N):
    """Archives on both sides of the shared-memory tile (256 rows), for every state_dim the kernel is built for: 2, 4, 8, 12."""
    eng = make(emu, env, n_agents=N, population=100)
    rng = np.random.default_rng(A)
    bc, archive = rng.normal(0, 1, (67, eng.state_dim)), rng.normal(0, 1, (A, eng.state_dim))
    for k in (1, 10, 32):
        assert same_bits(novelty(eng, bc, archive, k), nref.novelty(bc, archive, k))


def test_emu_novelty_duplicates_and_ties(emu):
    """Duplicated archive rows, offspring equal to archive rows (distance 0), and distances that tie."""
    eng = make(emu, "MountainCar-v0", population=64)
    base = np.array([[0.0, 0.0], [1.0, 0.0], [0.0, 1.0], [-1.0, 0.0], [0.0, -1.0], [3.0, 4.0]])
    archive = np.concatenate([base, base, base[:3]])
    bc = np.concatenate([base, [[0.5, 0.5], [2.0, 2.0], [-0.0, 0.0]], np.random.default_rng(2).normal(0, 2, (40, 2))])
    for k in (1, 2, 4, 5, 9, 15, 32):
        assert same_bits(novelty(eng, bc, archive, k), nref.novelty(bc, archive, k)), k


def test_emu_blend_equals_numpy(emu):
    eng = make(emu, "CartPole-v1", population=1000)
    rng = np.random.default_rng(5)
    fit, nov = rng.integers(0, 50, 999).astype(np.float64), rng.normal(0, 1, 999)
    sf = k23.centered_ref(k23.rank_ref(fit))
    sn = k23.centered_ref(k23.rank_ref(nov))
    # K2's own shapings (the kernels nsr_es blends)
    _, sf_k = eng.rank_desc(fit, shaped=True)
    _, sn_k = eng.rank_desc(nov, shaped=True, full_key=True)
    assert np.allclose(sf_k, sf, rtol=0, atol=1e-12) and np.allclose(sn_k, sn, rtol=0, atol=1e-12)
    for w in (0.0, 0.25, 0.5, 1.0 / 3.0, 0.9, 1.0):
        assert same_bits(blend(eng, sf_k, sn_k, w), nref.blend(sf_k, sn_k, w)), w
    assert same_bits(blend(eng, sf_k, sn_k, 0.0), sf_k)
    assert same_bits(blend(eng, sf_k, sn_k, 1.0), sn_k)


def test_emu_novelty_argument_errors(emu):
    eng = make(emu, "CartPole-v1", population=8, eval_ep_num=2)
    lib, h = eng.lib, eng._h
    fs, bc, arc, out = np.zeros((8, 2, 4)), np.zeros((8, 4)), np.zeros((3, 4)), np.zeros(8)

    def err(rc):
        assert rc != 0
        return lib.ses_last_error().decode()
    assert "null handle" in err(lib.ses_behavior(None, _p(fs), 8, _p(bc), None))
    assert "required" in err(lib.ses_behavior(h, None, 8, _p(bc), None))
    assert "required" in err(lib.ses_behavior(h, _p(fs), 8, None, None))
    for n in (0, 9, -1):
        assert "population" in err(lib.ses_behavior(h, _p(fs), n, _p(bc), None))
        assert "population" in err(lib.ses_novelty(h, _p(bc), n, _p(arc), 3, 2, _p(out), None))
        assert "population" in err(lib.ses_blend_shaped(h, _p(out), _p(out), n, 0.5, _p(out), None))
    assert "null handle" in err(lib.ses_novelty(None, _p(bc), 8, _p(arc), 3, 2, _p(out), None))
    for args in ((None, _p(arc), _p(out)), (_p(bc), None, _p(out)), (_p(bc), _p(arc), None)):
        assert "required" in err(lib.ses_novelty(h, args[0], 8, args[1], 3, 2, args[2], None))
    for k in (0, 33, -1):
        assert "k must be" in err(lib.ses_novelty(h, _p(bc), 8, _p(arc), 3, k, _p(out), None))
    assert "n_archive" in err(lib.ses_novelty(h, _p(bc), 8, _p(arc), 0, 2, _p(out), None))
    assert "null handle" in err(lib.ses_blend_shaped(None, _p(out), _p(out), 8, 0.5, _p(out), None))
    assert "required" in err(lib.ses_blend_shaped(h, None, _p(out), 8, 0.5, _p(out), None))
    for w in (-0.1, 1.5, float("nan")):
        assert "w must be" in err(lib.ses_blend_shaped(h, _p(out), _p(out), 8, w, _p(out), None))
    assert np.all(bc == 0) and np.all(out == 0)          # nothing was launched

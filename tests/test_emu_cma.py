"""sep_cma_es's kernels (DESIGN.md section 4.11) on the SIMT emulator of tests/simt_emu, against the numpy restatement of
tests/cma_reference.py: the samples (contiguous slices and block-cyclic shards, in local order), the weight scatter, and
updates bit for bit except sigma (<= 2 ulp), for mu in {1, lambda // 2, lambda} with a population ragged against both the
level-0 block (32) and the level-1 group (2048 offspring), on three parameter counts.  Also the argument checks."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))

import cma_reference as cref  # noqa: E402
import k23_reference as k23  # noqa: E402
from test_emu_evaluate import make  # noqa: E402

from simple_es_b200.engine import cma_params, owned_ids, sep_cma_constants, sep_cma_threshold  # noqa: E402

SEED = 7


@pytest.fixture(scope="module")
def emu():
    from simt_emu import emu_engine
    emu_engine.load()
    return emu_engine.EmuEngine


def same_bits(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and np.array_equal(a.view(np.uint8), b.view(np.uint8))


def cma_engine(emu, D, P, **kw):
    env, _, _, gru, N = k23.ENVS[D]
    return make(emu, env, gru, False, N, seed=SEED, population=P, group=P, n_head=0, eval_ep_num=1, **kw)


def _p(a):
    return None if a is None else C.c_void_p(a.ctypes.data)


def cma_sample(eng, generation, mean, c, sigma):
    """ses_cma_sample on the emulated handle: [n_local, D] float32 samples from float64 mean [D], c [D], sigma [1]."""
    out = np.full((eng.n_local, eng.D), np.nan, dtype=np.float32)
    mean, c, sigma = (np.ascontiguousarray(a, dtype=np.float64) for a in (mean, c, sigma))
    eng._check(eng.lib.ses_cma_sample(eng._h, int(generation), _p(mean), _p(c), _p(sigma), _p(out), None))
    return out


def cma_update(eng, generation, order, k, s, mean, c, p_sigma, p_c, sigma, parent):
    """ses_cma_update on the emulated handle, in place on the float64 arrays s [P], mean / c / p_sigma / p_c [D], sigma [1] and
    the float32 parent [D]."""
    for a, dt in ((s, np.float64), (mean, np.float64), (c, np.float64), (p_sigma, np.float64), (p_c, np.float64),
                  (sigma, np.float64), (parent, np.float32)):
        assert a.dtype == dt and a.flags.c_contiguous
    w, order = np.ascontiguousarray(k["weights"], dtype=np.float64), np.ascontiguousarray(order, dtype=np.int32)
    eng._check(eng.lib.ses_cma_update(eng._h, int(generation), _p(order), _p(w), int(k["mu"]), cma_params(k),
                                      sep_cma_threshold(k, generation), _p(s), _p(mean), _p(c), _p(p_sigma), _p(p_c), _p(sigma),
                                      _p(parent), None))


def random_state(D, rng):
    return (rng.normal(0, 0.3, D), rng.uniform(0.2, 3.0, D), rng.normal(0, 1, D), rng.normal(0, 0.5, D), np.array([0.7]))


@pytest.mark.parametrize("D", [195, 226, 581])
@pytest.mark.parametrize("shard", [None, (0, 1), (1, 3, 4), (2, 3, 5)], ids=["all", "slice", "cyclic-1-of-3", "cyclic-2-of-3"])
def test_emu_cma_sample_equals_numpy(emu, twin, D, shard):
    """Row l is the sample of the l-th id the handle owns: a contiguous slice [13, 60), or a block-cyclic share."""
    P, gen = 77, 9
    if shard is None:
        eng, ids = cma_engine(emu, D, P), np.arange(P)
    elif len(shard) == 2:
        eng, ids = cma_engine(emu, D, P, id_begin=13, id_end=60), np.arange(13, 60)
    else:
        eng, ids = cma_engine(emu, D, P, shard=shard), owned_ids(P, *shard)
    mean, c, _, _, sigma = random_state(D, np.random.default_rng(D))
    got = cma_sample(eng, gen, mean, c, sigma)
    want = cref.sample(mean, c, sigma[0], cref.normals(twin, SEED, gen, ids, D))
    assert same_bits(got, want)
    eng.close()


def one_update(eng, twin, k, gen, order, st, z):
    """Run ses_cma_update on copies of st and the numpy step from st; return (device state, reference state, s, h_sigma)."""
    P = eng.P
    mean, c, ps, pc, sigma = (np.array(x, dtype=np.float64) for x in st)
    parent = np.full(eng.D, np.nan, dtype=np.float32)
    s = np.full(P, np.nan)
    cma_update(eng, gen, order, k, s, mean, c, ps, pc, sigma, parent)
    s_ref = cref.weights(order, k["weights"], k["mu"], P)
    t1, t2 = cref.tables(s_ref, z)
    ref = cref.update(t1, t2, k, sep_cma_threshold(k, gen), *st[:4], st[4][0])
    return (mean, c, ps, pc, sigma, parent), ref, (s, s_ref)


def check_update(got, ref):
    for name, g, w in zip(("mean", "c", "p_sigma", "p_c"), got[:4], ref[:4]):
        assert same_bits(g, w), name
    assert same_bits(got[5], ref[5]), "parent"
    assert cref.ulps(got[4][0], ref[4]) <= 2, (got[4][0], ref[4])


@pytest.mark.parametrize("D", [195, 226, 581])
@pytest.mark.parametrize("mu_kind", ["one", "half", "all"])
def test_emu_cma_update_equals_numpy(emu, twin, D, mu_kind):
    """P = 2085: 65 full level-0 blocks and a partial one, two level-1 groups (the second partial).  Two updates: generation
    0 from a long p_sigma (h_sigma = 0), then generation 60 from the device's state with p_sigma shortened (h_sigma = 1)."""
    P = 2085
    mu = {"one": 1, "half": P // 2, "all": P}[mu_kind]
    k = sep_cma_constants(D, P, mu)
    eng = cma_engine(emu, D, P)
    rng = np.random.default_rng(100 * D + mu)
    mean, c, ps, pc, sigma = random_state(D, rng)
    st = (mean, c, 30.0 * ps, pc, sigma)
    hs = []
    for gen in (0, 60):
        order = rng.permutation(P).astype(np.int32)
        z = cref.normals(twin, SEED, gen, range(P), D)
        got, ref, (s, s_ref) = one_update(eng, twin, k, gen, order, st, z)
        assert same_bits(s, s_ref), "weight scatter"
        assert np.count_nonzero(s) == mu and same_bits(s[order[:mu]], k["weights"])
        check_update(got, ref)
        hs.append(ref[6])
        mean, c, ps, pc, sigma = got[:5]
        st = (mean, c, 0.01 * ps, pc, sigma)
    assert hs == [False, True]
    eng.close()


def test_emu_cma_update_sharded_engine_equals_whole(emu, twin):
    """A handle that owns a block-cyclic share still updates from every row (order and fitness cover the population)."""
    D, P, gen = 226, 300, 4
    k = sep_cma_constants(D, P, 150)
    st = random_state(D, np.random.default_rng(3))
    order = np.random.default_rng(4).permutation(P).astype(np.int32)
    z = cref.normals(twin, SEED, gen, range(P), D)
    outs = []
    for kw in ({}, {"shard": (1, 2, 8)}):
        eng = cma_engine(emu, D, P, **kw)
        got, ref, _ = one_update(eng, twin, k, gen, order, st, z)
        check_update(got, ref)
        outs.append(got)
        eng.close()
    for a, b in zip(*outs):
        assert same_bits(a, b)


def test_emu_cma_argument_errors(emu):
    D, P = 226, 40
    eng = cma_engine(emu, D, P)
    lib, h = eng.lib, eng._h
    k = sep_cma_constants(D, P, 20)
    mean, c, ps, pc, sigma = random_state(D, np.random.default_rng(0))
    out, s, parent = np.zeros((P, D), np.float32), np.zeros(P), np.zeros(D, np.float32)
    order, w = np.arange(P, dtype=np.int32), k["weights"]

    def err(rc):
        assert rc != 0
        return lib.ses_last_error().decode()

    def update(handle, mu, **kw):
        a = dict(order=_p(order), w=_p(w), params=cma_params(k), s=_p(s), mean=_p(mean), c=_p(c), ps=_p(ps), pc=_p(pc), sigma=_p(sigma),
                 parent=_p(parent))
        a.update(kw)
        return lib.ses_cma_update(handle, 0, a["order"], a["w"], mu, a["params"], 1.0, a["s"], a["mean"], a["c"], a["ps"], a["pc"],
                                  a["sigma"], a["parent"], None)
    assert "null handle" in err(lib.ses_cma_sample(None, 0, _p(mean), _p(c), _p(sigma), _p(out), None))
    for i in range(4):
        args = [_p(mean), _p(c), _p(sigma), _p(out)]
        args[i] = None
        assert "required" in err(lib.ses_cma_sample(h, 0, *args, None))
    assert "null handle" in err(update(None, 20))
    for key in ("order", "w", "params", "s", "mean", "c", "ps", "pc", "sigma", "parent"):
        assert "null argument" in err(update(h, 20, **{key: None}))
    for mu in (0, -1, P + 1):
        assert "mu=" in err(update(h, mu))
    assert np.all(out == 0) and np.all(s == 0) and np.all(parent == 0)         # nothing was launched
    eng.close()
    for kw in ({"n_head": 1}, {"group": P // 2, "n_parents": 2}, {"antithetic": True}):
        env, _, _, gru, N = k23.ENVS[D]
        bad = make(emu, env, gru, False, N, seed=SEED, population=P, **dict({"group": P, "n_head": 0, "eval_ep_num": 1}, **kw))
        assert "layout" in err(bad.lib.ses_cma_sample(bad._h, 0, _p(mean), _p(c), _p(sigma), _p(out), None))
        assert "layout" in err(update(bad._h, 20))
        bad.close()

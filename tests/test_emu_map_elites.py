"""MAP-Elites (map_elites, DESIGN.md section 4.12) on the SIMT emulator of tests/simt_emu, through the C ABI, against the
numpy restatement of tests/map_elites_reference.py and the C twin, bit for bit:

* K1 with the map_elites layout (group = 1, n_head = 0: every offspring perturbed from its own parent row) on the slot kernel
  (CartPole, MountainCar, simple_spread), the CartPole-GRU kernel and the generic GRU kernel, final states included.
* ses_map_insert on hand-built populations: one cell for all, ties inside a cell, a candidate equal to the incumbent, NaN
  fitness and behaviour, out-of-range and infinite behaviour, a single cell, and 1 to 4 descriptor dimensions.
* ses_map_select at 0, 1, 2, 3, several hundred and all cells occupied; a block-cyclic shard against a whole handle.
* The argument checks.
"""
import ctypes as C
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))

import map_elites_reference as mref  # noqa: E402
from test_emu_evaluate import make  # noqa: E402

SEED = 11


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


def map_engine(emu, env="CartPole-v1", gru=False, N=1, P=32, E=2, **kw):
    return make(emu, env, gru, False, N, seed=SEED, population=P, group=1, n_head=0, n_parents=P, eval_ep_num=E, **kw)


def insert(eng, gen, sigma, parents, order, fitness, bc, spec, a):
    """ses_map_insert in place on the archive dict a (F, B, born, W numpy arrays)."""
    parents, order = np.ascontiguousarray(parents, np.float32), np.ascontiguousarray(order, np.int32)
    fitness, bc = np.ascontiguousarray(fitness, np.float64), np.ascontiguousarray(bc, np.float64)
    eng._check(eng.lib.ses_map_insert(eng._h, int(gen), float(sigma), _p(parents), _p(order), _p(fitness), _p(bc),
                                      C.byref(spec.ctype()), _p(a["F"]), _p(a["B"]), _p(a["born"]), _p(a["W"]), None))


def select(eng, gen, spec, a, seed_row):
    stats = np.full(4, -7.0)
    parents = np.full((eng.P, eng.D), np.nan, dtype=np.float32)
    eng._check(eng.lib.ses_map_select(eng._h, int(gen), C.byref(spec.ctype()), _p(a["F"]), _p(a["W"]),
                                      _p(np.ascontiguousarray(seed_row, np.float32)), _p(stats), _p(parents), None))
    return stats, parents


def same_archive(a, b):
    for k in ("F", "B", "born", "W"):
        assert same_bits(a[k], b[k]), k
    return True


def check_stats(stats, F):
    n_occ, best, bf, qd = mref.stats(F)
    assert stats[0] == n_occ and stats[1] == best
    assert same_bits(stats[2:3], np.array([bf])) and same_bits(stats[3:4], np.array([qd]))


# ---------------------------------------------------------------------------------------------------- K1 with the layout
def twin_population(twin, env, gru, N, parents, sigma, gen, P, E):
    kw = dict(sigma=sigma, seed=SEED, gen=gen, group=1, n_head=0, id0=0, n=P, E=E, final=True)
    if env.startswith("CartPole"):
        return twin.population_cartpole(parents, gru=gru, max_step=500, **kw)
    if env == "simple_spread":
        return twin.population_mpe(parents, N=N, gru=gru, **kw)
    return twin.population_classic(env, parents, gru=gru, **kw)


@pytest.mark.parametrize("env,gru,N", [("CartPole-v1", False, 1), ("MountainCar-v0", False, 1), ("simple_spread", False, 3),
                                       ("CartPole-v1", True, 1), ("MountainCar-v0", True, 1), ("Acrobot-v1", True, 1)],
                         ids=["cartpole-slot", "mountaincar-slot", "spread3-slot", "cartpole-gru", "mountaincar-gru-generic",
                              "acrobot-gru-generic"])
def test_emu_k1_one_parent_row_per_offspring_equals_twin(emu, twin, env, gru, N):
    """P distinct parent rows, every offspring perturbed: fitness, steps and final states equal the twin's."""
    P, E, gen, sigma = 37, 2, 3, 0.4
    eng = map_engine(emu, env, gru, N, P=P, E=E)
    parents = np.random.default_rng(5).normal(0, 0.6, (P, eng.D)).astype(np.float32)
    fs = np.full((P, E, eng.state_dim), np.nan)
    eng._check(eng.lib.ses_set_final_states(eng._h, _p(fs)))
    fit, steps = eng.rollout(gen, sigma, parents)
    tf, ts, tfs = twin_population(twin, env, gru, N, parents, sigma, gen, P, E)
    assert same_bits(fit, tf) and np.array_equal(steps, ts)
    assert same_bits(fs, tfs)
    assert len(np.unique(fs.reshape(P, -1), axis=0)) > 1          # the rows differ
    eng.close()


# ---------------------------------------------------------------------------------------------------- insertion
def run_insert(emu, twin, fitness, bc, spec, env="CartPole-v1", N=1, archive=None, gen=4, sigma=0.3, eng=None):
    """One insertion on the emulator and in numpy from the same archive; both archives (asserted equal) are returned."""
    P = len(fitness)
    own = eng is None
    if own:
        eng = map_engine(emu, env, False, N, P=P)
    sd, D = eng.state_dim, eng.D
    parents = np.random.default_rng(gen).normal(0, 1, (P, D)).astype(np.float32)
    fitness = np.asarray(fitness, dtype=np.float64)
    bc = np.asarray(bc, dtype=np.float64).reshape(P, sd)
    order = twin.rank_desc(fitness)
    a = mref.empty(spec, sd, D) if archive is None else {k: v.copy() for k, v in archive.items()}
    want, entered = mref.insert(a, spec, order, fitness, bc, gen, lambda ids: twin.materialize(parents, sigma, SEED, gen, 1, 0, ids))
    insert(eng, gen, sigma, parents, order, fitness, bc, spec, a)
    assert same_archive(a, want)
    if own:
        eng.close()
    return a, entered


def test_emu_insert_all_offspring_in_one_cell(emu, twin):
    spec = mref.Spec([0, 2], [-1, -1], [1, 1], [4, 4])
    P = 20
    bc = np.tile([0.1, 9.0, 0.3, -4.0], (P, 1))
    fit = np.arange(P, dtype=np.float64) * 0.5
    a, entered = run_insert(emu, twin, fit, bc, spec)
    assert entered == [P - 1] and np.count_nonzero(~np.isnan(a["F"])) == 1


def test_emu_insert_ties_follow_the_rank_order(emu, twin):
    """Equal fitness in a cell: K2 ranks ties by descending index, so the highest id is the candidate."""
    spec = mref.Spec([1], [0], [1], [2])
    P = 12
    bc = np.zeros((P, 4))
    bc[:, 1] = np.where(np.arange(P) % 2 == 0, 0.25, 0.75)
    a, entered = run_insert(emu, twin, np.full(P, 3.0), bc, spec)
    assert sorted(entered) == [P - 2, P - 1]
    assert list(a["born"][:, 1]) == [P - 2, P - 1]


def test_emu_insert_equal_candidate_keeps_the_incumbent(emu, twin):
    spec = mref.Spec([0], [0], [1], [3])
    P = 9
    bc = np.zeros((P, 4))
    bc[:, 0] = (np.arange(P) % 3 + 0.5) / 3
    fit = np.array([1, 2, 3, 4, 5, 6, 7, 8, 9], dtype=np.float64)
    eng = map_engine(emu, P=P)
    a, _ = run_insert(emu, twin, fit, bc, spec, gen=0, eng=eng)
    # generation 1: cell 0 ties its incumbent (7), cell 1 beats it (9 > 8), cell 2 falls short (1 < 9)
    fit2 = np.array([7, 9, 1, 0, 0, 0, 0, 0, 0], dtype=np.float64)
    b, entered = run_insert(emu, twin, fit2, bc, spec, archive=a, gen=1, eng=eng)
    assert entered == [1]
    assert b["born"][0].tolist() == [0, 6] and b["born"][1].tolist() == [1, 1] and b["born"][2].tolist() == [0, 8]
    eng.close()


def test_emu_insert_nan_fitness_and_nan_behaviour_are_unplaced(emu, twin):
    spec = mref.Spec([0, 1], [0, 0], [1, 1], [2, 2])
    P = 8
    bc = np.full((P, 4), 0.2)
    fit = np.arange(P, dtype=np.float64)
    fit[7] = np.nan                   # would rank first among the NaN-free ... and is skipped
    bc[6, 1] = np.nan                 # NaN in a descriptor coordinate
    bc[5, 3] = np.nan                 # NaN outside the descriptor: still placed
    a, entered = run_insert(emu, twin, fit, bc, spec)
    assert entered == [5]


def test_emu_insert_out_of_range_and_infinite_behaviour_land_in_edge_cells(emu, twin):
    spec = mref.Spec([0, 1], [-1, -1], [1, 1], [5, 3])
    vals = [-np.inf, -1e300, -5.0, -1.0, 1.0, 5.0, 1e300, np.inf, 5e-324, -5e-324, 0.0]
    bc = np.array([[x, y, 0, 0] for x in vals for y in vals[::3]], dtype=np.float64)
    P = len(bc)
    fit = np.random.default_rng(2).permutation(P).astype(np.float64)
    a, _ = run_insert(emu, twin, fit, bc, spec)
    assert not np.isnan(a["F"][[0, 2, 12, 14]]).any()      # the four corners


def test_emu_insert_single_cell(emu, twin):
    spec = mref.Spec([3], [-2], [2], [1])
    P = 10
    bc = np.random.default_rng(1).normal(0, 3, (P, 4))
    a, entered = run_insert(emu, twin, np.random.default_rng(1).normal(0, 1, P), bc, spec)
    assert len(entered) == 1 and a["F"].shape == (1,)


@pytest.mark.parametrize("n_dims", [1, 2, 3, 4])
def test_emu_insert_descriptor_dimensions(emu, twin, n_dims):
    """simple_spread N = 3 (12 final-state coordinates): the dims in a scrambled order, a second generation on top."""
    dims = [7, 2, 11, 0][:n_dims]
    cells = [3, 5, 2, 4][:n_dims]
    spec = mref.Spec(dims, [-1.0] * n_dims, [1.0] * n_dims, cells)
    P = 60
    rng = np.random.default_rng(n_dims)
    eng = map_engine(emu, "simple_spread", False, 3, P=P)
    a = None
    for gen in (0, 1):
        bc = rng.uniform(-1.2, 1.2, (P, 12))
        fit = np.round(rng.normal(0, 2, P), 1)               # some ties
        a, _ = run_insert(emu, twin, fit, bc, spec, archive=a, gen=gen, eng=eng)
    assert np.count_nonzero(~np.isnan(a["F"])) > 1
    eng.close()


# ---------------------------------------------------------------------------------------------------- selection
@pytest.mark.parametrize("n_occ", [0, 1, 2, 3, 300, 1024])
def test_emu_select_equals_numpy(emu, twin, n_occ):
    spec = mref.Spec([0, 1], [0, 0], [1, 1], [32, 32])
    P, gen = 70, 6
    eng = map_engine(emu, P=P)
    rng = np.random.default_rng(n_occ)
    a = mref.empty(spec, 4, eng.D)
    occ = np.sort(rng.choice(spec.n_cells, n_occ, replace=False))
    a["F"][occ] = np.round(rng.normal(0, 50, n_occ), 0)    # ties for the best cell
    a["W"][:] = rng.normal(0, 1, a["W"].shape).astype(np.float32)
    seed_row = rng.normal(0, 1, eng.D).astype(np.float32)
    stats, parents = select(eng, gen, spec, a, seed_row)
    check_stats(stats, a["F"])
    assert same_bits(parents, mref.select(twin, a, P, gen, SEED, seed_row))
    if n_occ >= 3:
        assert len(set(mref.select_cells(twin, a["F"], P, gen, SEED))) > 1
    eng.close()


def test_emu_select_qd_order_and_best_tie(emu, twin):
    """Magnitudes whose sum depends on the order, and the best fitness in two cells: the lower index wins."""
    spec = mref.Spec([0], [0], [1], [3000])
    eng = map_engine(emu, P=4)
    a = mref.empty(spec, 4, eng.D)
    a["F"][::3] = np.tile([1e16, 1.0, -1e16, 3.0, 0.1], 200)
    a["F"][2100] = a["F"][2700] = 5e16
    stats, _ = select(eng, 0, spec, a, np.zeros(eng.D, np.float32))
    check_stats(stats, a["F"])
    assert stats[1] == 2100
    eng.close()


def test_emu_sharded_handle_builds_the_same_archive(emu, twin):
    """A rank of a block-cyclic shard holds the full parent table and fitness: its archive and selection equal a whole handle's."""
    spec = mref.Spec([0, 2], [-0.2, -0.2], [0.2, 0.2], [6, 6])
    P = 50
    rng = np.random.default_rng(9)
    fit, bc = rng.normal(0, 1, P), rng.normal(0, 0.1, (P, 4))
    outs = []
    for kw in ({}, {"shard": (1, 3, 4)}):
        eng = map_engine(emu, P=P, **kw)
        a, _ = run_insert(emu, twin, fit, bc, spec, eng=eng)
        outs.append((a, select(eng, 5, spec, a, np.zeros(eng.D, np.float32))))
        eng.close()
    (a0, (s0, p0)), (a1, (s1, p1)) = outs
    assert same_archive(a0, a1) and same_bits(s0, s1) and same_bits(p0, p1)


# ---------------------------------------------------------------------------------------------------- argument checks
def test_emu_map_argument_errors(emu):
    P = 16
    eng = map_engine(emu, P=P)
    lib, h, D = eng.lib, eng._h, eng.D
    spec = mref.Spec([0, 1], [0, 0], [1, 1], [4, 4])
    a = mref.empty(spec, 4, D)
    parents, order = np.zeros((P, D), np.float32), np.arange(P, dtype=np.int32)
    fit, bc = np.zeros(P), np.zeros((P, 4))
    seed_row, stats, out = np.zeros(D, np.float32), np.zeros(4), np.zeros((P, D), np.float32)

    def err(rc):
        assert rc != 0
        return lib.ses_last_error().decode()

    def ins(handle, sp, **kw):
        x = dict(parents=_p(parents), order=_p(order), fit=_p(fit), bc=_p(bc), F=_p(a["F"]), B=_p(a["B"]), born=_p(a["born"]), W=_p(a["W"]))
        x.update(kw)
        return lib.ses_map_insert(handle, 0, 0.1, x["parents"], x["order"], x["fit"], x["bc"], sp, x["F"], x["B"], x["born"], x["W"], None)

    def sel(handle, sp, **kw):
        x = dict(F=_p(a["F"]), W=_p(a["W"]), seed=_p(seed_row), stats=_p(stats), out=_p(out))
        x.update(kw)
        return lib.ses_map_select(handle, 0, sp, x["F"], x["W"], x["seed"], x["stats"], x["out"], None)

    good = C.byref(spec.ctype())
    assert "null handle" in err(ins(None, good)) and "null handle" in err(sel(None, good))
    assert "null argument" in err(ins(h, None)) and "null argument" in err(sel(h, None))
    for key in ("parents", "order", "fit", "bc", "F", "B", "born", "W"):
        assert "null argument" in err(ins(h, good, **{key: None}))
    for key in ("F", "W", "seed", "stats", "out"):
        assert "null argument" in err(sel(h, good, **{key: None}))
    bad_specs = [
        (mref.Spec([0, 1], [0, 0], [1, 1], [4, 4]), {"n_dims": 0}, "n_dims"),
        (mref.Spec([0, 1], [0, 0], [1, 1], [4, 4]), {"n_dims": 5}, "n_dims"),
        (mref.Spec([0, 4], [0, 0], [1, 1], [4, 4]), {}, "outside the final state"),
        (mref.Spec([-1, 1], [0, 0], [1, 1], [4, 4]), {}, "outside the final state"),
        (mref.Spec([1, 1], [0, 0], [1, 1], [4, 4]), {}, "distinct"),
        (mref.Spec([0, 1], [0, 1], [1, 1], [4, 4]), {}, "width > 0"),
        (mref.Spec([0, 1], [0, np.inf], [1, np.inf], [4, 4]), {}, "finite"),
        (mref.Spec([0, 1], [0, np.nan], [1, 1], [4, 4]), {}, "finite"),
        (mref.Spec([0, 1], [0, 0], [1, 1], [4, 0]), {}, "cells[1]"),
        (mref.Spec([0, 1, 2], [0, 0, 0], [1, 1, 1], [1024, 1024, 2]), {}, "2^20"),
    ]
    for sp, patch, msg in bad_specs:
        st = sp.ctype()
        for k, v in patch.items():
            setattr(st, k, v)
        assert msg in err(ins(h, C.byref(st))), msg
        assert msg in err(sel(h, C.byref(st))), msg
    assert np.isnan(a["F"]).all() and np.all(out == 0) and np.all(stats == 0)       # nothing was launched
    eng.close()
    # the weight cap: CartPole-GRU (D = 6562) allows 163 630 cells
    gru = map_engine(emu, "CartPole-v1", True, P=4)
    assert "4 GiB" in err(ins(gru._h, C.byref(mref.Spec([0, 1], [0, 0], [1, 1], [512, 320]).ctype())))
    gru.close()
    for kw in ({"n_head": 1}, {"group": 2, "n_parents": P // 2}, {"antithetic": True}):
        bad = make(emu, "CartPole-v1", seed=SEED, population=P, **dict({"group": 1, "n_head": 0, "n_parents": P, "eval_ep_num": 2}, **kw))
        assert "layout" in err(ins(bad._h, good)) and "layout" in err(sel(bad._h, good))
        bad.close()

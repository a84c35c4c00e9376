"""K2 and K3 on the host SIMT emulator (tests/simt_emu) against the plain numpy references of tests/k23_reference.py, at
the shapes and values where they go wrong; plus the twin's rank against numpy.  The GPU twin of this file is
tests/test_gpu_k23_reference.py.  The emulator has no cooperative launch, so the persistent K2 build is GPU-only, and the
emulated sort is slow: sizes stop at 33000 and the large ones run the hardest key families only."""
import numpy as np
import pytest

import k23_reference as ref


class Emu:
    def __init__(self, monkeypatch, k2_fused=1):
        from simt_emu import emu_engine
        emu_engine.load()
        self.cls = emu_engine.EmuEngine
        monkeypatch.setenv("SES_K2_FUSED", str(k2_fused))       # read when the handle is created

    def engine(self, D, P, group=None, n_head=1, n_parents=1, seed=0, antithetic=False, **kw):
        name, obs, act, gru, agents = ref.ENVS[D]
        return self.cls(env_name=name, obs_dim=obs, act_dim=act, gru=gru, n_agents=agents, population=P,
                        group=P if group is None else group, n_head=n_head, n_parents=n_parents, seed=seed, antithetic=antithetic, **kw)

    @staticmethod
    def rank(eng, r, full_key):
        if r.size < 2:
            return eng.rank_desc(r, full_key=full_key), None
        return eng.rank_desc(r, shaped=True, full_key=full_key)

    @staticmethod
    def adam(eng, gen, sigma, lr, t, shaped, mu, m, v, eps):
        mu, m, v = mu.copy(), m.copy(), v.copy()
        g = eng.update_openai(gen, sigma, lr, t, shaped, mu, m, v, eps_override=eps)
        return g, mu, m, v

    @staticmethod
    def sgd(eng, gen, sigma, lr, shaped, mu, v, momentum, eps):
        mu, v = mu.copy(), v.copy()
        g = eng.update_openai_sgd(gen, sigma, lr, shaped, mu, v, momentum=momentum, eps_override=eps)
        return g, mu, v

    @staticmethod
    def materialize(eng, gen, sigma, parents, ids):
        return eng.materialize(gen, sigma, parents, ids)

    @staticmethod
    def elite_mean(eng, gen, sigma, parents, order, k):
        return eng.elite_mean(gen, sigma, parents, order, k)


EMU_SIZES = [n for n in ref.RANK_SIZES if n <= 33000]
EMU_PARTIAL = [(n, P) for n, P in ref.RANK_PARTIAL if n <= 33000]
HARD = ("special", "nan", "descending")                  # the families the emulator runs above 4097 keys


# ------------------------------------------------------------------------------------- K2
@pytest.mark.parametrize("fused", [0, 1])
@pytest.mark.parametrize("n,P", [(n, n) for n in EMU_SIZES] + EMU_PARTIAL)
def test_emu_rank_matches_numpy(n, P, fused, monkeypatch):
    """Separate kernels (0) and the fused build (1): numpy's permutation and the reference's centered ranks."""
    fe = Emu(monkeypatch, fused)
    eng = fe.engine(226, max(P, 2))
    for kind, r in ref.key_families(n, np.random.default_rng(n + P)).items():
        if n <= 4097 or kind in HARD:
            ref.check_rank(fe, eng, r, "%s n=%d of %d" % (kind, n, P))


@pytest.mark.parametrize("fused", [0, 1])
def test_emu_rank_nan_example(fused, monkeypatch):
    """Every NaN, whatever its sign, ranks above +inf (descending index among NaNs), as in numpy."""
    fe = Emu(monkeypatch, fused)
    order, _ = fe.rank(fe.engine(226, 10), ref.NAN_EXAMPLE, True)
    assert order.tolist() == ref.NAN_EXAMPLE_ORDER


def test_twin_rank_matches_numpy(twin):
    """The twin's comparator is a strict weak order with NaNs present, so finite values keep their order too."""
    assert twin.rank_desc(ref.NAN_EXAMPLE).tolist() == ref.NAN_EXAMPLE_ORDER
    for n in (2, 33, 1000):
        for kind, r in ref.key_families(n, np.random.default_rng(n)).items():
            assert np.array_equal(twin.rank_desc(r), ref.rank_ref(r)), (kind, n)


@pytest.mark.parametrize("fused", [0, 1])
@pytest.mark.parametrize("env,E", [("CartPole-v1", 5), ("CartPole-v1", 1), ("MountainCar-v0", 5), ("Acrobot-v1", 7)])
def test_emu_rank_integer_keys(env, E, fused, monkeypatch):
    """The integer-key path (step-count envs): step totals over the whole range, both ends, with key_bits as the host picks it."""
    fe = Emu(monkeypatch, fused)
    D = {"CartPole-v1": 226, "MountainCar-v0": 195, "Acrobot-v1": 323}[env]
    for n in (257, 4097, 33000):
        eng = fe.engine(D, n, eval_ep_num=E)
        assert eng.key_bits == ref.key_bits_host(E, eng.max_step) and eng.key_scale == E
        r = ref.step_totals(n, E, eng.max_step, np.random.default_rng(n + E))
        ref.check_rank(fe, eng, r, "%s E=%d n=%d" % (env, E, n), full_key=False)


# ------------------------------------------------------------------------------------- K3
@pytest.mark.parametrize("D", sorted(ref.ENVS))
@pytest.mark.parametrize("P", [2, 31, 32, 33, 2047, 2048, 2049])
def test_emu_grad_adam_sgd_match_exact_sums(D, P, monkeypatch):
    fe = Emu(monkeypatch)
    ref.run_k3_override(fe, D, P, tied=P % 2 == 1, seed=D + P)


@pytest.mark.parametrize("D", [195, 323])
def test_emu_grad_more_than_64_groups(D, monkeypatch):
    """P = 64 * 2048 + 1: 4097 level-0 blocks, 65 level-1 groups, the last holding one offspring."""
    fe = Emu(monkeypatch)
    ref.run_k3_override(fe, D, 64 * 2048 + 1, tied=D == 195, seed=D)


@pytest.mark.parametrize("antithetic", [False, True])
@pytest.mark.parametrize("n_head,group", [(1, None), (3, None), (1, 97), (3, 97)])
def test_emu_grad_regenerated_noise(twin, n_head, group, antithetic, monkeypatch):
    ref.run_k3_regenerated(Emu(monkeypatch), twin.normals, n_head, antithetic, group)


@pytest.mark.parametrize("antithetic", [False, True])
@pytest.mark.parametrize("n_head", [1, 3])
def test_emu_materialize_and_elite_mean(twin, n_head, antithetic, monkeypatch):
    ref.run_materialize_elite(Emu(monkeypatch), twin.normals, n_head, antithetic)

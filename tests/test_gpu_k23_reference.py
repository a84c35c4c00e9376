"""K2 and K3 on the B200 against the plain numpy references of tests/k23_reference.py, at the shapes and values where they
go wrong: every tile and path switch of the sort in all three builds (separate kernels, fused, persistent), special keys,
D % 4 != 0, the edges of the gradient's reduction tree.  The emulator runs the same checks (tests/test_emu_k23_reference.py)
except the persistent sort, which exists only on the GPU."""
import numpy as np
import pytest

import k23_reference as ref

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

# SES_K2_FUSED, SES_K2_PERSISTENT; K2 launches of one float64-key sort with centered ranks (8 radix passes)
BUILDS = {"separate": ("0", "0", 18), "fused": ("1", "0", 9), "persistent": ("1", "1", 1)}


def _cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


class Gpu:
    def __init__(self, monkeypatch, build="persistent"):
        fused, persistent, _ = BUILDS[build]
        monkeypatch.setenv("SES_K2_FUSED", fused)               # read when the handle is created
        monkeypatch.setenv("SES_K2_PERSISTENT", persistent)

    @staticmethod
    def engine(D, P, group=None, n_head=1, n_parents=1, seed=0, antithetic=False, eval_ep_num=5):
        from simple_es_b200.engine import CONTINUOUS_ENVS, RolloutEngine
        name, obs, act, gru, agents = ref.ENVS[D]
        return RolloutEngine(name, obs, act, gru, False, None, eval_ep_num, P, P if group is None else group, n_head, n_parents,
                             seed=seed, n_agents=agents, antithetic=antithetic, discrete_action=name not in CONTINUOUS_ENVS,
                             test_build=True)

    @staticmethod
    def rank(eng, r, full_key):
        if r.size < 2:
            return eng.rank_desc(_cuda(r), full_key=full_key).cpu().numpy(), None
        order, shaped = eng.rank_desc(_cuda(r), shaped=True, full_key=full_key)
        return order.cpu().numpy(), shaped.cpu().numpy()

    @staticmethod
    def adam(eng, gen, sigma, lr, t, shaped, mu, m, v, eps):
        mu, m, v = _cuda(mu), _cuda(m), _cuda(v)
        g = torch.empty_like(mu)
        eng.update_openai(gen, sigma, lr, t, _cuda(shaped), mu, m, v, eps_override=None if eps is None else _cuda(eps), grad_out=g)
        return tuple(x.cpu().numpy() for x in (g, mu, m, v))

    @staticmethod
    def sgd(eng, gen, sigma, lr, shaped, mu, v, momentum, eps):
        mu, v = _cuda(mu), _cuda(v)
        g = torch.empty_like(mu)
        eng.update_openai_sgd(gen, sigma, lr, _cuda(shaped), mu, v, momentum=momentum, eps_override=None if eps is None else _cuda(eps),
                              grad_out=g)
        return tuple(x.cpu().numpy() for x in (g, mu, v))

    @staticmethod
    def materialize(eng, gen, sigma, parents, ids):
        return eng.materialize(gen, sigma, _cuda(parents), _cuda(ids)).cpu().numpy()

    @staticmethod
    def elite_mean(eng, gen, sigma, parents, order, k):
        return eng.elite_mean(gen, sigma, _cuda(parents), _cuda(order), k).cpu().numpy()


LARGEST = ref.RANK_SIZES[-1]


# ------------------------------------------------------------------------------------- K2
@pytest.mark.parametrize("build", list(BUILDS))
@pytest.mark.parametrize("n,P", [(n, n) for n in ref.RANK_SIZES] + ref.RANK_PARTIAL)
def test_rank_matches_numpy(n, P, build, monkeypatch):
    """numpy's permutation and the reference's centered ranks, every key family, in the build that was asked for (the
    persistent sort may refuse a cooperative launch that does not fit; only at the largest size is either path accepted)."""
    fe = Gpu(monkeypatch, build)
    eng = fe.engine(226, max(P, 2))
    for kind, r in ref.key_families(n, np.random.default_rng(n + P)).items():
        l0 = eng.launches
        ref.check_rank(fe, eng, r, "%s n=%d of %d, %s" % (kind, n, P, build))
        if n >= 2 and n != LARGEST:
            assert eng.launches - l0 == BUILDS[build][2], (kind, "launches")


@pytest.mark.parametrize("build", list(BUILDS))
def test_rank_nan_example(build, monkeypatch):
    """Every NaN, whatever its sign, ranks above +inf (descending index among NaNs), as in numpy."""
    fe = Gpu(monkeypatch, build)
    order, _ = fe.rank(fe.engine(226, 10), ref.NAN_EXAMPLE, True)
    assert order.tolist() == ref.NAN_EXAMPLE_ORDER


@pytest.mark.parametrize("build", list(BUILDS))
@pytest.mark.parametrize("env,E", [("CartPole-v1", 5), ("CartPole-v1", 1), ("MountainCar-v0", 5), ("Acrobot-v1", 7)])
def test_rank_integer_keys(env, E, build, monkeypatch):
    """The integer-key path (step-count envs): step totals over the whole range, both ends, with key_bits as the host picks it."""
    fe = Gpu(monkeypatch, build)
    D = {"CartPole-v1": 226, "MountainCar-v0": 195, "Acrobot-v1": 323}[env]
    for n in (257, 4097, 33000, (1 << 18) + 1):
        eng = fe.engine(D, n, eval_ep_num=E)
        assert eng.key_bits == ref.key_bits_host(E, eng.max_step) and eng.key_scale == E
        r = ref.step_totals(n, E, eng.max_step, np.random.default_rng(n + E))
        ref.check_rank(fe, eng, r, "%s E=%d n=%d" % (env, E, n), full_key=False)


# ------------------------------------------------------------------------------------- K3
@pytest.mark.parametrize("D", sorted(ref.ENVS))
@pytest.mark.parametrize("P", [2, 31, 32, 33, 2047, 2048, 2049])
def test_grad_adam_sgd_match_exact_sums(D, P, monkeypatch):
    ref.run_k3_override(Gpu(monkeypatch), D, P, tied=P % 2 == 1, seed=D + P)


@pytest.mark.parametrize("D", [195, 323])
def test_grad_more_than_64_groups(D, monkeypatch):
    """P = 64 * 2048 + 1: 4097 level-0 blocks, 65 level-1 groups, the last holding one offspring."""
    ref.run_k3_override(Gpu(monkeypatch), D, 64 * 2048 + 1, tied=D == 195, seed=D)


@pytest.mark.parametrize("antithetic", [False, True])
@pytest.mark.parametrize("n_head,group", [(1, None), (3, None), (1, 97), (3, 97)])
def test_grad_regenerated_noise(twin, n_head, group, antithetic, monkeypatch):
    ref.run_k3_regenerated(Gpu(monkeypatch), twin.normals, n_head, antithetic, group)


@pytest.mark.parametrize("antithetic", [False, True])
@pytest.mark.parametrize("n_head", [1, 3])
def test_materialize_and_elite_mean(twin, n_head, antithetic, monkeypatch):
    ref.run_materialize_elite(Gpu(monkeypatch), twin.normals, n_head, antithetic)

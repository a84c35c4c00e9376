"""Novelty search with reward (nsr_es, DESIGN.md section 4.10) at full size on the B200, bit for bit.

1. The final-state (FINAL) instances of K1 on every launch path of the scheduler: every [P][E][state_dim] row against the
   twin's final states (oracle/twin.py, population_* with final=True), fitness and steps equal to the plain launch's.  The
   launch shapes are derived from the occupancy a FINAL launch of the test build reports (the FINAL instances can use more
   registers than the plain ones), and each asserts through the geometry hook the path it was chosen for.
2. ses_behavior, ses_novelty (all 24 (state_dim, list capacity) instances, archives past one 256-row tile) and
   ses_blend_shaped against the numpy restatements of tests/novelty_reference.py.
3. nsr_es generations resumed with an archive of 1023 rows (four tiles, then five, across a capacity doubling) against the
   host restatement.

Offspring i has the same weights and episodes whatever P is (one parent, group >= P), so one twin table per population serves
every shape.  Every twin and numpy vector is computed once per module, on every host thread."""
import os
import sys
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest
import yaml

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))

import bench  # noqa: E402
import novelty_reference as nref  # noqa: E402
from test_gpu_full_size_envs import CLASSIC, POPULATIONS, _lanes, _residency_bound, gru_pumping_parent  # noqa: E402
from test_gpu_k1_full_size import P_HEAD, _shape, _tail_start  # noqa: E402
from test_gpu_novelty import centered  # noqa: E402

NT = os.cpu_count() or 1
GEN = 2                                          # generation of the classic-control populations (as test_gpu_full_size_envs)


def same_bits(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and np.array_equal(a.view(np.uint8), b.view(np.uint8))


def _cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _host(*ts):
    return tuple(t.cpu().numpy() for t in ts)


def _engine(env, P, E, gru=False, n_agents=1, pomdp=False, max_step=None, **kw):
    from simple_es_b200.engine import RolloutEngine
    if env == "CartPole-v1":
        obs, act, max_step = 4, 2, 500
    elif env == "simple_spread":
        obs, act = 6 * n_agents, 5
    else:
        obs, act = CLASSIC[env][:2]
    args = dict(n_agents=n_agents, discrete_action=env != "Pendulum-v0")
    args.update(kw)
    return RolloutEngine(env, obs, act, gru, pomdp, max_step, E, P, P, 1, 1, **args)


def final_launch(eng, gen, sigma, mu, fs=None):
    """A plain launch, then the FINAL launch into a buffer pre-filled with NaN: (fit, steps) of each, and the buffer."""
    parents = _cuda(mu)
    plain = _host(*eng.rollout(gen, sigma, parents))
    if fs is None:
        fs = torch.full((eng.P, eng.E, eng.state_dim), float("nan"), dtype=torch.float64, device="cuda")
    eng.set_final_states(fs)
    final = _host(*eng.rollout(gen, sigma, parents))
    eng.set_final_states(None)
    return plain, final, fs.cpu().numpy()


def check_final(label, plain, final, got, table, P):
    """fitness and steps of the FINAL launch equal the plain launch's; every row of the buffer equals the twin's."""
    tf, ts, tfs = table
    assert same_bits(final[0], plain[0]) and same_bits(final[1], plain[1]), label
    assert same_bits(final[1], ts[:P]) and same_bits(final[0], tf[:P]), label
    assert same_bits(got, tfs[:P]), (label, int(np.isnan(got).any(axis=(1, 2)).sum()), int((got != tfs[:P]).any(axis=(1, 2)).sum()))
    return "%d rows of [%d][%d] equal the twin" % (got.shape[0], got.shape[1], got.shape[2])


def run_both_builds(label, make, gen, sigma, mu, table, P):
    """The test build (geometry after its FINAL launch), then the product build; both against the twin."""
    t = make(True)
    plain, final, got = final_launch(t, gen, sigma, mu)
    torch.cuda.synchronize()
    g = t.test_k1_geometry()
    t.close()
    msg = check_final(label + " (test build)", plain, final, got, table, P)
    eng = make(False)
    plain, final, got = final_launch(eng, gen, sigma, mu)
    eng.close()
    check_final(label, plain, final, got, table, P)
    print("\n%s: %s; geometry after the FINAL launch %s" % (label, msg, g))
    return g


# ------------------------------------------------------------------------------------- twin tables, once per module
class Tables:
    def __init__(self, twin):
        self.twin, self.cache = twin, {}

    def get(self, key, fn):
        if key not in self.cache:
            self.cache[key] = fn()
        return self.cache[key]


@pytest.fixture(scope="module")
def tables(twin):
    return Tables(twin)


@pytest.fixture(scope="module")
def state():
    return bench.bench_state()


def _cartpole_table(tables, state, E, P, gen0=False):
    P = max(P, P_HEAD) if E == 5 else P
    if gen0:
        key, mu, sigma, gen = ("cp_gen0", E), np.zeros((1, bench.D), np.float32), 0.2, 0
    else:
        key, mu, sigma, gen = ("cp30", E), state["mu"][None], state["sigma"], 30
    cached = tables.cache.get(key)
    if cached is None or cached[0].size < P:
        tables.cache[key] = tables.twin.population_cartpole(mu, sigma=sigma, seed=0, gen=gen, group=P, n_head=1, n=P, E=E,
                                                            nthreads=NT, final=True)
    return tables.cache[key]


def _mpe_table(twin, mu, N, P, E, gru=False, **kw):
    """population_mpe with final states over every offspring, in id windows on host threads."""
    step = max(256, -(-P // (4 * NT)))
    windows = [(lo, min(P, lo + step)) for lo in range(0, P, step)]
    with ThreadPoolExecutor(NT) as ex:
        parts = list(ex.map(lambda w: twin.population_mpe(mu, N=N, gru=gru, group=P, n_head=1, id0=w[0], n=w[1] - w[0], E=E,
                                                          final=True, **kw), windows))
    return tuple(np.concatenate([p[i] for p in parts]) for i in range(3))


# ------------------------------------------------------------------------------------- A. CartPole MLP: every launch path
@pytest.fixture(scope="module")
def geometry_final(state):
    """The occupancy of the CartPole FINAL instance: one converged FINAL launch of the test build at the headline size."""
    eng = _engine("CartPole-v1", P_HEAD, 5, seed=0, test_build=True)
    final_launch(eng, 30, state["sigma"], state["mu"][None])
    torch.cuda.synchronize()
    g = eng.test_k1_geometry()
    eng.close()
    print("\nCartPole FINAL geometry at P = %d, E = 5: %s, R = %d episodes" % (P_HEAD, g, g["resident_warps"] * 32))
    return g


CP_SHAPES = ["one_round", "past_one_round", "below_2R", "past_2R_queue_a_0", "past_2R_queue_a_1", "headline", "sparse",
             "E1", "E3", "E7", "E32"]


def _sparse_P(num_sms):
    """One full CTA of 4 warps x 32 lanes per SM plus 3 episodes per warp of a second CTA: the sparse class."""
    return (num_sms * 4 * 32 + num_sms * 4 * 3) // 5


@pytest.mark.parametrize("shape", CP_SHAPES)
def test_cartpole_final_states_on_every_launch_path(tables, state, geometry_final, shape):
    """Converged populations at the FINAL instance's own round and tail boundaries, the headline, a launch of sparse warps
    (the 2- and 4-lane straggler phase), and E = 1, 3, 7, 32 with queue A non-empty."""
    R = geometry_final["resident_warps"] * 32
    if shape == "sparse":
        P, E = _sparse_P(torch.cuda.get_device_properties(0).multi_processor_count), 5
    else:
        P, E = _shape(shape, R)
    n_ep = P * E
    table = _cartpole_table(tables, state, E, P)
    g = run_both_builds("CartPole %s: P = %d, E = %d, episodes = %d" % (shape, P, E, n_ep),
                        lambda tb: _engine("CartPole-v1", P, E, seed=0, test_build=tb), 30, state["sigma"], state["mu"][None],
                        table, P)
    Rk = g["resident_warps"] * 32
    assert g["lanes"] == 32
    if E == 5:
        assert g["resident_warps"] == geometry_final["resident_warps"]
    if shape == "sparse":
        assert g["sparse_rank"] >= 0 and g["tail_start"] == 0, g
        return
    assert g["sparse_rank"] < 0 and g["tail_start"] == _tail_start(n_ep, E, g["resident_warps"]), g
    path = {"one_round": n_ep <= Rk, "past_one_round": Rk < n_ep <= 2 * Rk, "below_2R": Rk < n_ep <= 2 * Rk,
            "past_2R_queue_a_0": n_ep > 2 * Rk and g["tail_start"] == 0,
            "past_2R_queue_a_1": n_ep > 2 * Rk and g["tail_start"] == E}.get(shape, g["tail_start"] > 0)
    assert path, "shape %s no longer runs the path it was chosen for: %s" % (shape, g)


def test_cartpole_final_states_after_a_ragged_launch(tables):
    """A generation-0 population at P = 65536 on one handle: the first launch reads "long" (unknown) and takes a queue B; the
    FINAL launch after it reads the first one's short episodes as "ragged" and takes none."""
    table = _cartpole_table(tables, None, 5, P_HEAD, gen0=True)
    assert table[1].mean() / 5 < 0.25 * 500
    for tb in (True, False):
        eng = _engine("CartPole-v1", P_HEAD, 5, seed=0, test_build=tb)
        plain, final, got = final_launch(eng, 0, 0.2, np.zeros((1, bench.D), np.float32))
        if tb:
            torch.cuda.synchronize()
            g = eng.test_k1_geometry()
            print("\ngeneration 0 after a ragged launch: geometry %s" % g)
            assert g["sparse_rank"] < 0 and g["tail_start"] == _tail_start(P_HEAD * 5, 5, g["resident_warps"], tail=False), g
        eng.close()
        check_final("generation 0, test build %s" % tb, plain, final, got, table, P_HEAD)


@pytest.mark.parametrize("N", [2, 4, 8])
def test_cyclic_shares_write_one_final_state_buffer(tables, state, N):
    """The headline population as N block-cyclic shares, each handle writing its rows into one buffer: the buffer equals the
    single handle's and the twin's.  One handle alone leaves every row it does not own NaN."""
    from simple_es_b200.engine import cyclic_block, owned_ids
    tf, ts, tfs = _cartpole_table(tables, state, 5, P_HEAD)
    mu, sigma = state["mu"][None], state["sigma"]
    B = cyclic_block(P_HEAD, N)
    fs = torch.full((P_HEAD, 5, 4), float("nan"), dtype=torch.float64, device="cuda")
    fit = torch.full((P_HEAD,), float("nan"), dtype=torch.float64, device="cuda")
    steps = torch.full((P_HEAD,), -1, dtype=torch.int64, device="cuda")
    for r in range(N):
        eng = _engine("CartPole-v1", P_HEAD, 5, seed=0, shard=(r, N, B))
        eng.set_final_states(fs)
        eng.rollout(30, sigma, _cuda(mu), fitness=fit, steps=steps)
        eng.close()
    got, fit, steps = _host(fs, fit, steps)
    single = _engine("CartPole-v1", P_HEAD, 5, seed=0)
    _, _, one = final_launch(single, 30, sigma, mu)
    single.close()
    assert same_bits(got, one) and same_bits(got, tfs) and same_bits(fit, tf) and same_bits(steps, ts), N
    alone = torch.full((P_HEAD, 5, 4), float("nan"), dtype=torch.float64, device="cuda")
    eng = _engine("CartPole-v1", P_HEAD, 5, seed=0, shard=(N - 1, N, B))
    eng.set_final_states(alone)
    eng.rollout(30, sigma, _cuda(mu))
    eng.close()
    alone = alone.cpu().numpy()
    mine = owned_ids(P_HEAD, N - 1, N, B)
    rest = np.ones(P_HEAD, bool)
    rest[mine] = False
    assert same_bits(alone[mine], tfs[mine]) and np.isnan(alone[rest]).all(), N
    print("\nN = %d shares: %d rows equal the twin; one handle alone: %d rows written, %d left NaN" % (N, P_HEAD, mine.size, rest.sum()))


# ------------------------------------------------------------------------------------- A. classic control on the slot kernel
@pytest.fixture(scope="module")
def occupancy_final():
    """Resident warps of the FINAL slot-kernel instance of (env, E): one small FINAL launch of the test build."""
    cache = {}

    def get(env, E):
        if (env, E) not in cache:
            eng = _engine(env, 64, E, seed=7, test_build=True)
            mu, sigma = POPULATIONS[env]
            final_launch(eng, GEN, sigma, mu)
            torch.cuda.synchronize()
            cache[env, E] = eng.test_k1_geometry()["resident_warps"]
            eng.close()
        return cache[env, E]
    return get


SLOT_SHAPES = {"E5_below_R": (5, "below"), "E5_past_R": (5, "past"), "E1": (1, 2.5), "E5": (5, 2.5), "E7": (7, 2.5), "E32": (32, 2.5)}


def _slot_P(shape, R):
    E, rounds = SLOT_SHAPES[shape]
    if rounds == "below":
        return R // E
    if rounds == "past":
        return R // E + 1
    return -(-int(rounds * R) // E) + 1


@pytest.mark.parametrize("shape", list(SLOT_SHAPES))
@pytest.mark.parametrize("env", list(CLASSIC))
def test_classic_final_states_across_rounds(tables, occupancy_final, env, shape):
    """The ragged MountainCar / Acrobot / Pendulum populations just below and past one round of the FINAL instance and at 2.5
    rounds for E = 1, 5, 7, 32."""
    E, rounds = SLOT_SHAPES[shape]
    R = occupancy_final(env, E) * _lanes(E)
    P = _slot_P(shape, R)
    Pmax = max(_slot_P(s, occupancy_final(env, SLOT_SHAPES[s][0]) * _lanes(SLOT_SHAPES[s][0]))
               for s in SLOT_SHAPES if SLOT_SHAPES[s][0] == E)
    mu, sigma = POPULATIONS[env]
    table = tables.get((env, E), lambda: tables.twin.population_classic(env, mu, sigma=sigma, seed=7, gen=GEN, group=Pmax, n_head=1,
                                                                         n=Pmax, E=E, nthreads=NT, final=True))
    n_ep = P * E
    g = run_both_builds("%s %s: P = %d, E = %d, %.2f rounds of R = %d" % (env, shape, P, E, n_ep / R, R),
                        lambda tb: _engine(env, P, E, seed=7, test_build=tb), GEN, sigma, mu, table, P)
    assert g["resident_warps"] * _lanes(E) == R and g["lanes"] == _lanes(E)
    assert g["tail_start"] == n_ep and g["sparse_rank"] < 0
    path = n_ep <= R if rounds == "below" else R < n_ep <= 2 * R if rounds == "past" else n_ep > rounds * R
    assert path, (shape, n_ep, R)


# ------------------------------------------------------------------------------------- A. simple_spread, the GRU kernels
@pytest.mark.parametrize("E", [5, 2, 4])
@pytest.mark.parametrize("N", [2, 3])
def test_spread_final_states_every_offspring(tables, N, E):
    """simple_spread at P = 16384: the 6-slot instances (E = 5) and the 8-slot instances (E = 2, 4)."""
    P = 16384
    mu = np.random.default_rng(N).normal(0, 0.3, (1, 6 * N * 32 + 32 + 165)).astype(np.float32)
    table = tables.get(("spread", N, E), lambda: _mpe_table(tables.twin, mu, N, P, E, sigma=0.2, seed=4, gen=2, init_mode=1))
    g = run_both_builds("simple_spread N = %d, E = %d: P = %d" % (N, E, P),
                        lambda tb: _engine("simple_spread", P, E, n_agents=N, seed=4, init_mode="fresh", test_build=tb), 2, 0.2, mu,
                        table, P)
    assert g["lanes"] == _lanes(E) and g["tail_start"] == P * E and g["sparse_rank"] < 0


@pytest.mark.parametrize("E", [5, 7])
@pytest.mark.parametrize("pomdp", [False, True])
def test_cartpole_gru_final_states_past_one_round(tables, pomdp, E):
    """The CartPole-GRU kernel with more offspring than the device holds warps, at E = 5 (one lockstep chunk) and E = 7 (a
    full chunk of 5 and a partial chunk of 2)."""
    P = _residency_bound() + 1031
    D = 6562
    mu = np.random.default_rng(5).normal(0, 0.3, (1, D)).astype(np.float32)
    table = tables.get(("cp_gru", pomdp, E), lambda: tables.twin.population_cartpole(
        mu, gru=True, pomdp=pomdp, sigma=0.5, seed=2, gen=3, group=P, n_head=1, n=P, E=E, nthreads=NT, final=True))
    eng = _engine("CartPole-v1", P, E, gru=True, pomdp=pomdp, seed=2)
    plain, final, got = final_launch(eng, 3, 0.5, mu)
    eng.close()
    msg = check_final("CartPole GRU pomdp %s E = %d" % (pomdp, E), plain, final, got, table, P)
    print("\nCartPole GRU, pomdp %s, E = %d, P = %d > %d warps: %s, %d distinct step totals" % (pomdp, E, P, _residency_bound(), msg,
                                                                                               len(np.unique(table[1]))))


GRU_ENVS = {"mountaincar": ("MountainCar-v0", 1, None), "acrobot": ("Acrobot-v1", 1, None), "pendulum": ("Pendulum-v0", 1, 60),
            "spread2": ("simple_spread", 2, None), "spread3": ("simple_spread", 3, None)}


@pytest.mark.parametrize("case", list(GRU_ENVS))
def test_generic_gru_final_states_past_one_round(tables, case):
    """The generic GRU kernel on all five envs at P = 10 503, above the 9472 warps 148 SMs can hold: some warp takes a
    second offspring and must store its rows, not the first one's."""
    env, N, max_step = GRU_ENVS[case]
    P, E = _residency_bound() + 1031, 5
    eng = _engine(env, P, E, gru=True, n_agents=N, max_step=max_step, seed=5, init_mode="fresh")
    if env == "MountainCar-v0":
        mu, sigma = gru_pumping_parent()[None], 0.3
    else:
        mu = np.random.default_rng(1).normal(0, 0.3, (1, eng.D)).astype(np.float32)
        sigma = 1.0 if env != "simple_spread" else 0.5
    kw = dict(sigma=sigma, seed=5, gen=3, init_mode=1)
    if env == "simple_spread":
        table = _mpe_table(tables.twin, mu, N, P, E, gru=True, **kw)
    else:
        table = tables.twin.population_classic(env, mu, gru=True, group=P, n_head=1, n=P, E=E, max_step=max_step, nthreads=NT,
                                               final=True, **kw)
    plain, final, got = final_launch(eng, 3, sigma, mu)
    eng.close()
    msg = check_final("generic GRU %s" % case, plain, final, got, table, P)
    print("\ngeneric GRU %s: P = %d > %d warps: %s" % (case, P, _residency_bound(), msg))


# ------------------------------------------------------------------------------------- B. the novelty kernels against numpy
# state_dim -> (env, n_agents, population)
SD_HANDLES = {2: ("MountainCar-v0", 1, 65536), 4: ("CartPole-v1", 1, 65536), 8: ("simple_spread", 2, 16384),
              12: ("simple_spread", 3, 16384)}
KS = [1, 2, 3, 4, 5, 8, 9, 16, 17, 32]            # both ends of every list capacity KC in {1, 2, 4, 8, 16, 32}
A_MAX = 4097


def _archive_sizes(k):
    return sorted({a for a in (1, k - 1, k, 255, 256, 257, 513, A_MAX) if a >= 1})


def _novelty_inputs(rng, n, sd):
    """Behaviours and a 4097-row archive (whose prefixes are the smaller archives): rows near archive rows, exact duplicates
    (distance 0), integer lattice points (ties at the k-th place), magnitudes from 1e-160 to 1e160 (squares that underflow to
    subnormals or 0, or overflow to inf) and rows at 1e200 whose every distance is inf."""
    A = A_MAX
    arch = rng.normal(0, 1, (A, sd))
    arch[A // 4:A // 2] = rng.integers(-2, 3, (A // 2 - A // 4, sd))
    arch[A // 2:A // 2 + A // 8] = arch[:A // 8]
    wide = rng.uniform(-160, 160, (A // 8, sd))
    arch[A - A // 8:] = np.sign(rng.normal(size=wide.shape)) * 10.0 ** wide
    arch[A - 64:A - 32] = 1e-160 * rng.normal(size=(32, sd))
    arch = arch[rng.permutation(A)]
    bc = rng.normal(0, 1, (n, sd))
    fam = rng.integers(0, 7, n)
    src = arch[rng.integers(0, A, n)]
    bc[fam == 0] = src[fam == 0] + rng.normal(0, 1e-9, (int((fam == 0).sum()), sd))
    bc[fam == 1] = src[fam == 1]
    bc[fam == 2] = rng.integers(-2, 3, (int((fam == 2).sum()), sd))
    w = rng.uniform(-160, 160, (int((fam == 3).sum()), sd))
    bc[fam == 3] = np.sign(rng.normal(size=w.shape)) * 10.0 ** w
    bc[fam == 4] = 1e200
    bc[fam == 5] = 1e-160 * rng.normal(size=(int((fam == 5).sum()), sd))
    return bc, arch


@pytest.mark.parametrize("sd", list(SD_HANDLES))
def test_novelty_every_instance_against_numpy(sd):
    """k_novelty<SD, KC> for every KC (k = 1 .. 32 at both ends of each capacity), archives of 1, k - 1, k, 255, 256, 257,
    513 and 4097 rows (one to seventeen tiles), n = 1, 63, 65 and P: every value equals nref.novelty_table's."""
    env, N, P = SD_HANDLES[sd]
    eng = _engine(env, P, 5, n_agents=N, seed=0)
    assert eng.state_dim == sd
    bc, arch = _novelty_inputs(np.random.default_rng(sd), P, sd)
    sizes = sorted({a for k in KS for a in _archive_sizes(k)})
    want = nref.novelty_table(bc, arch, sizes, KS, threads=min(NT, 16))
    bc_d, arch_d = _cuda(bc), _cuda(arch)
    out = torch.empty(P, dtype=torch.float64, device="cuda")
    checked = 0
    for k in KS:
        for a in _archive_sizes(k):
            for n in (1, 63, 65, P):
                out.fill_(float("nan"))
                eng.novelty(bc_d[:n], arch_d, a, k, out=out[:n])
                got = out[:n].cpu().numpy()
                assert same_bits(got, want[a, k][:n]), (sd, k, a, n, int((got != want[a, k][:n]).sum()))
                checked += n
    v = want[A_MAX, 32]
    print("\nnovelty, state_dim %d: %d values of %d launches equal numpy; at k = 32, |A| = 4097: %d inf, %d zero-distance rows at k = 1"
          % (sd, checked, len(KS) * 4 * 8, int(np.isinf(v).sum()), int((want[A_MAX, 1] == 0).sum())))
    assert np.isinf(v).any() and (want[A_MAX, 1] == 0).any()
    eng.close()


@pytest.mark.parametrize("sd", list(SD_HANDLES))
def test_behavior_every_state_dim_against_numpy(sd):
    """k_behavior at E = 1, 2, 5, 32, n = P, with final states whose magnitudes cancel (+-1e16 beside values near 1), so
    that any other order of the episode sum changes bits."""
    env, N, P = SD_HANDLES[sd]
    rng = np.random.default_rng(100 + sd)
    for E in (1, 2, 5, 32):
        eng = _engine(env, P, E, n_agents=N, seed=0)
        fs = rng.normal(0, 1, (P, E, sd)) * 10.0 ** rng.integers(-3, 17, (P, E, sd))
        fs[:, ::3] *= -1.0
        got = eng.behavior(_cuda(fs)).cpu().numpy()
        eng.close()
        want = nref.behavior(fs)
        assert same_bits(got, want), (sd, E, int((got != want).sum()))
        if E >= 5:                                   # the data can tell the order apart
            assert not same_bits(nref.behavior(fs[:, ::-1]), want)
    print("\nbehaviour, state_dim %d: %d rows x 4 episode counts equal numpy" % (sd, P))


def test_blend_on_real_centered_ranks():
    """k_blend_shaped at w = 0, 2^-53, 0.5, 1 - 2^-53 and 1 on K2's centered ranks of fitness with ties and of novelty:
    equal to nref.blend; w = 0 returns shaped_f and w = 1 returns shaped_n bit for bit."""
    P = 65536
    eng = _engine("CartPole-v1", P, 5, seed=0)
    rng = np.random.default_rng(7)
    fit = rng.integers(0, 2500, P).astype(np.float64) / 5
    nov = rng.exponential(1.0, P)
    _, sf = eng.rank_desc(_cuda(fit), shaped=True)
    _, sn = eng.rank_desc(_cuda(nov), shaped=True, full_key=True)
    sf_h, sn_h = _host(sf, sn)
    assert same_bits(sf_h, centered(fit)) and same_bits(sn_h, centered(nov))
    for w in (0.0, 2.0 ** -53, 0.5, 1.0 - 2.0 ** -53, 1.0):
        got = eng.blend_shaped(sf, sn, w).cpu().numpy()
        assert same_bits(got, nref.blend(sf_h, sn_h, w)), w
    assert same_bits(eng.blend_shaped(sf, sn, 0.0).cpu().numpy(), sf_h)
    assert same_bits(eng.blend_shaped(sf, sn, 1.0).cpu().numpy(), sn_h)
    eng.close()


# ------------------------------------------------------------------------------------- C. nsr_es at full size
ARCHIVE_ROWS = 1023                              # + 1 per generation: 1024 rows (four full tiles), then 1025 in a grown buffer


def _nsr(conf, P, k, seed, network=None, engine_cfg=None, name="nsr_es"):
    from simple_es_b200.strategies import STRATEGIES
    cfg = yaml.load(open(os.path.join(ROOT, "conf", conf)), Loader=yaml.FullLoader)
    strat = dict(cfg["strategy"], name=name, offspring_num=P)
    strat.pop("novelty_weight", None)
    strat.pop("novelty_k", None)
    if name == "nsr_es":
        strat.update(novelty_weight=0.5, novelty_k=k)
    return STRATEGIES[name](strat, cfg["env"], dict(cfg["network"], **(network or {})), 5, seed, 0,
                            dict(cfg["engine"], **(engine_cfg or {})))


# run -> (conf, P, k, seed, network override, engine override, generation-30 state)
NSR_RUNS = {"cartpole": ("cartpole_openai.yaml", P_HEAD, 32, 0, None, None, True),
            "spread3": ("simplespread.yaml", 16384, 10, 4, {"num_state": 18}, {"n_agents": 3}, False),
            "mountaincar_gru": ("mountaincar_nsr.yaml", 16384, 17, 3, {"gru": True}, None, False)}


def _twin_final(tables, run, s, mu, sigma, gen):
    """The twin's final states of the whole population the strategy rolled out (every row)."""
    tw = tables.twin
    if run == "cartpole":
        assert gen == 30
        return _cartpole_table(tables, bench.bench_state(), 5, P_HEAD)[2]
    if run == "spread3":
        return _mpe_table(tw, mu, 3, s.P, 5, sigma=sigma, seed=4, gen=gen, init_mode=1)[2]
    return tw.population_classic("MountainCar-v0", mu, gru=True, sigma=sigma, seed=3, gen=gen, group=s.P, n_head=1, n=s.P, E=5,
                                 init_mode=1, nthreads=NT, final=True)[2]


@pytest.mark.parametrize("run", list(NSR_RUNS))
def test_nsr_es_resumed_with_a_large_archive(tables, run):
    """Three nsr_es generations resumed from a state whose archive holds 1023 rows: the final states of the first
    generation (every row) equal the twin's; every generation's bc, novelty, shaped vector and mu / m / v equal the host
    restatement (numpy behaviours, archive and novelty, centered ranks, the blend, then ses_update_openai on the host's
    vector)."""
    conf, P, k, seed, net, ecfg, gen30 = NSR_RUNS[run]
    s = _nsr(conf, P, k, seed, net, ecfg)
    st = s.state()
    rng = np.random.default_rng(11)
    if gen30:
        cs = bench.converged_state()
        st.update({key: cs[key] for key in ("generation", "sigma", "curr_sigma", "parents", "m", "v", "t")})
    else:
        st["parents"] = torch.from_numpy(rng.normal(0, 0.3, tuple(st["parents"].shape)).astype(np.float32))
    sd = s.engine.state_dim
    archive = rng.normal(0, 1, (ARCHIVE_ROWS, sd)) * rng.uniform(0.01, 2.0, sd)
    archive[ARCHIVE_ROWS // 2:ARCHIVE_ROWS // 2 + 40] = archive[:40]
    st["archive"] = torch.from_numpy(archive)
    s.load_state(st)
    ref = _nsr(conf, P, k, seed, net, ecfg, name="openai_es")
    archive = list(archive)
    for i in range(3):
        torch.cuda.synchronize()
        mu0, m0, v0 = (t.cpu().numpy().copy() for t in (s.parents, s.m, s.v))
        gen, t0, sigma0 = s.generation, s.t, s.sigma
        s.step()
        torch.cuda.synchronize()
        fs = s.final_states.cpu().numpy()
        if i == 0:
            want = _twin_final(tables, run, s, mu0, sigma0, gen)
            assert same_bits(fs, want), (run, int((fs != want).any(axis=(1, 2)).sum()))
        bc = nref.behavior(fs)
        assert same_bits(s.bc.cpu().numpy(), bc), (run, i)
        archive.append(bc[0])
        assert s.n_archive == len(archive) and s.archive.shape[0] == (1024 if len(archive) <= 1024 else 2048)
        nov = nref.novelty_table(bc, np.asarray(archive), [len(archive)], [k], threads=min(NT, 16))[len(archive), k]
        assert same_bits(s.novelty.cpu().numpy(), nov), (run, i)
        shaped = nref.blend(centered(s.fitness.cpu().numpy()), centered(nov), 0.5)
        assert same_bits(s.shaped.cpu().numpy(), shaped), (run, i)
        mu, m, v = (_cuda(a) for a in (mu0[0], m0, v0))
        ref.engine.update_openai(gen, sigma0, s.lr, t0 + 1, _cuda(shaped), mu, m, v)
        torch.cuda.synchronize()
        assert same_bits(s.parents[0].cpu().numpy(), mu.cpu().numpy()), (run, i)
        assert same_bits(s.m.cpu().numpy(), m.cpu().numpy()) and same_bits(s.v.cpu().numpy(), v.cpu().numpy()), (run, i)
    assert same_bits(s.archive[:s.n_archive].cpu().numpy(), np.asarray(archive))
    print("\nnsr_es %s: P = %d, k = %d, state_dim %d, archive %d -> %d rows (capacity %d); %d final-state rows equal the twin"
          % (run, P, k, sd, ARCHIVE_ROWS, s.n_archive, s.archive.shape[0], P))

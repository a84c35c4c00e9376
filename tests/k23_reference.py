"""Plain numpy references for K2 (rank, centered ranks) and K3 (gradient, Adam / SGD, elite mean, materialise).

The bit-exact tests compare every kernel with the C twin (oracle/ses_twin*.c), which was written to the same contract as
the kernels, so a mistake both share passes them.  These references are independent of the twin: each restates the
operation from its definition (numpy's own sort, the reference's centered-rank formula, float64 or extended-precision
sums), and the tests compare the kernels with them within stated rounding bounds.  Only the Philox normals come from the
twin (`normals`): they are pinned by the Philox known-answer test and by the kernel-against-twin normals tests.
"""
import numpy as np

U32 = 2.0 ** -24                     # unit roundoff of float32
U64 = 2.0 ** -53                     # unit roundoff of float64


# ------------------------------------------------------------------------------------- K2
def rank_ref(r):
    """order[k] = offspring of rank k (0 = best): np.flip(np.argsort(r, kind="stable")).  numpy sorts every NaN, whatever
    its sign or payload, after +inf, and -0.0 equal to +0.0; ties keep index order, so the flip ranks them by descending
    index."""
    return np.flip(np.argsort(np.asarray(r, dtype=np.float64), kind="stable")).astype(np.int32)


def centered_ref(order):
    """The reference's centered ranks (offspring_strategies.py:392-398): the offspring of rank k (0 = best) gets
    (P-1-k)/(P-1) - 0.5, then the vector is standardised with numpy's mean and (population) std."""
    order = np.asarray(order)
    P = order.size
    ranks = np.empty(P, dtype=np.float64)
    ranks[order] = np.arange(P - 1, -1, -1, dtype=np.float64)
    y = ranks / (P - 1) - 0.5
    return (y - y.mean()) / y.std()


# ------------------------------------------------------------------------------------- population layout
def layout_ref(P, group, n_head, antithetic):
    """(parent, perturbed, noise_id, sign) of offspring 0..P-1.  Groups of `group` consecutive ids share parent id // group;
    the first `n_head` slots of a group are the parent itself (no noise); with antithetic sampling the perturbed slots come
    in pairs, the second of a pair reusing the first one's noise with the sign flipped."""
    ids = np.arange(P, dtype=np.int64)
    slot = ids % group
    perturbed = slot >= n_head
    odd = ((slot - n_head) % 2 == 1) & perturbed if antithetic else np.zeros(P, dtype=bool)
    return ids // group, perturbed, ids - odd, np.where(odd, -1.0, 1.0).astype(np.float32)


def noise_rows(normals, seed, gen, P, D, group, n_head, antithetic, ids=None):
    """eps[j] of the offspring `ids` (default all), float32 [n, D]; zero rows for unperturbed ones.  normals(seed, gen, id, D)
    is the Philox stream of one noise id."""
    _, perturbed, nid, sign = layout_ref(P, group, n_head, antithetic)
    ids = np.arange(P) if ids is None else np.asarray(ids)
    eps = np.zeros((ids.size, D), dtype=np.float32)
    for r, j in enumerate(ids):
        if perturbed[j]:
            eps[r] = sign[j] * normals(seed, gen, int(nid[j]), D)       # times +-1: exact
    return eps


# ------------------------------------------------------------------------------------- K3
def grad_ref(eps, F, rows=2048):
    """(S, err, mag) per column: S = sum_j eps[j] * F[j] in np.longdouble, err a bound on |S - exact sum|, mag = sum_j
    |eps[j]| |F[j]|.  Every product and every addition rounds once with relative error <= finfo(longdouble).eps / 2, and no
    term passes through more than P + 1 of them in any summation order, so |S - exact| <= (P + 1) eps_ld * mag (x87 extended
    precision: 2^-63 * P * mag; where longdouble is float64 the bound is simply looser)."""
    eps = np.asarray(eps, dtype=np.float32)
    F = np.asarray(F, dtype=np.float64)
    P, D = eps.shape
    S = np.zeros(D, dtype=np.longdouble)
    mag = np.zeros(D, dtype=np.float64)
    for a in range(0, P, rows):
        e = eps[a:a + rows].astype(np.longdouble)
        f = F[a:a + rows].astype(np.longdouble)[:, None]
        S += (e * f).sum(axis=0)
        mag += np.abs(F[a:a + rows]) @ np.abs(eps[a:a + rows].astype(np.float64))
    mag *= 1.0 + 1e-12                                    # the float64 sum of magnitudes is itself rounded
    err = (P + 1) * float(np.finfo(np.longdouble).eps) * mag
    return S, err, mag


def grad_bounds(S, err, mag, P, update_factor):
    """[lo, hi] of the float32 gradient the contract allows (DESIGN.md section 4.6): the float64 tree sum s, rounded once to
    float32, times float32(update_factor), rounded.  s lies within P * 2^-52 * mag of the exact sum (each of the at most
    P - 1 fma / adds on a term's path rounds once, relative 2^-53), so round32(s) lies between the roundings of the ends of
    that interval, and so does the scaled product (rounding and scaling are monotone).  Unless the exact sum sits within the
    bound of a float32 rounding boundary, lo == hi: the one float32 the contract produces."""
    tree = P * 2.0 ** -52 * mag
    uf = np.float32(update_factor)
    w = np.longdouble(err) + np.longdouble(tree)
    a = (S - w).astype(np.float32) * uf                  # float32 * float32: one IEEE rounding
    b = (S + w).astype(np.float32) * uf
    return np.minimum(a, b), np.maximum(a, b)


def adam_step_size(lr, t, beta1=0.99, beta2=0.999):
    """optimizers.py:43-47: the step size a of Adam step t (t counted from 1)."""
    return lr * np.sqrt(1 - beta2 ** t) / (1 - beta1 ** t)


def adam_ref(theta, m, v, g, a, beta1=0.99, beta2=0.999, epsilon=1e-8):
    """optimizers.py:42-57 + :13-24 in float64: m = b1 m + (1 - b1) g, v = b2 v + (1 - b2) g^2, theta += -a m / (sqrt(v) + eps).
    Returns (theta, m, v, step) in float64."""
    theta, m, v, g = (np.asarray(x, dtype=np.float64) for x in (theta, m, v, g))
    m = beta1 * m + (1.0 - beta1) * g
    v = beta2 * v + (1.0 - beta2) * (g * g)
    step = -a * m / (np.sqrt(v) + epsilon)
    return theta + step, m, v, step


def sgd_ref(theta, v, g, stepsize, momentum):
    """SGD with momentum in float64: v = mom v + (1 - mom) g, theta += -stepsize v.  Returns (theta, v, step)."""
    theta, v, g = (np.asarray(x, dtype=np.float64) for x in (theta, v, g))
    v = momentum * v + (1.0 - momentum) * g
    step = -stepsize * v
    return theta + step, v, step


def materialize_ref(parents, sigma, eps, parent_of):
    """parent + sigma * eps per row, in float64 (the exact value up to 2^-53 relative; the float32 result is this rounded
    once).  parents [n_parents, D], eps [n, D] (zero rows for unperturbed offspring), parent_of [n]."""
    p = np.asarray(parents, dtype=np.float64)[np.asarray(parent_of)]
    return p + np.float64(np.float32(sigma)) * np.asarray(eps, dtype=np.float64)


def elite_mean_ref(rows):
    """float64 mean of the materialised elite rows [k, D] (float32)."""
    return np.asarray(rows, dtype=np.float64).mean(axis=0)


def ulp32(x):
    """Spacing of float32 at |x| (the gap to the next larger float32)."""
    return np.spacing(np.abs(np.asarray(x, dtype=np.float32))).astype(np.float64)


# ------------------------------------------------------------------------------------- cases and checks
# Shared by tests/test_gpu_k23_reference.py (B200) and tests/test_emu_k23_reference.py (host SIMT emulator).  A front end
# `fe` wraps one engine flavour with numpy in / numpy out:
#   fe.engine(D, P, group=None, n_head=1, n_parents=1, seed=0, antithetic=False, eval_ep_num=5)
#   fe.rank(eng, r, full_key) -> (order, shaped or None)
#   fe.adam(eng, gen, sigma, lr, t, shaped, mu, m, v, eps) -> (grad, mu, m, v)
#   fe.sgd(eng, gen, sigma, lr, shaped, mu, v, momentum, eps) -> (grad, mu, v)
#   fe.materialize(eng, gen, sigma, parents, ids)              fe.elite_mean(eng, gen, sigma, parents, order, k)

# parameter count -> (env name, obs, act, gru, agents): one entry per env / policy pair (D % 4 = 1, 3, 2, 3, 1, 1, 2)
ENVS = {161: ("Pendulum-v0", 3, 1, False, 1), 195: ("MountainCar-v0", 2, 3, False, 1), 226: ("CartPole-v1", 4, 2, False, 1),
        323: ("Acrobot-v1", 6, 3, False, 1), 581: ("simple_spread", 12, 5, False, 2), 773: ("simple_spread", 18, 5, False, 3),
        6562: ("CartPole-v1", 4, 2, True, 1)}

# the rank sizes: both sides of every tile (256 / 512 / 1024 / 4096 keys), of the 512-key tiles' limit (population 2^15) and
# of the 4096-key tiles' threshold (n = 2^18); (n, population) with n < population on both sides of both limits
RANK_SIZES = [1, 2, 3, 31, 32, 33, 255, 256, 257, 511, 512, 513, 1023, 1024, 1025, 4095, 4096, 4097, 16384, 32767, 32768, 32769,
              (1 << 18) - 1, 1 << 18, (1 << 18) + 1, (1 << 20) + 7]
RANK_PARTIAL = [(100, 40000), (32768, 32769), (1 << 18, (1 << 18) + 5)]

DBL_MAX = float(np.finfo(np.float64).max)
NAN_BITS = (0x7FF8000000000000, 0xFFF8000000000000, 0x7FF0000000000001, 0xFFF0000000000123)   # +-qNaN, +sNaN, -NaN payload


def _bits(b):
    return np.asarray(b, dtype=np.uint64).view(np.float64)


def key_families(n, rng):
    """float64 fitness vectors where a radix sort goes wrong: a converged population (all equal), special values, keys that
    differ only in the lowest mantissa bit (the first digit pass) or only in the top byte (the last), presorted vectors with
    ties (stability), alternating signs, and NaNs of both signs among finite values and infinities."""
    i = np.arange(n)
    asc = np.sort(rng.integers(-(n // 4) - 1, n // 4 + 2, n)).astype(np.float64)
    special = np.array([np.inf, -np.inf, 0.0, -0.0, 5e-324, -5e-324, DBL_MAX, -DBL_MAX, 1.0, -1.0])
    nan = rng.normal(0, 1, n)
    pick = rng.random(n)
    nan[pick < 0.05] = np.inf
    nan[(pick >= 0.05) & (pick < 0.1)] = -np.inf
    for k, b in enumerate(NAN_BITS):
        nan[(pick >= 0.1 + 0.05 * k) & (pick < 0.15 + 0.05 * k)] = _bits(b)
    nan[n // 2] = _bits(NAN_BITS[1])
    return {
        "equal": np.full(n, 0.1),
        "special": special[rng.integers(0, special.size, n)],
        "lowbit": _bits(0x3FF8000000000000 + rng.integers(0, 2, n).astype(np.uint64)),
        "topbyte": _bits((rng.integers(0, 256, n).astype(np.uint64) << np.uint64(56)) | np.uint64(0x00123456789ABCDE)),
        "ascending": asc,
        "descending": asc[::-1].copy(),
        "alternating": np.where(i % 2 == 0, 1.0, -1.0) * (i // 2),
        "nan": nan,
    }


# The NaN example: numpy ranks every NaN best (descending index among them), -0.0 equal to +0.0
NAN_EXAMPLE = np.array([1.0, _bits(NAN_BITS[1]), 2.0, np.nan, -np.inf, np.inf, -0.0, 0.0, 5e-324, -5e-324])
NAN_EXAMPLE_ORDER = [3, 1, 5, 2, 0, 8, 7, 6, 9, 4]


def check_rank(fe, eng, r, what, full_key=True):
    """Permutation equal to numpy's, centered ranks within 1e-12 of the reference's formula."""
    want = rank_ref(r)
    order, shaped = fe.rank(eng, r, full_key)
    if not np.array_equal(order, want):
        bad = int(np.flatnonzero(order != want)[0])
        raise AssertionError("%s: rank %d of %d is offspring %d (fitness %r), numpy has %d (fitness %r)"
                             % (what, bad, r.size, order[bad], r[order[bad]], want[bad], r[want[bad]]))
    if shaped is not None:
        np.testing.assert_allclose(shaped, centered_ref(want), rtol=1e-12, atol=1e-15, err_msg=what)


def key_bits_host(E, max_step):
    """key_bits as ses_generation_openai_host chooses it: the least k with 2^k > E * max_step."""
    k = 0
    while (1 << k) <= E * max_step:
        k += 1
    return k


def step_totals(n, E, max_step, rng):
    """Fitness = (signed step total) / E over the integer-key range, both ends included."""
    vmax = E * max_step
    s = rng.integers(-vmax, vmax + 1, n)
    ends = np.array([vmax, -vmax, 0, 1, -1, vmax - 1, 1 - vmax])[:n]
    s[rng.permutation(n)[:ends.size]] = ends
    return s / E


def check_grad(g, eps, F, update_factor):
    S, err, mag = grad_ref(eps, F)
    lo, hi = grad_bounds(S, err, mag, eps.shape[0], update_factor)
    bad = np.flatnonzero((g < lo) | (g > hi))
    assert bad.size == 0, "gradient[%d] = %r outside [%r, %r] (%d of %d parameters)" % (bad[0], g[bad[0]], lo[bad[0]], hi[bad[0]],
                                                                                       bad.size, g.size)


def check_adam(mu, m, v, g, a, got, beta1=0.99, beta2=0.999, epsilon=1e-8):
    """Kernel's (mu, m, v) after one Adam step from the kernel's own gradient g, against adam_ref in float64.  The kernel
    runs m and v in float32 with float32(beta): <= 3 roundings of relative 2^-24 on each of the two terms of m (4 of v),
    the step in float64 from those (sqrt, + eps, in float32: 3 more), theta rounded once to float32."""
    mu_k, m_k, v_k = (np.asarray(x, dtype=np.float64) for x in got)
    th, mr, vr, step = adam_ref(mu, m, v, g, a, beta1, beta2, epsilon)
    g = np.asarray(g, dtype=np.float64)
    bm = 4 * U32 * (beta1 * np.abs(np.asarray(m, np.float64)) + (1 - beta1) * np.abs(g))
    bv = 6 * U32 * (beta2 * np.asarray(v, np.float64) + (1 - beta2) * g * g)
    assert np.all(np.abs(m_k - mr) <= bm), "Adam m"
    assert np.all(np.abs(v_k - vr) <= bv), "Adam v"
    bstep = a * bm / (np.sqrt(vr) + epsilon) + 8 * U32 * np.abs(step)
    bmu = bstep + 0.5 * ulp32(mu_k) + 4 * U64 * (np.abs(np.asarray(mu, np.float64)) + np.abs(step))
    assert np.all(np.abs(mu_k - th) <= bmu), "Adam mu: worst %.3g of its bound" % np.max(np.abs(mu_k - th) / bmu)


def check_sgd(mu, v, g, lr, momentum, got):
    """v and mu in float32 (four separately rounded operations, float32(momentum) and float32(-lr)) against sgd_ref."""
    mu_k, v_k = (np.asarray(x, dtype=np.float64) for x in got)
    th, vr, step = sgd_ref(mu, v, g, lr, momentum)
    bv = 4 * U32 * (momentum * np.abs(np.asarray(v, np.float64)) + (1 - momentum) * np.abs(np.asarray(g, np.float64)))
    assert np.all(np.abs(v_k - vr) <= bv), "SGD v"
    bmu = lr * bv + 3 * U32 * np.abs(step) + 0.5 * ulp32(mu_k)
    assert np.all(np.abs(mu_k - th) <= bmu), "SGD mu: worst %.3g of its bound" % np.max(np.abs(mu_k - th) / bmu)


def run_k3_override(fe, D, P, tied, seed):
    """Gradient from given eps rows (eps_override) and shaped fitness, then Adam and SGD from the kernel's gradient."""
    rng = np.random.default_rng(seed)
    eng = fe.engine(D, P, seed=seed)
    fit = np.round(rng.normal(0, 2, P)) if tied else rng.normal(0, 1, P)
    shaped = centered_ref(rank_ref(fit))
    eps = rng.normal(0, 1, (P, D)).astype(np.float32)
    lr, sigma, t = 0.05, 0.1, 3
    uf = -(lr / (P * sigma))                             # offspring_strategies.py:406-408
    mu = rng.normal(0, 1, D).astype(np.float32)
    m = rng.normal(0, 0.01, D).astype(np.float32)
    v = np.abs(rng.normal(0, 0.01, D)).astype(np.float32)
    g, *got = fe.adam(eng, 1, sigma, lr, t, shaped, mu, m, v, eps)
    check_grad(g, eps, shaped, uf)
    check_adam(mu, m, v, g, adam_step_size(lr, t), got)
    for momentum in (0.9, 0.0):
        g2, *got = fe.sgd(eng, 1, sigma, lr, shaped, mu, v, momentum, eps)
        assert np.array_equal(g2, g), "the SGD build reduces the gradient differently"
        check_sgd(mu, v, g, lr, momentum, got)


def run_k3_regenerated(fe, normals, n_head, antithetic, group, seed=11, gen=6):
    """Gradient with the noise regenerated from the layout (no eps_override) against the exact sum over eps rows built
    from layout_ref and the Philox normals; unperturbed rows must contribute exactly nothing."""
    D, P = 195, 2 * 2048 + 37                            # 130 level-0 blocks -> 3 level-1 groups, the last one ragged
    group = P if group is None else group
    rng = np.random.default_rng(seed + n_head)
    eng = fe.engine(D, P, group=group, n_head=n_head, n_parents=(P - 1) // group + 1, seed=seed, antithetic=antithetic)
    eps = noise_rows(normals, seed, gen, P, D, group, n_head, antithetic)
    lr, sigma = 0.1, 0.3
    zeros = np.zeros(D, np.float32)
    shaped = centered_ref(rank_ref(rng.normal(0, 1, P)))
    g = fe.adam(eng, gen, sigma, lr, 1, shaped, zeros, zeros, zeros, None)[0]
    check_grad(g, eps, shaped, -(lr / (P * sigma)))
    perturbed = layout_ref(P, group, n_head, antithetic)[1]
    heads_only = np.where(perturbed, 0.0, rng.normal(0, 1e3, P))
    g = fe.adam(eng, gen, sigma, lr, 1, heads_only, zeros, zeros, zeros, None)[0]
    assert np.all(g == 0.0), "unperturbed offspring contribute to the gradient"


def run_materialize_elite(fe, normals, n_head, antithetic, seed=23, gen=4):
    """Weights of head and perturbed offspring, and the elite mean for k in {1, 2, 3, 7, 64, P}, against float64
    references: a materialised weight is parent + sigma*eps rounded once (<= half a float32 ulp); the elite mean a float32
    running sum of k rows (<= (k - 1) roundings of relative 2^-24), each row itself within 2^-24, then one division."""
    D, group, n_par = 195, 97, 2
    P = group * n_par
    sigma = 0.37
    rng = np.random.default_rng(seed)
    parents = rng.normal(0, 1, (n_par, D)).astype(np.float32)
    eng = fe.engine(D, P, group=group, n_head=n_head, n_parents=n_par, seed=seed, antithetic=antithetic)
    parent_of, perturbed = layout_ref(P, group, n_head, antithetic)[:2]
    ids = np.array([0, n_head - 1, n_head, n_head + 1, n_head + 2, group - 1, group, group + n_head, P - 1], dtype=np.int32)
    out = fe.materialize(eng, gen, sigma, parents, ids)
    ref = materialize_ref(parents, sigma, noise_rows(normals, seed, gen, P, D, group, n_head, antithetic, ids), parent_of[ids])
    assert np.array_equal(out[~perturbed[ids]], parents[parent_of[ids][~perturbed[ids]]]), "a head is not its parent"
    bound = 0.5 * ulp32(out) + 2 * U64 * np.abs(ref)
    assert np.all(np.abs(out - ref) <= bound), "materialise: worst %.3g of its bound" % np.max(np.abs(out - ref) / bound)
    order = rng.permutation(P).astype(np.int32)
    for k in (1, 2, 3, 7, 64, P):
        got = fe.elite_mean(eng, gen, sigma, parents, order, k).astype(np.float64)
        rows = materialize_ref(parents, sigma, noise_rows(normals, seed, gen, P, D, group, n_head, antithetic, order[:k]),
                               parent_of[order[:k]])
        ref = elite_mean_ref(rows)
        bound = (k + 1) * U32 * np.abs(rows).mean(axis=0) + 0.5 * ulp32(got)
        assert np.all(np.abs(got - ref) <= bound), "elite mean k=%d: worst %.3g of its bound" % (k, np.max(np.abs(got - ref) / bound))

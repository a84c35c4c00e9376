"""numpy restatement of sep_cma_es (DESIGN.md section 4.11): steps 1 (sample), 3 (weights), 4 (the two reduction tables) and
5 (the update), float64 with every operation rounded once and every sum in the kernels' order, so that the kernels must match
it bit for bit -- except sigma, which goes through the device exp (<= 1 ulp) and is held to 2 ulp.

Level 0 of the tables is a chain of fused multiply-adds.  numpy has none, so `fma` emulates it exactly: Dekker's product
splits a*b into two doubles, and the sum of those and c is rounded once with Boldo and Melquiond's rounding-to-odd step
("Emulation of FMA and correctly rounded sums: proved algorithms using rounding to odd", IEEE TC 57(4), 2008).
"""
import numpy as np

GB0, GB1 = 32, 64               # level-0 blocks of offspring, level-1 groups of blocks (csrc/update.cuh)
CMA_THREADS = 256               # k_cma_final's threads: the tree of |p_sigma|^2 (csrc/cma.cuh)


def _split(a):
    t = 134217729.0 * a          # 2^27 + 1: Veltkamp's split into two halves of 26 bits
    hi = t - (t - a)
    return hi, a - hi


def _two_sum(a, b):
    s = a + b
    bb = s - a
    return s, (a - (s - bb)) + (b - bb)


def _two_prod(a, b):
    p = a * b
    ah, al = _split(a)
    bh, bl = _split(b)
    return p, ((ah * bh - p) + ah * bl + al * bh) + al * bl


def fma(a, b, c):
    """round(a * b + c) once, elementwise, for finite float64 operands whose product neither overflows nor underflows."""
    a, b, c = (np.asarray(x, dtype=np.float64) for x in (a, b, c))
    uh, ul = _two_prod(a, b)
    th, tl = _two_sum(c, uh)
    v, e = _two_sum(tl, ul)
    even = (v.view(np.int64) & 1) == 0
    v = np.where((e != 0) & even, np.nextafter(v, np.where(e > 0, np.inf, -np.inf)), v)      # round to odd
    return th + v


def normals(twin, seed, gen, ids, D):
    """z [len(ids), D] float32: the Philox normals of each id in generation gen (what K1's sampling and K3 re-derive)."""
    return np.stack([twin.normals(int(seed) & 0xFFFFFFFF, int(gen), int(i), int(D)) for i in ids])


def sample(mean, c, sigma, z):
    """Step 1: (float)(mean + sigma (sqrt(c) z)) per row of z."""
    return (mean[None, :] + sigma * (np.sqrt(c)[None, :] * z.astype(np.float64))).astype(np.float32)


def weights(order, w, mu, P):
    """Step 3: s[order[r]] = w[r] for r < mu, 0 otherwise."""
    s = np.zeros(P)
    s[np.asarray(order[:mu], dtype=np.int64)] = w[:mu]
    return s


def tables(s, z):
    """Step 4, levels 0 and 1: ([nb1, D] sum_j s_j z_jd, [nb1, D] sum_j s_j z_jd^2) per group of 64 blocks of 32 offspring.
    z: [P, D] float32 in id order."""
    P, D = z.shape
    nb0 = (P + GB0 - 1) // GB0
    nb1 = (nb0 + GB1 - 1) // GB1
    zz = np.zeros((nb0 * GB0, D))
    zz[:P] = z
    ss = np.zeros(nb0 * GB0)
    ss[:P] = s
    zz = zz.reshape(nb0, GB0, D)
    ss = ss.reshape(nb0, GB0)
    a = np.zeros((nb0, D))
    q = np.zeros((nb0, D))
    for k in range(GB0):
        f = ss[:, k:k + 1]
        e = zz[:, k, :]
        a = fma(e, f, a)
        q = fma(e * e, f, q)
    out = []
    for part in (a, q):
        t1 = np.zeros((nb1, D))
        for g in range(nb1):
            t = 0.0
            for b in range(g * GB1, min(nb0, (g + 1) * GB1)):
                t = t + part[b]
            t1[g] = t
        out.append(t1)
    return out[0], out[1]


def level2(t):
    s = np.zeros(t.shape[1])
    for g in range(t.shape[0]):
        s = s + t[g]
    return s


def norm_tree(p):
    """sqrt of sum p_d^2: per thread t of CMA_THREADS the sequential sum over d = t, t + T, ..., then a halving tree."""
    T = CMA_THREADS
    n = -(-p.size // T) * T
    sq = np.zeros(max(n, T))
    sq[:p.size] = p * p
    acc = np.zeros(T)
    for r in range(sq.size // T):
        acc = acc + sq[r * T:(r + 1) * T]
    h = T // 2
    while h > 0:
        acc = acc[:h] + acc[h:2 * h]
        h //= 2
    return np.sqrt(acc[0])


def update(t1, t2, k, threshold, mean, c, p_sigma, p_c, sigma):
    """Step 5 from the level-1 tables: (mean, c, p_sigma, p_c, sigma, parent float32, h_sigma).  k: sep_cma_constants."""
    zm, Q = level2(t1), level2(t2)
    D = mean.size
    zm, Q = zm[:D], Q[:D]
    ps = k["one_m_cs"] * p_sigma + k["k_sigma"] * zm
    norm = norm_tree(ps)
    hs = bool(norm < threshold)
    y = np.sqrt(c) * zm
    m = mean + sigma * y
    pc = k["one_m_cc"] * p_c + (k["k_c"] if hs else 0.0) * y
    r1 = pc * pc + (0.0 if hs else k["cc2"]) * c
    c2 = (k["c_keep"] * c + k["c1"] * r1) + (k["cmu"] * c) * Q
    sig = sigma * np.exp(k["damp"] * (norm / k["chi"] - 1.0))
    return m, c2, ps, pc, np.float64(sig), m.astype(np.float32), hs


def ulps(a, b):
    """|a - b| in units of the last place of float64 (same sign, finite)."""
    ia, ib = np.asarray(a, dtype=np.float64).view(np.int64), np.asarray(b, dtype=np.float64).view(np.int64)
    return np.abs(ia - ib)

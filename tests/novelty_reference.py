"""References for novelty search with reward (nsr_es, DESIGN.md section 4.10).

* Final states: the CPU twin's own single-episode rollouts with traces (oracle/twin.py, E = 1, trace as long as the
  episode) under the training keying -- the offspring's weights from `twin.materialize`, episode e's initial state from the
  env's `*_init(seed, init_mode, gen, id, e)` -- so the last trace row is the state after the episode's last step.
* Behaviour, novelty and the blend: numpy restatements of the contract, each float64 operation separately rounded and every
  sum in the contract's order, so the kernels must match them bit for bit.
"""
import numpy as np

from eval_reference import CAPS


def final_states(twin, env, parents, ids, E, sigma, seed, gen, group, n_head, gru=False, pomdp=False, n_agents=2,
                 init_mode=0, antithetic=False):
    """[len(ids)][E][state_dim] f64: the state after the last step of episode e of offspring ids[i] of generation gen."""
    ids = np.asarray(ids, dtype=np.int32)
    twin.set_antithetic(antithetic)
    try:
        W = twin.materialize(np.ascontiguousarray(parents, dtype=np.float32), sigma, seed, gen, group, n_head, ids)
    finally:
        twin.set_antithetic(False)
    T = CAPS[env]
    rows = []
    for i, idx in enumerate(ids):
        per = []
        for e in range(E):
            if env.startswith("CartPole"):
                st = twin.cartpole_init(seed, init_mode, gen, int(idx), e)
                n, tr, _ = twin.rollout_cartpole(W[i], gru=gru, pomdp=pomdp, E=1, max_step=T, init=np.asarray(st)[None], trace_steps=T)
            elif env == "simple_spread":
                st = twin.spread_init(seed, init_mode, gen, int(idx), e, n_agents)
                _, n, tr, _ = twin.rollout_mpe(W[i], N=n_agents, E=1, max_cycles=T, init=np.asarray(st)[None], trace_steps=T, gru=gru)
            else:
                st = twin.classic_init(env, seed, init_mode, gen, int(idx), e)
                _, n, tr, _ = twin.rollout_classic(env, W[i], E=1, max_step=T, init=np.asarray(st)[None], trace_steps=T, gru=gru)
            per.append(np.asarray(tr)[int(n) - 1])
        rows.append(per)
    return np.asarray(rows, dtype=np.float64)


def behavior(final):
    """bc[i] = (sum over e, in episode order, of final[i][e]) / E."""
    final = np.asarray(final, dtype=np.float64)
    s = final[:, 0].copy()
    for e in range(1, final.shape[1]):
        s = s + final[:, e]
    return s / float(final.shape[1])


def novelty(bc, archive, k):
    """novelty[i]: mean of the distances sqrt(sum_d (b_d - a_d)^2) (d in order) from bc[i] to its min(k, |A|) nearest
    archive rows, added in ascending order."""
    bc, archive = np.asarray(bc, dtype=np.float64), np.asarray(archive, dtype=np.float64)
    m = min(int(k), archive.shape[0])
    out = np.empty(bc.shape[0])
    for i in range(bc.shape[0]):
        diff = bc[i][None, :] - archive
        q = np.zeros(archive.shape[0])
        with np.errstate(over="ignore"):                     # squares past the float64 range are inf, as on the device
            for d in range(archive.shape[1]):
                q = q + diff[:, d] * diff[:, d]
        dist = np.sort(np.sqrt(q))[:m]
        s = 0.0
        for x in dist:
            s = s + x
        out[i] = s / float(m)
    return out


def novelty_table(bc, archive, sizes, ks, chunk=1024, threads=1):
    """{(a, k): novelty of bc against archive[:a] with k neighbours} for every a in sizes and k in ks: `novelty`, vectorised
    over rows of bc in chunks (on `threads` host threads) and sharing each chunk's distances between the archive prefixes.
    The same operations in the same order: q accumulated over d in order from +0, the square root, the min(k, a) smallest
    distances in ascending order, added left to right from +0 and divided by min(k, a)."""
    from concurrent.futures import ThreadPoolExecutor
    bc, archive = np.asarray(bc, dtype=np.float64), np.asarray(archive, dtype=np.float64)
    sizes, ks = [int(a) for a in sizes], [int(k) for k in ks]
    out = {(a, k): np.empty(bc.shape[0]) for a in sizes for k in ks}

    def part(lo):
        hi = min(bc.shape[0], lo + chunk)
        b = bc[lo:hi]
        q = np.zeros((hi - lo, max(sizes)))
        with np.errstate(over="ignore"):
            for d in range(archive.shape[1]):
                diff = b[:, d:d + 1] - archive[None, :max(sizes), d]
                q = q + diff * diff
        dist = np.sqrt(q)
        for a in sizes:
            mmax = min(max(ks), a)
            near = dist[:, :a] if mmax == a else np.partition(dist[:, :a], mmax - 1, axis=1)[:, :mmax]
            near = np.sort(near, axis=1)
            s = np.zeros(hi - lo)
            sums = []
            for j in range(mmax):
                s = s + near[:, j]
                sums.append(s)
            for k in ks:
                m = min(k, a)
                out[a, k][lo:hi] = sums[m - 1] / float(m)

    with ThreadPoolExecutor(max(1, threads)) as ex:
        list(ex.map(part, range(0, bc.shape[0], chunk)))
    return out


def blend(shaped_f, shaped_n, w):
    """(1 - w) shaped_f + w shaped_n, each operation rounded separately."""
    w = np.float64(w)
    return (np.float64(1.0) - w) * np.asarray(shaped_f, dtype=np.float64) + w * np.asarray(shaped_n, dtype=np.float64)

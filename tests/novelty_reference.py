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
        for d in range(archive.shape[1]):
            q = q + diff[:, d] * diff[:, d]
        dist = np.sort(np.sqrt(q))[:m]
        s = 0.0
        for x in dist:
            s = s + x
        out[i] = s / float(m)
    return out


def blend(shaped_f, shaped_n, w):
    """(1 - w) shaped_f + w shaped_n, each operation rounded separately."""
    w = np.float64(w)
    return (np.float64(1.0) - w) * np.asarray(shaped_f, dtype=np.float64) + w * np.asarray(shaped_n, dtype=np.float64)

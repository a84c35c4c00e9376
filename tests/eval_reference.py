"""Reference of policy evaluation (DESIGN.md section 4.9) for tests: the CPU twin's own single-episode rollouts
(oracle/twin.py, E = 1 with an explicit initial state) under a numpy restatement of the evaluation keying -- episode m
starts from Philox stream 2 at counter (m, 0, round, block) with the handle's seed, drawn by the env's reset
distribution."""
import math

import numpy as np

STREAM_EVAL = 2
K32 = 2.3283064365386963e-10          # 2^-32

# env name -> (obs_dim, act_dim) of the single-agent envs
DIMS = {"CartPole-v1": (4, 2), "CartPole-v0": (4, 2), "MountainCar-v0": (2, 3), "Acrobot-v1": (6, 3), "Pendulum-v0": (3, 1)}
CAPS = {"CartPole-v1": 500, "CartPole-v0": 200, "MountainCar-v0": 200, "Acrobot-v1": 500, "Pendulum-v0": 200, "simple_spread": 25}


def dims(env, n_agents=2):
    return (6 * n_agents, 5) if env == "simple_spread" else DIMS[env]


def eval_init(twin, env, seed, rnd, m, n_agents=2):
    """Initial state of evaluation episode m (the layout of the env's init_states rows)."""
    def draw(b):
        r = twin.philox([m, 0, rnd & 0xFFFFFFFF, b], [seed & 0xFFFFFFFF, STREAM_EVAL])
        return [(float(x) + 0.5) * K32 for x in r]
    if env.startswith("CartPole"):
        return np.array([u * 0.1 - 0.05 for u in draw(0)])
    if env == "MountainCar-v0":
        return np.array([draw(0)[0] * 0.2 - 0.6, 0.0])
    if env == "Pendulum-v0":
        u = draw(0)
        return np.array([u[0] * (2.0 * math.pi) - math.pi, u[1] * 2.0 - 1.0])
    if env == "Acrobot-v1":
        return np.array([u * 0.2 - 0.1 for u in draw(0)])
    if env == "simple_spread":
        return np.array([u * 2.0 - 1.0 for b in range(n_agents) for u in draw(b)])
    raise ValueError(env)


def evaluate(twin, env, policies, n_episodes, seed=0, rnd=0, gru=False, pomdp=False, n_agents=2, max_step=None,
             init_states=None):
    """(returns [n_pol][M] f64, lengths [n_pol][M] i32) as ses_evaluate defines them."""
    W = np.ascontiguousarray(policies, dtype=np.float32)
    W = W.reshape(-1, W.shape[-1])
    cap = CAPS[env]
    max_step = cap if not max_step else min(int(max_step), cap)
    M = int(n_episodes)
    ret = np.empty((W.shape[0], M))
    lng = np.empty((W.shape[0], M), dtype=np.int32)
    for m in range(M):
        st = np.asarray(init_states[m], dtype=np.float64) if init_states is not None else eval_init(twin, env, seed, rnd, m, n_agents)
        st = st[None]
        for j in range(W.shape[0]):
            if env.startswith("CartPole"):
                t, _, _ = twin.rollout_cartpole(W[j], gru=gru, pomdp=pomdp, E=1, max_step=max_step, init=st)
                r, n = float(t), t
            elif env == "simple_spread":
                r, n, _, _ = twin.rollout_mpe(W[j], N=n_agents, E=1, max_cycles=max_step, init=st, gru=gru)
            else:
                r, n = twin.rollout_classic(env, W[j], E=1, max_step=max_step, init=st, gru=gru)
            ret[j, m], lng[j, m] = r, n
    return ret, lng

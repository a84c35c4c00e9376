"""Reference of episode recording (DESIGN.md section 4.9) for tests: the CPU twin's single-episode rollouts with their traces
(oracle/twin.py, E = 1 with an explicit initial state) under the evaluation keying of tests/eval_reference.py."""
import numpy as np

from eval_reference import CAPS, eval_init


def record(twin, env, policies, n_episodes, seed=0, rnd=0, gru=False, pomdp=False, n_agents=2, max_step=None,
           init_states=None):
    """(initial [K][state_dim] f64, states [n_pol][K][T][state_dim] f64, actions [n_pol][K][T][n_agents] i32 (float32 for
    Pendulum), returns [n_pol][K][T] f64, lengths [n_pol][K] i32) as ses_record defines them, NaN / -1 past each episode's
    end.  States and actions are the twin's trace of the single-episode rollout; returns[t - 1] is the twin's return of the
    same episode truncated at max_step = t (truncation only ends an episode, so this is the running sum, exactly)."""
    W = np.ascontiguousarray(policies, dtype=np.float32)
    W = W.reshape(-1, W.shape[-1])
    T = CAPS[env] if not max_step else min(int(max_step), CAPS[env])
    K, NA = int(n_episodes), n_agents if env == "simple_spread" else 1
    sd = len(eval_init(twin, env, seed, rnd, 0, n_agents))        # the trace rows are as wide as the init_states rows
    initial = np.empty((K, sd))
    states = np.full((W.shape[0], K, T, sd), np.nan)
    actions = np.full((W.shape[0], K, T, NA), -1, dtype=np.int32)
    returns = np.full((W.shape[0], K, T), np.nan)
    lengths = np.empty((W.shape[0], K), dtype=np.int32)

    def run(w, st, steps, trace_steps=0):
        """(return, length, trace, actions [trace_steps][NA] i32) of one episode truncated at `steps`."""
        if env.startswith("CartPole"):
            n, tr, ac = twin.rollout_cartpole(w, gru=gru, pomdp=pomdp, E=1, max_step=steps, init=st, trace_steps=trace_steps)
            return float(n), n, tr, ac
        if env == "simple_spread":
            return twin.rollout_mpe(w, N=n_agents, E=1, max_cycles=steps, init=st, trace_steps=trace_steps, gru=gru)
        out = twin.rollout_classic(env, w, E=1, max_step=steps, init=st, trace_steps=trace_steps, gru=gru)
        if not trace_steps:
            return out[0], out[1], None, None
        return out[0], out[1], out[2], out[3].view(np.int32)

    for m in range(K):
        st = np.asarray(init_states[m], dtype=np.float64) if init_states is not None else eval_init(twin, env, seed, rnd, m, n_agents)
        initial[m] = st
        for j in range(W.shape[0]):
            r, n, tr, ac = run(W[j], st[None], T, T)
            lengths[j, m] = n
            states[j, m, :n] = tr[:n]
            actions[j, m, :n] = np.asarray(ac[:n], dtype=np.int32).reshape(n, NA)
            for t in range(1, n):
                returns[j, m, t - 1] = run(W[j], st[None], t)[0]
            returns[j, m, n - 1] = r
    return initial, states, actions, returns, lengths

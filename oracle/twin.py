"""ctypes binding of the CPU bit-twin oracle (oracle/ses_twin.c).

TEST INFRASTRUCTURE ONLY -- importable from tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs; never from simple-es_b200/.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "_build", "libses_twin.so")


def build(force=False):
    """Compile the twin with the committed Makefile (gcc only, seconds)."""
    srcs = [os.path.join(_HERE, f) for f in ("ses_twin.c", "ses_twin_mpe.c", "ses_twin_classic.c", "Makefile")]
    if not force and os.path.exists(_SO) and all(os.path.getmtime(_SO) >= os.path.getmtime(s) for s in srcs):
        return _SO
    subprocess.check_call(["make", "-s", "-C", _HERE], env={**os.environ, "CC": "/usr/bin/gcc"})
    return _SO


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_SO):
            build()
        _lib = C.CDLL(_SO)
        _lib.tw_rollout_cartpole.restype = C.c_int64
        if hasattr(_lib, "tw_rollout_mpe"):
            _lib.tw_rollout_mpe.restype = C.c_double
            _lib.tw_rollout_mpe_gru.restype = C.c_double
        if hasattr(_lib, "tw_rollout_classic"):
            _lib.tw_rollout_classic.restype = C.c_double
            _lib.tw_rollout_classic_gru.restype = C.c_double
    return _lib


def _p(a, t=None):
    if a is None:
        return None
    return a.ctypes.data_as(C.c_void_p)


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def set_antithetic(on):
    """Process-wide switch of the oracle's mirrored-sampling mode (engine.antithetic); tests reset it to False."""
    lib().tw_set_antithetic(int(bool(on)))


# ---------------------------------------------------------------------------- math hooks
def philox(ctr, key):
    ctr = np.ascontiguousarray(ctr, dtype=np.uint32)
    key = np.ascontiguousarray(key, dtype=np.uint32)
    out = np.zeros(4, dtype=np.uint32)
    lib().tw_philox(_p(ctr), _p(key), _p(out))
    return out


def tanhf(x):
    x = _f32(x); y = np.empty_like(x)
    lib().tw_tanhf_v(_p(x), _p(y), C.c_int64(x.size))
    return y


def sigmf(x):
    x = _f32(x); y = np.empty_like(x)
    lib().tw_sigmf_v(_p(x), _p(y), C.c_int64(x.size))
    return y


def lnf(x):
    x = _f32(x); y = np.empty_like(x)
    lib().tw_lnf_v(_p(x), _p(y), C.c_int64(x.size))
    return y


def sincos2pif(x):
    x = _f32(x); s = np.empty_like(x); c = np.empty_like(x)
    lib().tw_sincos2pif_v(_p(x), _p(s), _p(c), C.c_int64(x.size))
    return s, c


def sincos(x):
    x = _f64(x); s = np.empty_like(x); c = np.empty_like(x)
    lib().tw_sincos_v(_p(x), _p(s), _p(c), C.c_int64(x.size))
    return s, c


def normals(seed, gen, idx, D):
    out = np.empty(D, dtype=np.float32)
    lib().tw_normals(C.c_uint32(seed), C.c_uint32(gen), C.c_uint32(idx), C.c_int(D), _p(out))
    return out


def param_count(obs, act, gru):
    return int(lib().tw_param_count(C.c_int(obs), C.c_int(act), C.c_int(int(gru))))


# ---------------------------------------------------------------------------- population
def layout(strategy, P, offspring_num=None, elite_num=None):
    """(group, n_head) of the population index layout (SURVEY.md section 8 table)."""
    if strategy == "simple_evolution":
        return P, 2
    if strategy == "openai_es":
        return P, 1
    if strategy == "simple_genetic":
        return offspring_num // elite_num, 1
    raise ValueError(strategy)


def materialize(parents, sigma, seed, gen, group, n_head, ids):
    parents = _f32(parents)
    if parents.ndim == 1:
        parents = parents[None]
    D = parents.shape[1]
    ids = np.ascontiguousarray(ids, dtype=np.int32)
    out = np.empty((ids.size, D), dtype=np.float32)
    lib().tw_materialize(_p(parents), C.c_int(D), C.c_float(sigma), C.c_uint32(seed), C.c_uint32(gen),
                         C.c_int(group), C.c_int(n_head), _p(ids), C.c_int(ids.size), _p(out))
    return out


def policy_step(w, obs, act, gru, o, h=None):
    """One forward pass; returns (action, logits, new_h)."""
    w = _f32(w); o = _f32(o)
    hh = np.zeros(32, dtype=np.float32) if h is None else _f32(h).copy()
    logits = np.zeros(act, dtype=np.float32)
    a = lib().tw_policy_step(_p(w), C.c_int(obs), C.c_int(act), C.c_int(int(gru)), _p(o), _p(hh), _p(logits))
    return int(a), logits, hh


def cartpole_step(state, action):
    st = _f64(state).copy()
    d = lib().tw_cartpole_step_x(_p(st), C.c_int(int(action)))
    return st, bool(d)


def cartpole_init(seed, init_mode, gen, idx, e):
    st = np.empty(4, dtype=np.float64)
    lib().tw_cartpole_init(C.c_uint32(seed), C.c_int(init_mode), C.c_uint32(gen), C.c_uint32(idx), C.c_uint32(e), _p(st))
    return st


def rollout_cartpole(w, gru=False, pomdp=False, E=5, max_step=500, init=None, seed=0, init_mode=0, gen=0, idx=0,
                     trace_steps=0):
    """One offspring.  Returns (total_steps, trace[trace_steps,4], actions[trace_steps])."""
    w = _f32(w)
    init_a = None if init is None else _f64(init)
    trace = np.full((max(trace_steps, 1), 4), np.nan, dtype=np.float64)
    acts = np.full(max(trace_steps, 1), -1, dtype=np.int32)
    t = lib().tw_rollout_cartpole(_p(w), C.c_int(int(gru)), C.c_int(int(pomdp)), C.c_int(E), C.c_int(max_step),
                                  _p(init_a), C.c_uint32(seed), C.c_int(init_mode), C.c_uint32(gen), C.c_uint32(idx),
                                  _p(trace), _p(acts), C.c_int(trace_steps))
    return int(t), trace[:trace_steps], acts[:trace_steps]


def _final(on, n, E, sd):
    return np.full((n, E, sd), np.nan) if on else None


def population_cartpole(parents, gru=False, pomdp=False, sigma=0.0, seed=0, gen=0, group=1, n_head=1, id0=0, n=1,
                        E=5, max_step=500, W_override=None, init=None, init_mode=0, nthreads=1, final=False):
    """Fitness (float64) and total steps (int64) of offspring [id0, id0+n); final=True adds their final states
    [n][E][4] (the state after each episode's last step)."""
    parents = _f32(parents)
    Wo = None if W_override is None else _f32(W_override)
    init_a = None if init is None else _f64(init)
    fit = np.empty(n, dtype=np.float64)
    steps = np.empty(n, dtype=np.int64)
    fs = _final(final, n, E, 4)
    lib().tw_population_cartpole(_p(parents), C.c_int(int(gru)), C.c_int(int(pomdp)), C.c_float(sigma),
                                 C.c_uint32(seed), C.c_uint32(gen), C.c_int(group), C.c_int(n_head), C.c_int(id0),
                                 C.c_int(n), C.c_int(E), C.c_int(max_step), _p(Wo), _p(init_a), C.c_int(init_mode),
                                 _p(fit), _p(steps), C.c_int(nthreads), _p(fs))
    return (fit, steps, fs) if final else (fit, steps)


# ---------------------------------------------------------------------------- K2 / K3
def rank_desc(fitness):
    f = _f64(fitness)
    order = np.empty(f.size, dtype=np.int32)
    lib().tw_rank_desc(_p(f), C.c_int(f.size), _p(order))
    return order


def centered_rank(order):
    order = np.ascontiguousarray(order, dtype=np.int32)
    shaped = np.empty(order.size, dtype=np.float64)
    lib().tw_centered_rank(_p(order), C.c_int(order.size), _p(shaped))
    return shaped


def grad_openai(shaped, D, seed, gen, group, n_head, update_factor, eps=None):
    shaped = _f64(shaped)
    e = None if eps is None else _f32(eps)
    g = np.empty(D, dtype=np.float32)
    lib().tw_grad_openai(_p(shaped), C.c_int(shaped.size), C.c_int(D), C.c_uint32(seed), C.c_uint32(gen),
                         C.c_int(group), C.c_int(n_head), _p(e), C.c_double(update_factor), _p(g))
    return g


def adam(theta, m, v, g, a, beta1=0.99, beta2=0.999, epsilon=1e-8):
    """In-place on copies; returns (theta, m, v)."""
    theta = _f32(theta).copy(); m = _f32(m).copy(); v = _f32(v).copy(); g = _f32(g)
    lib().tw_adam(_p(theta), _p(m), _p(v), _p(g), C.c_int(theta.size), C.c_double(a), C.c_double(beta1),
                  C.c_double(beta2), C.c_double(epsilon))
    return theta, m, v


def sgd(theta, v, g, stepsize, momentum=0.9):
    """In-place on copies; returns (theta, v)."""
    theta = _f32(theta).copy(); v = _f32(v).copy(); g = _f32(g)
    lib().tw_sgd(_p(theta), _p(v), _p(g), C.c_int(theta.size), C.c_double(stepsize), C.c_double(momentum))
    return theta, v


def elite_mean(elites):
    elites = _f32(elites)
    k, D = elites.shape
    mu = np.empty(D, dtype=np.float32)
    lib().tw_elite_mean(_p(elites), C.c_int(k), C.c_int(D), _p(mu))
    return mu


# ---------------------------------------------------------------------------- MPE simple_spread
def logaddexp0(y):
    y = _f64(y); out = np.empty_like(y)
    lib().tw_logaddexp0_v(_p(y), _p(out), C.c_int64(y.size))
    return out


def spread_init(seed, init_mode, gen, idx, e, N=2):
    st = np.empty(4 * N, dtype=np.float64)
    lib().tw_spread_init(C.c_uint32(seed), C.c_int(init_mode), C.c_uint32(gen), C.c_uint32(idx), C.c_uint32(e), C.c_int(N), _p(st))
    return st


def spread_policy(w, N, o):
    w = _f32(w); o = _f32(o)
    logits = np.zeros(5, dtype=np.float32)
    a = lib().tw_spread_policy(_p(w), C.c_int(N), _p(o), _p(logits))
    return int(a), logits


def rollout_mpe(w, N=2, E=5, max_cycles=25, init=None, seed=0, init_mode=0, gen=0, idx=0, trace_steps=0, gru=False):
    """One offspring.  Returns (fitness, steps, trace[trace_steps,4N], actions[trace_steps,N])."""
    w = _f32(w)
    init_a = None if init is None else _f64(init)
    trace = np.full((max(trace_steps, 1), 4 * N), np.nan, dtype=np.float64)
    acts = np.full((max(trace_steps, 1), N), -1, dtype=np.int32)
    steps = C.c_int64(0)
    f = lib().tw_rollout_mpe_gru(C.c_int(int(bool(gru))), _p(w), C.c_int(N), C.c_int(E), C.c_int(max_cycles), _p(init_a), C.c_uint32(seed),
                                 C.c_int(init_mode), C.c_uint32(gen), C.c_uint32(idx), _p(trace), _p(acts), C.c_int(trace_steps),
                                 C.byref(steps))
    return float(f), int(steps.value), trace[:trace_steps], acts[:trace_steps]


def population_mpe(parents, N=2, sigma=0.0, seed=0, gen=0, group=1, n_head=1, id0=0, n=1, E=5, max_cycles=25,
                   W_override=None, init=None, init_mode=0, gru=False, final=False):
    """final=True adds the final states [n][E][4N] (agent positions, then velocities, as a trace row)."""
    parents = _f32(parents)
    Wo = None if W_override is None else _f32(W_override)
    init_a = None if init is None else _f64(init)
    fit = np.empty(n, dtype=np.float64)
    steps = np.empty(n, dtype=np.int64)
    fs = _final(final, n, E, 4 * N)
    lib().tw_population_mpe_gru(C.c_int(int(bool(gru))), _p(parents), C.c_int(N), C.c_float(sigma), C.c_uint32(seed), C.c_uint32(gen),
                                C.c_int(group), C.c_int(n_head), C.c_int(id0), C.c_int(n), C.c_int(E), C.c_int(max_cycles), _p(Wo),
                                _p(init_a), C.c_int(init_mode), _p(fit), _p(steps), _p(fs))
    return (fit, steps, fs) if final else (fit, steps)


# ---------------------------------------------------------------------------- classic control (ses_twin_classic.c)
CLASSIC_ENVS = {"MountainCar-v0": 2, "Acrobot-v1": 3, "Pendulum-v0": 4}
CONTINUOUS_ENVS = ("Pendulum-v0",)          # tanh head (networks/neural_network.py:32-33): actions are float32


def classic_dims(env):
    """(obs, act, state_dim, time_limit) of a classic-control env name."""
    o, a, sd, cap = C.c_int(), C.c_int(), C.c_int(), C.c_int()
    assert lib().tw_classic_dims(CLASSIC_ENVS[env], C.byref(o), C.byref(a), C.byref(sd), C.byref(cap)) == 0
    return o.value, a.value, sd.value, cap.value


def sincos_full(x):
    x = _f64(x)
    s, c = np.empty_like(x), np.empty_like(x)
    lib().tw_sincos_full_v(_p(x), _p(s), _p(c), C.c_int64(x.size))
    return s, c


def classic_step(env, state, action):
    st = _f64(state).copy()
    r = C.c_double()
    if env in CONTINUOUS_ENVS:
        done = lib().tw_classic_step_continuous(CLASSIC_ENVS[env], _p(st), C.c_double(float(action)), C.byref(r))
    else:
        done = lib().tw_classic_step(CLASSIC_ENVS[env], _p(st), int(action), C.byref(r))
    return st, r.value, bool(done)


def classic_init(env, seed, init_mode, gen, idx, e):
    sd = classic_dims(env)[2]
    st = np.zeros(sd)
    lib().tw_classic_init(CLASSIC_ENVS[env], C.c_uint32(seed), int(init_mode), C.c_uint32(gen), C.c_uint32(idx), C.c_uint32(e), _p(st))
    return st


def rollout_classic(env, w, E=5, max_step=None, init=None, seed=0, init_mode=0, gen=0, idx=0, trace_steps=0, gru=False):
    """fitness, steps[, trace, actions] of one offspring (continuous envs: actions are float32)."""
    obs, act, sd, cap = classic_dims(env)
    max_step = cap if max_step is None else min(int(max_step), cap)
    w = _f32(w)
    init = None if init is None else _f64(init)
    trace = np.full((trace_steps, sd), np.nan) if trace_steps else None
    actions = np.full(trace_steps, -1, dtype=np.int32) if trace_steps else None
    steps = C.c_int64()
    f = lib().tw_rollout_classic_gru(CLASSIC_ENVS[env], int(bool(gru)), _p(w), int(E), int(max_step), _p(init), C.c_uint32(seed),
                                     int(init_mode), C.c_uint32(gen), C.c_uint32(idx), _p(trace), _p(actions), int(trace_steps),
                                     C.byref(steps))
    if trace_steps:
        if env in CONTINUOUS_ENVS:
            actions = actions.view(np.float32)
        return f, steps.value, trace, actions
    return f, steps.value


def population_classic(env, parents, sigma=0.0, seed=0, gen=0, group=1, n_head=1, id0=0, n=1, E=5, max_step=None,
                       W_override=None, init=None, init_mode=0, nthreads=8, gru=False, final=False):
    """final=True adds the final states [n][E][state_dim]."""
    obs, act, sd, cap = classic_dims(env)
    max_step = cap if max_step is None else min(int(max_step), cap)
    parents = _f32(parents)
    W_override = None if W_override is None else _f32(W_override)
    init = None if init is None else _f64(init)
    fitness = np.zeros(n)
    steps = np.zeros(n, dtype=np.int64)
    fs = _final(final, n, E, sd)
    lib().tw_population_classic_gru(CLASSIC_ENVS[env], int(bool(gru)), _p(parents), C.c_float(sigma), C.c_uint32(seed), C.c_uint32(gen),
                                    int(group), int(n_head), int(id0), int(n), int(E), int(max_step), _p(W_override), _p(init),
                                    int(init_mode), _p(fitness), _p(steps), int(nthreads), _p(fs))
    return (fitness, steps, fs) if final else (fitness, steps)

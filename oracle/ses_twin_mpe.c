/*
 * ses_twin_mpe.c -- CPU bit-twin of the PettingZoo MPE simple_spread rollout (oracle, TEST
 * INFRASTRUCTURE ONLY; see the header of ses_twin.c for the rules and the parity status).
 *
 * Restates (citations relative to /root/reference):
 *   - PettingzooWrapper.reset/step, team reward = sum of agent rewards   envs/pettingzoo_wrapper.py:22-58
 *   - the episode / fitness loop with one policy copy per agent id       learning_strategies/evolution/loop.py:108-125,
 *                                                                         learning_strategies/evolution/utils.py:4-8
 *   - MPE simple_spread_v2 (N agents, N landmarks, local_ratio 0.5, max_cycles 25, discrete actions):
 *     un-vendored / unpinned third-party code, restated from the published algorithm
 *     (SURVEY.md Appendix A.2) -- PARITY UNPINNED at that boundary; pinned only against the
 *     float64 numpy restatement oracle/pyref.py::SimpleSpreadShim driven by the reference's own
 *     RolloutWorker + GymEnvModel (tests/golden/rollout_spread_*.npz).
 *
 * Numerical contract: as ses_twin.c (separately rounded IEEE ops, fused only where fma() is
 * written); exp / log1p inside numpy's logaddexp are replaced by the polynomial kernels below,
 * which the CUDA kernel mirrors bit for bit.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define TW_EXPORT __attribute__((visibility("default")))
#define HID 32
#define MAXN 3

/* from ses_twin.c */
void tw_philox(const uint32_t *ctr, const uint32_t *key, uint32_t *out);
int tw_param_count(int obs, int act, int gru);
float tw_fc2_row(const float *w2row, const float *x, float bias);
int tw_policy_step(const float *w, int obs, int act, int gru, const float *o, float *h, float *logits);
void tw_perturb(const float *parent, int D, float sigma, uint32_t seed, uint32_t gen, uint32_t id, int perturbed, float *w);
void tw_tanhf_v(const float *x, float *y, int64_t n);

static inline float u2f(uint32_t u) { float f; memcpy(&f, &u, 4); return f; }
static inline double ll2d(int64_t v) { double d; memcpy(&d, &v, 8); return d; }

/* exp(t) for t <= 0; values below exp(-700) are flushed to 0 */
static double tw_exp_neg(double t)
{
    if (t < -700.0) return 0.0;
    int k = (int)(t * 1.4426950408889634 - 0.5);
    double kf = (double)k;
    double r = fma(-kf, 6.93147180369123816490e-01, t);
    r = fma(-kf, 1.90821492927058770002e-10, r);
    double p = 1.6059043836821613e-10;            /* 1/13! */
    p = fma(p, r, 2.08767569878681e-09);          /* 1/12! */
    p = fma(p, r, 2.505210838544172e-08);         /* 1/11! */
    p = fma(p, r, 2.7557319223985888e-07);        /* 1/10! */
    p = fma(p, r, 2.7557319223985893e-06);        /* 1/9!  */
    p = fma(p, r, 2.4801587301587302e-05);        /* 1/8!  */
    p = fma(p, r, 0.00019841269841269841);        /* 1/7!  */
    p = fma(p, r, 0.0013888888888888889);         /* 1/6!  */
    p = fma(p, r, 0.0083333333333333332);         /* 1/5!  */
    p = fma(p, r, 0.041666666666666664);          /* 1/4!  */
    p = fma(p, r, 0.16666666666666666);           /* 1/3!  */
    p = fma(p, r, 0.5);
    p = fma(p, r, 1.0);
    p = fma(p, r, 1.0);
    return p * ll2d((int64_t)(k + 1023) << 52);
}

/* ln(u) for u in [1, 2] */
static double tw_log_12(double u)
{
    double m = u, e = 0.0;
    if (u > 1.4142135623730951) { m = u * 0.5; e = 0.6931471805599453; }
    double s = (m - 1.0) / (m + 1.0);
    double z = s * s;
    double q = 1.0 / 21.0;
    q = fma(q, z, 1.0 / 19.0);
    q = fma(q, z, 1.0 / 17.0);
    q = fma(q, z, 1.0 / 15.0);
    q = fma(q, z, 1.0 / 13.0);
    q = fma(q, z, 1.0 / 11.0);
    q = fma(q, z, 1.0 / 9.0);
    q = fma(q, z, 1.0 / 7.0);
    q = fma(q, z, 1.0 / 5.0);
    q = fma(q, z, 1.0 / 3.0);
    q = q * z;
    double r2 = 2.0 * s;
    return e + fma(r2, q, r2);
}

/* log1p(v) for v in [0, 1] */
static double tw_log1p_01(double v)
{
    double u = 1.0 + v;
    double c = (v - (u - 1.0)) / u;
    return tw_log_12(u) + c;
}

/* numpy.logaddexp(0, y) */
static double tw_logaddexp0(double y)
{
    if (y < 0.0) return tw_log1p_01(tw_exp_neg(y));
    return y + tw_log1p_01(tw_exp_neg(-y));
}

TW_EXPORT void tw_logaddexp0_v(const double *y, double *out, int64_t n)
{
    for (int64_t i = 0; i < n; ++i) out[i] = tw_logaddexp0(y[i]);
}

/* ------------------------------------------------------------------------------------ */
typedef struct {
    double apos[MAXN][2], avel[MAXN][2], lpos[MAXN][2];
} spread_state;

/* observation of agent i (simple_spread Scenario.observation), float64 -> float32 */
static void spread_obs(const spread_state *s, int N, int i, float *o)
{
    int c = 0;
    o[c++] = (float)s->avel[i][0]; o[c++] = (float)s->avel[i][1];
    o[c++] = (float)s->apos[i][0]; o[c++] = (float)s->apos[i][1];
    for (int l = 0; l < N; ++l) { o[c++] = (float)(s->lpos[l][0] - s->apos[i][0]); o[c++] = (float)(s->lpos[l][1] - s->apos[i][1]); }
    for (int j = 0; j < N; ++j) if (j != i) { o[c++] = (float)(s->apos[j][0] - s->apos[i][0]); o[c++] = (float)(s->apos[j][1] - s->apos[i][1]); }
    for (int j = 0; j < N; ++j) if (j != i) { o[c++] = 0.0f; o[c++] = 0.0f; }     /* silent agents: comm = 0 */
}

static int argmax_softmax(const float *z, int act)
{
    float zmax = z[0];
    for (int m = 1; m < act; ++m) zmax = fmaxf(zmax, z[m]);
    for (int m = 0; m < act; ++m)
        if (zmax - z[m] <= u2f(0x33000000u)) return m;
    return 0;
}

/* shared-MLP policy (networks/neural_network.py:20-36, gru = False) */
static int spread_policy(const float *w, int obs, const float *o, float *logits)
{
    const float *W1 = w, *b1 = W1 + HID * obs, *W2 = b1 + HID, *b2 = W2 + 5 * HID;
    float pre[HID], x[HID];
    for (int j = 0; j < HID; ++j) {
        float a = b1[j];
        for (int k = 0; k < obs; ++k) a = fmaf(W1[j * obs + k], o[k], a);
        pre[j] = a;
    }
    tw_tanhf_v(pre, x, HID);
    float z[5];
    for (int m = 0; m < 5; ++m) {
        z[m] = tw_fc2_row(W2 + m * HID, x, b2[m]);          /* four blocks of eight hidden units (ses_twin.c) */
        if (logits) logits[m] = z[m];
    }
    return argmax_softmax(z, 5);
}

/* one world step (MPE core.World.step) + team reward (pettingzoo_wrapper.py:45-53) */
static double spread_step(spread_state *s, int N, const int *act)
{
    double F[MAXN][2];
    for (int i = 0; i < N; ++i) {
        double ux = 0.0, uy = 0.0;
        if (act[i] == 1) ux = -1.0;
        if (act[i] == 2) ux = 1.0;
        if (act[i] == 3) uy = -1.0;
        if (act[i] == 4) uy = 1.0;
        F[i][0] = ux * 5.0; F[i][1] = uy * 5.0;
    }
    for (int a = 0; a < N; ++a)
        for (int b = a + 1; b < N; ++b) {
            double dx = s->apos[a][0] - s->apos[b][0], dy = s->apos[a][1] - s->apos[b][1];
            double dist = sqrt(dx * dx + dy * dy);
            double pen = tw_logaddexp0(-(dist - 0.3) / 0.001) * 0.001;
            double fx = ((100.0 * dx) / dist) * pen, fy = ((100.0 * dy) / dist) * pen;
            F[a][0] = F[a][0] + fx; F[a][1] = F[a][1] + fy;
            F[b][0] = F[b][0] - fx; F[b][1] = F[b][1] - fy;
        }
    for (int i = 0; i < N; ++i)
        for (int d = 0; d < 2; ++d) {
            s->avel[i][d] = s->avel[i][d] * 0.75;                       /* 1 - damping */
            s->avel[i][d] = s->avel[i][d] + (F[i][d] / 1.0) * 0.1;
            s->apos[i][d] = s->apos[i][d] + s->avel[i][d] * 0.1;
        }
    double glob = 0.0;
    for (int l = 0; l < N; ++l) {
        double best = 0.0;
        for (int a = 0; a < N; ++a) {
            double dx = s->apos[a][0] - s->lpos[l][0], dy = s->apos[a][1] - s->lpos[l][1];
            double d = sqrt(dx * dx + dy * dy);
            if (a == 0 || d < best) best = d;
        }
        glob = glob - best;
    }
    double total = 0.0;
    for (int i = 0; i < N; ++i) {
        double local = 0.0;
        for (int a = 0; a < N; ++a) {                                   /* 2021 sources: includes a == i */
            double dx = s->apos[a][0] - s->apos[i][0], dy = s->apos[a][1] - s->apos[i][1];
            if (sqrt(dx * dx + dy * dy) < 0.3) local = local - 1.0;
        }
        total = total + (glob * 0.5 + local * 0.5);
    }
    return total;
}

/* initial positions of episode e: agents then landmarks, U(-1,1), Philox stream 1, counter block b */
TW_EXPORT void tw_spread_init(uint32_t seed, int init_mode, uint32_t gen, uint32_t id, uint32_t e, int N, double *st /* [4N] */)
{
    for (int b = 0; 4 * b < 4 * N; ++b) {
        uint32_t ctr[4] = { e, init_mode ? id : 0u, init_mode ? gen : 0u, (uint32_t)b };
        uint32_t key[2] = { seed, 1u };
        uint32_t r[4];
        tw_philox(ctr, key, r);
        for (int k = 0; k < 4; ++k) {
            double u = ((double)r[k] + 0.5) * 2.3283064365386963e-10;
            st[4 * b + k] = u * 2.0 - 1.0;
        }
    }
}

/* One offspring, E episodes of max_cycles steps.  Returns fitness = (sum_e R_e) / E with R_e the
 * sequential float64 sum of the team rewards of episode e (loop.py:111-125).
 * init: [E][4N] explicit positions (agents then landmarks) or NULL -> Philox.
 * trace: optional [trace_steps][4N] (agent pos, agent vel) after each step of episode 0;
 * actions: optional [trace_steps][N]. */
TW_EXPORT double tw_rollout_mpe_gru(int gru, const float *w, int N, int E, int max_cycles, const double *init, uint32_t seed,
                                    int init_mode, uint32_t gen, uint32_t id, double *trace, int32_t *actions, int trace_steps,
                                    int64_t *steps_out);
static double mpe_rollout(int gru, const float *w, int N, int E, int max_cycles, const double *init, uint32_t seed, int init_mode,
                          uint32_t gen, uint32_t id, double *trace, int32_t *actions, int trace_steps, int64_t *steps_out,
                          double *final);

TW_EXPORT double tw_rollout_mpe(const float *w, int N, int E, int max_cycles, const double *init, uint32_t seed,
                                int init_mode, uint32_t gen, uint32_t id, double *trace, int32_t *actions, int trace_steps,
                                int64_t *steps_out)
{
    return tw_rollout_mpe_gru(0, w, N, E, max_cycles, init, seed, init_mode, gen, id, trace, actions, trace_steps, steps_out);
}

/* gru = 1: the recurrent policy.  wrap_agentid (learning_strategies/evolution/utils.py:4-8) deep-copies the network once per
 * agent id: shared weights, ONE HIDDEN STATE PER AGENT, all reset at the start of every episode (loop.py:114-116). */
TW_EXPORT double tw_rollout_mpe_gru(int gru, const float *w, int N, int E, int max_cycles, const double *init, uint32_t seed,
                                    int init_mode, uint32_t gen, uint32_t id, double *trace, int32_t *actions, int trace_steps,
                                    int64_t *steps_out)
{
    return mpe_rollout(gru, w, N, E, max_cycles, init, seed, init_mode, gen, id, trace, actions, trace_steps, steps_out, NULL);
}

/* final: optional [E][4N] (agent pos, agent vel) after each episode's last step, laid out as a trace row. */
static double mpe_rollout(int gru, const float *w, int N, int E, int max_cycles, const double *init, uint32_t seed, int init_mode,
                          uint32_t gen, uint32_t id, double *trace, int32_t *actions, int trace_steps, int64_t *steps_out,
                          double *final)
{
    const int obs = 6 * N;
    double total = 0.0;
    int64_t nsteps = 0;
    for (int e = 0; e < E; ++e) {
        double st[4 * MAXN];
        float hid[MAXN][HID];
        spread_state s;
        memset(hid, 0, sizeof(hid));
        if (init) memcpy(st, init + (size_t)4 * N * e, sizeof(double) * 4 * N);
        else tw_spread_init(seed, init_mode, gen, id, (uint32_t)e, N, st);
        for (int i = 0; i < N; ++i) {
            s.apos[i][0] = st[2 * i]; s.apos[i][1] = st[2 * i + 1];
            s.avel[i][0] = 0.0; s.avel[i][1] = 0.0;
            s.lpos[i][0] = st[2 * N + 2 * i]; s.lpos[i][1] = st[2 * N + 2 * i + 1];
        }
        double R = 0.0;
        for (int t = 0; t < max_cycles; ++t) {
            int act[MAXN];
            float o[6 * MAXN];
            for (int i = 0; i < N; ++i) {
                spread_obs(&s, N, i, o);
                act[i] = gru ? tw_policy_step(w, obs, 5, 1, o, hid[i], NULL) : spread_policy(w, obs, o, NULL);
            }
            R = R + spread_step(&s, N, act);
            ++nsteps;
            if (e == 0 && t < trace_steps) {
                if (trace) for (int i = 0; i < N; ++i) {
                    trace[(size_t)t * 4 * N + 2 * i] = s.apos[i][0]; trace[(size_t)t * 4 * N + 2 * i + 1] = s.apos[i][1];
                    trace[(size_t)t * 4 * N + 2 * N + 2 * i] = s.avel[i][0]; trace[(size_t)t * 4 * N + 2 * N + 2 * i + 1] = s.avel[i][1];
                }
                if (actions) for (int i = 0; i < N; ++i) actions[(size_t)t * N + i] = act[i];
            }
        }
        if (final) for (int i = 0; i < N; ++i) {
            double *f = final + (size_t)4 * N * e;
            f[2 * i] = s.apos[i][0]; f[2 * i + 1] = s.apos[i][1];
            f[2 * N + 2 * i] = s.avel[i][0]; f[2 * N + 2 * i + 1] = s.avel[i][1];
        }
        total = total + R;
    }
    if (steps_out) *steps_out = nsteps;
    return total / (double)E;
}

TW_EXPORT void tw_population_mpe_gru(int gru, const float *parents, int N, float sigma, uint32_t seed, uint32_t gen, int group, int n_head,
                                     int id0, int n, int E, int max_cycles, const float *W_override, const double *init,
                                     int init_mode, double *fitness, int64_t *steps, double *final)
{
    const int D = tw_param_count(6 * N, 5, gru);
    float *w = (float *)malloc(sizeof(float) * (size_t)D);
    for (int j = 0; j < n; ++j) {
        int id = id0 + j;
        if (W_override) memcpy(w, W_override + (size_t)j * D, sizeof(float) * (size_t)D);
        else tw_perturb(parents + (size_t)(id / group) * D, D, sigma, seed, gen, (uint32_t)id, (id % group) - n_head + 1, w);
        fitness[j] = mpe_rollout(gru, w, N, E, max_cycles, init, seed, init_mode, gen, (uint32_t)id, NULL, NULL, 0, &steps[j],
                                 final ? final + (size_t)j * E * 4 * N : NULL);
    }
    free(w);
}

TW_EXPORT void tw_population_mpe(const float *parents, int N, float sigma, uint32_t seed, uint32_t gen, int group, int n_head,
                                 int id0, int n, int E, int max_cycles, const float *W_override, const double *init,
                                 int init_mode, double *fitness, int64_t *steps)
{
    tw_population_mpe_gru(0, parents, N, sigma, seed, gen, group, n_head, id0, n, E, max_cycles, W_override, init, init_mode, fitness, steps, NULL);
}

TW_EXPORT int tw_spread_policy(const float *w, int N, const float *o, float *logits) { return spread_policy(w, 6 * N, o, logits); }

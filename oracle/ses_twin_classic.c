/*
 * ses_twin_classic.c -- CPU bit-twin of the classic-control rollouts beyond CartPole (oracle, TEST
 * INFRASTRUCTURE ONLY; see the header of ses_twin.c for the rules and the parity status).
 *
 * Environments any reference config can name through GymWrapper (envs/gym_wrapper.py:8-45 passes the
 * name straight to gym.make) with the discrete-action policy head (networks/neural_network.py:29-31):
 *   env 2  MountainCar-v0   obs 2, 3 actions, reward -1 per step, TimeLimit 200
 *   env 3  Acrobot-v1       obs 6, 3 actions, reward -1 per step (0 on the terminal step), TimeLimit 500
 * and, with the continuous-action head (`discrete_action: False`, networks/neural_network.py:32-33: tanh of fc2):
 *   env 4  Pendulum-v0      obs 3, 1 action in (-1, 1) used as the torque, reward -(th_norm^2 + .1 thdot^2 + .001 u^2),
 *                           never terminates, TimeLimit 200
 * Each of them also with the recurrent policy (`gru: True`): the hidden state is reset per episode
 * (loop.py:114-116 -> GymEnvModel.reset, neural_network.py:38-40).
 *
 * Restates (citations relative to /root/reference):
 *   - GymWrapper.reset/step, max_step truncation                 envs/gym_wrapper.py:23-45
 *   - the episode / fitness loop                                 learning_strategies/evolution/loop.py:108-125
 *   - gym classic_control/mountain_car.py and acrobot.py (gym ~0.18-0.21): un-vendored, unpinned
 *     third-party code restated from the published algorithm (DESIGN.md Appendix) -- PARITY UNPINNED
 *     at that boundary; pinned only against the float64 Python restatement oracle/pyref.py
 *     (MountainCarShim / AcrobotShim, libm sin/cos) driven by the reference's own RolloutWorker +
 *     GymEnvModel (tests/golden/rollout_mountaincar.npz, rollout_acrobot.npz).
 *
 * Numerical contract: as ses_twin.c (separately rounded IEEE ops, fused only where fma() is written).
 * libm's sin / cos are replaced by tw_sincos_full below (Cody-Waite reduction by pi/2 in two parts with
 * fma, Taylor kernels to x^17 / x^16 on [-pi/4, pi/4]; <= 1 ulp from glibc for the |x| < 100 these
 * environments produce), which the CUDA kernels mirror bit for bit.
 */
#include <math.h>
#include <pthread.h>
#include <stdatomic.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define TW_EXPORT __attribute__((visibility("default")))
#define HID 32

#define ENV_MOUNTAINCAR 2
#define ENV_ACROBOT 3
#define ENV_PENDULUM 4       /* continuous action: the policy's tanh head (networks/neural_network.py:32-33) */

/* from ses_twin.c */
void tw_philox(const uint32_t *ctr, const uint32_t *key, uint32_t *out);
int tw_param_count(int obs, int act, int gru);
void tw_perturb(const float *parent, int D, float sigma, uint32_t seed, uint32_t gen, uint32_t id, int perturbed, float *w);
int tw_policy_step(const float *w, int obs, int act, int gru, const float *o, float *h, float *logits);
void tw_tanhf_v(const float *x, float *y, int64_t n);

/* ------------------------------------------------------------------------------------ */
/* float64 sin / cos, full range (|x| * 2/pi must fit an int32; here |x| < 100)           */
/* ------------------------------------------------------------------------------------ */
static inline double tw_sin_kernel(double r)
{
    double z = r * r;
    double p = 2.8114572543455206e-15;         /*  1/17! */
    p = fma(p, z, -7.6471637318198164e-13);    /* -1/15! */
    p = fma(p, z, 1.6059043836821613e-10);     /*  1/13! */
    p = fma(p, z, -2.505210838544172e-08);     /* -1/11! */
    p = fma(p, z, 2.7557319223985893e-06);     /*  1/9!  */
    p = fma(p, z, -0.00019841269841269841);    /* -1/7!  */
    p = fma(p, z, 0.0083333333333333332);      /*  1/5!  */
    p = fma(p, z, -0.16666666666666666);       /* -1/3!  */
    return fma(r * z, p, r);
}

static inline double tw_cos_kernel(double r)
{
    double z = r * r;
    double p = 4.7794773323873853e-14;         /*  1/16! */
    p = fma(p, z, -1.1470745597729725e-11);    /* -1/14! */
    p = fma(p, z, 2.08767569878681e-09);       /*  1/12! */
    p = fma(p, z, -2.7557319223985888e-07);    /* -1/10! */
    p = fma(p, z, 2.4801587301587302e-05);     /*  1/8!  */
    p = fma(p, z, -0.0013888888888888889);     /* -1/6!  */
    p = fma(p, z, 0.041666666666666664);       /*  1/4!  */
    double w = z * z;
    double t = fma(w, p, -(0.5 * z));
    return 1.0 + t;
}

static inline void tw_sincos_full(double x, double *sn, double *cs)
{
    int n = (int)nearbyint(x * 0.63661977236758138);      /* round-half-even(x * 2/pi) */
    double kf = (double)n;
    double r = fma(-kf, 1.5707963267948966, x);            /* pi/2, high part */
    r = fma(-kf, 6.123233995736766e-17, r);                /* pi/2, low part  */
    double s = tw_sin_kernel(r), c = tw_cos_kernel(r);
    switch (n & 3) {
    case 0: *sn = s; *cs = c; break;
    case 1: *sn = c; *cs = -s; break;
    case 2: *sn = -s; *cs = -c; break;
    default: *sn = -c; *cs = s; break;
    }
}

static inline double tw_sin_full(double x) { double s, c; tw_sincos_full(x, &s, &c); return s; }
static inline double tw_cos_full(double x) { double s, c; tw_sincos_full(x, &s, &c); return c; }

TW_EXPORT void tw_sincos_full_v(const double *x, double *s, double *c, int64_t n)
{
    for (int64_t i = 0; i < n; ++i) tw_sincos_full(x[i], s + i, c + i);
}

static inline double clipd(double v, double lo, double hi) { return fmin(fmax(v, lo), hi); }

/* ------------------------------------------------------------------------------------ */
/* MountainCar-v0 (gym classic_control/mountain_car.py)                                    */
/* ------------------------------------------------------------------------------------ */
static int mountaincar_step(double st[2], int action, double *reward)
{
    double position = st[0], velocity = st[1];
    velocity = velocity + ((double)(action - 1) * 0.001 + tw_cos_full(3.0 * position) * (-0.0025));
    velocity = clipd(velocity, -0.07, 0.07);
    position = position + velocity;
    position = clipd(position, -1.2, 0.6);
    if (position == -1.2 && velocity < 0.0) velocity = 0.0;
    st[0] = position; st[1] = velocity;
    *reward = -1.0;
    return position >= 0.5 && velocity >= 0.0;
}

/* ------------------------------------------------------------------------------------ */
/* Acrobot-v1 (gym classic_control/acrobot.py, book_or_nips = "book", torque_noise_max = 0) */
/* ------------------------------------------------------------------------------------ */
#define ACRO_PI 3.141592653589793

static void acrobot_dsdt(const double s[4], double a, double ds[4])
{
    /* m1 = m2 = l1 = 1, lc1 = lc2 = 0.5, I1 = I2 = 1, g = 9.8; products of constants folded exactly
     * as Python evaluates them left to right (all of them are exact in binary except 1.5 * 9.8) */
    const double theta1 = s[0], theta2 = s[1], dtheta1 = s[2], dtheta2 = s[3];
    double sin2, cos2;
    tw_sincos_full(theta2, &sin2, &cos2);
    /* d1 = m1*lc1**2 + m2*(l1**2 + lc2**2 + 2*l1*lc2*cos(theta2)) + I1 + I2 */
    double d1 = ((0.25 + (1.25 + 1.0 * cos2)) + 1.0) + 1.0;
    /* d2 = m2*(lc2**2 + l1*lc2*cos(theta2)) + I2 */
    double d2 = (0.25 + 0.5 * cos2) + 1.0;
    /* phi2 = m2*lc2*g*cos(theta1 + theta2 - pi/2) */
    double phi2 = 4.9 * tw_cos_full((theta1 + theta2) - ACRO_PI / 2.0);
    /* phi1 = -m2*l1*lc2*dtheta2**2*sin(theta2) - 2*m2*l1*lc2*dtheta2*dtheta1*sin(theta2)
     *        + (m1*lc1 + m2*l1)*g*cos(theta1 - pi/2) + phi2 */
    double phi1 = (((-0.5 * (dtheta2 * dtheta2)) * sin2 - ((1.0 * dtheta2) * dtheta1) * sin2)
                   + (1.5 * 9.8) * tw_cos_full(theta1 - ACRO_PI / 2.0)) + phi2;
    /* book: ddtheta2 = (a + d2/d1*phi1 - m2*l1*lc2*dtheta1**2*sin(theta2) - phi2) / (m2*lc2**2 + I2 - d2**2/d1) */
    double ddtheta2 = (((a + (d2 / d1) * phi1) - (0.5 * (dtheta1 * dtheta1)) * sin2) - phi2)
                      / ((0.25 + 1.0) - (d2 * d2) / d1);
    double ddtheta1 = -(d2 * ddtheta2 + phi1) / d1;
    ds[0] = dtheta1; ds[1] = dtheta2; ds[2] = ddtheta1; ds[3] = ddtheta2;
}

static inline double acro_wrap(double x)
{
    const double diff = ACRO_PI - (-ACRO_PI);
    while (x > ACRO_PI) x = x - diff;
    while (x < -ACRO_PI) x = x + diff;
    return x;
}

static int acrobot_step(double st[4], int action, double *reward)
{
    const double torque = (double)(action - 1);            /* AVAIL_TORQUE = [-1, 0, +1] */
    const double dt = 0.2, dt2 = 0.2 / 2.0;
    double k1[4], k2[4], k3[4], k4[4], y[4];
    acrobot_dsdt(st, torque, k1);                          /* rk4(self._dsdt, s_augmented, [0, dt]) */
    for (int i = 0; i < 4; ++i) y[i] = st[i] + dt2 * k1[i];
    acrobot_dsdt(y, torque, k2);
    for (int i = 0; i < 4; ++i) y[i] = st[i] + dt2 * k2[i];
    acrobot_dsdt(y, torque, k3);
    for (int i = 0; i < 4; ++i) y[i] = st[i] + dt * k3[i];
    acrobot_dsdt(y, torque, k4);
    double ns[4];
    for (int i = 0; i < 4; ++i)
        ns[i] = st[i] + (dt / 6.0) * (((k1[i] + 2.0 * k2[i]) + 2.0 * k3[i]) + k4[i]);
    ns[0] = acro_wrap(ns[0]);
    ns[1] = acro_wrap(ns[1]);
    ns[2] = clipd(ns[2], -4.0 * ACRO_PI, 4.0 * ACRO_PI);
    ns[3] = clipd(ns[3], -9.0 * ACRO_PI, 9.0 * ACRO_PI);
    memcpy(st, ns, sizeof(ns));
    int terminal = (-tw_cos_full(ns[0]) - tw_cos_full(ns[1] + ns[0])) > 1.0;
    *reward = terminal ? 0.0 : -1.0;
    return terminal;
}

/* ------------------------------------------------------------------------------------ */
/* generic dispatch                                                                        */
/* ------------------------------------------------------------------------------------ */
/* ------------------------------------------------------------------------------------ */
/* Pendulum-v0 (gym classic_control/pendulum.py, gym ~0.18): max_speed 8, max_torque 2, dt .05, g 10, m = l = 1.  */
/* The action is the float32 tanh output of the policy widened to double (|u| < 1 < max_torque: the clip is the    */
/* identity); Python's float % is fmod with the divisor's sign, exact.                                             */
/* ------------------------------------------------------------------------------------ */
#define PEND_PI 3.141592653589793
static double pend_angle_normalize(double x)
{
    double m = fmod(x + PEND_PI, 2.0 * PEND_PI);              /* ((x + pi) % (2 pi)) - pi */
    if (m < 0.0) m = m + 2.0 * PEND_PI;
    return m - PEND_PI;
}

static int pendulum_step(double st[2], double u, double *reward)
{
    const double th = st[0], thdot = st[1];
    u = clipd(u, -2.0, 2.0);
    const double an = pend_angle_normalize(th);
    const double costs = an * an + 0.1 * (thdot * thdot) + 0.001 * (u * u);
    /* newthdot = thdot + (-3 g / (2 l) * sin(th + pi) + 3. / (m l^2) * u) * dt:  -3*10/(2*1) = -15.0, 3./(1*1) = 3.0 */
    double newthdot = thdot + (-15.0 * tw_sin_full(th + PEND_PI) + 3.0 * u) * 0.05;
    const double newth = th + newthdot * 0.05;
    newthdot = clipd(newthdot, -8.0, 8.0);
    st[0] = newth; st[1] = newthdot;
    *reward = -costs;
    return 0;
}

TW_EXPORT int tw_classic_continuous(int env) { return env == ENV_PENDULUM; }

TW_EXPORT int tw_classic_dims(int env, int *obs, int *act, int *state_dim, int *time_limit)
{
    switch (env) {
    case ENV_PENDULUM: *obs = 3; *act = 1; *state_dim = 2; *time_limit = 200; return 0;
    case ENV_MOUNTAINCAR: *obs = 2; *act = 3; *state_dim = 2; *time_limit = 200; return 0;
    case ENV_ACROBOT: *obs = 6; *act = 3; *state_dim = 4; *time_limit = 500; return 0;
    default: return -1;
    }
}

TW_EXPORT int tw_classic_step(int env, double *st, int action, double *reward)
{
    return env == ENV_MOUNTAINCAR ? mountaincar_step(st, action, reward) : acrobot_step(st, action, reward);
}

TW_EXPORT int tw_classic_step_continuous(int env, double *st, double u, double *reward)
{
    (void)env;
    return pendulum_step(st, u, reward);
}

static void classic_obs(int env, const double *st, float *o)
{
    if (env == ENV_MOUNTAINCAR) {
        o[0] = (float)st[0]; o[1] = (float)st[1];
    } else if (env == ENV_PENDULUM) {
        double sn, cs;
        tw_sincos_full(st[0], &sn, &cs);
        o[0] = (float)cs; o[1] = (float)sn; o[2] = (float)st[1];                 /* [cos th, sin th, thdot] */
    } else {
        double s0, c0, s1, c1;
        tw_sincos_full(st[0], &s0, &c0);
        tw_sincos_full(st[1], &s1, &c1);
        o[0] = (float)c0; o[1] = (float)s0; o[2] = (float)c1; o[3] = (float)s1; o[4] = (float)st[2]; o[5] = (float)st[3];
    }
}

TW_EXPORT void tw_classic_obs(int env, const double *st, float *o) { classic_obs(env, st, o); }

/* initial state of episode e from Philox stream 1 (same counter convention as tw_cartpole_init):
 * MountainCar: position ~ U(-0.6, -0.4), velocity 0;  Acrobot: U(-0.1, 0.1)^4 */
TW_EXPORT void tw_classic_init(int env, uint32_t seed, int init_mode, uint32_t gen, uint32_t id, uint32_t e, double *st)
{
    uint32_t ctr[4] = { e, init_mode ? id : 0u, init_mode ? gen : 0u, 0u };
    uint32_t key[2] = { seed, 1u };
    uint32_t r[4];
    tw_philox(ctr, key, r);
    if (env == ENV_MOUNTAINCAR) {
        double u = ((double)r[0] + 0.5) * 2.3283064365386963e-10;
        st[0] = u * 0.2 - 0.6;
        st[1] = 0.0;
    } else if (env == ENV_PENDULUM) {                              /* uniform(-[pi, 1], [pi, 1]) */
        double u0 = ((double)r[0] + 0.5) * 2.3283064365386963e-10, u1 = ((double)r[1] + 0.5) * 2.3283064365386963e-10;
        st[0] = u0 * (2.0 * PEND_PI) - PEND_PI;
        st[1] = u1 * 2.0 - 1.0;
    } else {
        for (int k = 0; k < 4; ++k) {
            double u = ((double)r[k] + 0.5) * 2.3283064365386963e-10;
            st[k] = u * 0.2 - 0.1;
        }
    }
}

TW_EXPORT double tw_rollout_classic_gru(int env, int gru, const float *w, int E, int max_step, const double *init, uint32_t seed,
                                        int init_mode, uint32_t gen, uint32_t id, double *trace, int32_t *actions,
                                        int trace_steps, int64_t *steps_out);
/* final: optional [E][state_dim] state after each episode's last step. */
static double classic_rollout(int env, int gru, const float *w, int E, int max_step, const double *init, uint32_t seed,
                              int init_mode, uint32_t gen, uint32_t id, double *trace, int32_t *actions, int trace_steps,
                              int64_t *steps_out, double *final);

/* One offspring: E episodes (loop.py:111-125).  Returns fitness = (sum over episodes, in episode order, of the
 * sequential float64 sum of the episode's rewards) / E.
 * init: [E][state_dim] explicit initial states or NULL -> Philox.  trace: optional [trace_steps][state_dim] states
 * after each of the first steps of episode 0; actions: optional [trace_steps]. */
TW_EXPORT double tw_rollout_classic(int env, const float *w, int E, int max_step, const double *init, uint32_t seed,
                                    int init_mode, uint32_t gen, uint32_t id, double *trace, int32_t *actions,
                                    int trace_steps, int64_t *steps_out)
{
    return tw_rollout_classic_gru(env, 0, w, E, max_step, init, seed, init_mode, gen, id, trace, actions, trace_steps, steps_out);
}

/* The same with the policy kind as a parameter: gru = 1 runs GymEnvModel's recurrent branch, hidden state zeroed at the start
 * of every episode.  Continuous envs: `actions` receives the float32 action's bit pattern. */
TW_EXPORT double tw_rollout_classic_gru(int env, int gru, const float *w, int E, int max_step, const double *init, uint32_t seed,
                                        int init_mode, uint32_t gen, uint32_t id, double *trace, int32_t *actions,
                                        int trace_steps, int64_t *steps_out)
{
    return classic_rollout(env, gru, w, E, max_step, init, seed, init_mode, gen, id, trace, actions, trace_steps, steps_out, NULL);
}

static double classic_rollout(int env, int gru, const float *w, int E, int max_step, const double *init, uint32_t seed,
                              int init_mode, uint32_t gen, uint32_t id, double *trace, int32_t *actions, int trace_steps,
                              int64_t *steps_out, double *final)
{
    int obs, act, sd, cap;
    if (tw_classic_dims(env, &obs, &act, &sd, &cap)) return NAN;
    const int continuous = tw_classic_continuous(env);
    double total = 0.0;
    int64_t nsteps = 0;
    for (int e = 0; e < E; ++e) {
        double st[4];
        float h[HID];
        memset(h, 0, sizeof(h));                                   /* model.reset() (loop.py:114-116) */
        if (init) memcpy(st, init + (size_t)sd * e, sizeof(double) * (size_t)sd);
        else tw_classic_init(env, seed, init_mode, gen, id, (uint32_t)e, st);
        double R = 0.0;
        int step = 0, done = 0;
        while (!done) {
            float o[8], logits[16];
            classic_obs(env, st, o);
            int a = tw_policy_step(w, obs, act, gru, o, h, logits);
            double r;
            if (continuous) {
                float u;                                           /* tanh head (neural_network.py:32-33), float32 */
                tw_tanhf_v(logits, &u, 1);
                memcpy(&a, &u, 4);
                done = tw_classic_step_continuous(env, st, (double)u, &r);
            } else {
                done = tw_classic_step(env, st, a, &r);
            }
            R = R + r;                                             /* loop.py:120-122 */
            ++step;                                                /* gym_wrapper.py:33 */
            if (step >= max_step) done = 1;                        /* gym_wrapper.py:37-39 / TimeLimit */
            if (e == 0 && step <= trace_steps) {
                if (trace) memcpy(trace + (size_t)sd * (step - 1), st, sizeof(double) * (size_t)sd);
                if (actions) actions[step - 1] = a;
            }
        }
        if (final) memcpy(final + (size_t)sd * e, st, sizeof(double) * (size_t)sd);
        nsteps += step;
        total = total + R;
    }
    if (steps_out) *steps_out = nsteps;
    return total / (double)E;
}

typedef struct {
    int env; const float *parents; float sigma; uint32_t seed, gen; int group, n_head, id0, n, E, max_step;
    const float *W_override; const double *init; int init_mode; double *fitness; int64_t *steps; int D;
    atomic_int next;
    int gru, sd;
    double *final;
} classic_job;

static void *classic_worker(void *arg)
{
    classic_job *jb = (classic_job *)arg;
    float *w = (float *)malloc(sizeof(float) * (size_t)jb->D);
    for (;;) {
        int j0 = atomic_fetch_add(&jb->next, 8);
        if (j0 >= jb->n) break;
        for (int j = j0; j < j0 + 8 && j < jb->n; ++j) {
            int id = jb->id0 + j;
            if (jb->W_override) memcpy(w, jb->W_override + (size_t)j * jb->D, sizeof(float) * (size_t)jb->D);
            else tw_perturb(jb->parents + (size_t)(id / jb->group) * jb->D, jb->D, jb->sigma, jb->seed, jb->gen, (uint32_t)id,
                            (id % jb->group) - jb->n_head + 1, w);
            jb->fitness[j] = classic_rollout(jb->env, jb->gru, w, jb->E, jb->max_step, jb->init, jb->seed, jb->init_mode, jb->gen,
                                             (uint32_t)id, NULL, NULL, 0, &jb->steps[j],
                                             jb->final ? jb->final + (size_t)j * jb->E * jb->sd : NULL);
        }
    }
    free(w);
    return NULL;
}

TW_EXPORT void tw_population_classic_gru(int env, int gru, const float *parents, float sigma, uint32_t seed, uint32_t gen, int group,
                                         int n_head, int id0, int n, int E, int max_step, const float *W_override,
                                         const double *init, int init_mode, double *fitness, int64_t *steps, int nthreads,
                                         double *final)
{
    int obs, act, sd, cap;
    if (tw_classic_dims(env, &obs, &act, &sd, &cap)) return;
    classic_job jb = { env, parents, sigma, seed, gen, group, n_head, id0, n, E, max_step, W_override, init, init_mode,
                       fitness, steps, tw_param_count(obs, act, gru), 0, gru, sd, final };
    if (nthreads < 1) nthreads = 1;
    if (nthreads > 256) nthreads = 256;
    pthread_t th[256];
    for (int t = 1; t < nthreads; ++t) pthread_create(&th[t], NULL, classic_worker, &jb);
    classic_worker(&jb);
    for (int t = 1; t < nthreads; ++t) pthread_join(th[t], NULL);
}

TW_EXPORT void tw_population_classic(int env, const float *parents, float sigma, uint32_t seed, uint32_t gen, int group,
                                     int n_head, int id0, int n, int E, int max_step, const float *W_override,
                                     const double *init, int init_mode, double *fitness, int64_t *steps, int nthreads)
{
    tw_population_classic_gru(env, 0, parents, sigma, seed, gen, group, n_head, id0, n, E, max_step, W_override, init, init_mode,
                              fitness, steps, nthreads, NULL);
}

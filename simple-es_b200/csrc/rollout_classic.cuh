// rollout_classic.cuh -- K1 environments beyond CartPole for the persistent slot kernel of rollout_slots.cuh:
// the classic-control tasks any reference config can name through GymWrapper (envs/gym_wrapper.py:8-45 hands the
// name to gym.make) with the discrete-action policy head (networks/neural_network.py:29-31).
//
//   MountainCarEnv  MountainCar-v0  obs 2, 3 actions, D = 195, reward -1 per step, TimeLimit 200
//   AcrobotEnv      Acrobot-v1      obs 6, 3 actions, D = 323, reward -1 per step (0 on the terminal step), TimeLimit 500
//
// Replaces GymEnvModel.forward (networks/neural_network.py:20-36), GymWrapper.reset/step (envs/gym_wrapper.py:23-45)
// and gym's classic_control/mountain_car.py / acrobot.py (un-vendored third party; restated in DESIGN.md Appendix).
// float64 physics in registers, float32 policy off the slot table (flat parameter order), one lane = one episode.
// The arithmetic is the contract of oracle/ses_twin_classic.c, operation for operation.
#pragma once
#include "rollout_cartpole_mlp.cuh"

namespace ses {

// ---------------------------------------------------------------------------------------------
// float64 sin / cos, full range (|x| * 2/pi must fit an int32): Cody-Waite reduction by pi/2 in two parts with fma,
// Taylor kernels to x^17 / x^16 on [-pi/4, pi/4]; <= 1 ulp from glibc on |x| < 100
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void sincos64_full(double x, double &sn, double &cs)
{
    const int n = __double2int_rn(__dmul_rn(x, 0.63661977236758138));
    const double kf = (double)n;
    double r = fma(-kf, 1.5707963267948966, x);
    r = fma(-kf, 6.123233995736766e-17, r);
    const double z = __dmul_rn(r, r);
    double p = 2.8114572543455206e-15;
    p = fma(p, z, -7.6471637318198164e-13);
    p = fma(p, z, 1.6059043836821613e-10);
    p = fma(p, z, -2.505210838544172e-08);
    p = fma(p, z, 2.7557319223985893e-06);
    p = fma(p, z, -0.00019841269841269841);
    p = fma(p, z, 0.0083333333333333332);
    p = fma(p, z, -0.16666666666666666);
    const double s = fma(__dmul_rn(r, z), p, r);
    double q = 4.7794773323873853e-14;
    q = fma(q, z, -1.1470745597729725e-11);
    q = fma(q, z, 2.08767569878681e-09);
    q = fma(q, z, -2.7557319223985888e-07);
    q = fma(q, z, 2.4801587301587302e-05);
    q = fma(q, z, -0.0013888888888888889);
    q = fma(q, z, 0.041666666666666664);
    const double c = __dadd_rn(1.0, fma(__dmul_rn(z, z), q, -__dmul_rn(0.5, z)));
    const int k = n & 3;
    const double s0 = (k & 1) ? c : s, c0 = (k & 1) ? s : c;
    sn = (k & 2) ? -s0 : s0;                       // k=0: s  1: c  2: -s  3: -c
    cs = (k == 1 || k == 2) ? -c0 : c0;            // k=0: c  1: -s 2: -c  3: s
}

__device__ __forceinline__ double cos64_full(double x) { double s, c; sincos64_full(x, s, c); return c; }
__device__ __forceinline__ double clip64(double v, double lo, double hi) { return fmin(fmax(v, lo), hi); }

// ---------------------------------------------------------------------------------------------
// the policy of a single-agent env off the flat slot table: W1 [32][OBS] | b1 [32] | W2 [ACT][32] | b2 [ACT].
// Hidden units in blocks of 4 (OBS consecutive quads of W1, one quad of b1, one quad per W2 row); tanh on
// packed pairs; every accumulator sees its products in ascending index order, one rounding per fma.
// ---------------------------------------------------------------------------------------------
template <int OBS, int ACT, int NQ, int S>
__device__ __forceinline__ void mlp_logits_flat(const float4 (&w)[NQ][S], int slot, const float (&o)[OBS], float (&z)[ACT])
{
    constexpr int O_B1 = HID * OBS, O_W2 = O_B1 + HID, O_B2 = O_W2 + ACT * HID;
    static_assert(O_B1 % 4 == 0 && O_W2 % 4 == 0 && O_B2 % 4 == 0 && ACT <= 4, "blocks are quad aligned");
    {
        const float4 b = w[O_B2 / 4][slot];
        const float bz[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
        for (int m = 0; m < ACT; ++m) z[m] = bz[m];
    }
    float sblk[ACT];                                   // fc2 block sums (contract 4.4: four blocks of eight hidden units)
#pragma unroll
    for (int m = 0; m < ACT; ++m) sblk[m] = 0.0f;
#pragma unroll
    for (int jq = 0; jq < HID / 4; ++jq) {
        float wr[4 * OBS];
#pragma unroll
        for (int q = 0; q < OBS; ++q) {
            const float4 t = w[jq * OBS + q][slot];
            wr[4 * q] = t.x; wr[4 * q + 1] = t.y; wr[4 * q + 2] = t.z; wr[4 * q + 3] = t.w;
        }
        const float4 b1 = w[O_B1 / 4 + jq][slot];
        float a[4] = {b1.x, b1.y, b1.z, b1.w};
#pragma unroll
        for (int u = 0; u < 4; ++u)
#pragma unroll
            for (int k = 0; k < OBS; ++k) a[u] = fmaf(wr[u * OBS + k], o[k], a[u]);
        const float2 h01 = tanh32x2<false>(make_float2(a[0], a[1])), h23 = tanh32x2<false>(make_float2(a[2], a[3]));
        const float h[4] = {h01.x, h01.y, h23.x, h23.y};
#pragma unroll
        for (int m = 0; m < ACT; ++m) {
            const float4 t = w[O_W2 / 4 + m * (HID / 4) + jq][slot];
            sblk[m] = fmaf(t.x, h[0], sblk[m]); sblk[m] = fmaf(t.y, h[1], sblk[m]); sblk[m] = fmaf(t.z, h[2], sblk[m]); sblk[m] = fmaf(t.w, h[3], sblk[m]);
            if (jq & 1) { z[m] = __fadd_rn(z[m], sblk[m]); sblk[m] = 0.0f; }
        }
    }
}

// discrete head (neural_network.py:29-31)
template <int OBS, int ACT, int NQ, int S>
__device__ __forceinline__ int mlp_policy_flat(const float4 (&w)[NQ][S], int slot, const float (&o)[OBS])
{
    float z[ACT];
    mlp_logits_flat<OBS, ACT, NQ, S>(w, slot, o, z);
    // argmax(softmax(z)) with the float32 collapse rule (neural_network.py:30-31; ses_common.cuh argmax_softmax2)
    float zmax = z[0];
#pragma unroll
    for (int m = 1; m < ACT; ++m) zmax = fmaxf(zmax, z[m]);
    int act = ACT - 1;
#pragma unroll
    for (int m = ACT - 2; m >= 0; --m)
        if (__fsub_rn(zmax, z[m]) <= __uint_as_float(0x33000000u)) act = m;
    return act;
}

// uniform in (0, 1) from one Philox word, as cartpole_init
__device__ __forceinline__ double unit64(uint32_t r) { return __dmul_rn(__dadd_rn((double)r, 0.5), 2.3283064365386963e-10); }

// ---------------------------------------------------------------------------------------------
// MountainCar-v0
// ---------------------------------------------------------------------------------------------
struct MountainCarEnv {
    static constexpr int OBS = 2, ACT = 3;
    static constexpr int D = param_count(OBS, ACT, 0), NQ = (D + 3) / 4;     // 195, 49
    static constexpr int STATE_DIM = 2, N_AGENTS = 1;
    static constexpr bool UNIT_REWARD = false;
    static constexpr bool LANES32_OK = false;     // the launcher may give all 32 lanes episodes (rollout_slots.cuh scheduler)
    struct State { double pos, vel, ret; };

    template <uint32_t STREAM = STREAM_INIT>
    __device__ static __forceinline__ void init(State &s, const RolloutParams &p, int id, int ep)
    {
        if (p.init_states) {
            s.pos = p.init_states[2 * ep]; s.vel = p.init_states[2 * ep + 1];
        } else {
            const uint4 r = philox4x32_10((uint32_t)ep, p.init_mode ? (uint32_t)id : 0u, p.init_mode ? p.gen : 0u, 0u, p.seed, STREAM);
            s.pos = __dsub_rn(__dmul_rn(unit64(r.x), 0.2), 0.6);       // U(-0.6, -0.4)
            s.vel = 0.0;
        }
        s.ret = 0.0;
    }

    template <int S>
    __device__ static __forceinline__ void store_quad(float4 (&w)[NQ][S], int q, int s, const float4 v) { w[q][s] = v; }
    template <int S>
    __device__ static __forceinline__ void bind(State &, const float4 (&)[NQ][S], int) {}

    // the env seen by a policy kernel: observations of every agent, and one step under the chosen actions
    static constexpr int OBS_EFF = OBS;
    static constexpr bool CONTINUOUS = false;
    __device__ static __forceinline__ void observe(const State &s, float (&o)[N_AGENTS][OBS_EFF]) { o[0][0] = (float)s.pos; o[0][1] = (float)s.vel; }

    template <int S>
    __device__ static __forceinline__ bool step(State &s, const float4 (&w)[NQ][S], int slot, const RolloutParams &, int *actions)
    {
        float o[N_AGENTS][OBS_EFF];
        observe(s, o);
        actions[0] = mlp_policy_flat<OBS, ACT, NQ, S>(w, slot, o[0]);
        return advance(s, actions);
    }

    __device__ static __forceinline__ bool advance(State &s, const int *actions)
    {
        const int a = actions[0];
        double v = __dadd_rn(s.vel, __dadd_rn(__dmul_rn((double)(a - 1), 0.001), __dmul_rn(cos64_full(__dmul_rn(3.0, s.pos)), -0.0025)));
        v = clip64(v, -0.07, 0.07);
        double x = clip64(__dadd_rn(s.pos, v), -1.2, 0.6);
        if (x == -1.2 && v < 0.0) v = 0.0;
        s.pos = x; s.vel = v;
        s.ret = __dadd_rn(s.ret, -1.0);
        return x >= 0.5 && v >= 0.0;
    }

    __device__ static __forceinline__ void store_trace(const State &s, double *row) { row[0] = s.pos; row[1] = s.vel; }
    __device__ static __forceinline__ void store_init(const State &s, double *row) { store_trace(s, row); }
};

// ---------------------------------------------------------------------------------------------
// Pendulum-v0 with the continuous-action head: action = tanh(fc2(...)) (neural_network.py:32-33), one float32 in (-1, 1)
// used as the torque.  gym classic_control/pendulum.py (gym ~0.18; DESIGN.md Appendix): never terminates (TimeLimit 200),
// reward -(angle_normalize(th)^2 + .1 thdot^2 + .001 u^2), obs [cos th, sin th, thdot].
// ---------------------------------------------------------------------------------------------
struct PendulumEnv {
    static constexpr int OBS = 3, ACT = 1;
    static constexpr int D = param_count(OBS, ACT, 0), NQ = (D + 3) / 4;     // 161, 41
    static constexpr int STATE_DIM = 2, N_AGENTS = 1;
    static constexpr bool UNIT_REWARD = false;
    static constexpr bool LANES32_OK = false;
    static constexpr double PI = 3.141592653589793;
    struct State { double th, thd, ret; };

    template <uint32_t STREAM = STREAM_INIT>
    __device__ static __forceinline__ void init(State &s, const RolloutParams &p, int id, int ep)
    {
        if (p.init_states) {
            s.th = p.init_states[2 * ep]; s.thd = p.init_states[2 * ep + 1];
        } else {                                                       // uniform(-[pi, 1], [pi, 1])
            const uint4 r = philox4x32_10((uint32_t)ep, p.init_mode ? (uint32_t)id : 0u, p.init_mode ? p.gen : 0u, 0u, p.seed, STREAM);
            s.th = __dsub_rn(__dmul_rn(unit64(r.x), __dmul_rn(2.0, PI)), PI);
            s.thd = __dsub_rn(__dmul_rn(unit64(r.y), 2.0), 1.0);
        }
        s.ret = 0.0;
    }

    template <int S>
    __device__ static __forceinline__ void store_quad(float4 (&w)[NQ][S], int q, int s, const float4 v) { w[q][s] = v; }
    template <int S>
    __device__ static __forceinline__ void bind(State &, const float4 (&)[NQ][S], int) {}

    static constexpr int OBS_EFF = OBS;
    static constexpr bool CONTINUOUS = true;
    __device__ static __forceinline__ void observe(const State &s, float (&o)[N_AGENTS][OBS_EFF])
    {
        double sn, cs;
        sincos64_full(s.th, sn, cs);
        o[0][0] = (float)cs; o[0][1] = (float)sn; o[0][2] = (float)s.thd;
    }

    template <int S>
    __device__ static __forceinline__ bool step(State &s, const float4 (&w)[NQ][S], int slot, const RolloutParams &, int *actions)
    {
        float o[N_AGENTS][OBS_EFF];
        observe(s, o);
        float z[ACT];
        mlp_logits_flat<OBS, ACT, NQ, S>(w, slot, o[0], z);
        const float uf = tanh32_fast_t<false>(z[0]);                   // == the contract's tanh32 for every input (exhaustive test)
        actions[0] = __float_as_int(uf);                               // traces carry the float32 action's bit pattern
        return advance(s, actions);
    }

    // actions[0]: bit pattern of the float32 action in (-1, 1)
    __device__ static __forceinline__ bool advance(State &s, const int *actions)
    {
        const float uf = __int_as_float(actions[0]);
        const double u = clip64((double)uf, -2.0, 2.0);
        double m = fmod(__dadd_rn(s.th, PI), __dmul_rn(2.0, PI));      // Python's float %: fmod, then the divisor's sign
        if (m < 0.0) m = __dadd_rn(m, __dmul_rn(2.0, PI));
        const double an = __dsub_rn(m, PI);
        const double costs = __dadd_rn(__dadd_rn(__dmul_rn(an, an), __dmul_rn(0.1, __dmul_rn(s.thd, s.thd))), __dmul_rn(0.001, __dmul_rn(u, u)));
        double s2, c2;
        sincos64_full(__dadd_rn(s.th, PI), s2, c2);
        double nthd = __dadd_rn(s.thd, __dmul_rn(__dadd_rn(__dmul_rn(-15.0, s2), __dmul_rn(3.0, u)), 0.05));
        s.th = __dadd_rn(s.th, __dmul_rn(nthd, 0.05));
        s.thd = clip64(nthd, -8.0, 8.0);
        s.ret = __dadd_rn(s.ret, -costs);
        return false;
    }

    __device__ static __forceinline__ void store_trace(const State &s, double *row) { row[0] = s.th; row[1] = s.thd; }
    __device__ static __forceinline__ void store_init(const State &s, double *row) { store_trace(s, row); }
};

// ---------------------------------------------------------------------------------------------
// Acrobot-v1 (book dynamics, RK4 over dt = 0.2, no torque noise)
// ---------------------------------------------------------------------------------------------
struct AcrobotEnv {
    static constexpr int OBS = 6, ACT = 3;
    static constexpr int D = param_count(OBS, ACT, 0), NQ = (D + 3) / 4;     // 323, 81
    static constexpr int STATE_DIM = 4, N_AGENTS = 1;
    static constexpr bool UNIT_REWARD = false;
    static constexpr bool LANES32_OK = false;     // the launcher may give all 32 lanes episodes (rollout_slots.cuh scheduler)
    static constexpr double PI = 3.141592653589793;
    // sc = { sin th1, cos th1, sin th2, cos th2 } of the current state: computed once per step (terminal test) and reused
    // by the next step's observation and first RK4 stage (same function, same argument: same bits as recomputing)
    struct State { double s[4]; double sc[4]; double ret; };

    template <uint32_t STREAM = STREAM_INIT>
    __device__ static __forceinline__ void init(State &st, const RolloutParams &p, int id, int ep)
    {
        if (p.init_states) {
#pragma unroll
            for (int k = 0; k < 4; ++k) st.s[k] = p.init_states[4 * ep + k];
        } else {
            const uint4 r = philox4x32_10((uint32_t)ep, p.init_mode ? (uint32_t)id : 0u, p.init_mode ? p.gen : 0u, 0u, p.seed, STREAM);
            st.s[0] = __dsub_rn(__dmul_rn(unit64(r.x), 0.2), 0.1);       // U(-0.1, 0.1)^4
            st.s[1] = __dsub_rn(__dmul_rn(unit64(r.y), 0.2), 0.1);
            st.s[2] = __dsub_rn(__dmul_rn(unit64(r.z), 0.2), 0.1);
            st.s[3] = __dsub_rn(__dmul_rn(unit64(r.w), 0.2), 0.1);
        }
        sincos64_full(st.s[0], st.sc[0], st.sc[1]);
        sincos64_full(st.s[1], st.sc[2], st.sc[3]);
        st.ret = 0.0;
    }

    template <int S>
    __device__ static __forceinline__ void store_quad(float4 (&w)[NQ][S], int q, int s, const float4 v) { w[q][s] = v; }
    template <int S>
    __device__ static __forceinline__ void bind(State &, const float4 (&)[NQ][S], int) {}

    // _dsdt of acrobot.py with m1 = m2 = l1 = 1, lc1 = lc2 = 0.5, I1 = I2 = 1, g = 9.8 (this translation unit is
    // compiled with -fmad=false: every operator below is one separately rounded IEEE operation, in Python's order)
    template <bool CACHED>
    __device__ static __forceinline__ void dsdt(const double (&y)[4], double a, double (&ds)[4], double sin2c = 0.0, double cos2c = 0.0)
    {
        const double theta1 = y[0], theta2 = y[1], dtheta1 = y[2], dtheta2 = y[3];
        double sin2 = sin2c, cos2 = cos2c;
        if constexpr (!CACHED) sincos64_full(theta2, sin2, cos2);
        const double d1 = ((0.25 + (1.25 + cos2)) + 1.0) + 1.0;
        const double d2 = (0.25 + 0.5 * cos2) + 1.0;
        const double phi2 = 4.9 * cos64_full((theta1 + theta2) - PI / 2.0);
        const double phi1 = (((-0.5 * (dtheta2 * dtheta2)) * sin2 - (dtheta2 * dtheta1) * sin2)
                             + (1.5 * 9.8) * cos64_full(theta1 - PI / 2.0)) + phi2;
        const double ddtheta2 = (((a + (d2 / d1) * phi1) - (0.5 * (dtheta1 * dtheta1)) * sin2) - phi2)
                                / (1.25 - (d2 * d2) / d1);
        const double ddtheta1 = -(d2 * ddtheta2 + phi1) / d1;
        ds[0] = dtheta1; ds[1] = dtheta2; ds[2] = ddtheta1; ds[3] = ddtheta2;
    }

    __device__ static __forceinline__ double wrap(double x)
    {
        const double diff = PI - (-PI);
        while (x > PI) x = x - diff;
        while (x < -PI) x = x + diff;
        return x;
    }

    static constexpr int OBS_EFF = OBS;
    static constexpr bool CONTINUOUS = false;
    __device__ static __forceinline__ void observe(const State &st, float (&o)[N_AGENTS][OBS_EFF])
    {
        o[0][0] = (float)st.sc[1]; o[0][1] = (float)st.sc[0]; o[0][2] = (float)st.sc[3]; o[0][3] = (float)st.sc[2];
        o[0][4] = (float)st.s[2]; o[0][5] = (float)st.s[3];
    }

    template <int S>
    __device__ static __forceinline__ bool step(State &st, const float4 (&w)[NQ][S], int slot, const RolloutParams &, int *actions)
    {
        float o[N_AGENTS][OBS_EFF];
        observe(st, o);
        actions[0] = mlp_policy_flat<OBS, ACT, NQ, S>(w, slot, o[0]);
        return advance(st, actions);
    }

    __device__ static __forceinline__ bool advance(State &st, const int *actions)
    {
        const int act = actions[0];
        const double torque = (double)(act - 1);
        const double dt = 0.2, dt2 = 0.2 / 2.0;
        double k1[4], k2[4], k3[4], k4[4], y[4];
        dsdt<true>(st.s, torque, k1, st.sc[2], st.sc[3]);
#pragma unroll
        for (int i = 0; i < 4; ++i) y[i] = st.s[i] + dt2 * k1[i];
        dsdt<false>(y, torque, k2);
#pragma unroll
        for (int i = 0; i < 4; ++i) y[i] = st.s[i] + dt2 * k2[i];
        dsdt<false>(y, torque, k3);
#pragma unroll
        for (int i = 0; i < 4; ++i) y[i] = st.s[i] + dt * k3[i];
        dsdt<false>(y, torque, k4);
        double ns[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) ns[i] = st.s[i] + (dt / 6.0) * (((k1[i] + 2.0 * k2[i]) + 2.0 * k3[i]) + k4[i]);
        ns[0] = wrap(ns[0]);
        ns[1] = wrap(ns[1]);
        ns[2] = clip64(ns[2], -4.0 * PI, 4.0 * PI);
        ns[3] = clip64(ns[3], -9.0 * PI, 9.0 * PI);
#pragma unroll
        for (int i = 0; i < 4; ++i) st.s[i] = ns[i];
        sincos64_full(ns[0], st.sc[0], st.sc[1]);
        sincos64_full(ns[1], st.sc[2], st.sc[3]);
        const bool terminal = (-st.sc[1] - cos64_full(ns[1] + ns[0])) > 1.0;
        st.ret = st.ret + (terminal ? 0.0 : -1.0);
        return terminal;
    }

    __device__ static __forceinline__ void store_trace(const State &st, double *row)
    {
        row[0] = st.s[0]; row[1] = st.s[1]; row[2] = st.s[2]; row[3] = st.s[3];
    }
    __device__ static __forceinline__ void store_init(const State &st, double *row) { store_trace(st, row); }
};

}  // namespace ses

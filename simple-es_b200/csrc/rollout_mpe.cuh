// rollout_mpe.cuh -- K1 environment: PettingZoo MPE simple_spread (N agents, N landmarks) with the
// shared 32-hidden MLP policy (obs 6N, 5 discrete actions; D = 581 for N = 2, 773 for N = 3),
// plugged into the persistent slot kernel of rollout_slots.cuh.
//
// Replaces PettingzooWrapper.reset/step (envs/pettingzoo_wrapper.py:22-58), the one-model-copy-per
// agent rollout (learning_strategies/evolution/utils.py:4-8, loop.py:114-123) and the MPE
// simple_spread_v2 world (un-vendored third party, SURVEY.md Appendix A.2): float64 physics,
// observations rounded to float32, team reward = sum of the agents' rewards
// (0.5 * global + 0.5 * local), fixed 25-cycle episodes.
//
// A lane owns one episode: 6N doubles of world state in registers.  The N agents share the
// offspring's weights, so both forward passes run off the same LDS.128 of a weight quad.
#pragma once
#include <cstdio>
#include "rollout_cartpole_mlp.cuh"

namespace ses {

// exp(t), t <= 0; below exp(-700) flushed to 0 (contract: oracle/ses_twin_mpe.c tw_exp_neg)
__device__ __forceinline__ double exp_neg64(double t)
{
    if (t < -700.0) return 0.0;
    const int k = __double2int_rz(__dsub_rn(__dmul_rn(t, 1.4426950408889634), 0.5));
    const double kf = (double)k;
    double r = fma(-kf, 6.93147180369123816490e-01, t);
    r = fma(-kf, 1.90821492927058770002e-10, r);
    double p = 1.6059043836821613e-10;
    p = fma(p, r, 2.08767569878681e-09);
    p = fma(p, r, 2.505210838544172e-08);
    p = fma(p, r, 2.7557319223985888e-07);
    p = fma(p, r, 2.7557319223985893e-06);
    p = fma(p, r, 2.4801587301587302e-05);
    p = fma(p, r, 0.00019841269841269841);
    p = fma(p, r, 0.0013888888888888889);
    p = fma(p, r, 0.0083333333333333332);
    p = fma(p, r, 0.041666666666666664);
    p = fma(p, r, 0.16666666666666666);
    p = fma(p, r, 0.5);
    p = fma(p, r, 1.0);
    p = fma(p, r, 1.0);
    return __dmul_rn(p, __longlong_as_double((long long)(k + 1023) << 52));
}

// ln(u), u in [1, 2]
__device__ __forceinline__ double log_12_64(double u)
{
    double m = u, e = 0.0;
    if (u > 1.4142135623730951) { m = __dmul_rn(u, 0.5); e = 0.6931471805599453; }
    const double s = __ddiv_rn(__dsub_rn(m, 1.0), __dadd_rn(m, 1.0));
    const double z = __dmul_rn(s, s);
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
    q = __dmul_rn(q, z);
    const double r2 = __dmul_rn(2.0, s);
    return __dadd_rn(e, fma(r2, q, r2));
}

__device__ __forceinline__ double log1p_01_64(double v)
{
    const double u = __dadd_rn(1.0, v);
    const double c = __ddiv_rn(__dsub_rn(v, __dsub_rn(u, 1.0)), u);
    return __dadd_rn(log_12_64(u), c);
}

// numpy.logaddexp(0, y)
__device__ __forceinline__ double logaddexp0_64(double y)
{
    if (y < 0.0) return log1p_01_64(exp_neg64(y));
    return __dadd_rn(y, log1p_01_64(exp_neg64(-y)));
}

template <int N>
struct SpreadEnv {
    static constexpr int OBS = 6 * N, ACT = 5;
    static constexpr int D = param_count(OBS, ACT, 0), NQ = (D + 3) / 4;
    static constexpr int STATE_DIM = 4 * N, N_AGENTS = N;
    static constexpr bool UNIT_REWARD = false;
    static constexpr bool LANES32_OK = false;     // the launcher may give all 32 lanes episodes (rollout_slots.cuh scheduler)
    static constexpr int OBS_EFF = OBS - 2 * (N - 1);      // trailing comm entries are always 0 (silent agents)
    // flat offsets (floats): W1 [32][OBS] | b1 [32] | W2 [5][32] | b2 [5]
    static constexpr int O_B1 = HID * OBS, O_W2 = O_B1 + HID, O_B2 = O_W2 + ACT * HID;
    static_assert(O_B1 % 4 == 0 && O_W2 % 4 == 0 && O_B2 % 4 == 0, "blocks are quad aligned");

    struct State {
        double apos[N][2], avel[N][2], lpos[N][2];
        double ret;                                          // sequential sum of the episode's team rewards
    };

    template <uint32_t STREAM = STREAM_INIT>
    __device__ static __forceinline__ void init(State &s, const RolloutParams &p, int id, int ep)
    {
        double v[4 * N];
        if (p.init_states) {
#pragma unroll
            for (int k = 0; k < 4 * N; ++k) v[k] = p.init_states[(size_t)4 * N * ep + k];
        } else {
#pragma unroll
            for (int b = 0; b < N; ++b) {
                const uint4 r = philox4x32_10((uint32_t)ep, p.init_mode ? (uint32_t)id : 0u, p.init_mode ? p.gen : 0u, (uint32_t)b,
                                              p.seed, STREAM);
                const double k32 = 2.3283064365386963e-10;
                v[4 * b + 0] = __dsub_rn(__dmul_rn(__dmul_rn(__dadd_rn((double)r.x, 0.5), k32), 2.0), 1.0);
                v[4 * b + 1] = __dsub_rn(__dmul_rn(__dmul_rn(__dadd_rn((double)r.y, 0.5), k32), 2.0), 1.0);
                v[4 * b + 2] = __dsub_rn(__dmul_rn(__dmul_rn(__dadd_rn((double)r.z, 0.5), k32), 2.0), 1.0);
                v[4 * b + 3] = __dsub_rn(__dmul_rn(__dmul_rn(__dadd_rn((double)r.w, 0.5), k32), 2.0), 1.0);
            }
        }
#pragma unroll
        for (int i = 0; i < N; ++i) {
            s.apos[i][0] = v[2 * i]; s.apos[i][1] = v[2 * i + 1];
            s.avel[i][0] = 0.0; s.avel[i][1] = 0.0;
            s.lpos[i][0] = v[2 * N + 2 * i]; s.lpos[i][1] = v[2 * N + 2 * i + 1];
        }
        s.ret = 0.0;
    }

    template <int S>
    __device__ static __forceinline__ void store_quad(float4 (&w)[NQ][S], int q, int s, const float4 v) { w[q][s] = v; }

    template <int S>
    __device__ static __forceinline__ void bind(State &, const float4 (&)[NQ][S], int) {}

    static constexpr bool CONTINUOUS = false;
    // observations (Scenario.observation): [vel, pos, landmarks - pos, others - pos, comm = 0], f64 -> f32
    __device__ static __forceinline__ void observe(const State &s, float (&o)[N][OBS_EFF])
    {
#pragma unroll
        for (int i = 0; i < N; ++i) {
            int c = 0;
            o[i][c++] = (float)s.avel[i][0]; o[i][c++] = (float)s.avel[i][1];
            o[i][c++] = (float)s.apos[i][0]; o[i][c++] = (float)s.apos[i][1];
#pragma unroll
            for (int l = 0; l < N; ++l) {
                o[i][c++] = (float)__dsub_rn(s.lpos[l][0], s.apos[i][0]);
                o[i][c++] = (float)__dsub_rn(s.lpos[l][1], s.apos[i][1]);
            }
#pragma unroll
            for (int j = 0; j < N; ++j)
                if (j != i) {
                    o[i][c++] = (float)__dsub_rn(s.apos[j][0], s.apos[i][0]);
                    o[i][c++] = (float)__dsub_rn(s.apos[j][1], s.apos[i][1]);
                }
        }
    }

    template <int S>
    __device__ static __forceinline__ bool step(State &s, const float4 (&w)[NQ][S], int slot, const RolloutParams &, int *actions)
    {
        float o[N][OBS_EFF];
        observe(s, o);
        // shared MLP, all agents off the same weight loads; logits in the contract's sequential order.
        // Agents 0 and 1 run as the two halves of packed FFMA2 operations (same weight, two observations);
        // a third agent runs scalar.  Same operations, same order, one rounding each as the oracle.
        constexpr int NS = N - 2;                              // agents beyond the packed pair
        float2 op[OBS_EFF];
#pragma unroll
        for (int k = 0; k < OBS_EFF; ++k) op[k] = make_float2(o[0][k], o[1][k]);
        float2 zp[ACT];
        float zs[NS > 0 ? NS : 1][ACT];
        {
            const float4 ba = w[O_B2 / 4][slot], bb = w[O_B2 / 4 + 1][slot];
            const float bz[ACT] = {ba.x, ba.y, ba.z, ba.w, bb.x};
#pragma unroll
            for (int m = 0; m < ACT; ++m) {
                zp[m] = make_float2(bz[m], bz[m]);
#pragma unroll
                for (int i = 0; i < NS; ++i) zs[i][m] = bz[m];
            }
        }
        // fc2 in four blocks of eight hidden units (contract 4.4): block sums sp / ss live over two iterations of the inner loop
#pragma unroll 1
        for (int g = 0; g < HID / 8; ++g) {
        float2 sp[ACT];
        float ss[NS > 0 ? NS : 1][ACT];
#pragma unroll
        for (int m = 0; m < ACT; ++m) {
            sp[m] = make_float2(0.0f, 0.0f);
#pragma unroll
            for (int i = 0; i < NS; ++i) ss[i][m] = 0.0f;
        }
#pragma unroll 1
        for (int jq = 2 * g; jq < 2 * g + 2; ++jq) {
            // 4 hidden units = OBS consecutive quads of W1
            float wr[4 * OBS];
#pragma unroll
            for (int q = 0; q < OBS; ++q) {
                const float4 t = w[jq * OBS + q][slot];
                wr[4 * q] = t.x; wr[4 * q + 1] = t.y; wr[4 * q + 2] = t.z; wr[4 * q + 3] = t.w;
            }
            const float4 b1 = w[O_B1 / 4 + jq][slot];
            const float bias[4] = {b1.x, b1.y, b1.z, b1.w};
            float w2[ACT][4];
#pragma unroll
            for (int m = 0; m < ACT; ++m) {
                const float4 t = w[O_W2 / 4 + m * (HID / 4) + jq][slot];
                w2[m][0] = t.x; w2[m][1] = t.y; w2[m][2] = t.z; w2[m][3] = t.w;
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                float2 a = make_float2(bias[u], bias[u]);
#pragma unroll
                for (int k = 0; k < OBS_EFF; ++k) a = __ffma2_rn(make_float2(wr[u * OBS + k], wr[u * OBS + k]), op[k], a);
                // the skipped comm inputs are exactly 0: fmaf(w, 0, a) == a
                const float2 h = tanh32x2<false>(a);
#pragma unroll
                for (int m = 0; m < ACT; ++m) sp[m] = __ffma2_rn(make_float2(w2[m][u], w2[m][u]), h, sp[m]);
#pragma unroll
                for (int i = 0; i < NS; ++i) {
                    float as = bias[u];
#pragma unroll
                    for (int k = 0; k < OBS_EFF; ++k) as = fmaf(wr[u * OBS + k], o[2 + i][k], as);
                    const float hs = tanh32_fast_t<false>(as);
#pragma unroll
                    for (int m = 0; m < ACT; ++m) ss[i][m] = fmaf(w2[m][u], hs, ss[i][m]);
                }
            }
        }
#pragma unroll
        for (int m = 0; m < ACT; ++m) {
            zp[m] = __fadd2_rn(zp[m], sp[m]);
#pragma unroll
            for (int i = 0; i < NS; ++i) zs[i][m] = __fadd_rn(zs[i][m], ss[i][m]);
        }
        }
        float z[N][ACT];
#pragma unroll
        for (int m = 0; m < ACT; ++m) {
            z[0][m] = zp[m].x; z[1][m] = zp[m].y;
#pragma unroll
            for (int i = 0; i < NS; ++i) z[2 + i][m] = zs[i][m];
        }
        // argmax(softmax(z)) with the float32 collapse rule (neural_network.py:30-31)
#pragma unroll
        for (int i = 0; i < N; ++i) {
            float zmax = z[i][0];
#pragma unroll
            for (int m = 1; m < ACT; ++m) zmax = fmaxf(zmax, z[i][m]);
            int a = ACT - 1;
#pragma unroll
            for (int m = ACT - 2; m >= 0; --m)
                if (__fsub_rn(zmax, z[i][m]) <= __uint_as_float(0x33000000u)) a = m;
            actions[i] = a;
        }
        return advance(s, actions);
    }

    // world step (MPE core.World.step) under the agents' actions + the team reward
    __device__ static __forceinline__ bool advance(State &s, const int *actions)
    {
        double F[N][2];
#pragma unroll
        for (int i = 0; i < N; ++i) {
            const int a = actions[i];
            const double ux = a == 1 ? -1.0 : (a == 2 ? 1.0 : 0.0);
            const double uy = a == 3 ? -1.0 : (a == 4 ? 1.0 : 0.0);
            F[i][0] = __dmul_rn(ux, 5.0); F[i][1] = __dmul_rn(uy, 5.0);
        }
#pragma unroll
        for (int a = 0; a < N; ++a)
#pragma unroll
            for (int b = a + 1; b < N; ++b) {
                const double dx = __dsub_rn(s.apos[a][0], s.apos[b][0]), dy = __dsub_rn(s.apos[a][1], s.apos[b][1]);
                const double dist = __dsqrt_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)));
                const double pen = __dmul_rn(logaddexp0_64(__ddiv_rn(-__dsub_rn(dist, 0.3), 0.001)), 0.001);
                const double fx = __dmul_rn(__ddiv_rn(__dmul_rn(100.0, dx), dist), pen);
                const double fy = __dmul_rn(__ddiv_rn(__dmul_rn(100.0, dy), dist), pen);
                F[a][0] = __dadd_rn(F[a][0], fx); F[a][1] = __dadd_rn(F[a][1], fy);
                F[b][0] = __dsub_rn(F[b][0], fx); F[b][1] = __dsub_rn(F[b][1], fy);
            }
#pragma unroll
        for (int i = 0; i < N; ++i)
#pragma unroll
            for (int d = 0; d < 2; ++d) {
                double v = __dmul_rn(s.avel[i][d], 0.75);
                v = __dadd_rn(v, __dmul_rn(F[i][d], 0.1));
                s.avel[i][d] = v;
                s.apos[i][d] = __dadd_rn(s.apos[i][d], __dmul_rn(v, 0.1));
            }
        // rewards (Scenario.global_reward / reward; the 2021 sources count the agent's own "collision")
        // The oracle takes min_a sqrt(d2) per landmark and tests sqrt(d2) < 0.3 for every ordered agent pair.  sqrt is
        // monotone and correctly rounded, so (same bits, 6 instead of 21 square roots at N = 3):
        //   min_a sqrt(d2_a) == sqrt(min_a d2_a);   sqrt(d2) < 0.3  <=>  d2 < D2_COLLIDE, the smallest double whose root
        //   is >= 0.3 (0x3fb70a3d70a3d709);   d2(a, i) == d2(i, a) bit for bit;   d2(i, i) == 0 always collides.
        double glob = 0.0;
#pragma unroll
        for (int l = 0; l < N; ++l) {
            double best2 = 0.0;
#pragma unroll
            for (int a = 0; a < N; ++a) {
                const double dx = __dsub_rn(s.apos[a][0], s.lpos[l][0]), dy = __dsub_rn(s.apos[a][1], s.lpos[l][1]);
                const double d2 = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
                if (a == 0 || d2 < best2) best2 = d2;
            }
            glob = __dsub_rn(glob, __dsqrt_rn(best2));
        }
        const double D2_COLLIDE = __longlong_as_double(0x3fb70a3d70a3d709ll);
        bool hit[N][N];
#pragma unroll
        for (int i = 0; i < N; ++i) {
            hit[i][i] = true;
#pragma unroll
            for (int a = i + 1; a < N; ++a) {
                const double dx = __dsub_rn(s.apos[a][0], s.apos[i][0]), dy = __dsub_rn(s.apos[a][1], s.apos[i][1]);
                hit[i][a] = hit[a][i] = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)) < D2_COLLIDE;
            }
        }
        double total = 0.0;
#pragma unroll
        for (int i = 0; i < N; ++i) {
            double local = 0.0;
#pragma unroll
            for (int a = 0; a < N; ++a)
                if (hit[i][a]) local = __dsub_rn(local, 1.0);
            total = __dadd_rn(total, __dadd_rn(__dmul_rn(glob, 0.5), __dmul_rn(local, 0.5)));
        }
        s.ret = __dadd_rn(s.ret, total);
        return false;                                         // the episode ends by max_cycles only
    }

    __device__ static __forceinline__ void store_trace(const State &s, double *row)
    {
#pragma unroll
        for (int i = 0; i < N; ++i) {
            row[2 * i] = s.apos[i][0]; row[2 * i + 1] = s.apos[i][1];
            row[2 * N + 2 * i] = s.avel[i][0]; row[2 * N + 2 * i + 1] = s.avel[i][1];
        }
    }

    // init_states layout: agent positions, then landmark positions (the velocities start at 0)
    __device__ static __forceinline__ void store_init(const State &s, double *row)
    {
#pragma unroll
        for (int i = 0; i < N; ++i) {
            row[2 * i] = s.apos[i][0]; row[2 * i + 1] = s.apos[i][1];
            row[2 * N + 2 * i] = s.lpos[i][0]; row[2 * N + 2 * i + 1] = s.lpos[i][1];
        }
    }
};

}  // namespace ses

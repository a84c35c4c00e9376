// update.cuh -- K3: strategy updates that re-derive the noise instead of storing it.
//
//   openai_es : g = sum_j eps_j F_j, scale, Adam      (offspring_strategies.py:401-416, optimizers.py:13-57)
//   evolution : mu = mean of the k best offspring      (offspring_strategies.py:241-250)
//   genetic   : elite table = weights of the k best    (offspring_strategies.py:114-116)
//
// The reduction tree of the gradient is fixed (DESIGN.md section 4.6) so that every rank and the
// CPU oracle produce the same bits: float64 accumulation,
//   level 0: blocks of 32 consecutive offspring, sequential fma in offspring order
//   level 1: groups of 64 consecutive block partials, sequential add
//   level 2: sequential add over groups, one rounding to float32, scale, Adam.
#pragma once
#include "ses_common.cuh"

namespace ses {

constexpr int GB0 = 32;
constexpr int GB1 = 64;

struct PeerRows { double *p[8]; };

// quads per CTA of k_grad_partial (CTA = 64 blocks x GQC quads).  A pure launch-shape parameter: 2 (928 CTAs of 128 threads at
// P = 65536, 6.3 per SM) balances the 148 SMs better than 4 (480 CTAs, 3.2 per SM): 59 -> 54 us per update on a B200.
constexpr int GQC = 2;

// levels 0 and 1 fused: CTA <-> (group g, chunk of GQC quads); thread <-> (block b of the group, quad q).
// Level 0 runs in registers (32 sequential fma per parameter), the 64 block partials of the group meet in
// shared memory and are added sequentially in block order (level 1).  part1[g][DP] float64.
// Groups [g_begin, g_end) only: with several ranks each computes its share of the groups and stores the rows
// into every peer's part1 buffer over NVLink (peer_part1), so that all ranks finish with the same table.
// SQ (sep_cma_es, DESIGN.md section 4.11): a second table of sum_j shaped_j eps_jd^2 (eps^2 formed exactly in float64) in the
// same pass, at part1 + nb1 * DP, mirrored to the peers likewise.  Rows with shaped_j == 0 are skipped: their fma would add
// an exact zero to a sum that is never -0.0, so both tables keep their bits.
template <bool SQ = false>
__global__ void __launch_bounds__(GB1 * GQC) k_grad_partial(const double *__restrict__ shaped, int P, int D, int NQ, uint32_t seed,
                                                            uint32_t gen, Layout layout, const float *__restrict__ eps_override,
                                                            double *__restrict__ part1, int nb0, int g_begin, int n_chunks,
                                                            int n_peers, PeerRows peers, const PeerSync sync)
{
    __shared__ double sp[SQ ? 2 : 1][GB1][GQC * 4];
    const int g = g_begin + blockIdx.x / n_chunks;
    const int qc = blockIdx.x % n_chunks;
    const int bb = threadIdx.x / GQC, qq = threadIdx.x % GQC;
    const int b = g * GB1 + bb, q = qc * GQC + qq;
    double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
    [[maybe_unused]] double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
    if (b < nb0 && q < NQ) {
        const int j1 = min(P, (b + 1) * GB0);
        for (int j = b * GB0; j < j1; ++j) {
            if constexpr (SQ) {
                if (shaped[j] == 0.0) continue;
            }
            float4 e;
            if (eps_override) {
                const float *row = eps_override + (size_t)j * D;
                const int d = 4 * q;
                e.x = d + 0 < D ? row[d + 0] : 0.0f;
                e.y = d + 1 < D ? row[d + 1] : 0.0f;
                e.z = d + 2 < D ? row[d + 2] : 0.0f;
                e.w = d + 3 < D ? row[d + 3] : 0.0f;
            } else {
                if (!layout.perturbed(j)) continue;           // eps == 0 (offspring_strategies.py:302-308)
                float sg;
                const uint32_t nid = layout.noise_id(j, sg);
                e = normal4(seed, (uint32_t)q, nid, gen);
                e.x = __fmul_rn(e.x, sg); e.y = __fmul_rn(e.y, sg); e.z = __fmul_rn(e.z, sg); e.w = __fmul_rn(e.w, sg);
            }
            const double f = shaped[j];
            a0 = fma((double)e.x, f, a0);
            a1 = fma((double)e.y, f, a1);
            a2 = fma((double)e.z, f, a2);
            a3 = fma((double)e.w, f, a3);
            if constexpr (SQ) {
                s0 = fma(__dmul_rn((double)e.x, (double)e.x), f, s0);
                s1 = fma(__dmul_rn((double)e.y, (double)e.y), f, s1);
                s2 = fma(__dmul_rn((double)e.z, (double)e.z), f, s2);
                s3 = fma(__dmul_rn((double)e.w, (double)e.w), f, s3);
            }
        }
    }
    sp[0][bb][qq * 4 + 0] = a0; sp[0][bb][qq * 4 + 1] = a1; sp[0][bb][qq * 4 + 2] = a2; sp[0][bb][qq * 4 + 3] = a3;
    if constexpr (SQ) {
        sp[1][bb][qq * 4 + 0] = s0; sp[1][bb][qq * 4 + 1] = s1; sp[1][bb][qq * 4 + 2] = s2; sp[1][bb][qq * 4 + 3] = s3;
    }
    __syncthreads();
    if (threadIdx.x < GQC * 4) {
        const int d = qc * GQC * 4 + threadIdx.x;
        if (d < NQ * 4) {
            const int nb = min(GB1, nb0 - g * GB1);
            double t = 0.0;
            for (int k = 0; k < nb; ++k) t = __dadd_rn(t, sp[0][k][threadIdx.x]);
            const size_t o = (size_t)g * (NQ * 4) + d;
            part1[o] = t;
            for (int r = 0; r < n_peers; ++r) peers.p[r][o] = t;
            if constexpr (SQ) {
                double t2 = 0.0;
                for (int k = 0; k < nb; ++k) t2 = __dadd_rn(t2, sp[1][k][threadIdx.x]);
                const size_t o2 = o + (size_t)((nb0 + GB1 - 1) / GB1) * (NQ * 4);      // + nb1 * DP: the second table
                part1[o2] = t2;
                for (int r = 0; r < n_peers; ++r) peers.p[r][o2] = t2;
            }
        }
        if (n_peers > 0) __threadfence_system();                   // the rows before this CTA's arrival below
    }
    // sharded over ranks: the last CTA of the launch runs the flag barrier, so the launch's completion publishes every rank's
    // rows (PeerSync, ses_common.cuh).  The arrival counter resets itself.
    if (sync.world > 1) {
        __shared__ int last_s;
        __syncthreads();
        if (threadIdx.x == 0) {
            __threadfence_system();
            last_s = atomicAdd(sync.done, 1) == sync.expected - 1;
            if (last_s) atomicExch(sync.done, 0);
        }
        __syncthreads();
        if (last_s && threadIdx.x < 32) { __threadfence(); peer_flag_barrier(sync, threadIdx.x); }
    }
}

// level 2 + scale + Adam with the dtypes numpy>=2 gives the reference (m, v float32 with separately
// rounded products, step float64, theta rounded once to float32).
__global__ void __launch_bounds__(256) k_grad_final_adam(const double *__restrict__ part1, int nb1, int DP, int D, float update_factor,
                                                         double a, float b1, float ob1, float b2, float ob2, float ep,
                                                         float *__restrict__ mu, float *__restrict__ m, float *__restrict__ v,
                                                         float *__restrict__ grad_out)
{
    const int d = blockIdx.x * blockDim.x + threadIdx.x;
    if (d >= D) return;
    double s = 0.0;
    for (int g = 0; g < nb1; ++g) s = __dadd_rn(s, part1[(size_t)g * DP + d]);
    const float gr = __fmul_rn((float)s, update_factor);        // offspring_strategies.py:413-414
    if (grad_out) grad_out[d] = gr;
    const float mn = __fadd_rn(__fmul_rn(b1, m[d]), __fmul_rn(ob1, gr));                 // optimizers.py:48-49
    const float vn = __fadd_rn(__fmul_rn(b2, v[d]), __fmul_rn(ob2, __fmul_rn(gr, gr)));  // optimizers.py:50-53
    m[d] = mn;
    v[d] = vn;
    const double step = __ddiv_rn(__dmul_rn(-a, (double)mn), (double)__fadd_rn(__fsqrt_rn(vn), ep));  // :56
    mu[d] = (float)__dadd_rn((double)mu[d], step);              // optimizers.py:22-24
}

// level 2 + scale + SGD with momentum.  optimizers.py has Adam only; its header names OpenAI's es_distributed/optimizers.py
// as the source, whose SGD is  v = momentum * v + (1 - momentum) * g;  step = -stepsize * v.  With the reference's
// list-of-float32-arrays idiom under numpy >= 2 every operand is float32 (Python floats are weak scalars): four
// separately rounded float32 operations and a float32 `theta += step`.  Opt-in (engine.optimizer: sgd).
__global__ void __launch_bounds__(256) k_grad_final_sgd(const double *__restrict__ part1, int nb1, int DP, int D, float update_factor,
                                                        float neg_stepsize, float mom, float omm, float *__restrict__ mu,
                                                        float *__restrict__ v, float *__restrict__ grad_out)
{
    const int d = blockIdx.x * blockDim.x + threadIdx.x;
    if (d >= D) return;
    double s = 0.0;
    for (int g = 0; g < nb1; ++g) s = __dadd_rn(s, part1[(size_t)g * DP + d]);
    const float gr = __fmul_rn((float)s, update_factor);
    if (grad_out) grad_out[d] = gr;
    const float vn = __fadd_rn(__fmul_rn(mom, v[d]), __fmul_rn(omm, gr));
    v[d] = vn;
    mu[d] = __fadd_rn(mu[d], __fmul_rn(neg_stepsize, vn));
}

// weights of selected offspring: out[j][D] = parent(ids[j]) + sigma * eps(gen, ids[j])
__global__ void __launch_bounds__(256) k_materialize(const float *__restrict__ parents, const float *__restrict__ w_override,
                                                     Shard shard, int D, int NQ, float sigma, uint32_t seed, uint32_t gen,
                                                     Layout layout, const int *__restrict__ ids, int n, float *__restrict__ out)
{
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n * NQ) return;
    const int j = t / NQ, q = t - j * NQ;
    const int id = ids[j];
    float4 w;
    if (w_override) {
        const float *row = w_override + (size_t)shard.id_to_local(id) * D;
        const int d = 4 * q;
        w.x = d + 0 < D ? row[d + 0] : 0.0f;
        w.y = d + 1 < D ? row[d + 1] : 0.0f;
        w.z = d + 2 < D ? row[d + 2] : 0.0f;
        w.w = d + 3 < D ? row[d + 3] : 0.0f;
    } else {
        { float sg; const uint32_t nid = layout.noise_id(id, sg);
              w = offspring_quad(parents + (size_t)layout.parent(id) * D, D, q, layout.perturbed(id), __fmul_rn(sigma, sg), seed, nid, gen); }
    }
    float *o = out + (size_t)j * D + 4 * q;
    const int d = 4 * q;
    if (d + 0 < D) o[0] = w.x;
    if (d + 1 < D) o[1] = w.y;
    if (d + 2 < D) o[2] = w.z;
    if (d + 3 < D) o[3] = w.w;
}

// simple_evolution: float32 running sum of the k best in rank order, then / k
__global__ void __launch_bounds__(64) k_elite_mean(const float *__restrict__ parents, const float *__restrict__ w_override, Shard shard,
                                                   int D, int NQ, float sigma, uint32_t seed, uint32_t gen, Layout layout,
                                                   const int *__restrict__ order, int k, float *__restrict__ mu_out)
{
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= NQ) return;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int e = 0; e < k; ++e) {
        const int id = order[e];
        float4 w;
        if (w_override) {
            const float *row = w_override + (size_t)shard.id_to_local(id) * D;
            const int d = 4 * q;
            w.x = d + 0 < D ? row[d + 0] : 0.0f;
            w.y = d + 1 < D ? row[d + 1] : 0.0f;
            w.z = d + 2 < D ? row[d + 2] : 0.0f;
            w.w = d + 3 < D ? row[d + 3] : 0.0f;
        } else {
            { float sg; const uint32_t nid = layout.noise_id(id, sg);
              w = offspring_quad(parents + (size_t)layout.parent(id) * D, D, q, layout.perturbed(id), __fmul_rn(sigma, sg), seed, nid, gen); }
        }
        if (e == 0) acc = w;
        else {
            acc.x = __fadd_rn(acc.x, w.x); acc.y = __fadd_rn(acc.y, w.y);
            acc.z = __fadd_rn(acc.z, w.z); acc.w = __fadd_rn(acc.w, w.w);
        }
    }
    const float kf = (float)k;
    const int d = 4 * q;
    if (d + 0 < D) mu_out[d + 0] = __fdiv_rn(acc.x, kf);
    if (d + 1 < D) mu_out[d + 1] = __fdiv_rn(acc.y, kf);
    if (d + 2 < D) mu_out[d + 2] = __fdiv_rn(acc.z, kf);
    if (d + 3 < D) mu_out[d + 3] = __fdiv_rn(acc.w, kf);
}

}  // namespace ses

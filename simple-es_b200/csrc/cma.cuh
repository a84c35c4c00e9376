// cma.cuh -- separable CMA-ES (sep_cma_es, DESIGN.md section 4.11): the kernels on each side of K1.
//
//   k_cma_sample  : offspring weights x_j = m + sigma * (sqrt(c) * z_j), the table K1 rolls out as w_override
//   k_cma_weights : recombination weight of every offspring id from K2's order
//   k_cma_final   : level 2 of the two tables of k_grad_partial<true>, then the update of m, c, p_sigma, p_c and sigma
//
// Every quantity is float64 with each operation separately rounded (sigma also goes through the device exp), so every rank
// of a multi-GPU run computes the same state and a numpy restatement (tests/cma_reference.py) reproduces it.
#pragma once
#include "ses_common.cuh"

namespace ses {

constexpr int CMA_THREADS = 256;          // k_cma_final: one CTA; the norm of p_sigma is reduced by a tree over these threads

struct CmaParams {                        // the host constants of ses_cma_params (include/ses_b200.h)
    double one_m_cs, k_sigma, one_m_cc, k_c, cc2, c_keep, c1, cmu, damp, chi;
};

// thread <-> (local index l, parameter quad q): out[l][4q .. 4q+3] for the id this handle's slice holds at l
__global__ void __launch_bounds__(256) k_cma_sample(const double *__restrict__ mean, const double *__restrict__ c,
                                                    const double *__restrict__ sigma, Shard shard, int D, int NQ, uint32_t seed,
                                                    uint32_t gen, float *__restrict__ out)
{
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (long long)shard.n_local * NQ) return;
    const int l = (int)(t / NQ), q = (int)(t - (long long)l * NQ);
    const float4 z = normal4(seed, (uint32_t)q, (uint32_t)shard.local_to_id(l), gen);
    const double s = *sigma;
    const float zz[4] = {z.x, z.y, z.z, z.w};
    float *o = out + (size_t)l * D;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int d = 4 * q + k;
        if (d < D) o[d] = (float)__dadd_rn(mean[d], __dmul_rn(s, __dmul_rn(__dsqrt_rn(c[d]), (double)zz[k])));
    }
}

// s[order[r]] = w[r] for r < mu, 0 otherwise
__global__ void __launch_bounds__(256) k_cma_weights(const int *__restrict__ order, const double *__restrict__ w, int mu, int P,
                                                     double *__restrict__ s)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r < P) s[order[r]] = r < mu ? w[r] : 0.0;
}

// One CTA.  part1 [nb1][DP] holds sum_j s_j z_jd per group, part1 + nb1 * DP the same for z_jd^2; level 2 adds the groups in
// order.  Pass 1 updates p_sigma and its squared norm (per thread sequential over d = t, t + T, ..., then a halving tree over
// the T threads); pass 2 updates m, p_c and c with the old sigma and the old c; thread 0 writes the new sigma last (every
// thread has read the old one before the tree's first barrier).
__global__ void __launch_bounds__(CMA_THREADS) k_cma_final(const double *__restrict__ part1, int nb1, int DP, int D, CmaParams pr,
                                                           double threshold, double *__restrict__ mean, double *__restrict__ c,
                                                           double *__restrict__ ps, double *__restrict__ pc, double *__restrict__ sigma,
                                                           float *__restrict__ parent)
{
    __shared__ double red[CMA_THREADS];
    const int t = threadIdx.x;
    const double *part2 = part1 + (size_t)nb1 * DP;
    const double sig = *sigma;
    double nrm = 0.0;
    for (int d = t; d < D; d += CMA_THREADS) {
        double zm = 0.0;
        for (int g = 0; g < nb1; ++g) zm = __dadd_rn(zm, part1[(size_t)g * DP + d]);
        const double p = __dadd_rn(__dmul_rn(pr.one_m_cs, ps[d]), __dmul_rn(pr.k_sigma, zm));
        ps[d] = p;
        nrm = __dadd_rn(nrm, __dmul_rn(p, p));
    }
    red[t] = nrm;
    __syncthreads();
    for (int h = CMA_THREADS / 2; h > 0; h >>= 1) {
        if (t < h) red[t] = __dadd_rn(red[t], red[t + h]);
        __syncthreads();
    }
    const double norm = __dsqrt_rn(red[0]);
    const bool hs = norm < threshold;
    for (int d = t; d < D; d += CMA_THREADS) {
        double zm = 0.0, Q = 0.0;
        for (int g = 0; g < nb1; ++g) {
            zm = __dadd_rn(zm, part1[(size_t)g * DP + d]);
            Q = __dadd_rn(Q, part2[(size_t)g * DP + d]);
        }
        const double cd = c[d];
        const double y = __dmul_rn(__dsqrt_rn(cd), zm);
        const double m = __dadd_rn(mean[d], __dmul_rn(sig, y));
        mean[d] = m;
        parent[d] = (float)m;
        const double p = __dadd_rn(__dmul_rn(pr.one_m_cc, pc[d]), __dmul_rn(hs ? pr.k_c : 0.0, y));
        pc[d] = p;
        const double r1 = __dadd_rn(__dmul_rn(p, p), __dmul_rn(hs ? 0.0 : pr.cc2, cd));
        c[d] = __dadd_rn(__dadd_rn(__dmul_rn(pr.c_keep, cd), __dmul_rn(pr.c1, r1)), __dmul_rn(__dmul_rn(pr.cmu, cd), Q));
    }
    if (t == 0) *sigma = __dmul_rn(sig, exp(__dmul_rn(pr.damp, __dsub_rn(__ddiv_rn(norm, pr.chi), 1.0))));
}

}  // namespace ses

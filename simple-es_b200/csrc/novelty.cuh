// novelty.cuh -- novelty search with reward (nsr_es, DESIGN.md section 4.10): behaviour characterisations, k-nearest-neighbour
// novelty against the archive, and the blend of the fitness and novelty shapings.
//
// Every result is defined bit for bit (float64, each operation separately rounded, sums in a fixed order), so that every rank
// of a multi-GPU run computes the same vector and a numpy restatement reproduces it.
#pragma once
#include "ses_common.cuh"

namespace ses {

constexpr int NOVELTY_MAX_K = 32;
constexpr int NOVELTY_THREADS = 64;       // one offspring per thread; small blocks so that P = 16384 still spreads over every SM
constexpr int NOVELTY_TILE = 256;         // archive rows staged in shared memory per pass

// bc[i][d] = (sum over e, in episode order, of final[i][e][d]) / E
__global__ void k_behavior(const double *final_states, int n, int E, int sd, double *bc)
{
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (size_t)n * sd) return;
    const size_t i = t / sd;
    const int d = (int)(t - i * sd);
    const double *f = final_states + i * E * sd + d;
    double s = f[0];
    for (int e = 1; e < E; ++e) s = __dadd_rn(s, f[(size_t)e * sd]);
    bc[t] = __ddiv_rn(s, (double)E);
}

// novelty[i] = mean of the Euclidean distances from bc[i] to its min(k, n_archive) nearest archive rows, summed in ascending
// order.  The list keeps SQUARED distances (the square root is monotone, so the k smallest squares are the squares of the k
// smallest distances) and takes the root of the k survivors only.  KC >= k: the list's capacity, a compile-time size so that
// it lives in registers.  Entries k .. KC-1 hold -inf, which no candidate beats, so the list keeps exactly k entries and the
// k-th smallest so far is the list's maximum: found without indexing the list by k, which would move it to local memory.
// SD: state_dim (2, 4, 8 or 12), a compile-time size so that a candidate costs SD difference-square-adds and nothing more.
template <int SD, int KC>
__global__ void __launch_bounds__(NOVELTY_THREADS) k_novelty(const double *bc, int n, const double *archive, int n_archive, int k,
                                                             double *novelty)
{
    __shared__ double tile[NOVELTY_TILE * SD];
    const int i = blockIdx.x * NOVELTY_THREADS + threadIdx.x;
    const bool live = i < n;
    double b[SD];
#pragma unroll
    for (int d = 0; d < SD; ++d) b[d] = live ? bc[(size_t)i * SD + d] : 0.0;
    const double inf = __longlong_as_double(0x7ff0000000000000ll);
    double best[KC];
#pragma unroll
    for (int j = 0; j < KC; ++j) best[j] = j < k ? inf : -inf;
    double thr = inf;                                         // the k-th smallest so far: a candidate must beat it
    for (int a0 = 0; a0 < n_archive; a0 += NOVELTY_TILE) {
        const int rows = min(NOVELTY_TILE, n_archive - a0);
        __syncthreads();
        for (int t = threadIdx.x; t < rows * SD; t += NOVELTY_THREADS) tile[t] = archive[(size_t)a0 * SD + t];
        __syncthreads();
        if (!live) continue;
        for (int r = 0; r < rows; ++r) {
            const double *a = tile + r * SD;
            double q = 0.0;
#pragma unroll
            for (int d = 0; d < SD; ++d) {
                const double diff = __dsub_rn(b[d], a[d]);
                q = __dadd_rn(q, __dmul_rn(diff, diff));
            }
            if (q < thr) {                                    // insert into the ascending list
#pragma unroll
                for (int j = 0; j < KC; ++j) {
                    if (q < best[j]) { const double o = best[j]; best[j] = q; q = o; }
                }
                thr = -inf;
#pragma unroll
                for (int j = 0; j < KC; ++j) thr = fmax(thr, best[j]);
            }
        }
    }
    if (!live) return;
    const int m = min(k, n_archive);
    double s = 0.0;
#pragma unroll
    for (int j = 0; j < KC; ++j) if (j < m) s = __dadd_rn(s, __dsqrt_rn(best[j]));
    novelty[i] = __ddiv_rn(s, (double)m);
}

// out[i] = (1 - w) shaped_f[i] + w shaped_n[i], each operation rounded separately: w = 0 gives shaped_f exactly
__global__ void k_blend_shaped(const double *shaped_f, const double *shaped_n, int n, double w, double *out)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    out[i] = __dadd_rn(__dmul_rn(__dsub_rn(1.0, w), shaped_f[i]), __dmul_rn(w, shaped_n[i]));
}

}  // namespace ses

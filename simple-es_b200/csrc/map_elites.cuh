// map_elites.cuh -- MAP-Elites (map_elites, DESIGN.md section 4.12): a grid archive of elite policies, one per behaviour cell.
//
//   k_map_claim   : every placed offspring offers the key P - rank to its cell (atomicMax: the best-ranked offspring wins)
//   k_map_commit  : each cell's winner enters iff the cell is empty or its fitness beats the incumbent's; resets the claims
//   k_map_weights : the weights of every offspring that entered, regenerated from the parent table as K1 rolled them out
//   k_map_compact : one CTA: the occupied cells in ascending index, their count, the best cell and the QD score
//   k_map_gather  : parent row i := the elite of the occupied cell that Philox draw i picks (or the seed row while empty)
//
// Every result is defined bit for bit (float64 cell map with each operation separately rounded, a fixed summation order for
// the QD score, integer keys for the claims), so every rank of a multi-GPU run holds the same archive and a numpy restatement
// (tests/map_elites_reference.py) reproduces it.
#pragma once
#include "ses_common.cuh"

namespace ses {

constexpr int MAP_MAX_DIMS = 4;
constexpr int MAP_COMPACT_THREADS = 1024;   // k_map_compact: one CTA; thread t sums the QD score over the cells c = t (mod 1024)

struct MapSpec {                            // ses_map_spec (include/ses_b200.h), checked by the host
    int n_dims;
    int dims[MAP_MAX_DIMS];
    double low[MAP_MAX_DIMS], width[MAP_MAX_DIMS];
    int cells[MAP_MAX_DIMS];
};

// Cell of the behaviour row b, row-major over the descriptor dimensions; -1 (unplaced) if a descriptor coordinate is NaN.
// The edge tests run in double before the conversion, so +-inf and out-of-range values land in the edge cells.
__device__ __forceinline__ int map_cell(const double *b, const MapSpec &s)
{
    int c = 0;
#pragma unroll
    for (int j = 0; j < MAP_MAX_DIMS; ++j) {          // unrolled: the spec stays in parameter space, not in a local copy
        if (j >= s.n_dims) break;
        const double x = b[s.dims[j]];
        if (x != x) return -1;
        const double sc = __dmul_rn(__ddiv_rn(__dsub_rn(x, s.low[j]), s.width[j]), (double)s.cells[j]);
        const int k = sc < 1.0 ? 0 : (sc >= (double)(s.cells[j] - 1) ? s.cells[j] - 1 : (int)sc);
        c = c * s.cells[j] + k;
    }
    return c;
}

// cell of offspring i, or -1 when its fitness or a descriptor coordinate is NaN
__device__ __forceinline__ int map_placed_cell(const double *fitness, const double *bc, int sd, const MapSpec &s, int i)
{
    const double f = fitness[i];
    return f != f ? -1 : map_cell(bc + (size_t)i * sd, s);
}

// thread r: offspring order[r] offers P - r to its cell; claim[] is all zero before the launch (k_map_commit restores that)
__global__ void __launch_bounds__(256) k_map_claim(const int *__restrict__ order, const double *__restrict__ fitness,
                                                   const double *__restrict__ bc, int P, int sd, MapSpec s, int *claim)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= P) return;
    const int c = map_placed_cell(fitness, bc, sd, s, order[r]);
    if (c >= 0) atomicMax(claim + c, P - r);
}

// thread r: if offspring i = order[r] won its cell's claim, reset the claim and enter iff the cell is empty (F NaN) or
// fitness_i > F (strict: a tie keeps the incumbent).  enter[r] := the cell it entered, or -1.  A loser reads the winner's key
// or the 0 the winner wrote back; it matches neither.
__global__ void __launch_bounds__(256) k_map_commit(const int *__restrict__ order, const double *__restrict__ fitness,
                                                    const double *__restrict__ bc, int P, int sd, MapSpec s, int *claim, uint32_t gen,
                                                    double *__restrict__ F, double *__restrict__ B, int *__restrict__ born,
                                                    int *__restrict__ enter)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= P) return;
    const int i = order[r];
    const int c = map_placed_cell(fitness, bc, sd, s, i);
    int entered = -1;
    if (c >= 0 && claim[c] == P - r) {
        claim[c] = 0;
        const double f = fitness[i], old = F[c];
        if (old != old || f > old) {
            F[c] = f;
            for (int d = 0; d < sd; ++d) B[(size_t)c * sd + d] = bc[(size_t)i * sd + d];
            born[2 * c] = (int)gen;
            born[2 * c + 1] = i;
            entered = c;
        }
    }
    enter[r] = entered;
}

// block r: W[enter[r]] := the weights offspring order[r] had in generation gen -- offspring_quad of its parent row, exactly
// what K1 and k_materialize compute
__global__ void __launch_bounds__(128) k_map_weights(const float *__restrict__ parents, const int *__restrict__ order,
                                                     const int *__restrict__ enter, int D, int NQ, float sigma, uint32_t seed,
                                                     uint32_t gen, Layout layout, float *__restrict__ W)
{
    const int c = enter[blockIdx.x];
    if (c < 0) return;
    const int id = order[blockIdx.x];
    float sg;
    const uint32_t nid = layout.noise_id(id, sg);
    const float *prow = parents + (size_t)layout.parent(id) * D;
    float *o = W + (size_t)c * D;
    for (int q = threadIdx.x; q < NQ; q += blockDim.x) {
        const float4 w = offspring_quad(prow, D, q, layout.perturbed(id), __fmul_rn(sigma, sg), seed, nid, gen);
        const int d = 4 * q;
        if (d + 0 < D) o[d + 0] = w.x;
        if (d + 1 < D) o[d + 1] = w.y;
        if (d + 2 < D) o[d + 2] = w.z;
        if (d + 3 < D) o[d + 3] = w.w;
    }
}

// One CTA of MAP_COMPACT_THREADS.  list[0 .. n_occ) := the occupied cells (F not NaN) in ascending index.
// stats[0] = n_occ, stats[1] = c* (the largest F, ties to the lowest index; -1 while empty), stats[2] = F[c*] (NaN while
// empty), stats[3] = the QD score: thread t adds F[c] over the occupied c = t (mod 1024) in ascending c from +0.0, then a
// halving tree red[t] += red[t + h], h = 512, 256, ..., 1.
__global__ void __launch_bounds__(MAP_COMPACT_THREADS) k_map_compact(const double *__restrict__ F, int n_cells, int *__restrict__ list,
                                                                     double *__restrict__ stats)
{
    __shared__ int warp_n[MAP_COMPACT_THREADS / 32];
    __shared__ double red_q[MAP_COMPACT_THREADS], red_f[MAP_COMPACT_THREADS];
    __shared__ int red_c[MAP_COMPACT_THREADS];
    const double nan = __longlong_as_double(0x7ff8000000000000ll);
    const int t = threadIdx.x, lane = t & 31, w = t >> 5;
    int base = 0, bc = -1;
    double qd = 0.0, bf = nan;
    for (int c0 = 0; c0 < n_cells; c0 += MAP_COMPACT_THREADS) {
        const int c = c0 + t;
        const double f = c < n_cells ? F[c] : nan;
        const bool occ = f == f;
        if (occ) {
            qd = __dadd_rn(qd, f);
            if (bc < 0 || f > bf) { bf = f; bc = c; }
        }
        const unsigned m = __ballot_sync(0xffffffffu, occ);
        if (lane == 0) warp_n[w] = __popc(m);
        __syncthreads();
        int off = base, total = 0;
        for (int k = 0; k < MAP_COMPACT_THREADS / 32; ++k) {
            off += k < w ? warp_n[k] : 0;
            total += warp_n[k];
        }
        if (occ) list[off + __popc(m & lanemask_lt())] = c;
        base += total;
        __syncthreads();
    }
    red_q[t] = qd;
    red_f[t] = bf;
    red_c[t] = bc;
    __syncthreads();
    for (int h = MAP_COMPACT_THREADS / 2; h > 0; h >>= 1) {
        if (t < h) {
            red_q[t] = __dadd_rn(red_q[t], red_q[t + h]);
            const int ca = red_c[t], cb = red_c[t + h];
            const double fa = red_f[t], fb = red_f[t + h];
            if (cb >= 0 && (ca < 0 || fb > fa || (fb == fa && cb < ca))) { red_f[t] = fb; red_c[t] = cb; }
        }
        __syncthreads();
    }
    if (t == 0) {
        stats[0] = (double)base;
        stats[1] = (double)red_c[0];
        stats[2] = red_f[0];
        stats[3] = red_q[0];
    }
}

// block i: parent row i := W[list[(r_i * n_occ) >> 32]] with r_i = word 0 of Philox(i, gen, 0, 0; seed, STREAM_SELECT), or
// seed_row while the archive is empty (stats[0] = n_occ from k_map_compact)
__global__ void __launch_bounds__(256) k_map_gather(const float *__restrict__ W, const int *__restrict__ list, const double *__restrict__ stats,
                                                    const float *__restrict__ seed_row, int D, uint32_t seed, uint32_t gen,
                                                    float *__restrict__ parents)
{
    const unsigned long long n_occ = (unsigned long long)stats[0];
    const float *src = seed_row;
    if (n_occ > 0) {
        const unsigned long long r = philox4x32_10((uint32_t)blockIdx.x, gen, 0u, 0u, seed, STREAM_SELECT).x;
        src = W + (size_t)list[(r * n_occ) >> 32] * D;
    }
    float *dst = parents + (size_t)blockIdx.x * D;
    for (int d = threadIdx.x; d < D; d += blockDim.x) dst[d] = src[d];
}

}  // namespace ses

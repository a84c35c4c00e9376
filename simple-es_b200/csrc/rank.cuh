// rank.cuh -- K2: descending rank of the fitness vector, centered-rank shaping.
//
// Replaces np.flip(np.argsort(np.array(rewards))) (offspring_strategies.py:112,234,380) and the
// centered-rank loop + standardisation (offspring_strategies.py:392-398).
//
// Tie order is pinned (SURVEY.md quirk Q6): descending fitness, ties by DESCENDING index, which
// equals np.flip(np.argsort(r, kind="stable")).  Implementation: the input is presented in
// reverse index order with keys that ascend when fitness descends, then sorted with a STABLE
// least-significant-digit radix sort (8-bit digits; 8 passes for a full float64 key, ceil((k+1)/8)
// when the caller bounds fitness*scale to an integer of magnitude < 2^k, e.g. CartPole's step totals or the
// negative step totals of MountainCar / Acrobot).
// HBM-trivial (<= 12 MB at P = 2^20); what matters is launch count and stability.
#pragma once
#include "ses_common.cuh"

namespace ses {

constexpr int SORT_THREADS = 256;
constexpr int SORT_WARPS = SORT_THREADS / 32;
// keys per thread: 4 (1024-key tiles, more CTAs in flight) up to 2^18 keys, 16 (4096-key tiles, fewer per-tile
// histograms to walk) above
constexpr int SORT_ITEMS_SMALL = 4, SORT_ITEMS_LARGE = 16;
__host__ __device__ constexpr int sort_tile(int items) { return SORT_THREADS * items; }

// Every NaN, whatever its sign and payload, is keyed as +qNaN: above +inf, ties by descending index, as numpy ranks NaNs
// (np.argsort puts them last).  The bit transform alone would send a NaN with the sign bit set to the bottom.
constexpr unsigned long long SORT_KEY_NAN = 0x7ff8000000000000ull;

// position p holds offspring i = n-1-p; key ascends when fitness descends
__global__ void k_sort_init(const double *__restrict__ fitness, int n, int key_bits, double key_scale,
                            unsigned long long *__restrict__ keys, int *__restrict__ vals)
{
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    const int i = n - 1 - p;
    const double f = __dadd_rn(fitness[i], 0.0);   // -0.0 -> +0.0: numpy compares them equal
    unsigned long long k;
    if (key_bits == 0) {
        const unsigned long long b = isnan(f) ? SORT_KEY_NAN : (unsigned long long)__double_as_longlong(f);
        const unsigned long long asc = (b >> 63) ? ~b : (b | 0x8000000000000000ull);
        k = ~asc;
    } else {
        // integer key in (-2^key_bits, 2^key_bits), biased to [1, 2^(key_bits+1)); never NaN: the host picks this path
        // only for the step-count envs, whose fitness is a step total over E
        const long long v = __double2ll_rn(__dmul_rn(f, key_scale)) + (1ll << key_bits);
        k = ((2ull << key_bits) - 1ull) - (unsigned long long)v;
    }
    keys[p] = k;
    vals[p] = i;
}

// per-CTA digit histogram -> hist[cta][256]; digit totals -> tot[256] (zeroed by the host)
template <int SORT_ITEMS>
__global__ void __launch_bounds__(SORT_THREADS) k_sort_hist(const unsigned long long *__restrict__ keys, int n, int shift,
                                                            int *__restrict__ hist, int *__restrict__ tot)
{
    constexpr int SORT_TILE = SORT_THREADS * SORT_ITEMS;
    __shared__ int h[256];
    h[threadIdx.x] = 0;
    __syncthreads();
    const int base = blockIdx.x * SORT_TILE;
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int it = 0; it < SORT_ITEMS; ++it) {
        const int p = base + it * SORT_THREADS + threadIdx.x;
        // warp-aggregated: a converged CartPole population puts every key in one bin
        const int d = p < n ? (int)((keys[p] >> shift) & 255ull) : 256 + lane;
        const unsigned peers = __match_any_sync(0xffffffffu, d);
        if (p < n && lane == __ffs(peers) - 1) atomicAdd(&h[d], __popc(peers));
    }
    __syncthreads();
    const int c = h[threadIdx.x];
    hist[blockIdx.x * 256 + threadIdx.x] = c;
    if (c) atomicAdd(&tot[threadIdx.x], c);
}

// stable scatter of one tile: CTA c owns keys [c*TILE, ...), warp w the 32*ITEMS consecutive keys
// [c*TILE + w*32*ITEMS, ...) in ITEMS chunks of 32 (so "earlier position" == lower (warp, chunk, lane)).
template <int SORT_ITEMS>
__global__ void __launch_bounds__(SORT_THREADS) k_sort_scatter(const unsigned long long *__restrict__ keys_in,
                                                               const int *__restrict__ vals_in, int n, int shift,
                                                               const int *__restrict__ hist, const int *__restrict__ tot,
                                                               unsigned long long *__restrict__ keys_out,
                                                               int *__restrict__ vals_out)
{
    constexpr int SORT_TILE = SORT_THREADS * SORT_ITEMS, SORT_WSEG = 32 * SORT_ITEMS;
    __shared__ int digit_base[256];
    __shared__ int whist[SORT_WARPS][256];
    __shared__ int scan_tmp[256];
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const unsigned FULL = 0xffffffffu;
    const unsigned lt = lanemask_lt();

    // (a) global base of digit d for this CTA: sum_{d'<d} tot[d'] + sum_{c<cta} hist[c][d]
    {
        const int t = tot[tid];
        scan_tmp[tid] = t;
        __syncthreads();
        for (int off = 1; off < 256; off <<= 1) {             // Hillis-Steele inclusive scan
            int v = tid >= off ? scan_tmp[tid - off] : 0;
            __syncthreads();
            scan_tmp[tid] += v;
            __syncthreads();
        }
        int b = scan_tmp[tid] - t;
        for (int c = 0; c < (int)blockIdx.x; ++c) b += hist[c * 256 + tid];
        digit_base[tid] = b;
    }
    for (int i = tid; i < SORT_WARPS * 256; i += SORT_THREADS) (&whist[0][0])[i] = 0;
    __syncthreads();

    // (b) load this warp's segment, count digits
    unsigned long long key[SORT_ITEMS];
    int val[SORT_ITEMS];
    const int seg = blockIdx.x * SORT_TILE + w * SORT_WSEG;
#pragma unroll
    for (int it = 0; it < SORT_ITEMS; ++it) {
        const int p = seg + it * 32 + lane;
        const bool ok = p < n;
        key[it] = ok ? keys_in[p] : 0ull;
        val[it] = ok ? vals_in[p] : -1;
        const int d = ok ? (int)((key[it] >> shift) & 255ull) : (256 + lane);
        const unsigned peers = __match_any_sync(FULL, d);
        if (ok && lane == __ffs(peers) - 1) whist[w][d] += __popc(peers);
        __syncwarp();
    }
    __syncthreads();
    // (c) exclusive scan over warps per digit, seeded with the digit's global base
    {
        int run = digit_base[tid];
#pragma unroll
        for (int ww = 0; ww < SORT_WARPS; ++ww) {
            const int t = whist[ww][tid];
            whist[ww][tid] = run;
            run += t;
        }
    }
    __syncthreads();
    // (d) second walk: stable positions
#pragma unroll
    for (int it = 0; it < SORT_ITEMS; ++it) {
        const bool ok = val[it] >= 0;
        const int d = ok ? (int)((key[it] >> shift) & 255ull) : (256 + lane);
        const unsigned peers = __match_any_sync(FULL, d);
        const int leader = __ffs(peers) - 1;
        int b = 0;
        if (ok && lane == leader) { b = whist[w][d]; whist[w][d] = b + __popc(peers); }
        b = __shfl_sync(FULL, b, leader);
        if (ok) {
            const int pos = b + __popc(peers & lt);
            keys_out[pos] = key[it];
            vals_out[pos] = val[it];
        }
        __syncwarp();
    }
}

// ---------------------------------------------------------------------------------------------
// Fused variant (SES_K2_FUSED, DESIGN.md section 5.4): the same stable LSD sort with the launch count cut from
// 2 + 2*passes to 1 + passes (integer keys: 3 kernels instead of 6; float64 keys: 9 instead of 18).  K2 is latency
// bound -- every kernel is a few microseconds of work -- so launches are what it costs.
//   * sort_key(): the key of position p straight from the fitness vector (k_sort_init fused into the first histogram
//     and the first scatter: the initial (key, index) arrays are never written);
//   * every scatter pass also builds the NEXT pass's per-tile digit histograms and digit totals, keyed by the tile the
//     key lands in (warp-aggregated global atomics), so only pass 0 needs a histogram kernel;
//   * the last scatter writes the centered rank of each offspring from its final position (k_shape_centered fused).
// Positions, stability argument and the resulting permutation are exactly those of the unfused kernels above.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long sort_key(const double *__restrict__ fitness, int n, int p, int key_bits, double key_scale)
{
    const double f = __dadd_rn(fitness[n - 1 - p], 0.0);   // position p holds offspring n-1-p; -0.0 -> +0.0
    if (key_bits == 0) {
        const unsigned long long b = isnan(f) ? SORT_KEY_NAN : (unsigned long long)__double_as_longlong(f);
        const unsigned long long asc = (b >> 63) ? ~b : (b | 0x8000000000000000ull);
        return ~asc;
    }
    // integer keys: never NaN (step-count envs only, see k_sort_init)
    const long long v = __double2ll_rn(__dmul_rn(f, key_scale)) + (1ll << key_bits);
    return ((2ull << key_bits) - 1ull) - (unsigned long long)v;
}

// inclusive prefix sum over the 256 threads of a sort CTA: warp shuffles + one pass over the 8 warp totals (two barriers instead
// of the sixteen of a shared-memory Hillis-Steele scan); tmp: >= SORT_WARPS ints of shared memory
__device__ __forceinline__ int sort_scan256(int v, int *tmp)
{
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    int x = v;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const int y = __shfl_up_sync(0xffffffffu, x, off);
        if (lane >= off) x += y;
    }
    __syncthreads();                                               // tmp may still be read by a previous use
    if (lane == 31) tmp[w] = x;
    __syncthreads();
    int add = 0;
#pragma unroll
    for (int ww = 0; ww < SORT_WARPS; ++ww) add += ww < w ? tmp[ww] : 0;
    return x + add;
}

// pass-0 histogram straight from the fitness vector (one tile = one CTA)
template <int SORT_ITEMS>
__device__ __forceinline__ void sort_hist_first_tile(const double *__restrict__ fitness, int n, int key_bits, double key_scale, int *hist)
{
    constexpr int SORT_TILE = SORT_THREADS * SORT_ITEMS;
    __shared__ int h[256];
    h[threadIdx.x] = 0;
    __syncthreads();
    const int base = blockIdx.x * SORT_TILE;
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int it = 0; it < SORT_ITEMS; ++it) {
        const int p = base + it * SORT_THREADS + threadIdx.x;
        const int d = p < n ? (int)(sort_key(fitness, n, p, key_bits, key_scale) & 255ull) : 256 + lane;
        const unsigned peers = __match_any_sync(0xffffffffu, d);
        if (p < n && lane == __ffs(peers) - 1) atomicAdd(&h[d], __popc(peers));
    }
    __syncthreads();
    hist[blockIdx.x * 256 + threadIdx.x] = h[threadIdx.x];
}

template <int SORT_ITEMS>
__global__ void __launch_bounds__(SORT_THREADS) k_sort_hist_first(const double *__restrict__ fitness, int n, int key_bits, double key_scale,
                                                                  int *__restrict__ hist)
{
    sort_hist_first_tile<SORT_ITEMS>(fitness, n, key_bits, key_scale, hist);
}

// loads of data other CTAs of the SAME launch wrote (the persistent kernel below): L2 only, an SM's L1 may hold a stale line
template <bool COHERENT, class T>
__device__ __forceinline__ T sort_ld(const T *p) { if constexpr (COHERENT) return __ldcg(p); else return *p; }

// one stable scatter pass; `first`: keys come from the fitness vector; `last`: no next pass -- write the permutation
// (vals_out) and, if shaped != nullptr, the centered ranks; otherwise also accumulate hist_next (zeroed by the host) for
// the digit at shift + 8.  Digit totals are the column sums of the tile histograms (no separate table).
template <int SORT_ITEMS, bool COHERENT>
__device__ __forceinline__ void sort_scatter_fused_tile(const double *__restrict__ fitness, int key_bits, double key_scale,
                                                        const unsigned long long *keys_in, const int *vals_in, int n, int shift, int first, int last,
                                                        const int *hist, int *hist_next, unsigned long long *keys_out, int *vals_out,
                                                        double stdv, double *shaped)
{
    constexpr int SORT_TILE = SORT_THREADS * SORT_ITEMS, SORT_WSEG = 32 * SORT_ITEMS;
    __shared__ int digit_base[256];
    __shared__ int whist[SORT_WARPS][256];
    __shared__ int scan_tmp[256];
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const unsigned FULL = 0xffffffffu;
    const unsigned lt = lanemask_lt();

    {   // (a) global base of digit d for this CTA: sum_{d'<d} tot[d'] + sum_{c<cta} hist[c][d], tot[d] = sum_c hist[c][d]
        int t = 0, below = 0;
        for (int c = 0; c < (int)gridDim.x; ++c) {
            const int v = sort_ld<COHERENT>(hist + c * 256 + tid);
            t += v;
            if (c < (int)blockIdx.x) below += v;
        }
        digit_base[tid] = sort_scan256(t, scan_tmp) - t + below;
    }
    for (int i = tid; i < SORT_WARPS * 256; i += SORT_THREADS) (&whist[0][0])[i] = 0;
    __syncthreads();

    // (b) load this warp's segment, count digits
    unsigned long long key[SORT_ITEMS];
    int val[SORT_ITEMS];
    const int seg = blockIdx.x * SORT_TILE + w * SORT_WSEG;
#pragma unroll
    for (int it = 0; it < SORT_ITEMS; ++it) {
        const int p = seg + it * 32 + lane;
        const bool ok = p < n;
        if (first) {
            key[it] = ok ? sort_key(fitness, n, p, key_bits, key_scale) : 0ull;
            val[it] = ok ? n - 1 - p : -1;
        } else {
            key[it] = ok ? sort_ld<COHERENT>(keys_in + p) : 0ull;
            val[it] = ok ? sort_ld<COHERENT>(vals_in + p) : -1;
        }
        const int d = ok ? (int)((key[it] >> shift) & 255ull) : (256 + lane);
        const unsigned peers = __match_any_sync(FULL, d);
        if (ok && lane == __ffs(peers) - 1) whist[w][d] += __popc(peers);
        __syncwarp();
    }
    __syncthreads();
    {   // (c) exclusive scan over warps per digit, seeded with the digit's global base
        int run = digit_base[tid];
#pragma unroll
        for (int ww = 0; ww < SORT_WARPS; ++ww) {
            const int t = whist[ww][tid];
            whist[ww][tid] = run;
            run += t;
        }
    }
    __syncthreads();
    // (d) second walk: stable positions; next pass's histograms, or the final outputs
#pragma unroll
    for (int it = 0; it < SORT_ITEMS; ++it) {
        const bool ok = val[it] >= 0;
        const int d = ok ? (int)((key[it] >> shift) & 255ull) : (256 + lane);
        const unsigned peers = __match_any_sync(FULL, d);
        const int leader = __ffs(peers) - 1;
        int b = 0;
        if (ok && lane == leader) { b = whist[w][d]; whist[w][d] = b + __popc(peers); }
        b = __shfl_sync(FULL, b, leader);
        const int pos = b + __popc(peers & lt);
        if (ok) vals_out[pos] = val[it];
        if (!last) {
            if (ok) keys_out[pos] = key[it];
            // histogram of the next digit, per destination tile: one atomic per distinct (tile, digit) in the warp
            const int dn = (int)((key[it] >> (shift + 8)) & 255ull);
            const int bin = ok ? (pos / SORT_TILE) * 256 + dn : -1 - lane;
            const unsigned same = __match_any_sync(FULL, bin);
            if (ok && lane == __ffs(same) - 1) atomicAdd(&hist_next[bin], __popc(same));
        } else if (shaped && ok) {
            // centered rank of the offspring that ends at rank `pos` (k_shape_centered)
            const double v = __dsub_rn(__ddiv_rn((double)(n - 1 - pos), (double)(n - 1)), 0.5);
            shaped[val[it]] = __ddiv_rn(v, stdv);
        }
        __syncwarp();
    }
}

template <int SORT_ITEMS>
__global__ void __launch_bounds__(SORT_THREADS) k_sort_scatter_fused(const double *__restrict__ fitness, int key_bits, double key_scale,
                                                                     const unsigned long long *__restrict__ keys_in,
                                                                     const int *__restrict__ vals_in, int n, int shift, int first, int last,
                                                                     const int *__restrict__ hist, int *__restrict__ hist_next,
                                                                     unsigned long long *__restrict__ keys_out, int *__restrict__ vals_out,
                                                                     double stdv, double *__restrict__ shaped)
{
    sort_scatter_fused_tile<SORT_ITEMS, false>(fitness, key_bits, key_scale, keys_in, vals_in, n, shift, first, last, hist, hist_next, keys_out, vals_out,
                                               stdv, shaped);
}

// ---------------------------------------------------------------------------------------------
// Persistent variant: the whole sort in ONE cooperative launch.  Every CTA keeps its tile through the pass-0 histogram and all
// scatter passes; the launch boundaries of the fused build (each worth ~3.6 us of a kernel that does a few microseconds of
// work) become grid barriers (an arrival counter in global memory, zeroed with the histograms; all CTAs are co-resident:
// cudaLaunchCooperativeKernel refuses the launch otherwise and the caller falls back to the fused build).  Data written by
// other CTAs earlier in the launch is read through L2 (sort_ld<true>).  Same tile code, same positions, same permutation.
// Used for float64 keys (8 passes: 82 -> 64 us at P = 16384 with 512-key tiles); for integer keys (2 passes) the fused build is as fast.
// ---------------------------------------------------------------------------------------------
struct SortBuffers {
    unsigned long long *keys[2];
    int *vals[2];            // ping-pong, arranged by the host so that the last pass writes the caller's order array
};

__device__ __forceinline__ void sort_grid_barrier(unsigned *bar, unsigned target)
{
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        atomicAdd(bar, 1u);
        while (*reinterpret_cast<volatile unsigned *>(bar) < target) __nanosleep(64);
        __threadfence();
    }
    __syncthreads();
}

template <int SORT_ITEMS>
__global__ void __launch_bounds__(SORT_THREADS) k_sort_persistent(const double *__restrict__ fitness, int n, int key_bits, double key_scale, int passes,
                                                                  SortBuffers buf, int *hist_all, int per_pass, unsigned *bar, double stdv,
                                                                  double *shaped)
{
    sort_hist_first_tile<SORT_ITEMS>(fitness, n, key_bits, key_scale, hist_all);
    sort_grid_barrier(bar, gridDim.x);
    for (int ps = 0; ps < passes; ++ps) {
        const int a = ps & 1, b = a ^ 1, last = ps == passes - 1;
        sort_scatter_fused_tile<SORT_ITEMS, true>(fitness, key_bits, key_scale, buf.keys[a], buf.vals[a], n, 8 * ps, ps == 0, last, hist_all + (size_t)per_pass * ps,
                                                  last ? nullptr : hist_all + (size_t)per_pass * (ps + 1), buf.keys[b], buf.vals[b], stdv, shaped);
        if (!last) sort_grid_barrier(bar, (unsigned)(ps + 2) * gridDim.x);
    }
}

// centered ranks, standardised with the closed-form mean (0) and population std of the table
// {i/(P-1) - 0.5} (offspring_strategies.py:392-398; DESIGN.md section 4.5).
__global__ void k_shape_centered(const int *__restrict__ order, int n, double stdv, double *__restrict__ shaped)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    const double v = __dsub_rn(__ddiv_rn((double)(n - 1 - r), (double)(n - 1)), 0.5);
    shaped[order[r]] = __ddiv_rn(v, stdv);
}

}  // namespace ses

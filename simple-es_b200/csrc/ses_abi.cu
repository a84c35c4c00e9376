// ses_abi.cu -- the C ABI of include/ses_b200.h over the sm_100a kernels in this directory.
// Host side only does argument checking, scratch management and launches; there is no CPU
// implementation of any entry point (no fallback): without a device every call fails.
#include "../../include/ses_b200.h"
#ifdef SES_BUILD_TESTS
#include "../../include/ses_b200_test.h"
#endif

#include <cuda_runtime.h>

#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "cma.cuh"
#include "map_elites.cuh"
#include "novelty.cuh"
#include "rank.cuh"
#include "rollout_cartpole_mlp.cuh"
#include "rollout_cartpole_gru.cuh"
#include "rollout_mpe.cuh"
#include "rollout_classic.cuh"
#include "rollout_gru_generic.cuh"
#include "ses_common.cuh"
#include "update.cuh"

using namespace ses;

// ------------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";

static int fail(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return -1;
}

#define CU(call)                                                                                       \
    do {                                                                                               \
        cudaError_t e__ = (call);                                                                      \
        if (e__ != cudaSuccess) return fail("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); \
    } while (0)

extern "C" const char *ses_last_error(void) { return g_err; }
extern "C" int ses_abi_version(void) { return SES_ABI_VERSION; }
extern "C" int ses_param_count(int32_t obs, int32_t act, int32_t gru) { return param_count(obs, act, gru); }

// ------------------------------------------------------------------------------------------------
// handle
// ------------------------------------------------------------------------------------------------
struct ses_handle {
    ses_config cfg;
    int D, NQ, DP;
    Shard shard;
    int state_dim;
    int num_sms;
    int eff_max_step;
    // scratch (device)
    int *work_counter = nullptr;
    // episode-length estimate of the slot kernels' last launch (read back asynchronously; never waited for)
    unsigned long long *k1_steps_host = nullptr;   // pinned
    cudaEvent_t k1_ev = nullptr;
    bool k1_ev_pending = false;
    long long k1_last_episodes = 0;
    double k1_mean_len = -1.0;     // < 0: unknown
    int *ep_acc = nullptr;         // [n_local][2]: steps / episodes of offspring split over warps (rollout_slots.cuh retire_slot)
    unsigned long long *keys[2] = {nullptr, nullptr};
    int *vals_scratch = nullptr;
    int *hist = nullptr;
    int *tot = nullptr;            // [8][256]
    int *hist_fused = nullptr;     // fused K2: [passes][tiles][256] tile histograms, zeroed per call
    int k2_fused = 1;
    int k2_persistent = 1;         // the whole sort in one cooperative launch (falls back to the fused build if the launch is refused)
    double *part1 = nullptr;
    int nb0 = 0, nb1 = 0, n_tiles = 0;
    // scratch for the host-buffer generation path
    float *h_parents = nullptr, *h_m = nullptr, *h_v = nullptr;
    double *h_fitness = nullptr, *h_shaped = nullptr;
    long long *h_steps = nullptr;
    int *h_order = nullptr;
    unsigned long long *h_total = nullptr;
    // scratch of the elite strategies' host-buffer generations (ses_generation_evolution_host / _genetic_host)
    float *e_parents = nullptr, *e_out = nullptr;      // [n_parents][D] each
    double *e_fitness = nullptr;
    long long *e_steps = nullptr;
    int *e_order = nullptr;
    unsigned long long *e_total = nullptr;
    // peer (NVLink P2P) fitness exchange: [2][P] doubles (double buffered by generation parity) + flags
    double *xbuf = nullptr;
    double *peer_x[MAX_PEERS] = {nullptr};
    int peer_rank = 0, peer_world = 0;
    unsigned long long peer_epoch = 0;
    int *peer_error = nullptr;
    long long peer_timeout_cycles = 20000000000ll;
    double *last_rollout_fitness = nullptr;       // exchange buffer the last fused-exchange rollout wrote (poisoned on a barrier timeout)
    int *grad_done = nullptr;                     // arrival counter of k_grad_partial's CTAs (self-resetting)
    int k1_geometry[8] = {0};                     // the last slot-kernel launch (ses_test_k1_geometry)
    bool peer_fold = false;                       // test build, SES_PEER_FOLD=1: the barriers run inside K1 / k_grad_partial (PeerSync)
    bool barrier_folded = false;                  // that rollout's launch ended with the flag barrier: the next ses_peer_barrier() is a no-op
    unsigned long long *step_counter = nullptr;   // caller-owned, optional (ses_set_step_counter)
    double *final_states = nullptr;               // caller-owned, optional [P][E][state_dim] (ses_set_final_states)
    // rollout launch configuration
    int lanes_used_override = 0;
    int ctas_per_sm = 0;
    int k1_variant = 7;
    int spread_slots8 = 0;
    int k1_split = 1;
    int k1_sparse = 1;
    int *eval_counter = nullptr;   // work counter of ses_evaluate / ses_record launches (allocated by the first call)
    // map_elites scratch (allocated by the first ses_map_* call, grown with the cell count): per-cell claims (all zero between
    // calls: k_map_commit resets every claim it reads), the occupied-cell list, and the cell each rank entered
    int *map_claim = nullptr, *map_list = nullptr, *map_enter = nullptr;
    int map_cells = 0;

    int64_t launches = 0;
};

static cudaStream_t S(void *s) { return reinterpret_cast<cudaStream_t>(s); }

static int env_int(const char *name, int dflt)
{
    const char *v = getenv(name);
    return v && *v ? atoi(v) : dflt;
}

extern "C" int ses_create(const ses_config *cfg, ses_handle **out)
{
    if (!cfg || !out) return fail("ses_create: null argument");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail("ses_create: no CUDA device (%s); this engine has no CPU fallback", cudaGetErrorString(e));
    if (cfg->device < 0 || cfg->device >= ndev) return fail("ses_create: device %d out of range (%d devices)", cfg->device, ndev);
    if (cfg->env < SES_ENV_CARTPOLE || cfg->env > SES_ENV_PENDULUM) return fail("ses_create: unknown env %d", cfg->env);
    if (cfg->env == SES_ENV_MOUNTAINCAR && (cfg->obs_dim != 2 || cfg->act_dim != 3))
        return fail("ses_create: MountainCar-v0 needs num_state=2, num_action=3 (got %d, %d)", cfg->obs_dim, cfg->act_dim);
    if (cfg->env == SES_ENV_ACROBOT && (cfg->obs_dim != 6 || cfg->act_dim != 3))
        return fail("ses_create: Acrobot-v1 needs num_state=6, num_action=3 (got %d, %d)", cfg->obs_dim, cfg->act_dim);
    if (cfg->env == SES_ENV_PENDULUM && (cfg->obs_dim != 3 || cfg->act_dim != 1))
        return fail("ses_create: Pendulum-v0 needs num_state=3, num_action=1 (got %d, %d)", cfg->obs_dim, cfg->act_dim);
    if ((cfg->env == SES_ENV_PENDULUM) != (cfg->continuous_action != 0))
        return fail("ses_create: the continuous-action head (discrete_action: False) is implemented for Pendulum-v0, and Pendulum-v0 needs it");
    // envs/gym_wrapper.py:11-19: the reference's POMDP wrapper exists for LunarLander and CartPole only (AssertionError otherwise)
    if ((cfg->env == SES_ENV_MOUNTAINCAR || cfg->env == SES_ENV_ACROBOT || cfg->env == SES_ENV_PENDULUM) && cfg->pomdp)
        return fail("ses_create: only CartPole supports pomdp (envs/gym_wrapper.py:11-19 raises for every other env)");
    if (cfg->env == SES_ENV_CARTPOLE && (cfg->obs_dim != 4 || cfg->act_dim != 2))
        return fail("ses_create: CartPole-v1 needs num_state=4, num_action=2 (got %d, %d)", cfg->obs_dim, cfg->act_dim);
    if (cfg->env == SES_ENV_SIMPLE_SPREAD) {
        if (cfg->n_agents < 2 || cfg->n_agents > 3) return fail("ses_create: simple_spread supports N=2 or N=3 agents (got %d)", cfg->n_agents);
        if (cfg->obs_dim != 6 * cfg->n_agents || cfg->act_dim != 5)
            return fail("ses_create: simple_spread N=%d needs num_state=%d, num_action=5", cfg->n_agents, 6 * cfg->n_agents);
    }
    if (cfg->eval_ep_num < 1 || cfg->eval_ep_num > 32) return fail("ses_create: eval_ep_num must be in [1, 32] (got %d)", cfg->eval_ep_num);
    if (cfg->population < 2) return fail("ses_create: population must be >= 2");
    // the work queue counts episodes in 32-bit integers (headroom for the requests that overshoot the end of the queue)
    if ((long long)cfg->population * cfg->eval_ep_num > (1ll << 30))
        return fail("ses_create: population x eval_ep_num = %lld exceeds 2^30 episodes per generation", (long long)cfg->population * cfg->eval_ep_num);
    if (cfg->group < 1 || cfg->n_head < 0 || cfg->n_parents < 1) return fail("ses_create: bad population layout");
    if (cfg->antithetic != 0 && cfg->antithetic != 1) return fail("ses_create: antithetic must be 0 or 1");
    if (cfg->id_begin < 0 || cfg->id_end > cfg->population || cfg->id_begin > cfg->id_end) return fail("ses_create: bad slice [%d, %d)", cfg->id_begin, cfg->id_end);
    if (cfg->shard_block < 0 || (cfg->shard_block > 0 && (cfg->shard_world < 1 || cfg->shard_rank < 0 || cfg->shard_rank >= cfg->shard_world)))
        return fail("ses_create: bad block-cyclic shard (block %d, rank %d of %d)", cfg->shard_block, cfg->shard_rank, cfg->shard_world);
    if (cfg->shard_block > 0 && (cfg->id_begin != 0 || cfg->id_end != cfg->population))
        return fail("ses_create: a block-cyclic shard needs id_begin = 0 and id_end = population");
    if ((cfg->population - 1) / cfg->group >= cfg->n_parents) return fail("ses_create: layout needs %d parents, table has %d", (cfg->population - 1) / cfg->group + 1, cfg->n_parents);

    CU(cudaSetDevice(cfg->device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, cfg->device));
    if (prop.major < 10) return fail("ses_create: device %d is sm_%d%d; this library is built for sm_100a only", cfg->device, prop.major, prop.minor);

    ses_handle *h = new ses_handle();
    h->cfg = *cfg;
    h->D = param_count(cfg->obs_dim, cfg->act_dim, cfg->gru);
    h->shard.id_begin = cfg->id_begin; h->shard.block = cfg->shard_block; h->shard.rank = cfg->shard_rank; h->shard.world = cfg->shard_world;
    if (cfg->shard_block > 0) {
        // ids owned: full blocks b = rank, rank + world, ... plus the part of the last (partial) block below P
        const long long B = cfg->shard_block, W = cfg->shard_world, Pn = cfg->population;
        long long n = 0;
        for (long long b = cfg->shard_rank; b * B < Pn; b += W) n += (b + 1) * B <= Pn ? B : Pn - b * B;
        h->shard.n_local = (int)n;
    } else {
        h->shard.n_local = cfg->id_end - cfg->id_begin;
    }
    h->NQ = (h->D + 3) / 4;
    h->DP = h->NQ * 4;
    h->state_dim = cfg->env == SES_ENV_SIMPLE_SPREAD ? 4 * cfg->n_agents : ((cfg->env == SES_ENV_MOUNTAINCAR || cfg->env == SES_ENV_PENDULUM) ? 2 : 4);
    h->num_sms = prop.multiProcessorCount;
    // gym registers CartPole-v1 with max_episode_steps=500 (TimeLimit); the wrapper's own max_step
    // (gym_wrapper.py:37-39) can only shorten it (CartPole-v0: the caller passes max_step <= 200).
    // simple_spread: max_cycles=25; MountainCar-v0: 200; Acrobot-v1: 500.
    static const int caps[5] = {500, 25, 200, 500, 200};
    const int env_cap = caps[cfg->env];
    h->eff_max_step = cfg->max_step > 0 ? (cfg->max_step < env_cap ? cfg->max_step : env_cap) : env_cap;
    h->lanes_used_override = env_int("SES_ROLLOUT_LANES", 0);
    h->ctas_per_sm = env_int("SES_ROLLOUT_CTAS_PER_SM", 0);
#ifdef SES_BUILD_TESTS
    // alternative kernels exist only in the test build (include/ses_b200_test.h)
    h->k1_variant = env_int("SES_K1_VARIANT", 7);
    h->spread_slots8 = env_int("SES_SPREAD_SLOTS8", 0);
    h->k2_fused = env_int("SES_K2_FUSED", 1);     // 1 + passes launches (default); 0: the separate kernels
#endif
    h->k2_persistent = env_int("SES_K2_PERSISTENT", 1);   // 1: one cooperative launch for the whole sort (default); 0: the fused build
    h->k1_split = env_int("SES_K1_SPLIT", 1);
    h->k1_sparse = env_int("SES_K1_SPARSE", 1);
    if (h->k1_variant < 0 || h->k1_variant > 7) h->k1_variant = 7;

    const int P = cfg->population;
    h->n_tiles = (P + sort_tile(SORT_ITEMS_SMALL) - 1) / sort_tile(SORT_ITEMS_SMALL);
    if (P <= (1 << 15)) h->n_tiles = (P + sort_tile(1) - 1) / sort_tile(1);    // the persistent kernel's 256-key tiles (ses_rank_desc)
    h->nb0 = (P + GB0 - 1) / GB0;
    h->nb1 = (h->nb0 + GB1 - 1) / GB1;
    CU(cudaMalloc(&h->work_counter, sizeof(int) * WORK_COUNTER_INTS));
    CU(cudaMallocHost(reinterpret_cast<void **>(&h->k1_steps_host), sizeof(unsigned long long)));
    CU(cudaEventCreateWithFlags(&h->k1_ev, cudaEventDisableTiming));
    CU(cudaMalloc(&h->ep_acc, sizeof(int) * 2 * (size_t)(h->shard.n_local > 0 ? h->shard.n_local : 1)));
    CU(cudaMemset(h->ep_acc, 0, sizeof(int) * 2 * (size_t)(h->shard.n_local > 0 ? h->shard.n_local : 1)));
    CU(cudaMalloc(&h->keys[0], sizeof(unsigned long long) * P));
    CU(cudaMalloc(&h->keys[1], sizeof(unsigned long long) * P));
    CU(cudaMalloc(&h->vals_scratch, sizeof(int) * P));
    CU(cudaMalloc(&h->hist, sizeof(int) * h->n_tiles * 256));
    CU(cudaMalloc(&h->tot, sizeof(int) * 8 * 256));
    CU(cudaMalloc(&h->hist_fused, sizeof(int) * (8 * (size_t)h->n_tiles * 256 + 1)));   // + the persistent kernel's grid-barrier counter
    CU(cudaMalloc(&h->part1, sizeof(double) * 2 * (size_t)h->nb1 * h->DP));     // two tables: k_grad_partial<true> (sep_cma_es)
    *out = h;
    return 0;
}

extern "C" int ses_destroy(ses_handle *h)
{
    if (!h) return 0;
    cudaSetDevice(h->cfg.device);
    cudaFree(h->work_counter);
    if (h->k1_steps_host) cudaFreeHost(h->k1_steps_host);
    if (h->k1_ev) cudaEventDestroy(h->k1_ev);
    cudaFree(h->ep_acc);
    cudaFree(h->keys[0]); cudaFree(h->keys[1]);
    cudaFree(h->vals_scratch); cudaFree(h->hist); cudaFree(h->tot); cudaFree(h->hist_fused);
    cudaFree(h->part1);
    for (int r = 0; r < h->peer_world; ++r)
        if (r != h->peer_rank && h->peer_x[r]) cudaIpcCloseMemHandle(h->peer_x[r]);
    cudaFree(h->xbuf); cudaFree(h->peer_error); cudaFree(h->grad_done);
    cudaFree(h->h_parents); cudaFree(h->h_m); cudaFree(h->h_v);
    cudaFree(h->h_fitness); cudaFree(h->h_shaped); cudaFree(h->h_steps); cudaFree(h->h_order); cudaFree(h->h_total);
    cudaFree(h->e_parents); cudaFree(h->e_out); cudaFree(h->e_fitness); cudaFree(h->e_steps); cudaFree(h->e_order); cudaFree(h->e_total);
    cudaFree(h->eval_counter);
    cudaFree(h->map_claim); cudaFree(h->map_list); cudaFree(h->map_enter);
    delete h;
    return 0;
}

extern "C" int64_t ses_launch_count(ses_handle *h) { return h ? h->launches : 0; }

extern "C" int ses_set_step_counter(ses_handle *h, uint64_t *counter_dev)
{
    if (!h) return fail("ses_set_step_counter: null handle");
    h->step_counter = reinterpret_cast<unsigned long long *>(counter_dev);
    return 0;
}

extern "C" int ses_set_final_states(ses_handle *h, double *final_states_dev)
{
    if (!h) return fail("ses_set_final_states: null handle");
    h->final_states = final_states_dev;
    return 0;
}

// ------------------------------------------------------------------------------------------------
// K1
// ------------------------------------------------------------------------------------------------
static ses::PeerSync peer_sync_next(ses_handle *h, double *poison_fitness);

template <class Env, int SL, int WARPS = 4>
static int launch_slots(ses_handle *h, RolloutParams &rp, int need_warps, bool trace, cudaStream_t st)
{
    using Smem = SlotSmem<Env, SL, !Env::UNIT_REWARD>;
#ifdef SES_BUILD_TESTS
    // SES_PEER_FOLD=1 (test build): the launch ends with the peer flag barrier (PeerSync, sentinel CTA).  Measured and not
    // adopted: two launches fewer per generation but 0.782 instead of 0.772 ms at N = 8 (profiles/r02_k1_experiments.md section 11)
    const bool fold = rp.n_peers > 0 && h->peer_fold && !trace && !rp.final_states;
    auto kernel = trace ? k_rollout_slots<Env, SL, WARPS, true> : fold ? k_rollout_slots<Env, SL, WARPS, false, true> : k_rollout_slots<Env, SL, WARPS, false>;
#else
    [[maybe_unused]] const bool fold = false;
    auto kernel = trace ? k_rollout_slots<Env, SL, WARPS, true> : k_rollout_slots<Env, SL, WARPS, false>;
#endif
    if (rp.final_states) kernel = k_rollout_slots<Env, SL, WARPS, false, false, false, true>;   // the final-state instance
    const size_t smem = WARPS * sizeof(Smem);
    rp.slots_cap = SL;
    CU(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0;
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, WARPS * 32, smem));
    if (per_sm < 1) return fail("rollout kernel does not fit on an SM (smem %zu B)", smem);
    if (h->ctas_per_sm > 0 && h->ctas_per_sm < per_sm) per_sm = h->ctas_per_sm;
    const int resident_warps = per_sm * h->num_sms * WARPS;
    // Lanes of a warp that take episodes.  E * floor(32 / E) (30 for E = 5) lets slots start and finish together.  Envs whose
    // queue can hand out single episodes (EPISODE_UNITS: CartPole) use all 32: in the bulk of a launch the last offspring of a
    // refill waits for the warp's next round, and once at most one round of episodes is left every warp takes exactly as many
    // episodes as it has idle lanes, so no left-over episodes cost an extra, nearly empty round (profiles/r02_k1_experiments.md).
    const int E = h->cfg.eval_ep_num;
    const long long n_ep = (long long)h->shard.n_local * E;
    const int lanes_even = E >= 32 ? 32 : E * (32 / E);
    constexpr bool EP_UNITS = EnvEpisodeUnits<Env>::value;
    int lanes = (EP_UNITS && SL >= (32 + E - 1) / E + 1) ? 32 : lanes_even;
    if (h->lanes_used_override > 0) lanes = h->lanes_used_override < 32 ? h->lanes_used_override : 32;
    rp.lanes_used = lanes;
    {   // Queue B (exact requests) holds the last two rounds' worth of episodes -- when episodes are long.  With short, ragged
        // episodes (a generation-0 population) lanes come free one or two at a time, every refill is a small whole-offspring
        // request, and those are cheapest on the aligned queue A (one atomic, no offspring shared between warps): no queue B.
        // Which regime a launch is in is read off the PREVIOUS launch's mean episode length (k1_mean_len: copied back
        // asynchronously, never waited for; unknown = long).  None of this can change a result.
        if (h->k1_ev_pending && cudaEventQuery(h->k1_ev) == cudaSuccess) {
            h->k1_ev_pending = false;
            if (h->k1_last_episodes > 0) h->k1_mean_len = (double)*h->k1_steps_host / (double)h->k1_last_episodes;
        }
        const bool ragged = h->k1_mean_len >= 0.0 && h->k1_mean_len < 0.25 * (double)h->eff_max_step;
        const int tail_rounds = env_int("SES_K1_TAIL", ragged ? 0 : 2);
        const long long tail = EP_UNITS ? (long long)resident_warps * 32 * tail_rounds : 0;
        long long t0 = n_ep > tail ? ((n_ep - tail) / E) * E : 0;
        if (EP_UNITS && n_ep <= (long long)resident_warps * 32) t0 = 0;      // a single round: exact from the start (sparse warps need it)
        rp.tail_start = EP_UNITS ? (int)t0 : (int)n_ep;
    }
    need_warps = (int)((n_ep + lanes - 1) / lanes);
    int grid = per_sm * h->num_sms;
    const int need = (need_warps + WARPS - 1) / WARPS;
    if (grid > need) grid = need;
    if (grid < 1) grid = 1;
    // A launch that does not fill the SMs (need < resident CTAs): give every SM the same CTAs -- `full` CTAs with full warps
    // plus one whose warps share the rest, a few episodes each, which the straggler phase runs on 4 / 2 lanes per episode
    // (see the kernel).  Only where the sparse warps end up with at most 16 episodes, i.e. where they can split.
    if constexpr (EnvSplit<Env>::value && EP_UNITS) {
        const int full = need / h->num_sms;                               // full CTAs per SM
        const long long rest = n_ep - (long long)full * h->num_sms * WARPS * lanes;
        if (h->k1_sparse && h->k1_split && !trace && h->lanes_used_override == 0 && need < per_sm * h->num_sms && full >= 1 && full < per_sm && rest > 0) {
            const int quota = (int)((rest + (long long)h->num_sms * WARPS - 1) / ((long long)h->num_sms * WARPS));
            if (quota <= 16) {
                rp.sparse_rank = full;
                rp.sparse_quota = quota;                                  // episodes per sparse warp
                grid = (full + 1) * h->num_sms;
            }
        }
        if (env_int("SES_K1_SPARSE_QUOTA", 0) > 0) {                      // experiments: force the sparse class and its share
            rp.sparse_rank = env_int("SES_K1_SPARSE_RANK", 0);
            rp.sparse_quota = env_int("SES_K1_SPARSE_QUOTA", 0);
            grid = (h->ctas_per_sm > 0 ? h->ctas_per_sm : per_sm) * h->num_sms;
            if (rp.sparse_rank <= 0) {                                    // no full CTAs: the shares alone must cover the launch
                const long long warps = (long long)grid * WARPS;
                const long long min_quota = (n_ep + warps - 1) / warps;
                if (rp.sparse_quota < min_quota) rp.sparse_quota = (int)min_quota;
                rp.sparse_rank = 0;
            }
        }
        if (rp.sparse_rank >= 0) rp.tail_start = 0;                       // shares are counted in episodes: the exact queue only
    }
    {
        const int g[8] = {grid, rp.lanes_used, rp.tail_start, rp.sparse_rank, rp.sparse_quota, per_sm, resident_warps, 0};
        memcpy(h->k1_geometry, g, sizeof(g));
    }
    if (fold) {
        rp.sync = peer_sync_next(h, rp.fitness);
        rp.sync.done = h->work_counter + WORK_COUNTER_DONE;
        rp.sync.expected = grid * WARPS;
        h->barrier_folded = true;
        grid += 1;                                                         // the sentinel CTA (rollout_slots.cuh)
    }
    kernel<<<grid, WARPS * 32, smem, st>>>(rp);
    CU(cudaGetLastError());
    h->launches += 1;
    if (!h->k1_ev_pending) {                                               // this launch's env-step count, for the next launches' geometry
        CU(cudaMemcpyAsync(h->k1_steps_host, h->work_counter + WORK_COUNTER_STEPS, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
        CU(cudaEventRecord(h->k1_ev, st));
        h->k1_ev_pending = true;
        h->k1_last_episodes = n_ep;
    }
    return 0;
}

// slots per warp: enough offspring to occupy 32 lanes (E >= 4: 8, E in {2,3}: 16, E = 1: 32)
template <class Env>
static int launch_slots_by_E(ses_handle *h, RolloutParams &rp, int need_warps, bool trace, cudaStream_t st)
{
    if (h->cfg.eval_ep_num >= 4) return launch_slots<Env, 8>(h, rp, need_warps, trace, st);
    if (h->cfg.eval_ep_num >= 2) return launch_slots<Env, 16>(h, rp, need_warps, trace, st);
    return launch_slots<Env, 32>(h, rp, need_warps, trace, st);
}

extern "C" int ses_rollout(ses_handle *h, uint32_t generation, float sigma, const float *parents_dev,
                           const float *w_override_dev, const double *init_states_dev, double *fitness_dev,
                           int64_t *steps_dev, double *trace_dev, int32_t *trace_actions_dev, int32_t n_trace,
                           void *stream)
{
    if (!h) return fail("ses_rollout: null handle");
    if (!fitness_dev || !steps_dev) return fail("ses_rollout: fitness_dev and steps_dev are required");
    if (!parents_dev && !w_override_dev) return fail("ses_rollout: need parents_dev or w_override_dev");
    if (n_trace > 0 && (!trace_dev || !trace_actions_dev)) return fail("ses_rollout: n_trace > 0 needs trace buffers");
    if (n_trace > 0 && h->final_states) return fail("ses_rollout: traces and final states (ses_set_final_states) cannot be stored in one launch");
    const ses_config &c = h->cfg;
    const int n_local = h->shard.n_local;
    if (n_local == 0) return 0;
    if (n_trace > n_local) n_trace = n_local;
    CU(cudaSetDevice(c.device));
    cudaStream_t st = S(stream);
    CU(cudaMemsetAsync(h->work_counter, 0, sizeof(int) * WORK_COUNTER_INTS, st));

    RolloutParams rp;
    rp.parents = parents_dev; rp.w_override = w_override_dev; rp.init_states = init_states_dev;
    rp.fitness = fitness_dev; rp.steps = reinterpret_cast<long long *>(steps_dev);
    rp.trace = trace_dev; rp.trace_actions = trace_actions_dev; rp.work_counter = h->work_counter; rp.ep_acc = h->ep_acc;
    rp.sigma = sigma; rp.seed = c.seed; rp.gen = generation;
    rp.layout.group = c.group; rp.layout.n_head = c.n_head; rp.layout.antithetic = c.antithetic;
    rp.shard = h->shard;
    rp.E = c.eval_ep_num; rp.max_step = h->eff_max_step; rp.pomdp = c.pomdp; rp.init_mode = c.init_mode;
    rp.n_trace = n_trace; rp.slots_cap = 0; rp.lanes_used = 32; rp.n_agents = c.n_agents;
    rp.total_steps = h->step_counter;
    rp.n_peers = 0;
    for (int r = 0; r < MAX_PEERS; ++r) rp.peer_fitness[r] = nullptr;
    if (h->peer_world > 1 && h->xbuf) {
        // fused exchange only when the caller rolls out into one of the two exchange buffers
        for (int parity = 0; parity < 2; ++parity)
            if (fitness_dev == h->xbuf + (size_t)parity * c.population)
                for (int r = 0; r < h->peer_world; ++r)
                    if (r != h->peer_rank) rp.peer_fitness[rp.n_peers++] = h->peer_x[r] + (size_t)parity * c.population;
        h->last_rollout_fitness = rp.n_peers > 0 ? fitness_dev : nullptr;
    }
    rp.sync.world = 0;
    rp.final_states = h->final_states;
    h->barrier_folded = false;

    // lanes per warp and the grid are chosen per kernel in launch_slots(); the GRU kernel maps a warp to one offspring
    rp.lanes_used = c.eval_ep_num >= 32 ? 32 : c.eval_ep_num * (32 / c.eval_ep_num);
    rp.tail_start = 0;
    rp.split_ok = h->k1_split;
    rp.sparse_rank = -1; rp.sparse_quota = 0;
    const int need_warps = 0;
    const bool tr = n_trace > 0;
    if (c.env == SES_ENV_CARTPOLE && !c.gru) {
        // slots per warp: enough offspring to occupy 32 lanes (E >= 4: 8, E in {2,3}: 16, E = 1: 32)
        if (c.eval_ep_num >= 4) {
#ifdef SES_BUILD_TESTS
            if (h->k1_variant == 0) return launch_slots<CartpoleMlpEnvT<0>, 8>(h, rp, need_warps, tr, st);
            if (h->k1_variant == 1) return launch_slots<CartpoleMlpEnvT<1>, 8>(h, rp, need_warps, tr, st);
            if (h->k1_variant == 2) return launch_slots<CartpoleMlpEnvT<2>, 8>(h, rp, need_warps, tr, st);
            if (h->k1_variant == 3) return launch_slots<CartpoleMlpEnvT<3>, 8>(h, rp, need_warps, tr, st);
            if (h->k1_variant == 4) return launch_slots<CartpoleMlpEnvT<4>, 8>(h, rp, need_warps, tr, st);
            if (h->k1_variant == 5) return launch_slots<CartpoleMlpEnvT<5>, 8>(h, rp, need_warps, tr, st);
            if (h->k1_variant == 6) return launch_slots<CartpoleMlpEnvT<6>, 8>(h, rp, need_warps, tr, st);
#endif
            return launch_slots<CartpoleMlpEnvT<7>, 8>(h, rp, need_warps, tr, st);
        }
        if (c.eval_ep_num >= 2) return launch_slots<CartpoleMlpEnvT<7>, 16>(h, rp, need_warps, tr, st);
        return launch_slots<CartpoleMlpEnvT<7>, 32>(h, rp, need_warps, tr, st);
    }
    if (c.env == SES_ENV_CARTPOLE && c.gru) return launch_rollout_cartpole_gru(h->num_sms, h->ctas_per_sm, rp, tr, st, &h->launches, g_err, sizeof(g_err));
    if (c.gru) {            // the recurrent policy on every other env: one generic warp-per-offspring kernel (rollout_gru_generic.cuh)
        switch (c.env) {
        case SES_ENV_MOUNTAINCAR: return launch_rollout_gru_generic<MountainCarEnv>(h->num_sms, h->ctas_per_sm, rp, tr, st, &h->launches, g_err, sizeof(g_err));
        case SES_ENV_ACROBOT: return launch_rollout_gru_generic<AcrobotEnv>(h->num_sms, h->ctas_per_sm, rp, tr, st, &h->launches, g_err, sizeof(g_err));
        case SES_ENV_PENDULUM: return launch_rollout_gru_generic<PendulumEnv>(h->num_sms, h->ctas_per_sm, rp, tr, st, &h->launches, g_err, sizeof(g_err));
        default:
            if (c.n_agents == 2) return launch_rollout_gru_generic<SpreadEnv<2>>(h->num_sms, h->ctas_per_sm, rp, tr, st, &h->launches, g_err, sizeof(g_err));
            return launch_rollout_gru_generic<SpreadEnv<3>>(h->num_sms, h->ctas_per_sm, rp, tr, st, &h->launches, g_err, sizeof(g_err));
        }
    }
    if (c.env == SES_ENV_MOUNTAINCAR) return launch_slots_by_E<MountainCarEnv>(h, rp, need_warps, tr, st);
    if (c.env == SES_ENV_ACROBOT) return launch_slots_by_E<AcrobotEnv>(h, rp, need_warps, tr, st);
    if (c.env == SES_ENV_PENDULUM) return launch_slots_by_E<PendulumEnv>(h, rp, need_warps, tr, st);
    // simple_spread episodes all last max_cycles steps, so a warp never holds more than ceil(lanes_used / E) offspring at
    // once: 6 slots instead of 8 for E >= 5 (and 2-warp CTAs for N = 3) put 12 / 10 warps on an SM instead of 8
    // (shared-memory capacity is what limits this kernel)
    if (c.eval_ep_num >= 5 && !h->spread_slots8) {
        if (c.n_agents == 2) return launch_slots<SpreadEnv<2>, 6>(h, rp, need_warps, tr, st);
        return launch_slots<SpreadEnv<3>, 6, 2>(h, rp, need_warps, tr, st);
    }
    if (c.n_agents == 2) return launch_slots<SpreadEnv<2>, 8>(h, rp, need_warps, tr, st);
    return launch_slots<SpreadEnv<3>, 8>(h, rp, need_warps, tr, st);
}

// ------------------------------------------------------------------------------------------------
// policy evaluation and recording (DESIGN.md section 4.9): the EVAL and TRACE && EVAL instances of the K1 kernels
// ------------------------------------------------------------------------------------------------
// The slot kernel with chunks of E = 32 episodes: one chunk fills a warp.  Whole chunks only (queue A), so a chunk's clipped
// episode count is exact; no sparse warps, no straggler phase.  `record`: the TRACE instance (ses_record).
template <class Env, int SL, int WARPS = 4>
static int launch_eval_slots(ses_handle *h, RolloutParams &rp, bool record, cudaStream_t st)
{
    using Smem = SlotSmem<Env, SL, !Env::UNIT_REWARD>;
    auto kernel = record ? k_rollout_slots<Env, SL, WARPS, true, false, true> : k_rollout_slots<Env, SL, WARPS, false, false, true>;
    const size_t smem = WARPS * sizeof(Smem);
    CU(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0;
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, WARPS * 32, smem));
    if (per_sm < 1) return fail("evaluation kernel does not fit on an SM (smem %zu B)", smem);
    rp.slots_cap = SL;
    rp.lanes_used = 32;
    rp.tail_start = rp.shard.n_local * rp.E;
    const int need = (rp.shard.n_local + WARPS - 1) / WARPS;                  // one chunk per warp at most at a time
    int grid = per_sm * h->num_sms;
    if (grid > need) grid = need;
    kernel<<<grid, WARPS * 32, smem, st>>>(rp);
    CU(cudaGetLastError());
    h->launches += 1;
    return 0;
}

// episodes per chunk (virtual offspring) of the kernel that evaluates this handle's env / network: a full warp for the slot
// kernel, the lockstep width for the GRU kernels
static int eval_chunk(const ses_config &c)
{
    if (!c.gru) return 32;
    switch (c.env) {
    case SES_ENV_CARTPOLE: return 5;
    case SES_ENV_MOUNTAINCAR: return GruGenConfig<MountainCarEnv>::EC;
    case SES_ENV_ACROBOT: return GruGenConfig<AcrobotEnv>::EC;
    case SES_ENV_PENDULUM: return GruGenConfig<PendulumEnv>::EC;
    default: return c.n_agents == 2 ? GruGenConfig<SpreadEnv<2>>::EC : GruGenConfig<SpreadEnv<3>>::EC;
    }
}

// The launch of ses_evaluate and ses_record: n_pol x n_episodes episodes as virtual offspring (policy, chunk).  rp carries
// the caller's output pointers; `record` selects the TRACE instance of each kernel family.
static int launch_eval(ses_handle *h, const char *fn, uint32_t round, const float *policies_dev, int32_t n_pol, int32_t n_episodes,
                       const double *init_states_dev, RolloutParams &rp, bool record, void *stream)
{
    if (n_pol < 1 || n_episodes < 1) return fail("%s: n_pol and n_episodes must be >= 1 (got %d, %d)", fn, n_pol, n_episodes);
    const ses_config &c = h->cfg;
    const int E = eval_chunk(c);
    const long long chunks = ((long long)n_episodes + E - 1) / E;
    // the work queue counts episodes in 32-bit integers, as in ses_rollout
    if ((long long)n_pol * chunks * E > (1ll << 30))
        return fail("%s: %d policies x %d episodes exceed 2^30 episodes per call", fn, n_pol, n_episodes);
    CU(cudaSetDevice(c.device));
    cudaStream_t st = S(stream);
    if (!h->eval_counter) CU(cudaMalloc(&h->eval_counter, sizeof(int) * WORK_COUNTER_INTS));
    CU(cudaMemsetAsync(h->eval_counter, 0, sizeof(int) * WORK_COUNTER_INTS, st));

    rp.parents = policies_dev; rp.init_states = init_states_dev; rp.work_counter = h->eval_counter;
    rp.seed = c.seed; rp.gen = round;
    rp.init_mode = 1;                                   // counter (m, 0, round, block): Env::init with id 0 and gen = round
    rp.layout.group = (int)chunks; rp.layout.n_head = (int)chunks; rp.layout.antithetic = 0;   // parent = policy, never perturbed
    rp.shard.id_begin = 0; rp.shard.n_local = (int)(n_pol * chunks); rp.shard.block = 0; rp.shard.rank = 0; rp.shard.world = 1;
    rp.E = E; rp.max_step = h->eff_max_step; rp.pomdp = c.pomdp; rp.n_agents = c.n_agents;
    rp.sparse_rank = -1; rp.split_ok = 0;
    rp.eval_episodes = n_episodes;

    if (c.env == SES_ENV_CARTPOLE && !c.gru) return launch_eval_slots<CartpoleMlpEnvT<7>, 8>(h, rp, record, st);
    if (c.env == SES_ENV_CARTPOLE) return launch_rollout_cartpole_gru_ec<5, true>(h->num_sms, h->ctas_per_sm, rp, record, st, &h->launches, g_err, sizeof(g_err));
    if (c.gru) {
        switch (c.env) {
        case SES_ENV_MOUNTAINCAR: return launch_rollout_gru_generic<MountainCarEnv, true>(h->num_sms, h->ctas_per_sm, rp, record, st, &h->launches, g_err, sizeof(g_err));
        case SES_ENV_ACROBOT: return launch_rollout_gru_generic<AcrobotEnv, true>(h->num_sms, h->ctas_per_sm, rp, record, st, &h->launches, g_err, sizeof(g_err));
        case SES_ENV_PENDULUM: return launch_rollout_gru_generic<PendulumEnv, true>(h->num_sms, h->ctas_per_sm, rp, record, st, &h->launches, g_err, sizeof(g_err));
        default:
            if (c.n_agents == 2) return launch_rollout_gru_generic<SpreadEnv<2>, true>(h->num_sms, h->ctas_per_sm, rp, record, st, &h->launches, g_err, sizeof(g_err));
            return launch_rollout_gru_generic<SpreadEnv<3>, true>(h->num_sms, h->ctas_per_sm, rp, record, st, &h->launches, g_err, sizeof(g_err));
        }
    }
    if (c.env == SES_ENV_MOUNTAINCAR) return launch_eval_slots<MountainCarEnv, 8>(h, rp, record, st);
    if (c.env == SES_ENV_ACROBOT) return launch_eval_slots<AcrobotEnv, 8>(h, rp, record, st);
    if (c.env == SES_ENV_PENDULUM) return launch_eval_slots<PendulumEnv, 8>(h, rp, record, st);
    if (c.n_agents == 2) return launch_eval_slots<SpreadEnv<2>, 6>(h, rp, record, st);   // shared-memory sizes as in ses_rollout
    return launch_eval_slots<SpreadEnv<3>, 6, 2>(h, rp, record, st);
}

extern "C" int ses_evaluate(ses_handle *h, uint32_t round, const float *policies_dev, int32_t n_pol, int32_t n_episodes,
                            const double *init_states_dev, double *returns_dev, int32_t *lengths_dev, void *stream)
{
    if (!h) return fail("ses_evaluate: null handle");
    if (!policies_dev || !returns_dev || !lengths_dev) return fail("ses_evaluate: policies_dev, returns_dev and lengths_dev are required");
    RolloutParams rp{};
    rp.eval_returns = returns_dev; rp.eval_lengths = lengths_dev;
    return launch_eval(h, "ses_evaluate", round, policies_dev, n_pol, n_episodes, init_states_dev, rp, false, stream);
}

extern "C" int ses_record(ses_handle *h, uint32_t round, const float *policies_dev, int32_t n_pol, int32_t n_episodes,
                          const double *init_states_dev, double *initial_dev, double *states_dev, int32_t *actions_dev,
                          double *returns_dev, int32_t *lengths_dev, void *stream)
{
    if (!h) return fail("ses_record: null handle");
    if (!policies_dev || !initial_dev || !states_dev || !actions_dev || !returns_dev || !lengths_dev)
        return fail("ses_record: policies_dev, initial_dev, states_dev, actions_dev, returns_dev and lengths_dev are required");
    RolloutParams rp{};
    rp.trace_initial = initial_dev; rp.trace = states_dev; rp.trace_actions = actions_dev; rp.trace_returns = returns_dev;
    rp.eval_lengths = lengths_dev;
    return launch_eval(h, "ses_record", round, policies_dev, n_pol, n_episodes, init_states_dev, rp, true, stream);
}

// ------------------------------------------------------------------------------------------------
// novelty search (DESIGN.md section 4.10): behaviour characterisations, archive novelty, blended shaping
// ------------------------------------------------------------------------------------------------
extern "C" int ses_behavior(ses_handle *h, const double *final_states_dev, int32_t n, double *bc_dev, void *stream)
{
    if (!h) return fail("ses_behavior: null handle");
    if (!final_states_dev || !bc_dev) return fail("ses_behavior: final_states_dev and bc_dev are required");
    if (n < 1 || n > h->cfg.population) return fail("ses_behavior: n=%d outside [1, population=%d]", n, h->cfg.population);
    CU(cudaSetDevice(h->cfg.device));
    const long long total = (long long)n * h->state_dim;
    k_behavior<<<(unsigned)((total + 255) / 256), 256, 0, S(stream)>>>(final_states_dev, n, h->cfg.eval_ep_num, h->state_dim, bc_dev);
    CU(cudaGetLastError());
    h->launches += 1;
    return 0;
}

template <int SD>
static void launch_novelty(const double *bc, int n, const double *archive, int n_archive, int k, double *novelty, cudaStream_t st)
{
    const int grid = (n + NOVELTY_THREADS - 1) / NOVELTY_THREADS;
    if (k <= 1) k_novelty<SD, 1><<<grid, NOVELTY_THREADS, 0, st>>>(bc, n, archive, n_archive, k, novelty);
    else if (k <= 2) k_novelty<SD, 2><<<grid, NOVELTY_THREADS, 0, st>>>(bc, n, archive, n_archive, k, novelty);
    else if (k <= 4) k_novelty<SD, 4><<<grid, NOVELTY_THREADS, 0, st>>>(bc, n, archive, n_archive, k, novelty);
    else if (k <= 8) k_novelty<SD, 8><<<grid, NOVELTY_THREADS, 0, st>>>(bc, n, archive, n_archive, k, novelty);
    else if (k <= 16) k_novelty<SD, 16><<<grid, NOVELTY_THREADS, 0, st>>>(bc, n, archive, n_archive, k, novelty);
    else k_novelty<SD, 32><<<grid, NOVELTY_THREADS, 0, st>>>(bc, n, archive, n_archive, k, novelty);
}

extern "C" int ses_novelty(ses_handle *h, const double *bc_dev, int32_t n, const double *archive_dev, int32_t n_archive, int32_t k,
                           double *novelty_dev, void *stream)
{
    if (!h) return fail("ses_novelty: null handle");
    if (!bc_dev || !archive_dev || !novelty_dev) return fail("ses_novelty: bc_dev, archive_dev and novelty_dev are required");
    if (n < 1 || n > h->cfg.population) return fail("ses_novelty: n=%d outside [1, population=%d]", n, h->cfg.population);
    if (n_archive < 1) return fail("ses_novelty: n_archive must be >= 1 (got %d)", n_archive);
    if (k < 1 || k > NOVELTY_MAX_K) return fail("ses_novelty: k must be in [1, %d] (got %d)", NOVELTY_MAX_K, k);
    CU(cudaSetDevice(h->cfg.device));
    switch (h->state_dim) {                     // MountainCar / Pendulum, CartPole / Acrobot, simple_spread N = 2, N = 3
    case 2: launch_novelty<2>(bc_dev, n, archive_dev, n_archive, k, novelty_dev, S(stream)); break;
    case 4: launch_novelty<4>(bc_dev, n, archive_dev, n_archive, k, novelty_dev, S(stream)); break;
    case 8: launch_novelty<8>(bc_dev, n, archive_dev, n_archive, k, novelty_dev, S(stream)); break;
    case 12: launch_novelty<12>(bc_dev, n, archive_dev, n_archive, k, novelty_dev, S(stream)); break;
    default: return fail("ses_novelty: no kernel for state_dim %d", h->state_dim);
    }
    CU(cudaGetLastError());
    h->launches += 1;
    return 0;
}

extern "C" int ses_blend_shaped(ses_handle *h, const double *shaped_f_dev, const double *shaped_n_dev, int32_t n, double w,
                                double *out_dev, void *stream)
{
    if (!h) return fail("ses_blend_shaped: null handle");
    if (!shaped_f_dev || !shaped_n_dev || !out_dev) return fail("ses_blend_shaped: shaped_f_dev, shaped_n_dev and out_dev are required");
    if (n < 1 || n > h->cfg.population) return fail("ses_blend_shaped: n=%d outside [1, population=%d]", n, h->cfg.population);
    if (!(w >= 0.0 && w <= 1.0)) return fail("ses_blend_shaped: w must be in [0, 1] (got %g)", w);
    CU(cudaSetDevice(h->cfg.device));
    k_blend_shaped<<<(n + 255) / 256, 256, 0, S(stream)>>>(shaped_f_dev, shaped_n_dev, n, w, out_dev);
    CU(cudaGetLastError());
    h->launches += 1;
    return 0;
}

// ------------------------------------------------------------------------------------------------
// peer fitness exchange (multi-GPU): IPC-mapped exchange buffers + a flag barrier over NVLink
// ------------------------------------------------------------------------------------------------
// [2][P] fitness, flags, then the gradient rows: two [nb1][DP] tables (the second one only for sep_cma_es's k_grad_partial<true>)
static size_t xbuf_doubles(const ses_handle *h) { return 2 * (size_t)h->cfg.population + 2 * MAX_PEERS + 2 * (size_t)h->nb1 * h->DP; }
static double *xbuf_part1(double *base, const ses_handle *h) { return base + 2 * (size_t)h->cfg.population + 2 * MAX_PEERS; }
static unsigned long long *xbuf_flags(double *base, const ses_handle *h) { return reinterpret_cast<unsigned long long *>(base + 2 * (size_t)h->cfg.population); }

extern "C" int ses_peer_export(ses_handle *h, void *ipc_handle_out)
{
    if (!h || !ipc_handle_out) return fail("ses_peer_export: null argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    CU(cudaSetDevice(h->cfg.device));
    if (!h->xbuf) {
        CU(cudaMalloc(&h->xbuf, sizeof(double) * xbuf_doubles(h)));
        CU(cudaMemset(h->xbuf, 0, sizeof(double) * xbuf_doubles(h)));
        CU(cudaMalloc(&h->peer_error, sizeof(int)));
        CU(cudaMemset(h->peer_error, 0, sizeof(int)));
        CU(cudaMalloc(&h->grad_done, sizeof(int)));
        CU(cudaMemset(h->grad_done, 0, sizeof(int)));
        CU(cudaDeviceSynchronize());
    }
    cudaIpcMemHandle_t mh;
    CU(cudaIpcGetMemHandle(&mh, h->xbuf));
    memcpy(ipc_handle_out, &mh, sizeof(mh));
    return 0;
}

extern "C" int ses_peer_attach(ses_handle *h, const void *ipc_handles, int32_t rank, int32_t world)
{
    if (!h || !ipc_handles) return fail("ses_peer_attach: null argument");
    if (world < 2 || world > MAX_PEERS || rank < 0 || rank >= world) return fail("ses_peer_attach: bad rank/world %d/%d (max %d ranks)", rank, world, MAX_PEERS);
    if (!h->xbuf) return fail("ses_peer_attach: call ses_peer_export first");
    CU(cudaSetDevice(h->cfg.device));
    const cudaIpcMemHandle_t *mh = static_cast<const cudaIpcMemHandle_t *>(ipc_handles);
    for (int r = 0; r < world; ++r) {
        if (r == rank) { h->peer_x[r] = h->xbuf; continue; }
        void *ptr = nullptr;
        CU(cudaIpcOpenMemHandle(&ptr, mh[r], cudaIpcMemLazyEnablePeerAccess));
        h->peer_x[r] = static_cast<double *>(ptr);
    }
    h->peer_rank = rank;
    h->peer_world = world;
    h->peer_epoch = 0;
    {
        cudaDeviceProp prop;
        CU(cudaGetDeviceProperties(&prop, h->cfg.device));
        const long long ms = env_int("SES_PEER_TIMEOUT_MS", 10000);
        h->peer_timeout_cycles = (ms > 0 ? ms : 10000) * (long long)prop.clockRate;      // clockRate is in kHz = cycles per ms
#ifdef SES_BUILD_TESTS
        h->peer_fold = env_int("SES_PEER_FOLD", 0) != 0;
#endif
    }
    return 0;
}

extern "C" int ses_peer_fitness_ptr(ses_handle *h, int32_t parity, double **out)
{
    if (!h || !out || !h->xbuf) return fail("ses_peer_fitness_ptr: exchange buffer not allocated");
    *out = h->xbuf + (size_t)(parity & 1) * h->cfg.population;
    return 0;
}

// one CTA, thread r <-> peer r: raise my flag in r's buffer, then wait for r's flag in mine.  A peer that does not arrive
// within `timeout_cycles` SM cycles (SES_PEER_TIMEOUT_MS, default 10 s at the nominal SM clock; a throttled clock only makes
// the wait longer) sets the sticky error flag AND poisons this generation's fitness vector with a NaN, so that nothing
// downstream can silently consume a partially filled vector; B200Loop calls ses_peer_check() every generation and raises.
__global__ void k_peer_barrier(const ses::PeerSync s) { ses::peer_flag_barrier(s, threadIdx.x); }

// `poison_fitness`: the exchange buffer of the generation this barrier publishes (nullptr for the gradient-row barrier)
// the next barrier of this rank (every rank runs the same sequence of barriers, so the epochs agree)
static ses::PeerSync peer_sync_next(ses_handle *h, double *poison_fitness)
{
    ses::PeerSync s;
    h->peer_epoch += 1;
    s.my_flags = xbuf_flags(h->xbuf, h);
    for (int r = 0; r < MAX_PEERS; ++r) s.peer_flags[r] = r < h->peer_world ? xbuf_flags(h->peer_x[r], h) : nullptr;
    s.rank = h->peer_rank; s.world = h->peer_world; s.epoch = h->peer_epoch; s.timeout_cycles = h->peer_timeout_cycles;
    s.error = h->peer_error; s.poison = poison_fitness; s.done = nullptr; s.expected = 0;
    return s;
}

static int peer_barrier_launch(ses_handle *h, void *stream, double *poison_fitness)
{
    if (!h || h->peer_world < 2) return fail("ses_peer_barrier: peers not attached");
    CU(cudaSetDevice(h->cfg.device));
    const PeerSync ps = peer_sync_next(h, poison_fitness);
    k_peer_barrier<<<1, 32, 0, S(stream)>>>(ps);
    h->launches += 1;
    CU(cudaGetLastError());
    return 0;
}

extern "C" int ses_peer_barrier(ses_handle *h, void *stream)
{
    if (!h) return fail("ses_peer_barrier: null handle");
    if (h->barrier_folded) {                 // the rollout that filled the exchange buffer ended with this barrier (PeerSync)
        h->barrier_folded = false;
        return 0;
    }
    return peer_barrier_launch(h, stream, h->last_rollout_fitness);
}

extern "C" int ses_peer_check(ses_handle *h)
{
    if (!h || !h->peer_error) return 0;
    int e = 0;
    CU(cudaMemcpy(&e, h->peer_error, sizeof(int), cudaMemcpyDeviceToHost));
    if (e) return fail("ses_peer_barrier timed out waiting for a peer GPU");
    return 0;
}

// ------------------------------------------------------------------------------------------------
// K2
// ------------------------------------------------------------------------------------------------
extern "C" int ses_rank_desc(ses_handle *h, const double *fitness_dev, int32_t n, int32_t key_bits, double key_scale,
                             int32_t *order_dev, double *shaped_dev, void *stream)
{
    if (!h) return fail("ses_rank_desc: null handle");
    if (!fitness_dev || !order_dev) return fail("ses_rank_desc: null buffer");
    if (n < 1 || n > h->cfg.population) return fail("ses_rank_desc: n=%d outside (0, population=%d]", n, h->cfg.population);
    if (key_bits < 0 || key_bits > 61) return fail("ses_rank_desc: key_bits must be in [0, 61]");
    CU(cudaSetDevice(h->cfg.device));
    cudaStream_t st = S(stream);
    const int passes = key_bits == 0 ? 8 : (key_bits + 1 + 7) / 8;      // integer keys carry one bias bit (sign)
    const bool small = n <= (1 << 18);
    const int tile = sort_tile(small ? SORT_ITEMS_SMALL : SORT_ITEMS_LARGE);
    const int tiles = (n + tile - 1) / tile;
    // ping-pong so that the last pass lands in order_dev
    int *vals[2];
    vals[0] = (passes % 2 == 0) ? order_dev : h->vals_scratch;
    vals[1] = (passes % 2 == 0) ? h->vals_scratch : order_dev;
    if (h->k2_fused) {
        // 1 + passes launches: pass-0 histogram from the fitness vector, then one scatter per pass that also builds the next
        // pass's histograms; the last one writes the permutation and the centered ranks (rank.cuh)
        if (shaped_dev && n < 2) return fail("ses_rank_desc: centered ranks need n >= 2");
        const double stdv = n >= 2 ? sqrt((double)(n + 1) / (12.0 * (double)(n - 1))) : 1.0;
        const size_t per_pass = (size_t)tiles * 256;                      // [tiles][256] tile histograms of one pass
#ifndef SES_SIMT_EMU
        // float64 keys (8 passes) only: 82 -> 64 us at P = 16384; with the 2 passes of integer keys the grid barriers, the
        // L2-only loads and the cooperative launch cost what the two launch boundaries did (26.0 -> 27.3 us at P = 65536)
        const bool persistent = h->k2_persistent && passes >= 4;
        // small populations: 512-key tiles put twice the CTAs on the latency-bound passes (P = 16384: 71.7 -> 63.6 us; 256-key tiles
        // 76.4 us: the per-tile histogram walk and the barrier grow with the CTA count); SES_K2_TILE_ITEMS = 1 | 2 | 4 for experiments
        const int items = persistent && h->cfg.population <= (1 << 15) ? env_int("SES_K2_TILE_ITEMS", 2) : 0;
        const int ptiles = items == 1 ? (n + sort_tile(1) - 1) / sort_tile(1) : items == 2 ? (n + sort_tile(2) - 1) / sort_tile(2) : tiles;
        const size_t ppass = (size_t)ptiles * 256;
        CU(cudaMemsetAsync(h->hist_fused, 0, sizeof(int) * (ppass * passes + 1), st));      // ppass >= per_pass: covers the fused build too
        if (persistent) {
            SortBuffers buf;
            buf.keys[0] = h->keys[0]; buf.keys[1] = h->keys[1]; buf.vals[0] = vals[0]; buf.vals[1] = vals[1];
            int *hist_all = h->hist_fused;
            unsigned *bar = reinterpret_cast<unsigned *>(h->hist_fused + ppass * passes);
            int n_arg = n, kb = key_bits, passes_arg = passes, pp = (int)ppass;
            double ks = key_scale, stdv_arg = stdv;
            void *args[] = {(void *)&fitness_dev, &n_arg, &kb, &ks, &passes_arg, &buf, &hist_all, &pp, &bar, &stdv_arg, (void *)&shaped_dev};
            const void *fn = items == 1 ? (const void *)k_sort_persistent<1> : items == 2 ? (const void *)k_sort_persistent<2>
                           : small ? (const void *)k_sort_persistent<SORT_ITEMS_SMALL> : (const void *)k_sort_persistent<SORT_ITEMS_LARGE>;
            const cudaError_t e = cudaLaunchCooperativeKernel(fn, dim3(ptiles), dim3(SORT_THREADS), args, 0, st);
            if (e == cudaSuccess) {
                h->launches += 1;
                return 0;
            }
            (void)cudaGetLastError();                              // refused (not co-resident, no cooperative launch): the fused build from now on
            h->k2_persistent = 0;
        }
#else
        CU(cudaMemsetAsync(h->hist_fused, 0, sizeof(int) * (per_pass * passes + 1), st));
#endif
        if (small) k_sort_hist_first<SORT_ITEMS_SMALL><<<tiles, SORT_THREADS, 0, st>>>(fitness_dev, n, key_bits, key_scale, h->hist_fused);
        else k_sort_hist_first<SORT_ITEMS_LARGE><<<tiles, SORT_THREADS, 0, st>>>(fitness_dev, n, key_bits, key_scale, h->hist_fused);
        h->launches += 1;
        for (int ps = 0; ps < passes; ++ps) {
            const int a = ps & 1, b = a ^ 1;
            const int first = ps == 0, last = ps == passes - 1;
            int *hp = h->hist_fused + per_pass * ps;
            int *hn = last ? nullptr : h->hist_fused + per_pass * (ps + 1);
            if (small)
                k_sort_scatter_fused<SORT_ITEMS_SMALL><<<tiles, SORT_THREADS, 0, st>>>(fitness_dev, key_bits, key_scale, h->keys[a], vals[a], n, 8 * ps, first, last,
                                                                                        hp, hn, h->keys[b], vals[b], stdv, shaped_dev);
            else
                k_sort_scatter_fused<SORT_ITEMS_LARGE><<<tiles, SORT_THREADS, 0, st>>>(fitness_dev, key_bits, key_scale, h->keys[a], vals[a], n, 8 * ps, first, last,
                                                                                        hp, hn, h->keys[b], vals[b], stdv, shaped_dev);
            h->launches += 1;
        }
        CU(cudaGetLastError());
        return 0;
    }
#ifndef SES_BUILD_TESTS
    return fail("ses_rank_desc: the separate-kernel K2 path exists only in the test build");
#else
    CU(cudaMemsetAsync(h->tot, 0, sizeof(int) * 8 * 256, st));
    k_sort_init<<<(n + 255) / 256, 256, 0, st>>>(fitness_dev, n, key_bits, key_scale, h->keys[0], vals[0]);
    h->launches += 1;
    for (int ps = 0; ps < passes; ++ps) {
        const int a = ps & 1, b = a ^ 1;
        if (small) {
            k_sort_hist<SORT_ITEMS_SMALL><<<tiles, SORT_THREADS, 0, st>>>(h->keys[a], n, 8 * ps, h->hist, h->tot + 256 * ps);
            k_sort_scatter<SORT_ITEMS_SMALL><<<tiles, SORT_THREADS, 0, st>>>(h->keys[a], vals[a], n, 8 * ps, h->hist, h->tot + 256 * ps, h->keys[b], vals[b]);
        } else {
            k_sort_hist<SORT_ITEMS_LARGE><<<tiles, SORT_THREADS, 0, st>>>(h->keys[a], n, 8 * ps, h->hist, h->tot + 256 * ps);
            k_sort_scatter<SORT_ITEMS_LARGE><<<tiles, SORT_THREADS, 0, st>>>(h->keys[a], vals[a], n, 8 * ps, h->hist, h->tot + 256 * ps, h->keys[b], vals[b]);
        }
        h->launches += 2;
    }
    if (shaped_dev) {
        if (n < 2) return fail("ses_rank_desc: centered ranks need n >= 2");
        const double stdv = sqrt((double)(n + 1) / (12.0 * (double)(n - 1)));
        k_shape_centered<<<(n + 255) / 256, 256, 0, st>>>(order_dev, n, stdv, shaped_dev);
        h->launches += 1;
    }
    CU(cudaGetLastError());
    return 0;
#endif
}

// ------------------------------------------------------------------------------------------------
// K3
// ------------------------------------------------------------------------------------------------
// levels 0 + 1 of the gradient (k_grad_partial, and the peer barrier when the rows are sharded over ranks);
// *part1_out is the [nb1][DP] table the level-2 kernels read.  sq: k_grad_partial<true>, whose second table (the squared
// noise) follows at *part1_out + nb1 * DP
static int grad_levels01(ses_handle *h, uint32_t generation, const double *shaped_dev, const float *eps_override_dev,
                         void *stream, double **part1_out, bool sq = false)
{
    cudaStream_t st = S(stream);
    const int P = h->cfg.population;
    Layout lay{h->cfg.group, h->cfg.n_head, h->cfg.antithetic};
    // all groups here, or -- with peers attached -- this rank's share of the groups, each row stored into every
    // peer's table over NVLink, then the flag barrier
    const bool shard = h->peer_world > 1 && h->xbuf && !eps_override_dev;
    double *part1 = shard ? xbuf_part1(h->xbuf, h) : h->part1;
    int g0 = 0, g1 = h->nb1;
    PeerRows peers;
    int n_peers = 0;
    for (int r = 0; r < 8; ++r) peers.p[r] = nullptr;
    if (shard) {
        g0 = (int)((long long)h->peer_rank * h->nb1 / h->peer_world);
        g1 = (int)((long long)(h->peer_rank + 1) * h->nb1 / h->peer_world);
        for (int r = 0; r < h->peer_world; ++r)
            if (r != h->peer_rank) peers.p[n_peers++] = xbuf_part1(h->peer_x[r], h);
    }
    const int n_chunks = (h->NQ + GQC - 1) / GQC;
    PeerSync sync;
    sync.world = 0;
    const bool fold = shard && h->peer_fold && g1 > g0;                  // the launch ends with the flag barrier
    if (fold) {
        sync = peer_sync_next(h, nullptr);
        sync.done = h->grad_done;
        sync.expected = (g1 - g0) * n_chunks;
    }
    if (g1 > g0) {
        auto kernel = sq ? k_grad_partial<true> : k_grad_partial<false>;
        kernel<<<(g1 - g0) * n_chunks, GB1 * GQC, 0, st>>>(shaped_dev, P, h->D, h->NQ, h->cfg.seed, generation, lay, eps_override_dev,
                                                          part1, h->nb0, g0, n_chunks, n_peers, peers, sync);
        h->launches += 1;
    }
    if (shard && !fold && peer_barrier_launch(h, stream, nullptr)) return -1;
    *part1_out = part1;
    return 0;
}

extern "C" int ses_update_openai(ses_handle *h, uint32_t generation, const double *shaped_dev,
                                 const float *eps_override_dev, double update_factor, double adam_a, double beta1,
                                 double beta2, double adam_eps, float *mu_dev, float *m_dev, float *v_dev,
                                 float *grad_out_dev, void *stream)
{
    if (!h) return fail("ses_update_openai: null handle");
    if (!shaped_dev || !mu_dev || !m_dev || !v_dev) return fail("ses_update_openai: null buffer");
    CU(cudaSetDevice(h->cfg.device));
    cudaStream_t st = S(stream);
    double *part1 = nullptr;
    if (grad_levels01(h, generation, shaped_dev, eps_override_dev, stream, &part1)) return -1;
    k_grad_final_adam<<<(h->D + 255) / 256, 256, 0, st>>>(part1, h->nb1, h->DP, h->D, (float)update_factor, adam_a, (float)beta1,
                                                         (float)(1.0 - beta1), (float)beta2, (float)(1.0 - beta2), (float)adam_eps,
                                                         mu_dev, m_dev, v_dev, grad_out_dev);
    h->launches += 1;
    CU(cudaGetLastError());
    return 0;
}

extern "C" int ses_update_openai_sgd(ses_handle *h, uint32_t generation, const double *shaped_dev,
                                     const float *eps_override_dev, double update_factor, double stepsize, double momentum,
                                     float *mu_dev, float *v_dev, float *grad_out_dev, void *stream)
{
    if (!h) return fail("ses_update_openai_sgd: null handle");
    if (!shaped_dev || !mu_dev || !v_dev) return fail("ses_update_openai_sgd: null buffer");
    if (!(momentum >= 0.0 && momentum < 1.0)) return fail("ses_update_openai_sgd: momentum must be in [0, 1)");
    CU(cudaSetDevice(h->cfg.device));
    cudaStream_t st = S(stream);
    double *part1 = nullptr;
    if (grad_levels01(h, generation, shaped_dev, eps_override_dev, stream, &part1)) return -1;
    k_grad_final_sgd<<<(h->D + 255) / 256, 256, 0, st>>>(part1, h->nb1, h->DP, h->D, (float)update_factor, (float)(-stepsize),
                                                        (float)momentum, (float)(1.0 - momentum), mu_dev, v_dev, grad_out_dev);
    h->launches += 1;
    CU(cudaGetLastError());
    return 0;
}

// ------------------------------------------------------------------------------------------------
// sep_cma_es (DESIGN.md section 4.11)
// ------------------------------------------------------------------------------------------------
static int cma_layout_ok(const ses_handle *h, const char *fn)
{
    if (h->cfg.group != h->cfg.population || h->cfg.n_head != 0 || h->cfg.antithetic)
        return fail("%s: needs the sep_cma_es layout (group = population, n_head = 0, no antithetic pairs); this handle has group %d, "
                    "n_head %d, antithetic %d", fn, h->cfg.group, h->cfg.n_head, h->cfg.antithetic);
    return 0;
}

extern "C" int ses_cma_sample(ses_handle *h, uint32_t generation, const double *mean_dev, const double *c_dev, const double *sigma_dev,
                              float *out_dev, void *stream)
{
    if (!h) return fail("ses_cma_sample: null handle");
    if (!mean_dev || !c_dev || !sigma_dev || !out_dev) return fail("ses_cma_sample: mean_dev, c_dev, sigma_dev and out_dev are required");
    if (cma_layout_ok(h, "ses_cma_sample")) return -1;
    if (h->shard.n_local == 0) return 0;
    CU(cudaSetDevice(h->cfg.device));
    const long long total = (long long)h->shard.n_local * h->NQ;
    k_cma_sample<<<(unsigned)((total + 255) / 256), 256, 0, S(stream)>>>(mean_dev, c_dev, sigma_dev, h->shard, h->D, h->NQ, h->cfg.seed,
                                                                          generation, out_dev);
    CU(cudaGetLastError());
    h->launches += 1;
    return 0;
}

extern "C" int ses_cma_update(ses_handle *h, uint32_t generation, const int32_t *order_dev, const double *weights_dev, int32_t mu,
                              const ses_cma_params *params, double threshold, double *s_dev, double *mean_dev, double *c_dev,
                              double *p_sigma_dev, double *p_c_dev, double *sigma_dev, float *parent_dev, void *stream)
{
    if (!h) return fail("ses_cma_update: null handle");
    if (!order_dev || !weights_dev || !params || !s_dev || !mean_dev || !c_dev || !p_sigma_dev || !p_c_dev || !sigma_dev || !parent_dev)
        return fail("ses_cma_update: null argument");
    if (cma_layout_ok(h, "ses_cma_update")) return -1;
    const int P = h->cfg.population;
    if (mu < 1 || mu > P) return fail("ses_cma_update: mu=%d outside [1, population=%d]", mu, P);
    CU(cudaSetDevice(h->cfg.device));
    cudaStream_t st = S(stream);
    k_cma_weights<<<(P + 255) / 256, 256, 0, st>>>(order_dev, weights_dev, mu, P, s_dev);
    h->launches += 1;
    double *part1 = nullptr;
    if (grad_levels01(h, generation, s_dev, nullptr, stream, &part1, true)) return -1;
    const CmaParams pr{params->one_m_cs, params->k_sigma, params->one_m_cc, params->k_c, params->cc2, params->c_keep, params->c1,
                       params->cmu, params->damp, params->chi};
    k_cma_final<<<1, CMA_THREADS, 0, st>>>(part1, h->nb1, h->DP, h->D, pr, threshold, mean_dev, c_dev, p_sigma_dev, p_c_dev, sigma_dev,
                                           parent_dev);
    h->launches += 1;
    CU(cudaGetLastError());
    return 0;
}

// ------------------------------------------------------------------------------------------------
// map_elites (DESIGN.md section 4.12)
// ------------------------------------------------------------------------------------------------
// The layout and the descriptor spec; *out := the spec as the kernels take it, *n_cells_out := the cell count
static int map_check(const ses_handle *h, const ses_map_spec *spec, const char *fn, MapSpec *out, int *n_cells_out)
{
    if (h->cfg.group != 1 || h->cfg.n_head != 0 || h->cfg.antithetic)
        return fail("%s: needs the map_elites layout (group = 1, n_head = 0, no antithetic pairs); this handle has group %d, n_head %d, "
                    "antithetic %d", fn, h->cfg.group, h->cfg.n_head, h->cfg.antithetic);
    if (spec->n_dims < 1 || spec->n_dims > MAP_MAX_DIMS) return fail("%s: n_dims must be in [1, %d] (got %d)", fn, MAP_MAX_DIMS, spec->n_dims);
    long long n = 1;
    for (int j = 0; j < spec->n_dims; ++j) {
        if (spec->dims[j] < 0 || spec->dims[j] >= h->state_dim)
            return fail("%s: dims[%d] = %d outside the final state [0, %d)", fn, j, spec->dims[j], h->state_dim);
        for (int k = 0; k < j; ++k)
            if (spec->dims[k] == spec->dims[j]) return fail("%s: dims[%d] = dims[%d] = %d: the dimensions must be distinct", fn, k, j, spec->dims[j]);
        if (!std::isfinite(spec->low[j]) || !std::isfinite(spec->width[j]) || !(spec->width[j] > 0.0))
            return fail("%s: dimension %d needs a finite low and a finite width > 0 (got low %g, width %g)", fn, j, spec->low[j], spec->width[j]);
        if (spec->cells[j] < 1) return fail("%s: cells[%d] must be >= 1 (got %d)", fn, j, spec->cells[j]);
        n *= spec->cells[j];
        if (n > (1ll << 20)) return fail("%s: more than 2^20 cells (%lld after dimension %d)", fn, n, j);
    }
    if (n * h->D * 4 > (1ll << 32))
        return fail("%s: %lld cells x %d parameters x 4 bytes = %lld bytes of elite weights exceed 4 GiB", fn, n, h->D, n * h->D * 4);
    out->n_dims = spec->n_dims;
    for (int j = 0; j < MAP_MAX_DIMS; ++j) {
        const bool used = j < spec->n_dims;
        out->dims[j] = used ? spec->dims[j] : 0;
        out->low[j] = used ? spec->low[j] : 0.0;
        out->width[j] = used ? spec->width[j] : 1.0;
        out->cells[j] = used ? spec->cells[j] : 1;
    }
    *n_cells_out = (int)n;
    return 0;
}

static int map_scratch(ses_handle *h, int n_cells, cudaStream_t st)
{
    if (!h->map_enter) CU(cudaMalloc(&h->map_enter, sizeof(int) * (size_t)h->cfg.population));
    if (n_cells > h->map_cells) {
        CU(cudaStreamSynchronize(st));          // the old scratch may still be read by earlier launches on this stream
        cudaFree(h->map_claim); cudaFree(h->map_list);
        h->map_claim = h->map_list = nullptr;
        h->map_cells = 0;
        CU(cudaMalloc(&h->map_claim, sizeof(int) * (size_t)n_cells));
        CU(cudaMalloc(&h->map_list, sizeof(int) * (size_t)n_cells));
        CU(cudaMemset(h->map_claim, 0, sizeof(int) * (size_t)n_cells));
        h->map_cells = n_cells;
    }
    return 0;
}

extern "C" int ses_map_insert(ses_handle *h, uint32_t generation, float sigma, const float *parents_dev, const int32_t *order_dev,
                              const double *fitness_dev, const double *bc_dev, const ses_map_spec *spec, double *F_dev, double *B_dev,
                              int32_t *born_dev, float *W_dev, void *stream)
{
    if (!h) return fail("ses_map_insert: null handle");
    if (!parents_dev || !order_dev || !fitness_dev || !bc_dev || !spec || !F_dev || !B_dev || !born_dev || !W_dev)
        return fail("ses_map_insert: null argument");
    MapSpec ms;
    int n_cells = 0;
    if (map_check(h, spec, "ses_map_insert", &ms, &n_cells)) return -1;
    CU(cudaSetDevice(h->cfg.device));
    cudaStream_t st = S(stream);
    if (map_scratch(h, n_cells, st)) return -1;
    const int P = h->cfg.population, grid = (P + 255) / 256;
    k_map_claim<<<grid, 256, 0, st>>>(order_dev, fitness_dev, bc_dev, P, h->state_dim, ms, h->map_claim);
    k_map_commit<<<grid, 256, 0, st>>>(order_dev, fitness_dev, bc_dev, P, h->state_dim, ms, h->map_claim, generation, F_dev, B_dev,
                                       born_dev, h->map_enter);
    const Layout lay{h->cfg.group, h->cfg.n_head, h->cfg.antithetic};
    k_map_weights<<<P, 128, 0, st>>>(parents_dev, order_dev, h->map_enter, h->D, h->NQ, sigma, h->cfg.seed, generation, lay, W_dev);
    CU(cudaGetLastError());
    h->launches += 3;
    return 0;
}

extern "C" int ses_map_select(ses_handle *h, uint32_t generation, const ses_map_spec *spec, const double *F_dev, const float *W_dev,
                              const float *seed_row_dev, double *stats_dev, float *parents_dev, void *stream)
{
    if (!h) return fail("ses_map_select: null handle");
    if (!spec || !F_dev || !W_dev || !seed_row_dev || !stats_dev || !parents_dev) return fail("ses_map_select: null argument");
    MapSpec ms;
    int n_cells = 0;
    if (map_check(h, spec, "ses_map_select", &ms, &n_cells)) return -1;
    CU(cudaSetDevice(h->cfg.device));
    cudaStream_t st = S(stream);
    if (map_scratch(h, n_cells, st)) return -1;
    k_map_compact<<<1, MAP_COMPACT_THREADS, 0, st>>>(F_dev, n_cells, h->map_list, stats_dev);
    k_map_gather<<<h->cfg.population, 256, 0, st>>>(W_dev, h->map_list, stats_dev, seed_row_dev, h->D, h->cfg.seed, generation, parents_dev);
    CU(cudaGetLastError());
    h->launches += 2;
    return 0;
}

extern "C" int ses_materialize(ses_handle *h, uint32_t generation, float sigma, const float *parents_dev,
                               const float *w_override_dev, const int32_t *ids_dev, int32_t n, float *out_dev, void *stream)
{
    if (!h) return fail("ses_materialize: null handle");
    if ((!parents_dev && !w_override_dev) || !ids_dev || !out_dev) return fail("ses_materialize: null buffer");
    if (n < 1) return 0;
    CU(cudaSetDevice(h->cfg.device));
    Layout lay{h->cfg.group, h->cfg.n_head, h->cfg.antithetic};
    const int t = n * h->NQ;
    k_materialize<<<(t + 255) / 256, 256, 0, S(stream)>>>(parents_dev, w_override_dev, h->shard, h->D, h->NQ, sigma, h->cfg.seed,
                                                          generation, lay, ids_dev, n, out_dev);
    h->launches += 1;
    CU(cudaGetLastError());
    return 0;
}

extern "C" int ses_update_elite_mean(ses_handle *h, uint32_t generation, float sigma, const float *parents_dev,
                                     const float *w_override_dev, const int32_t *order_dev, int32_t k, float *mu_out_dev,
                                     void *stream)
{
    if (!h) return fail("ses_update_elite_mean: null handle");
    if ((!parents_dev && !w_override_dev) || !order_dev || !mu_out_dev) return fail("ses_update_elite_mean: null buffer");
    if (k < 1 || k > h->cfg.population) return fail("ses_update_elite_mean: k=%d out of range", k);
    CU(cudaSetDevice(h->cfg.device));
    Layout lay{h->cfg.group, h->cfg.n_head, h->cfg.antithetic};
    k_elite_mean<<<(h->NQ + 63) / 64, 64, 0, S(stream)>>>(parents_dev, w_override_dev, h->shard, h->D, h->NQ, sigma, h->cfg.seed,
                                                          generation, lay, order_dev, k, mu_out_dev);
    h->launches += 1;
    CU(cudaGetLastError());
    return 0;
}

// ------------------------------------------------------------------------------------------------
// whole openai_es generation with host buffers (bench.py e2e)
// ------------------------------------------------------------------------------------------------
extern "C" int ses_generation_openai_host(ses_handle *h, uint32_t generation, float sigma, double learning_rate,
                                          int64_t adam_t, float *mu_host, float *m_host, float *v_host,
                                          double *fitness_host, int64_t *total_steps_host, void *stream)
{
    if (!h) return fail("ses_generation_openai_host: null handle");
    const ses_config &c = h->cfg;
    const int P = c.population;
    if (h->shard.n_local != P) return fail("ses_generation_openai_host: needs a single-slice handle");
    if (c.n_parents != 1) return fail("ses_generation_openai_host: openai_es has one parent (mu)");
    if (!mu_host || !m_host || !v_host || !fitness_host || !total_steps_host) return fail("ses_generation_openai_host: null buffer");
    CU(cudaSetDevice(c.device));
    cudaStream_t st = S(stream);
    if (!h->h_parents) {
        CU(cudaMalloc(&h->h_parents, sizeof(float) * h->D));
        CU(cudaMalloc(&h->h_m, sizeof(float) * h->D));
        CU(cudaMalloc(&h->h_v, sizeof(float) * h->D));
        CU(cudaMalloc(&h->h_fitness, sizeof(double) * P));
        CU(cudaMalloc(&h->h_shaped, sizeof(double) * P));
        CU(cudaMalloc(&h->h_steps, sizeof(long long) * P));
        CU(cudaMalloc(&h->h_order, sizeof(int) * P));
        CU(cudaMalloc(&h->h_total, sizeof(unsigned long long)));
    }
    const size_t db = sizeof(float) * h->D;
    CU(cudaMemcpyAsync(h->h_parents, mu_host, db, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(h->h_m, m_host, db, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(h->h_v, v_host, db, cudaMemcpyHostToDevice, st));
    CU(cudaMemsetAsync(h->h_total, 0, sizeof(unsigned long long), st));
    unsigned long long *saved_counter = h->step_counter;
    h->step_counter = h->h_total;
    const int rc_roll = ses_rollout(h, generation, sigma, h->h_parents, nullptr, nullptr, h->h_fitness, reinterpret_cast<int64_t *>(h->h_steps),
                                    nullptr, nullptr, 0, stream);
    h->step_counter = saved_counter;
    if (rc_roll) return -1;
    int key_bits = 0;
    double key_scale = 1.0;
    if (c.env != SES_ENV_SIMPLE_SPREAD && c.env != SES_ENV_PENDULUM) {     // fitness = +-steps / E with integer |steps| <= E * max_step
        const long long vmax = (long long)c.eval_ep_num * h->eff_max_step;
        while ((1ll << key_bits) <= vmax) ++key_bits;
        key_scale = (double)c.eval_ep_num;
    }
    if (ses_rank_desc(h, h->h_fitness, P, key_bits, key_scale, h->h_order, h->h_shaped, stream)) return -1;
    const double beta1 = 0.99, beta2 = 0.999;  // optimizers.py:31
    const double a = learning_rate * sqrt(1.0 - pow(beta2, (double)adam_t)) / (1.0 - pow(beta1, (double)adam_t));
    const double uf = -(learning_rate / ((double)P * (double)sigma));
    if (ses_update_openai(h, generation, h->h_shaped, nullptr, uf, a, beta1, beta2, 1e-8, h->h_parents, h->h_m, h->h_v, nullptr, stream))
        return -1;
    CU(cudaMemcpyAsync(fitness_host, h->h_fitness, sizeof(double) * P, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(mu_host, h->h_parents, db, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(m_host, h->h_m, db, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(v_host, h->h_v, db, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(total_steps_host, h->h_total, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return 0;
}

// ------------------------------------------------------------------------------------------------
// whole simple_evolution / simple_genetic generation with host buffers
// ------------------------------------------------------------------------------------------------
// shared part: H2D of the parent table, K1, K2 (permutation only); leaves the order in h->e_order
static int elite_generation_prologue(ses_handle *h, const char *who, uint32_t generation, float sigma, const float *parents_host,
                                     void *stream)
{
    const ses_config &c = h->cfg;
    const int P = c.population;
    if (h->shard.n_local != P) return fail("%s: needs a single-slice handle", who);
    CU(cudaSetDevice(c.device));
    cudaStream_t st = S(stream);
    const size_t pb = sizeof(float) * (size_t)c.n_parents * h->D;
    if (!h->e_parents) {
        CU(cudaMalloc(&h->e_parents, pb));
        CU(cudaMalloc(&h->e_out, pb));
        CU(cudaMalloc(&h->e_fitness, sizeof(double) * P));
        CU(cudaMalloc(&h->e_steps, sizeof(long long) * P));
        CU(cudaMalloc(&h->e_order, sizeof(int) * P));
        CU(cudaMalloc(&h->e_total, sizeof(unsigned long long)));
    }
    CU(cudaMemcpyAsync(h->e_parents, parents_host, pb, cudaMemcpyHostToDevice, st));
    CU(cudaMemsetAsync(h->e_total, 0, sizeof(unsigned long long), st));
    unsigned long long *saved_counter = h->step_counter;
    h->step_counter = h->e_total;
    const int rc_roll = ses_rollout(h, generation, sigma, h->e_parents, nullptr, nullptr, h->e_fitness, reinterpret_cast<int64_t *>(h->e_steps),
                                    nullptr, nullptr, 0, stream);
    h->step_counter = saved_counter;
    if (rc_roll) return -1;
    int key_bits = 0;
    double key_scale = 1.0;
    if (c.env != SES_ENV_SIMPLE_SPREAD && c.env != SES_ENV_PENDULUM) {     // fitness = +-steps / E with integer |steps| <= E * max_step
        const long long vmax = (long long)c.eval_ep_num * h->eff_max_step;
        while ((1ll << key_bits) <= vmax) ++key_bits;
        key_scale = (double)c.eval_ep_num;
    }
    return ses_rank_desc(h, h->e_fitness, P, key_bits, key_scale, h->e_order, nullptr, stream);
}

static int elite_generation_epilogue(ses_handle *h, float *parents_host, size_t bytes, double *fitness_host, int64_t *total_steps_host,
                                     void *stream)
{
    cudaStream_t st = S(stream);
    CU(cudaMemcpyAsync(fitness_host, h->e_fitness, sizeof(double) * h->cfg.population, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(parents_host, h->e_out, bytes, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(total_steps_host, h->e_total, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return 0;
}

extern "C" int ses_generation_evolution_host(ses_handle *h, uint32_t generation, float sigma, int32_t elite_num, float *mu_host,
                                             double *fitness_host, int64_t *total_steps_host, void *stream)
{
    if (!h) return fail("ses_generation_evolution_host: null handle");
    if (!mu_host || !fitness_host || !total_steps_host) return fail("ses_generation_evolution_host: null buffer");
    if (h->cfg.n_parents != 1) return fail("ses_generation_evolution_host: simple_evolution has one parent (mu)");
    if (elite_num < 1 || elite_num > h->cfg.population) return fail("ses_generation_evolution_host: elite_num=%d out of range", elite_num);
    if (elite_generation_prologue(h, "ses_generation_evolution_host", generation, sigma, mu_host, stream)) return -1;
    if (ses_update_elite_mean(h, generation, sigma, h->e_parents, nullptr, h->e_order, elite_num, h->e_out, stream)) return -1;
    return elite_generation_epilogue(h, mu_host, sizeof(float) * h->D, fitness_host, total_steps_host, stream);
}

extern "C" int ses_generation_genetic_host(ses_handle *h, uint32_t generation, float sigma, float *elites_host,
                                           double *fitness_host, int64_t *total_steps_host, void *stream)
{
    if (!h) return fail("ses_generation_genetic_host: null handle");
    if (!elites_host || !fitness_host || !total_steps_host) return fail("ses_generation_genetic_host: null buffer");
    const int k = h->cfg.n_parents;
    if (k > h->cfg.population) return fail("ses_generation_genetic_host: more elites than offspring");
    if (elite_generation_prologue(h, "ses_generation_genetic_host", generation, sigma, elites_host, stream)) return -1;
    if (ses_materialize(h, generation, sigma, h->e_parents, nullptr, h->e_order, k, h->e_out, stream)) return -1;
    return elite_generation_epilogue(h, elites_host, sizeof(float) * (size_t)k * h->D, fitness_host, total_steps_host, stream);
}

// ------------------------------------------------------------------------------------------------
// FP32 pipe peak: dependent-free FFMA streams, the denominator of K1's roofline (bench.py)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_ffma_peak(float *out, int iters, float a, float b)
{
    float x0 = threadIdx.x, x1 = x0 + 1.f, x2 = x0 + 2.f, x3 = x0 + 3.f, x4 = x0 + 4.f, x5 = x0 + 5.f, x6 = x0 + 6.f, x7 = x0 + 7.f;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            x0 = fmaf(x0, a, b); x1 = fmaf(x1, a, b); x2 = fmaf(x2, a, b); x3 = fmaf(x3, a, b);
            x4 = fmaf(x4, a, b); x5 = fmaf(x5, a, b); x6 = fmaf(x6, a, b); x7 = fmaf(x7, a, b);
        }
    }
    const float s = ((x0 + x1) + (x2 + x3)) + ((x4 + x5) + (x6 + x7));
    if (s == 123.456f) out[0] = s;
}

__global__ void __launch_bounds__(256) k_ffma2_peak(float *out, int iters, float a, float b)
{
    const float t = threadIdx.x;
    float2 x0 = make_float2(t, t + 1.f), x1 = make_float2(t + 2.f, t + 3.f), x2 = make_float2(t + 4.f, t + 5.f), x3 = make_float2(t + 6.f, t + 7.f);
    float2 x4 = make_float2(t + 8.f, t + 9.f), x5 = make_float2(t + 10.f, t + 11.f), x6 = make_float2(t + 12.f, t + 13.f), x7 = make_float2(t + 14.f, t + 15.f);
    const float2 a2 = make_float2(a, a), b2 = make_float2(b, b);
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            x0 = __ffma2_rn(x0, a2, b2); x1 = __ffma2_rn(x1, a2, b2); x2 = __ffma2_rn(x2, a2, b2); x3 = __ffma2_rn(x3, a2, b2);
            x4 = __ffma2_rn(x4, a2, b2); x5 = __ffma2_rn(x5, a2, b2); x6 = __ffma2_rn(x6, a2, b2); x7 = __ffma2_rn(x7, a2, b2);
        }
    }
    const float s = ((x0.x + x1.x) + (x2.x + x3.x)) + ((x4.x + x5.x) + (x6.x + x7.x)) + ((x0.y + x1.y) + (x2.y + x3.y)) + ((x4.y + x5.y) + (x6.y + x7.y));
    if (s == 123.456f) out[0] = s;
}

static int measure_peak(int32_t device, double *tflops_out, bool packed)
{
    CU(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    float *out = nullptr;
    CU(cudaMalloc(&out, sizeof(float)));
    cudaEvent_t e0, e1;
    CU(cudaEventCreate(&e0));
    CU(cudaEventCreate(&e1));
    const int grid = prop.multiProcessorCount * 8, threads = 256, iters = 4096;
    double best = 0.0;
    for (int rep = 0; rep < 5; ++rep) {
        CU(cudaEventRecord(e0));
        if (packed) k_ffma2_peak<<<grid, threads>>>(out, iters, 0.999f, 0.001f);
        else k_ffma_peak<<<grid, threads>>>(out, iters, 0.999f, 0.001f);
        CU(cudaEventRecord(e1));
        CU(cudaEventSynchronize(e1));
        float ms = 0.f;
        CU(cudaEventElapsedTime(&ms, e0, e1));
        const double fl = (double)grid * threads * (double)iters * 64.0 * 2.0 * (packed ? 2.0 : 1.0);
        const double tf = fl / (ms * 1e-3) / 1e12;
        if (rep > 0 && tf > best) best = tf;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(out);
    *tflops_out = best;
    return 0;
}

extern "C" int ses_measure_fp32x2_peak(int32_t device, double *tflops_out)
{
    if (!tflops_out) return fail("ses_measure_fp32x2_peak: null argument");
    return measure_peak(device, tflops_out, true);
}

extern "C" int ses_measure_fp32_peak(int32_t device, double *tflops_out)
{
    if (!tflops_out) return fail("ses_measure_fp32_peak: null argument");
    return measure_peak(device, tflops_out, false);
}

#ifdef SES_BUILD_TESTS
// ------------------------------------------------------------------------------------------------
// test hooks
// ------------------------------------------------------------------------------------------------
__global__ void k_test_math(int kind, const void *in, void *out, long long n)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (kind <= 4 || kind == 7) {
        const float x = static_cast<const float *>(in)[i];
        float y = 0.0f, s, c;
        switch (kind) {
        case 0: y = tanh32(x); break;
        case 1: y = sigm32(x); break;
        case 2: y = ln32(x); break;
        case 3: sincos2pi32(x, s, c); y = s; break;
        case 7: y = tanh32_fast(x); break;
        default: sincos2pi32(x, s, c); y = c; break;
        }
        static_cast<float *>(out)[i] = y;
    } else {
        const double x = static_cast<const double *>(in)[i];
        double y;
        if (kind == 5) y = sin64(x);
        else if (kind == 6) y = cos64(x);
        else { double s, c; sincos64_full(x, s, c); y = kind == 8 ? s : c; }
        static_cast<double *>(out)[i] = y;
    }
}

extern "C" int ses_test_math(int32_t kind, const void *in_dev, void *out_dev, int64_t n, void *stream)
{
    if (kind < 0 || kind > 9) return fail("ses_test_math: unknown kind %d", kind);
    if (n < 1) return 0;
    k_test_math<<<(unsigned)((n + 255) / 256), 256, 0, S(stream)>>>(kind, in_dev, out_dev, (long long)n);
    CU(cudaGetLastError());
    return 0;
}

__global__ void k_test_normals(uint32_t seed, uint32_t gen, uint32_t id, int D, float *out)
{
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (4 * q >= D) return;
    const float4 n = normal4(seed, (uint32_t)q, id, gen);
    const int d = 4 * q;
    out[d] = n.x;
    if (d + 1 < D) out[d + 1] = n.y;
    if (d + 2 < D) out[d + 2] = n.z;
    if (d + 3 < D) out[d + 3] = n.w;
}

extern "C" int ses_test_k1_geometry(ses_handle *h, int32_t *out_host)
{
    if (!h || !out_host) return fail("ses_test_k1_geometry: null argument");
    for (int i = 0; i < 8; ++i) out_host[i] = h->k1_geometry[i];
    return 0;
}

extern "C" int ses_test_normals(ses_handle *h, uint32_t generation, int32_t id, float *out_dev, void *stream)
{
    if (!h || !out_dev) return fail("ses_test_normals: null argument");
    CU(cudaSetDevice(h->cfg.device));
    k_test_normals<<<(h->NQ + 63) / 64, 64, 0, S(stream)>>>(h->cfg.seed, generation, (uint32_t)id, h->D, out_dev);
    CU(cudaGetLastError());
    return 0;
}

// every float32 bit pattern b in [lo_bits, hi_bits]: tanh32_fast(x) must equal tanh32(x) bit for bit
__global__ void k_tanh_fast_exhaustive(uint32_t lo_bits, uint32_t hi_bits, unsigned long long *mismatches)
{
    unsigned long long bad = 0;
    const unsigned long long n = (unsigned long long)hi_bits - lo_bits + 1ull;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (unsigned long long)gridDim.x * blockDim.x) {
        const float x = __uint_as_float(lo_bits + (uint32_t)i);
        const uint32_t a = __float_as_uint(tanh32_fast(x)), b = __float_as_uint(tanh32(x));
        const uint32_t an = __float_as_uint(tanh32_fast(-x)), bn = __float_as_uint(tanh32(-x));
        // +0 and -0 compare equal (the only inputs that can differ in the sign of a zero result are x = +-0)
        bad += ((a != b) && ((a | b) << 1) != 0) + ((an != bn) && ((an | bn) << 1) != 0);
    }
    if (bad) atomicAdd(mismatches, bad);
}

// packed tanh: x in the low half with a far-away value in the high half and vice versa -- both halves must equal tanh32
template <bool NEWTON>
__global__ void k_tanh_x2_exhaustive(uint32_t lo_bits, uint32_t hi_bits, unsigned long long *mismatches)
{
    unsigned long long bad = 0;
    const unsigned long long n = (unsigned long long)hi_bits - lo_bits + 1ull;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (unsigned long long)gridDim.x * blockDim.x) {
        const float x = __uint_as_float(lo_bits + (uint32_t)i);
        const float2 y = tanh32x2<NEWTON>(make_float2(x, -x));
        const uint32_t a = __float_as_uint(y.x), b = __float_as_uint(tanh32(x));
        const uint32_t an = __float_as_uint(y.y), bn = __float_as_uint(tanh32(-x));
        bad += ((a != b) && ((a | b) << 1) != 0) + ((an != bn) && ((an | bn) << 1) != 0);
        // the scalar form with the same NEWTON choice (odd episodes / agents)
        const uint32_t s = __float_as_uint(tanh32_fast_t<NEWTON>(x)), sn = __float_as_uint(tanh32_fast_t<NEWTON>(-x));
        bad += ((s != b) && ((s | b) << 1) != 0) + ((sn != bn) && ((sn | bn) << 1) != 0);
    }
    if (bad) atomicAdd(mismatches, bad);
}

extern "C" int ses_test_tanh_x2_exhaustive(int32_t newton, float lo, float hi, uint64_t *mismatches_host)
{
    if (!mismatches_host || !(lo >= 0.0f) || !(hi >= lo)) return fail("ses_test_tanh_x2_exhaustive: bad arguments");
    unsigned long long *d = nullptr;
    CU(cudaMalloc(&d, sizeof(unsigned long long)));
    CU(cudaMemset(d, 0, sizeof(unsigned long long)));
    uint32_t lb, hb;
    memcpy(&lb, &lo, 4); memcpy(&hb, &hi, 4);
    if (newton) k_tanh_x2_exhaustive<true><<<148 * 16, 256>>>(lb, hb, d);
    else k_tanh_x2_exhaustive<false><<<148 * 16, 256>>>(lb, hb, d);
    CU(cudaGetLastError());
    unsigned long long r = 0;
    CU(cudaMemcpy(&r, d, sizeof(r), cudaMemcpyDeviceToHost));
    cudaFree(d);
    *mismatches_host = r;
    return 0;
}

extern "C" int ses_test_tanh_fast_exhaustive(float lo, float hi, uint64_t *mismatches_host)
{
    if (!mismatches_host || !(lo >= 0.0f) || !(hi >= lo)) return fail("ses_test_tanh_fast_exhaustive: bad arguments");
    unsigned long long *d = nullptr;
    CU(cudaMalloc(&d, sizeof(unsigned long long)));
    CU(cudaMemset(d, 0, sizeof(unsigned long long)));
    uint32_t lb, hb;
    memcpy(&lb, &lo, 4); memcpy(&hb, &hi, 4);
    k_tanh_fast_exhaustive<<<148 * 16, 256>>>(lb, hb, d);
    CU(cudaGetLastError());
    unsigned long long r = 0;
    CU(cudaMemcpy(&r, d, sizeof(r), cudaMemcpyDeviceToHost));
    cudaFree(d);
    *mismatches_host = r;
    return 0;
}

// div_total_mass(x) vs __ddiv_rn(x, 1.1) on n pseudo-random doubles (random sign, mantissa, exponent in [-60, 60])
__global__ void k_div11_check(unsigned long long n, unsigned long long *mismatches)
{
    unsigned long long bad = 0;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (unsigned long long)gridDim.x * blockDim.x) {
        const uint4 r = philox4x32_10((uint32_t)i, (uint32_t)(i >> 32), 0x51u, 0u, 0xC0FFEEu, 7u);
        const unsigned long long mant = (((unsigned long long)r.x << 32) | r.y) & 0x000FFFFFFFFFFFFFull;
        const unsigned long long expo = 1023ull - 60ull + (r.z % 121u);
        const unsigned long long sign = (unsigned long long)(r.w & 1u) << 63;
        const double x = __longlong_as_double((long long)(sign | (expo << 52) | mant));
        bad += __double_as_longlong(div_total_mass(x)) != __double_as_longlong(__ddiv_rn(x, 1.1));
    }
    if (bad) atomicAdd(mismatches, bad);
}

// ddiv_fast(a, b) vs __ddiv_rn(a, b) on n pseudo-random operand pairs of cartpole_step's ranges: |a| in [1, 64) (random sign
// and mantissa), b in [0.5, 1)
__global__ void k_ddiv_fast_check(unsigned long long n, unsigned long long *mismatches)
{
    unsigned long long bad = 0;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (unsigned long long)gridDim.x * blockDim.x) {
        const uint4 r = philox4x32_10((uint32_t)i, (uint32_t)(i >> 32), 0x52u, 0u, 0xD1Du, 9u);
        const uint4 t = philox4x32_10((uint32_t)i, (uint32_t)(i >> 32), 0x53u, 0u, 0xD1Du, 9u);
        const unsigned long long ma = (((unsigned long long)r.x << 32) | r.y) & 0x000FFFFFFFFFFFFFull;
        const unsigned long long mb = (((unsigned long long)r.z << 32) | r.w) & 0x000FFFFFFFFFFFFFull;
        const unsigned long long ea = 1023ull + (t.x % 6u);                      // 2^0 .. 2^5
        const unsigned long long sa = (unsigned long long)(t.y & 1u) << 63;
        const double a = __longlong_as_double((long long)(sa | (ea << 52) | ma));
        const double b = __longlong_as_double((long long)((1022ull << 52) | mb));  // [0.5, 1)
        bad += __double_as_longlong(ddiv_fast(a, b)) != __double_as_longlong(__ddiv_rn(a, b));
    }
    if (bad) atomicAdd(mismatches, bad);
}

extern "C" int ses_test_ddiv_fast(uint64_t n, uint64_t *mismatches_host)
{
    if (!mismatches_host) return fail("ses_test_ddiv_fast: null argument");
    unsigned long long *d = nullptr;
    CU(cudaMalloc(&d, sizeof(unsigned long long)));
    CU(cudaMemset(d, 0, sizeof(unsigned long long)));
    k_ddiv_fast_check<<<148 * 16, 256>>>((unsigned long long)n, d);
    CU(cudaGetLastError());
    unsigned long long r = 0;
    CU(cudaMemcpy(&r, d, sizeof(r), cudaMemcpyDeviceToHost));
    cudaFree(d);
    *mismatches_host = r;
    return 0;
}

extern "C" int ses_test_div_total_mass(uint64_t n, uint64_t *mismatches_host)
{
    if (!mismatches_host) return fail("ses_test_div_total_mass: null argument");
    unsigned long long *d = nullptr;
    CU(cudaMalloc(&d, sizeof(unsigned long long)));
    CU(cudaMemset(d, 0, sizeof(unsigned long long)));
    k_div11_check<<<148 * 16, 256>>>((unsigned long long)n, d);
    CU(cudaGetLastError());
    unsigned long long r = 0;
    CU(cudaMemcpy(&r, d, sizeof(r), cudaMemcpyDeviceToHost));
    cudaFree(d);
    *mismatches_host = r;
    return 0;
}
#endif  // SES_BUILD_TESTS

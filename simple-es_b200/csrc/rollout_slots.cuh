// rollout_slots.cuh -- the persistent "warp owns S offspring slots, lane owns one episode" rollout
// kernel, generic over the environment / policy pair (CartPole-v1 MLP, simple_spread MLP).
//
// Replaces, per generation: the mp.Pool fan-out (loop.py:66-78), RolloutWorker (loop.py:108-125),
// GymEnvModel.forward (networks/neural_network.py:20-36), the env wrappers' reset/step
// (envs/gym_wrapper.py:23-45,69-77, envs/pettingzoo_wrapper.py:22-58), the third-party physics
// (SURVEY.md Appendix A) and the perturbation half of _gen_offsprings
// (offspring_strategies.py:53-60,169-176,312-326).
//
// Mapping (DESIGN.md section 5): persistent warps, no inter-warp communication.
//   * a warp owns S "offspring slots" in shared memory; a slot holds the D perturbed weights of one
//     offspring as float4 quads, slot-interleaved ([quad][slot]) so that an LDS.128 of one quad by 32
//     lanes touches at most S*16 B = one conflict-free wavefront (S = 8).
//   * a lane runs ONE episode at a time: env state in registers, fp32 policy from the slot's weights.
//     When its episode ends it is handed the next pending (slot, episode) pair by a warp-synchronous
//     scheduler (ballot + prefix), so lanes stay busy although CartPole episodes last 8..500 steps.
//   * refill is demand driven: the warp takes just enough new offspring ids from a global atomic
//     counter to occupy its idle lanes, never more.  Only `lanes_used` = E*floor(32/E) lanes take
//     work, so when every episode has the same length (a converged CartPole population, or
//     simple_spread's fixed 25 cycles) whole slots start and finish together, no episode is left
//     waiting for a later round, and the last round of a generation is packed into few full warps
//     while the others exit.
//   * the weights of a new offspring are re-derived from Philox(generation, id) by the whole warp:
//     there is no noise table, and nothing but 16 B per offspring ever goes to HBM.
//
// An Env type provides:
//   D, NQ, STATE_DIM, N_AGENTS, UNIT_REWARD (reward == 1.0 per step: fitness = steps / E exactly)
//   struct State;  init<STREAM = STREAM_INIT>(State&, p, id, ep)
//   store_quad<S>(w[NQ][S], q, s, float4)   place flat parameter quad q of slot s (an Env may permute the table)
//   bind<S>(State&, w[NQ][S], slot)          a lane was handed an episode of `slot` (an Env may cache weights in registers)
//   step<S>(State&, w[NQ][S], slot, p, int *actions) -> done   (also adds the step reward to State::ret)
//   store_trace(State&, double *row)
//   store_init(State&, double *row)          the initial state in the layout of init_states rows (recording)
#pragma once
#include "ses_common.cuh"

namespace ses {

constexpr int WORK_COUNTER_TAIL = 1 + 256;   // work_counter: [0] queue A, [1 + smid] CTA arrivals per SM, [WORK_COUNTER_TAIL] queue B
constexpr int WORK_COUNTER_STEPS = WORK_COUNTER_TAIL + 1;   // (8-byte aligned) env steps of this launch: the launcher's episode-length estimate
constexpr int WORK_COUNTER_DONE = WORK_COUNTER_STEPS + 2;   // warps of this launch that have finished (folded peer barrier)
constexpr int WORK_COUNTER_INTS = WORK_COUNTER_DONE + 1;

// The barrier of a rollout launch runs in a SENTINEL CTA (one CTA more than the launch needs, the last block index): it waits
// until every worker warp of the launch has counted itself out (WORK_COUNTER_DONE; the workers' peer stores are fenced before
// that), then raises and awaits the flags.  The worker code gains one atomic at its very end and nothing else: a call at the
// workers' tail instead (last-arriving warp runs the barrier) cost the throughput loop 3.6-9 % through a different register
// allocation (profiles/r02_k1_experiments.md section 11).
__device__ __noinline__ void peer_sync_sentinel(const PeerSync s)
{
    const int lane = threadIdx.x & 31;
    if (threadIdx.x >= 32) return;
    if (lane == 0)
        while (*reinterpret_cast<volatile int *>(s.done) < s.expected) __nanosleep(200);
    __syncwarp();
    __threadfence();
    peer_flag_barrier(s, lane);
}

struct RolloutParams {
    const float *parents;        // [n_parents][D]
    const float *w_override;     // optional [n_local][D]
    const double *init_states;   // optional [E][state_dim]
    double *fitness;             // [P]
    long long *steps;            // [P]
    double *trace;               // optional [n_trace][200][state_dim]
    int *trace_actions;          // optional [n_trace][200][n_agents]
    int *work_counter;           // zeroed before launch; counts EPISODES handed out (local offspring index * E + episode)
    int *ep_acc;                 // [n_local][2] {steps, episodes done} of offspring whose episodes ran in more than one warp
                                 // (EPISODE_UNITS envs; all zero between launches: the last part to finish resets its pair)
    unsigned long long *total_steps;   // optional: += env steps simulated by this launch
    float sigma;
    uint32_t seed;
    uint32_t gen;
    Layout layout;
    Shard shard;                 // this rank's slice: local index (work queue) <-> global offspring id
    int E;
    int max_step;
    int pomdp;
    int init_mode;
    int n_trace;
    int slots_cap;               // <= S: slots a warp may hold
    int lanes_used;              // lanes of a warp that take episodes (E*floor(32/E) by default)
    int n_agents;                // simple_spread only
    int n_peers;                 // fused fitness exchange: other ranks' exchange buffers (NVLink peer memory)
    double *peer_fitness[MAX_PEERS];
    int sparse_rank;             // >= 0: warps of the CTAs that arrive on their SM as number sparse_rank or later take at most
    int sparse_quota;            //       sparse_quota offspring in total ("fractional" warps of a launch that does not fill the SMs)
    int split_ok;                // Envs with step_split(): a warp left with few episodes and nothing to refill spreads each over 2 / 4 lanes
    int tail_start;              // episodes [0, tail_start) are handed out in whole offspring (queue A = work_counter[0]), the rest --
                                 // EPISODE_UNITS envs: the last round's worth -- in exact numbers (queue B = work_counter[WORK_COUNTER_TAIL])
    PeerSync sync;               // sync.world > 1: the launch ends with the peer flag barrier (slot kernels)
    // policy evaluation (the EVAL instances, ses_evaluate): offspring id = policy * layout.group + chunk, a chunk is episodes
    // [chunk E, chunk E + E) of the policy, clipped to eval_episodes
    double *eval_returns;        // [n_pol][eval_episodes] return of every episode
    int *eval_lengths;           // [n_pol][eval_episodes] its env steps
    int eval_episodes;
    // recording (the TRACE && EVAL instances, ses_record): every step of every episode; trace / trace_actions are then
    // [n_pol][eval_episodes][max_step][state_dim | n_agents] and eval_returns is unused
    double *trace_returns;       // [n_pol][eval_episodes][max_step] return after each step
    double *trace_initial;       // [eval_episodes][state_dim] initial states (layout of init_states rows), written by policy 0
    // final states (the FINAL instances, ses_set_final_states): the state after each training episode's last step, in the
    // layout of Env::store_trace, at row (global id) * E + episode of [P][E][state_dim]; only the ids this handle owns
    double *final_states;
};

// row of (offspring id, episode e) in the final-state buffer: 64-bit, P * E * state_dim passes 2^31
__device__ __forceinline__ double *final_row(const RolloutParams &p, int id, int e, int state_dim)
{
    return p.final_states + ((size_t)id * p.E + e) * state_dim;
}

// row of (episode m of policy j, step t) in the recording buffers: 64-bit, n_pol * eval_episodes * max_step * state_dim
// passes 2^31 quickly
__device__ __forceinline__ size_t record_row(const RolloutParams &p, int j, int m, int t)
{
    return ((size_t)j * p.eval_episodes + m) * p.max_step + t;
}

// recording: the state, actions and return after step `nstep`, at row r of the recording buffers
template <class Env>
__device__ __forceinline__ void record_step(const RolloutParams &p, const typename Env::State &st, const int *actions, size_t r, int nstep)
{
    Env::store_trace(st, p.trace + r * Env::STATE_DIM);
#pragma unroll
    for (int a = 0; a < Env::N_AGENTS; ++a) p.trace_actions[r * Env::N_AGENTS + a] = actions[a];
    if constexpr (Env::UNIT_REWARD) p.trace_returns[r] = (double)nstep;
    else p.trace_returns[r] = st.ret;
}

constexpr int MAX_E = 32;

// Fitness all-gather fused into the rollout: the lane that retires an offspring stores its fitness into the
// exchange buffer of every peer GPU (plain st.global on NVLink-mapped peer pointers), so no collective has
// to move the vector afterwards; the flag barrier at the end of the launch (PeerSync) or ses_peer_barrier() publishes the
// stores (DESIGN.md section 6).
__device__ __forceinline__ void publish_fitness(const RolloutParams &p, int id, double f)
{
    p.fitness[id] = f;
    if (p.n_peers > 0) {
#pragma unroll 1
        for (int r = 0; r < p.n_peers; ++r) p.peer_fitness[r][id] = f;
        __threadfence_system();
    }
}

template <class Env, int S, bool NeedRet>
struct __align__(16) SlotSmem;

template <class Env, int S>
struct __align__(16) SlotSmem<Env, S, false> {
    float4 w[Env::NQ][S];
    int off_id[S];
    int ep_first[S];             // the slot runs episodes [ep_first, ep_first + ep_cnt) of its offspring (all E of them unless the
    int ep_cnt[S];               // env is EPISODE_UNITS and the queue handed this warp a part)
    int ep_next[S];              // ... of which ep_next have been handed to lanes and ep_done have ended
    int ep_done[S];
    int steps[S];
    int more, in_tail, quota, pad_;   // the warp's scheduler state: kept here, not in registers, so that the throughput loop's
};                                    // register allocation does not depend on the scheduler's bookkeeping

template <class Env, int S>
struct __align__(16) SlotSmem<Env, S, true> {
    float4 w[Env::NQ][S];
    double ret[S][MAX_E];        // per-episode returns, summed in episode order when the slot retires
    int off_id[S];
    int ep_first[S];
    int ep_cnt[S];
    int ep_next[S];
    int ep_done[S];
    int steps[S];
    int more, in_tail, quota, pad_;
};

template <class Env, class = void> struct EnvEpisodeUnits { static constexpr bool value = false; };
template <class Env> struct EnvEpisodeUnits<Env, decltype((void)Env::EPISODE_UNITS)> { static constexpr bool value = Env::EPISODE_UNITS; };

// A slot's episodes have all ended: emit the offspring's fitness (loop.py:124).  An offspring whose E episodes ran in ONE warp
// is emitted directly.  EPISODE_UNITS envs (reward 1 per step: the return is an integer step count) may have run parts of an
// offspring in different warps: each part adds its steps, then its episode count, to the offspring's pair in ep_acc; the part
// that completes the count emits the sum (integer addition: exact in any order) and clears the pair for the next launch.
// EVAL: every episode stored its return and length when it ended; nothing is left to emit.
template <class Env, bool EVAL = false, class Smem>
__device__ __forceinline__ void retire_slot(Smem &sm, const RolloutParams &p, int s, unsigned long long &warp_steps)
{
    const int id = sm.off_id[s];
    const int stp = sm.steps[s];
    warp_steps += (unsigned long long)stp;
    if constexpr (EVAL) {
        sm.off_id[s] = -1;
        return;
    }
    bool whole = true;
    if constexpr (EnvEpisodeUnits<Env>::value) whole = sm.ep_cnt[s] == p.E;
    if (whole) {
        p.steps[id] = (long long)stp;
        double total;
        if constexpr (Env::UNIT_REWARD) {
            total = (double)stp;                                    // reward 1.0 per step
        } else {
            total = 0.0;
            for (int e = 0; e < p.E; ++e) total = __dadd_rn(total, sm.ret[s][e]);
        }
        publish_fitness(p, id, __ddiv_rn(total, (double)p.E));
    } else {
        int *a = p.ep_acc + 2 * (size_t)p.shard.id_to_local(id);
        const int cnt = sm.ep_cnt[s];
        atomicAdd(a, stp);
        __threadfence();                                            // the steps are visible before the count that announces them
        if (atomicAdd(a + 1, cnt) + cnt == p.E) {
            __threadfence();
            const int tot = atomicExch(a, 0);
            atomicExch(a + 1, 0);
            p.steps[id] = (long long)tot;
            publish_fitness(p, id, __ddiv_rn((double)tot, (double)p.E));
        }
    }
    sm.off_id[s] = -1;
}

template <class Env, class = void> struct EnvSplit { static constexpr bool value = false; };
template <class Env> struct EnvSplit<Env, decltype((void)Env::SPLIT)> { static constexpr bool value = Env::SPLIT; };

// Straggler phase of the slot kernel (Envs that provide step_split<K, S>()): the warp's queue is empty and it holds at most
// 32 / K running episodes, so every further warp-step would cost a full step's latency for a handful of lanes.  The running
// episodes are compacted -- episode g moves to lanes [K g, K g + K) with its state replicated -- and stepped by K lanes each
// until they end, or until so few are left that twice as many lanes per episode fit (K = 2 -> 4).  A finished episode is
// booked into its slot (steps, ep_done) exactly as the throughput loop does; the caller retires the slots afterwards.
template <class Env, int S, int K, bool FINAL = false, class Smem>
__device__ __forceinline__ void run_split(Smem &sm, int pomdp, int max_step, int lane, bool &active, int &slot, int &nstep, double &x,
                                          double &xd, double &th, double &thd, [[maybe_unused]] int *ep = nullptr,
                                          [[maybe_unused]] double *final_states = nullptr, [[maybe_unused]] int E = 0)
{
    static_assert(Env::UNIT_REWARD && Env::N_AGENTS == 1, "run_split: CartPole-like envs");
    const unsigned FULL = 0xffffffffu;
    const unsigned act_mask = __ballot_sync(FULL, active);
    const int n_act = __popc(act_mask);
    const int g = lane / K;
    const int src = g < n_act ? __fns(act_mask, 0, g + 1) : lane;         // lane that holds the g-th running episode
    x = __shfl_sync(FULL, x, src); xd = __shfl_sync(FULL, xd, src);
    th = __shfl_sync(FULL, th, src); thd = __shfl_sync(FULL, thd, src);
    slot = __shfl_sync(FULL, slot, src); nstep = __shfl_sync(FULL, nstep, src);
    if constexpr (FINAL) *ep = __shfl_sync(FULL, *ep, src);
    active = g < n_act;
    if (!active) slot = 0;                                                // idle groups step a dummy episode (result unused)
    typename Env::template SplitW<K> wr;
    Env::template split_load<K, S>(wr, sm.w, slot, lane);
    constexpr int RESPLIT = K < 4 ? 32 / (2 * K) : 0;
    for (;;) {
        const int n = __popc(__ballot_sync(FULL, active)) / K;
        if (n == 0 || n <= RESPLIT) break;
        int action;
        bool done = Env::template step_split<K>(x, xd, th, thd, wr, pomdp, lane, action);
        if (active) {
            ++nstep;
            if (nstep >= max_step) done = true;
            if (done) {
                if ((lane & (K - 1)) == 0) {
                    if constexpr (FINAL) {
                        double *row = final_states + ((size_t)sm.off_id[slot] * E + *ep) * 4;
                        row[0] = x; row[1] = xd; row[2] = th; row[3] = thd;
                    }
                    atomicAdd(&sm.steps[slot], nstep);
                    atomicAdd(&sm.ep_done[slot], 1);
                }
                active = false;
                slot = 0;
            }
        }
    }
    active = active && (lane & (K - 1)) == 0;                             // the leader lane keeps the episode
    __syncwarp();
}

// Kept out of line (and fed scalars only) so that the throughput loop of k_rollout_slots keeps the register allocation and
// instruction schedule it has without this phase: the loop is bound by register-operand delivery, and its speed moved by
// 4-5 % with the allocation ptxas happened to choose when this code was inlined after it (profiles/r02_k1_experiments.md).
template <class Env, int S, class Smem>
__device__ __noinline__ void split_phase(Smem *smp, int pomdp, int max_step, int slot, int nstep, double x, double xd, double th, double thd)
{
    Smem &sm = *smp;
    const int lane = threadIdx.x & 31;
    bool active = slot >= 0;
    if (__popc(__ballot_sync(0xffffffffu, active)) > 8)
        run_split<Env, S, 2>(sm, pomdp, max_step, lane, active, slot, nstep, x, xd, th, thd);      // returns when <= 8 are left
    if (__ballot_sync(0xffffffffu, active))
        run_split<Env, S, 4>(sm, pomdp, max_step, lane, active, slot, nstep, x, xd, th, thd);      // runs them to their end
}

// The straggler phase of the FINAL instances: as split_phase, and the lane that ends an episode stores its final state.  A
// function of its own so that split_phase keeps its signature and code.
template <class Env, int S, class Smem>
__device__ __noinline__ void split_phase_final(Smem *smp, int pomdp, int max_step, int slot, int nstep, double x, double xd, double th,
                                               double thd, int ep, double *final_states, int E)
{
    Smem &sm = *smp;
    const int lane = threadIdx.x & 31;
    bool active = slot >= 0;
    if (__popc(__ballot_sync(0xffffffffu, active)) > 8)
        run_split<Env, S, 2, true>(sm, pomdp, max_step, lane, active, slot, nstep, x, xd, th, thd, &ep, final_states, E);
    if (__ballot_sync(0xffffffffu, active))
        run_split<Env, S, 4, true>(sm, pomdp, max_step, lane, active, slot, nstep, x, xd, th, thd, &ep, final_states, E);
}

// PEER: the instance launched when the launch ends with the peer flag barrier (sentinel CTA + one atomic at the workers' end); a
// separate instance so that single-GPU launches keep the exact code they have without it.
// EVAL: the policy-evaluation instance (ses_evaluate): unperturbed policies, STREAM_EVAL initial states, per-episode returns and
// lengths instead of fitness; no straggler phase.  Separate so that the training instances keep their code.
// FINAL: the training instance that also stores the final state of every episode (p.final_states), written by the lane that
// ends the episode, in the throughput loop or the straggler phase.  Separate for the same reason.
template <class Env, int S, int WARPS, bool TRACE, bool PEER = false, bool EVAL = false, bool FINAL = false>
__global__ void __launch_bounds__(WARPS * 32) k_rollout_slots(const RolloutParams p)
{
    using Smem = SlotSmem<Env, S, !Env::UNIT_REWARD>;
    constexpr int NQ = Env::NQ, D = Env::D;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    Smem &sm = reinterpret_cast<Smem *>(smem_raw)[threadIdx.x >> 5];
    const int lane = threadIdx.x & 31;
    const unsigned FULL = 0xffffffffu;
    const unsigned lt = lanemask_lt();
    const bool usable = lane < p.lanes_used;

    if constexpr (PEER) {
        if (blockIdx.x == gridDim.x - 1) {                             // the sentinel CTA of a launch that ends with the peer barrier
            peer_sync_sentinel(p.sync);
            return;
        }
    }
    if (lane < S) { sm.off_id[lane] = -1; sm.ep_first[lane] = 0; sm.ep_cnt[lane] = 0; sm.ep_next[lane] = 0; sm.ep_done[lane] = 0; sm.steps[lane] = 0; }
    __syncwarp();
    // Sparse warps.  A launch whose episodes do not fill every resident warp (one rank's share of an 8-GPU run: 2.3 warps
    // per SM sub-partition) would leave some sub-partitions with three full warps and others with two; the former set the
    // time.  Instead every SM gets the same CTAs: those that arrive first take full loads, the CTA that arrives as number
    // sparse_rank shares what is left -- a few episodes per warp, which the straggler phase then runs on 2 or 4 lanes each,
    // at a fraction of a full warp's cost per step.  work_counter[1 + smid] counts the CTAs arriving on an SM.
    int quota0 = 0x7fffffff;
    if (p.sparse_rank >= 0) {
        __shared__ int cta_rank_s;
        if (threadIdx.x == 0) {
            unsigned smid;
            asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
            cta_rank_s = atomicAdd(p.work_counter + 1 + (smid & 255u), 1);
        }
        __syncthreads();
        if (cta_rank_s >= p.sparse_rank) quota0 = p.sparse_quota;
    }
    if (lane == 0) { sm.more = 1; sm.in_tail = p.tail_start <= 0; sm.quota = quota0; }
    __syncwarp();

    // per-lane episode state
    int slot = -1, nstep = 0;
    [[maybe_unused]] int ep = 0;
    typename Env::State st;
    unsigned long long warp_steps = 0;   // lanes < S: steps of the offspring they retired
    bool sched = true;         // warp-uniform: something changed that the scheduler must look at
    [[maybe_unused]] bool to_split = false;

    for (;;) {
        if (sched) {
            // ------------------------------------------------------------------ scheduler
            __syncwarp();
            // warp-uniform scheduler state (SlotSmem): more = the episode queues may still hold work; in_tail = queue A (whole
            // offspring) is exhausted, requests go to queue B; quota = what a sparse warp may still take
            bool more = sm.more != 0, in_tail = sm.in_tail != 0;
            int quota = sm.quota;
            int my_id = -1;
            if (lane < S) {
                my_id = sm.off_id[lane];
                if (my_id >= 0 && sm.ep_done[lane] == sm.ep_cnt[lane]) {   // every episode of the slot has ended
                    retire_slot<Env, EVAL>(sm, p, lane, warp_steps);
                    my_id = -1;
                }
            }
            const unsigned empty_mask = __ballot_sync(FULL, lane < p.slots_cap && my_id < 0);
            const int n_empty = __popc(empty_mask);
            const int pend_mine = (lane < S && my_id >= 0) ? (sm.ep_cnt[lane] - sm.ep_next[lane]) : 0;
            int pending = pend_mine;
#pragma unroll
            for (int o = 16; o; o >>= 1) pending += __shfl_xor_sync(FULL, pending, o);
            const unsigned idle_mask = __ballot_sync(FULL, usable && slot < 0);
            const int n_idle = __popc(idle_mask);
            // Demand-driven refill: just enough episodes to occupy the idle lanes (episode index = local offspring * E + episode).
            // The bulk of a launch, [0, tail_start), is handed out in WHOLE offspring from queue A: the request is rounded up to a
            // multiple of E and the episodes that find no lane wait in the slot for the warp's next round, so an offspring's
            // weights are derived once.  Envs whose returns are integer step counts (EPISODE_UNITS) hand out the last round's worth,
            // [tail_start, n_total), from queue B in EXACT numbers: a warp whose lanes came free together takes precisely that many
            // episodes (rounding up there would leave every warp a few episodes for one more, nearly empty, round), and a sparse
            // warp takes its small share.  An exact range may leave an offspring's episodes to two warps (retire_slot adds them up).
            const int n_total = p.shard.n_local * p.E;
            int want = n_idle - pending;
            bool exact = false;
            int cap = n_empty * p.E;                               // queue A is aligned: n E episodes are n offspring
            bool realign = false;
            if constexpr (EnvEpisodeUnits<Env>::value) {
                if (in_tail) {
                    // a lane or two coming free at a time (ragged episode lengths) still take whole offspring
                    exact = quota != 0x7fffffff || want >= 2 * p.E || n_empty == 1;
                    cap = n_empty > 0 ? (n_empty - 1) * p.E + 1 : 0;   // whatever the range's alignment it spans <= n_empty offspring
                    realign = !exact && want > 0 && more;
                }
            }
            if (realign) {
                // Queue B may stand in the middle of an offspring (an exact request left it there).  A whole-offspring request then
                // takes that offspring's remaining episodes first, so that its range ENDS on an offspring boundary and the queue is
                // aligned again for everybody: k E - m episodes, m = episodes of the front offspring already gone (read, not
                // reserved: if another warp gets in between, the next request of this kind repairs the alignment).
                int c = 0;
                if (lane == 0) c = *reinterpret_cast<volatile int *>(p.work_counter + WORK_COUNTER_TAIL);
                c = __shfl_sync(FULL, c, 0);
                const int m = c % p.E;
                const int k = min((want + m + p.E - 1) / p.E, n_empty - 1);
                want = k > 0 ? k * p.E - m : 0;
            } else if (!exact) {
                want = ((want + p.E - 1) / p.E) * p.E;
            }
            want = min(min(max(want, 0), cap), quota);
            if (quota == 0) more = false;                          // a sparse warp that has taken its share (the launcher sizes the
                                                                   // shares so that together they cover the launch)
            bool rerun = false;
            if (want > 0 && more) {
                int base = 0, got;
                if (!in_tail) {
                    if (lane == 0) base = atomicAdd(p.work_counter, want);
                    base = __shfl_sync(FULL, base, 0);             // first episode of the range this warp was given
                    got = max(0, min(want, p.tail_start - base));
                    if (base + want >= p.tail_start) {             // queue A is exhausted: go on with queue B
                        in_tail = true;
                        if (p.tail_start >= n_total) more = false;
                        rerun = got < want && more;                // ... at once if this request came up short
                    }
                } else {
                    if (lane == 0) base = atomicAdd(p.work_counter + WORK_COUNTER_TAIL, want);
                    base = p.tail_start + __shfl_sync(FULL, base, 0);
                    got = max(0, min(want, n_total - base));
                    if (base + want >= n_total) more = false;
                    if (quota != 0x7fffffff) { quota -= want; if (quota == 0) more = false; }
                }
                const int off0 = base / p.E;                       // local index of the first offspring the range touches
                const int n_off = got > 0 ? (base + got - 1) / p.E - off0 + 1 : 0;
                const int my_rank = __popc(empty_mask & lt);       // rank of this lane's slot among the empty ones
                const bool fill = ((empty_mask >> lane) & 1u) && my_rank < n_off;
                if (fill) {
                    const int ol = off0 + my_rank;
                    const int lo = max(base, ol * p.E) - ol * p.E;
                    int hi = min(base + got, (ol + 1) * p.E) - ol * p.E;
                    if constexpr (EVAL) hi = min(hi, p.eval_episodes - (ol % p.layout.group) * p.E);   // a partial last chunk
                    sm.off_id[lane] = p.shard.local_to_id(ol);
                    sm.ep_first[lane] = lo;
                    sm.ep_cnt[lane] = hi - lo;
                    sm.ep_next[lane] = 0;
                    sm.ep_done[lane] = 0;
                    sm.steps[lane] = 0;
                }
                const unsigned fill_mask = __ballot_sync(FULL, fill);
                __syncwarp();
                // regenerate the weights of the newly filled slots: (slot, quad) tasks over 32 lanes
                const int ntask = n_off * NQ;
                for (int t = lane; t < ntask; t += 32) {
                    const int k = t / NQ, q = t - k * NQ;
                    const int s = __fns(fill_mask, 0, k + 1);      // k-th filled slot
                    const int id = sm.off_id[s];
                    float4 wq;
                    if (p.w_override) {
                        const float *row = p.w_override + (size_t)p.shard.id_to_local(id) * D;
                        const int d = 4 * q;
                        wq.x = row[d];
                        wq.y = d + 1 < D ? row[d + 1] : 0.0f;
                        wq.z = d + 2 < D ? row[d + 2] : 0.0f;
                        wq.w = d + 3 < D ? row[d + 3] : 0.0f;
                    } else {
                        float sg;
                        const uint32_t nid = p.layout.noise_id(id, sg);
                        wq = offspring_quad(p.parents + (size_t)p.layout.parent(id) * D, D, q,
                                            p.layout.perturbed(id), __fmul_rn(p.sigma, sg), p.seed, nid, p.gen);
                    }
                    Env::template store_quad<S>(sm.w, q, s, wq);
                }
                __syncwarp();
            }
            // hand pending (slot, episode) pairs to idle lanes, in slot order (the barrier orders the retire / refill
            // writes of lanes < S to off_id / ep_next before every lane reads them: votes alone do not order memory)
            __syncwarp();
            const int r = __popc(idle_mask & lt);
            int acc = 0, my_slot = -1, my_ep = 0, my_prefix = 0, my_avail = 0;
#pragma unroll
            for (int s = 0; s < S; ++s) {
                const int nx = sm.ep_next[s];
                const int av = (sm.off_id[s] >= 0) ? (sm.ep_cnt[s] - nx) : 0;
                if (usable && slot < 0 && my_slot < 0 && r < acc + av) { my_slot = s; my_ep = sm.ep_first[s] + nx + (r - acc); }
                if (lane == s) { my_prefix = acc; my_avail = av; }
                acc += av;
            }
            __syncwarp();
            if (lane < S) sm.ep_next[lane] += max(0, min(my_avail, n_idle - my_prefix));
            __syncwarp();
            if (my_slot >= 0) {
                slot = my_slot; ep = my_ep; nstep = 0;
                if constexpr (EVAL) Env::template init<STREAM_EVAL>(st, p, 0, (sm.off_id[my_slot] % p.layout.group) * p.E + my_ep);
                else Env::init(st, p, sm.off_id[my_slot], my_ep);
                if constexpr (EVAL && TRACE) {                      // recording: the chunks of policy 0 store the initial states
                    const int vid = sm.off_id[my_slot];
                    if (vid < p.layout.group) Env::store_init(st, p.trace_initial + (size_t)(vid * p.E + my_ep) * Env::STATE_DIM);
                }
                Env::template bind<S>(st, sm.w, my_slot);
            }
            __syncwarp();
            if (lane == 0) { sm.more = more; sm.in_tail = in_tail; sm.quota = quota; }
            if (rerun) continue;                                   // queue A ran dry under this request: ask queue B for the rest
            const unsigned act_mask = __ballot_sync(FULL, slot >= 0);
            if (act_mask == 0) break;                              // queue empty and every lane idle
            if constexpr (EnvSplit<Env>::value && !TRACE && !EVAL) {
                // nothing left to hand out (queue empty, every pending pair has a lane) and few episodes running: leave the
                // throughput loop for the straggler phase below
                if (p.split_ok && !more && acc <= n_idle && __popc(act_mask) <= 16) { to_split = true; break; }
            }
        }

        bool just_done = false;
        if (slot >= 0) {
            // ------------------------------------------------------------------ one env step
            int actions[Env::N_AGENTS];
            bool done = Env::template step<S>(st, sm.w, slot, p, actions);
            ++nstep;                                               // gym_wrapper.py:33 / pettingzoo_wrapper.py:34
            if (nstep >= p.max_step) done = true;                  // gym_wrapper.py:37-39, TimeLimit / max_cycles
            if constexpr (TRACE && EVAL) {
                const int vid = sm.off_id[slot];
                record_step<Env>(p, st, actions, record_row(p, vid / p.layout.group, (vid % p.layout.group) * p.E + ep, nstep - 1), nstep);
            } else if constexpr (TRACE) {
                const int local = p.shard.id_to_local(sm.off_id[slot]);
                if (ep == 0 && local < p.n_trace && nstep <= 200) {
                    Env::store_trace(st, p.trace + ((size_t)local * 200 + (nstep - 1)) * Env::STATE_DIM);
#pragma unroll
                    for (int a = 0; a < Env::N_AGENTS; ++a) p.trace_actions[((size_t)local * 200 + (nstep - 1)) * Env::N_AGENTS + a] = actions[a];
                }
            }
            if (done) {
                if constexpr (EVAL) {
                    const int vid = sm.off_id[slot];
                    const size_t at = (size_t)(vid / p.layout.group) * p.eval_episodes + (vid % p.layout.group) * p.E + ep;
                    if constexpr (!TRACE) {                         // (recording stored the returns step by step)
                        if constexpr (Env::UNIT_REWARD) p.eval_returns[at] = (double)nstep;
                        else p.eval_returns[at] = st.ret;
                    }
                    p.eval_lengths[at] = nstep;
                } else if constexpr (!Env::UNIT_REWARD) {
                    sm.ret[slot][ep] = st.ret;
                }
                if constexpr (FINAL) Env::store_trace(st, final_row(p, sm.off_id[slot], ep, Env::STATE_DIM));
                atomicAdd(&sm.steps[slot], nstep);
                atomicAdd(&sm.ep_done[slot], 1);
                slot = -1;
                just_done = true;
            }
        }
        // the scheduler has work only right after an episode ended (a lane to re-arm, maybe a slot
        // to retire and refill); otherwise idle lanes stay idle and the warp keeps stepping
        sched = __ballot_sync(FULL, just_done) != 0;
    }
    if constexpr (EnvSplit<Env>::value && !TRACE && !EVAL) {
        // ------------------------------------------------------------------ straggler phase (kept out of the loop above so
        // that its code does not touch the throughput loop's register allocation and schedule)
        if (to_split) {
            if constexpr (FINAL) split_phase_final<Env, S, Smem>(&sm, p.pomdp, p.max_step, slot, nstep, st.x, st.xd, st.th, st.thd, ep, p.final_states, p.E);
            else split_phase<Env, S, Smem>(&sm, p.pomdp, p.max_step, slot, nstep, st.x, st.xd, st.th, st.thd);
            __syncwarp();
            if (lane < S && sm.off_id[lane] >= 0) retire_slot<Env>(sm, p, lane, warp_steps);   // every slot the warp still holds
        }
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) warp_steps += __shfl_xor_sync(FULL, warp_steps, o);
    if (lane == 0 && warp_steps) {
        if (p.total_steps) atomicAdd(p.total_steps, warp_steps);
        atomicAdd(reinterpret_cast<unsigned long long *>(p.work_counter + WORK_COUNTER_STEPS), warp_steps);
    }
    if constexpr (PEER) {
        if (lane == 0) {                                               // folded peer barrier: count this warp out (its peer
            __threadfence_system();                                    // stores first) for the sentinel CTA
            atomicAdd(p.work_counter + WORK_COUNTER_DONE, 1);
        }
    }
}

}  // namespace ses

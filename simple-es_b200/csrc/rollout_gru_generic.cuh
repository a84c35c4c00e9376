// rollout_gru_generic.cuh -- K1 with the recurrent policy (`gru: True`) for every environment other than CartPole:
// MountainCar-v0, Acrobot-v1, Pendulum-v0 (continuous head) and simple_spread N = 2 / 3 (one hidden state per agent).
//
// Replaces GymEnvModel's GRU branch (networks/neural_network.py:15-16,25-27,38-40; torch nn.GRU cell, SURVEY.md Appendix A.3)
// driven per agent copy as wrap_agentid builds them (learning_strategies/evolution/utils.py:4-8: one deepcopy per agent id --
// shared weights, one hidden state each), the episode loop (loop.py:108-125) and the wrappers' reset / step.
//
// Mapping: as rollout_cartpole_gru.cuh -- a WARP owns one offspring, its 26 kB of gate weights live in shared memory as
// packed pairs, lane j owns hidden unit j -- generalised over the environment: EC episodes of the offspring run in lockstep
// and every (episode, agent) pair is one "virtual" policy evaluation v = e * N_AGENTS + a, V = EC * N_AGENTS of them share
// each weight read.  Lane e (e < EC) owns the float64 state of episode e (Env::State), computes its agents' observations
// (Env::observe) and steps it (Env::advance); the logits of the V evaluations are computed by V * ACT lanes at once (one fc2
// row each, the contract's four blocks of eight) and gathered by the owner lanes with shuffles.
// The CartPole kernel keeps its own, tuned, file; this one trades its tricks for generality.
#pragma once
#include "rollout_cartpole_gru.cuh"
#include "rollout_classic.cuh"
#include "rollout_mpe.cuh"

namespace ses {

template <class Env>
struct GruLayout {
    static constexpr int OBS = Env::OBS, ACT = Env::ACT;
    // flat parameter offsets (nn.Module.parameters() order, networks/neural_network.py:12-17)
    static constexpr int O_W1 = 0, O_B1 = HID * OBS, O_WIH = O_B1 + HID, O_WHH = O_WIH + G3 * HID, O_BIH = O_WHH + G3 * HID,
                         O_BHH = O_BIH + G3, O_W2 = O_BHH + G3, O_B2 = O_W2 + ACT * HID, D = O_B2 + ACT;
    static_assert(D == param_count(OBS, ACT, 1), "GRU parameter layout");
    static constexpr int NQ = (D + 3) / 4;
};

template <class Env, int EC>
struct __align__(16) GruGenSmem {
    static constexpr int V = EC * Env::N_AGENTS;
    static constexpr int OBS_PAD = (Env::OBS_EFF + 3) / 4 * 4;
    float4 wrz_i[HID / 2][HID];    // { W_ir[j][k], W_iz[j][k], W_ir[j][k+1], W_iz[j][k+1] } at [k/2][j]  (rollout_cartpole_gru.cuh)
    float4 wrz_h[HID / 2][HID];
    float4 wn[HID / 2][HID];       // { W_in[j][k], W_hn[j][k], W_in[j][k+1], W_hn[j][k+1] }
    float w1t[Env::OBS][HID];      // fc1 transposed: w1t[k][j] = W1[j][k] (lane j walks a column: conflict free)
    float b1[HID];
    float bih[G3], bhh[G3];
    float w2[Env::ACT][HID];
    float b2[8];
    float2 xh[V][HID];             // { tanh(fc1)[k], h[k] } per evaluation
    float obuf[V][HID + 4];        // tanh(h') per evaluation
    float obs[V][OBS_PAD];         // observations, written by the owner lanes
};

// place flat parameter d of the offspring into the warp's tables
template <class Env, int EC>
__device__ __forceinline__ void gru_gen_store(GruGenSmem<Env, EC> &sm, int d, float val)
{
    using L = GruLayout<Env>;
    if (d < L::O_B1) {
        const int j = d / L::OBS, k = d - j * L::OBS;
        sm.w1t[k][j] = val;
    } else if (d < L::O_WIH) {
        sm.b1[d - L::O_B1] = val;
    } else if (d < L::O_BIH) {
        const int hh = d >= L::O_WHH;
        const int o = d - (hh ? L::O_WHH : L::O_WIH);
        const int row = o >> 5, k = o & 31, g = row >> 5, j = row & 31;          // torch gate order r, z, n
        float *base = reinterpret_cast<float *>(g == 2 ? &sm.wn[0][0] : (hh ? &sm.wrz_h[0][0] : &sm.wrz_i[0][0]));
        const int comp = g == 2 ? hh : g;
        base[((size_t)(k >> 1) * HID + j) * 4 + 2 * (k & 1) + comp] = val;
    } else if (d < L::O_BHH) {
        sm.bih[d - L::O_BIH] = val;
    } else if (d < L::O_W2) {
        sm.bhh[d - L::O_BHH] = val;
    } else if (d < L::O_B2) {
        const int o = d - L::O_W2;
        sm.w2[o >> 5][o & 31] = val;
    } else if (d < L::D) {
        sm.b2[d - L::O_B2] = val;
    }
}

// fc2 row under contract 4.4: four blocks of eight hidden units, block sums added to the bias in block order
__device__ __forceinline__ float fc2_row_blocks(const float *w, const float *x, float bias)
{
    float a = bias;
#pragma unroll
    for (int g = 0; g < HID / 8; ++g) {
        float sb = 0.0f;
#pragma unroll
        for (int j = 8 * g; j < 8 * g + 8; ++j) sb = fmaf(w[j], x[j], sb);
        a = __fadd_rn(a, sb);
    }
    return a;
}

// EVAL (ses_evaluate): one chunk of p.E == EC episodes per virtual offspring (policy * layout.group + chunk), the policy's last
// chunk partial; initial states from STREAM_EVAL, and every episode stores its return and length instead of a fitness.
// TRACE && EVAL (ses_record): every step of every episode is recorded as well (record_step; the owner lanes write).
// FINAL (training, ses_set_final_states): the owner lanes store each episode's final state.
template <class Env, int EC, int WARPS, bool TRACE, bool EVAL = false, bool FINAL = false>
__global__ void __launch_bounds__(WARPS * 32) k_rollout_gru_generic(const RolloutParams p)
{
    using Smem = GruGenSmem<Env, EC>;
    using L = GruLayout<Env>;
    constexpr int NA = Env::N_AGENTS, V = EC * NA, OE = Env::OBS_EFF, ACT = Env::ACT;
    static_assert(V * ACT <= 32, "one lane per (evaluation, action) logit");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    Smem &sm = reinterpret_cast<Smem *>(smem_raw)[threadIdx.x >> 5];
    const int lane = threadIdx.x & 31;
    const unsigned FULL = 0xffffffffu;

    unsigned long long warp_steps = 0;
    for (;;) {
        // ---------------------------------------------------------------- next offspring
        int local_idx = 0;
        if (lane == 0) local_idx = atomicAdd(p.work_counter, 1);
        local_idx = __shfl_sync(FULL, local_idx, 0);
        if (local_idx >= p.shard.n_local) break;
        const int id = p.shard.local_to_id(local_idx);
        __syncwarp();
        {
            const float *prow = p.w_override ? p.w_override + (size_t)local_idx * L::D : p.parents + (size_t)p.layout.parent(id) * L::D;
            const bool pert = p.w_override ? false : p.layout.perturbed(id);
            float sg;
            const uint32_t nid = p.layout.noise_id(id, sg);
            for (int q = lane; q < L::NQ; q += 32) {
                const float4 w = offspring_quad(prow, L::D, q, pert, __fmul_rn(p.sigma, sg), p.seed, nid, p.gen);
                gru_gen_store<Env, EC>(sm, 4 * q, w.x); gru_gen_store<Env, EC>(sm, 4 * q + 1, w.y);
                gru_gen_store<Env, EC>(sm, 4 * q + 2, w.z); gru_gen_store<Env, EC>(sm, 4 * q + 3, w.w);
            }
        }
        __syncwarp();
        const float b1 = sm.b1[lane];
        const float bir = sm.bih[lane], biz = sm.bih[HID + lane], bin = sm.bih[2 * HID + lane];
        const float bhr = sm.bhh[lane], bhz = sm.bhh[HID + lane], bhn = sm.bhh[2 * HID + lane];

        double total = 0.0;                                           // sum over episodes, in episode order, of the episode returns
        long long total_steps = 0;
        [[maybe_unused]] const int m0 = EVAL ? (id % p.layout.group) * p.E : 0;     // EVAL: the chunk's first episode
        for (int e0 = 0; e0 < p.E; e0 += EC) {
            const int ne = EVAL ? min(EC, p.eval_episodes - m0) : min(EC, p.E - e0);
            typename Env::State st;                                    // lane e < ne: episode e0 + e (other lanes: a harmless copy)
            if constexpr (EVAL) Env::template init<STREAM_EVAL>(st, p, 0, m0 + (lane < ne ? lane : 0));
            else Env::init(st, p, id, e0 + (lane < ne ? lane : 0));
            if constexpr (EVAL && TRACE) {                             // recording: the chunks of policy 0 store the initial states
                if (lane < ne && id < p.layout.group) Env::store_init(st, p.trace_initial + (size_t)(m0 + lane) * Env::STATE_DIM);
            }
            bool alive = lane < ne;
            int nstep = 0;
            float h[V];
#pragma unroll
            for (int v = 0; v < V; ++v) { h[v] = 0.0f; sm.xh[v][lane] = make_float2(0.0f, 0.0f); }      // model.reset() per agent copy
            // recording: row of this lane's episode (computed once: inside the loop the Acrobot instance spilled 32 B instead of 8)
            [[maybe_unused]] size_t rec = 0;
            if constexpr (EVAL && TRACE) rec = record_row(p, id / p.layout.group, m0 + lane, 0);
            unsigned alive_mask = __ballot_sync(FULL, alive);
            while (alive_mask) {
                // observations of every agent of every episode
                if (lane < EC) {
                    float o[NA][OE];
                    Env::observe(st, o);
#pragma unroll
                    for (int a = 0; a < NA; ++a)
#pragma unroll
                        for (int k = 0; k < OE; ++k) sm.obs[lane * NA + a][k] = o[a][k];
                }
                __syncwarp();
                // fc1 + tanh: lane j, every evaluation (skipped trailing inputs are exactly 0: fmaf(w, 0, a) == a)
#pragma unroll
                for (int v = 0; v < V; ++v) {
                    float a = b1;
#pragma unroll
                    for (int k = 0; k < OE; ++k) a = fmaf(sm.w1t[k][lane], sm.obs[v][k], a);
                    sm.xh[v][lane].x = tanh32_fast_t<false>(a);
                }
                __syncwarp();
                // gate pre-activations of lane j as pairs: { r_i, z_i } (W_ih x), { r_h, z_h } (W_hh h), { n_i, n_h }
                float2 grz_i[V], grz_h[V], gn[V];
#pragma unroll
                for (int v = 0; v < V; ++v) { grz_i[v] = make_float2(bir, biz); grz_h[v] = make_float2(bhr, bhz); gn[v] = make_float2(bin, bhn); }
#pragma unroll 2
                for (int kp = 0; kp < HID / 2; ++kp) {
                    const float4 a = sm.wrz_i[kp][lane], c = sm.wrz_h[kp][lane], n = sm.wn[kp][lane];
#pragma unroll
                    for (int v = 0; v < V; ++v) {
                        const float4 xv = *reinterpret_cast<const float4 *>(&sm.xh[v][2 * kp]);     // { x[k], h[k], x[k+1], h[k+1] }
                        grz_i[v] = __ffma2_rn(make_float2(a.x, a.y), make_float2(xv.x, xv.x), grz_i[v]);
                        grz_h[v] = __ffma2_rn(make_float2(c.x, c.y), make_float2(xv.y, xv.y), grz_h[v]);
                        gn[v] = __ffma2_rn(make_float2(n.x, n.y), make_float2(xv.x, xv.y), gn[v]);
                        grz_i[v] = __ffma2_rn(make_float2(a.z, a.w), make_float2(xv.z, xv.z), grz_i[v]);
                        grz_h[v] = __ffma2_rn(make_float2(c.z, c.w), make_float2(xv.w, xv.w), grz_h[v]);
                        gn[v] = __ffma2_rn(make_float2(n.z, n.w), make_float2(xv.z, xv.w), gn[v]);
                    }
                }
                __syncwarp();                                          // everyone has read xh before h is rewritten
                // GRU cell (torch gate order r, z, n) and the output non-linearity
#pragma unroll
                for (int v = 0; v < V; ++v) {
                    const float2 sres = __fadd2_rn(grz_i[v], grz_h[v]);
                    const float2 t = tanh32x2<false>(__fmul2_rn(make_float2(0.5f, 0.5f), sres));
                    const float2 rz = __ffma2_rn(make_float2(0.5f, 0.5f), t, make_float2(0.5f, 0.5f));       // sigm32
                    const float ng = tanh32_fast_t<false>(fmaf(rz.x, gn[v].y, gn[v].x));
                    h[v] = fmaf(rz.y, h[v], __fmul_rn(__fsub_rn(1.0f, rz.y), ng));
                    sm.xh[v][lane].y = h[v];
                    sm.obuf[v][lane] = tanh32_fast_t<false>(h[v]);
                }
                __syncwarp();
                // logits: lane v * ACT + m evaluates row m of fc2 for evaluation v; the owner lanes gather theirs
                float z = 0.0f;
                if (lane < V * ACT) {
                    const int v = lane / ACT, m = lane - v * ACT;
                    z = fc2_row_blocks(sm.w2[m], sm.obuf[v], sm.b2[m]);
                }
                float zz[NA][ACT];
                const int own = lane < EC ? lane : 0;
#pragma unroll
                for (int a = 0; a < NA; ++a)
#pragma unroll
                    for (int m = 0; m < ACT; ++m) zz[a][m] = __shfl_sync(FULL, z, (own * NA + a) * ACT + m);
                if (alive) {
                    int actions[NA];
#pragma unroll
                    for (int a = 0; a < NA; ++a) {
                        if constexpr (Env::CONTINUOUS) {
                            actions[a] = __float_as_int(tanh32_fast_t<false>(zz[a][0]));       // tanh head (neural_network.py:32-33)
                        } else {
                            // argmax(softmax(z)) with the float32 collapse rule (neural_network.py:30-31)
                            float zmax = zz[a][0];
#pragma unroll
                            for (int m = 1; m < ACT; ++m) zmax = fmaxf(zmax, zz[a][m]);
                            int act = ACT - 1;
#pragma unroll
                            for (int m = ACT - 2; m >= 0; --m)
                                if (__fsub_rn(zmax, zz[a][m]) <= __uint_as_float(0x33000000u)) act = m;
                            actions[a] = act;
                        }
                    }
                    bool done = Env::advance(st, actions);
                    ++nstep;
                    if (nstep >= p.max_step) done = true;
                    if constexpr (TRACE && EVAL) {
                        record_step<Env>(p, st, actions, rec + (nstep - 1), nstep);
                    } else if constexpr (TRACE) {
                        if (e0 + lane == 0 && local_idx < p.n_trace && nstep <= 200) {
                            Env::store_trace(st, p.trace + ((size_t)local_idx * 200 + (nstep - 1)) * Env::STATE_DIM);
#pragma unroll
                            for (int a = 0; a < NA; ++a) p.trace_actions[((size_t)local_idx * 200 + (nstep - 1)) * NA + a] = actions[a];
                        }
                    }
                    if (done) alive = false;
                }
                alive_mask = __ballot_sync(FULL, alive);
            }
            if constexpr (FINAL) {
                if (lane < ne) Env::store_trace(st, final_row(p, id, e0 + lane, Env::STATE_DIM));
            }
            if constexpr (EVAL) {
                if (lane < ne) {
                    const size_t at = (size_t)(id / p.layout.group) * p.eval_episodes + m0 + lane;
                    if constexpr (!TRACE) p.eval_returns[at] = st.ret;     // (recording stored the returns step by step)
                    p.eval_lengths[at] = nstep;
                }
            }
            // returns of the chunk's episodes in episode order; steps
#pragma unroll
            for (int e = 0; e < EC; ++e) {
                const double r = __shfl_sync(FULL, st.ret, e);
                if (e < ne) total = __dadd_rn(total, r);
            }
            int n = lane < ne ? nstep : 0;
#pragma unroll
            for (int o = 16; o; o >>= 1) n += __shfl_xor_sync(FULL, n, o);
            total_steps += n;
        }
        warp_steps += (unsigned long long)total_steps;
        if (lane == 0 && !EVAL) {
            p.steps[id] = total_steps;
            publish_fitness(p, id, __ddiv_rn(total, (double)p.E));
        }
    }
    if (p.total_steps && lane == 0 && warp_steps) atomicAdd(p.total_steps, warp_steps);
}

// EC: as many episodes in lockstep as the logits' lane budget (32 / (N_AGENTS * ACT)) allows, at most 5
template <class Env>
struct GruGenConfig {
    static constexpr int EC_MAX = 32 / (Env::N_AGENTS * Env::ACT);
    static constexpr int EC = EC_MAX < 5 ? EC_MAX : 5;
    static constexpr int WARPS = 3;
};

template <class Env, bool EVAL = false>
static int launch_rollout_gru_generic(int num_sms, int ctas_per_sm, const RolloutParams &rp, bool trace, cudaStream_t st, int64_t *launches,
                                      char *err, size_t errlen)
{
    constexpr int EC = GruGenConfig<Env>::EC, WARPS = GruGenConfig<Env>::WARPS;
    const size_t smem = WARPS * sizeof(GruGenSmem<Env, EC>);
    auto kern = EVAL ? (trace ? k_rollout_gru_generic<Env, EC, WARPS, true, true> : k_rollout_gru_generic<Env, EC, WARPS, false, true>)
              : trace ? k_rollout_gru_generic<Env, EC, WARPS, true>
              : rp.final_states ? k_rollout_gru_generic<Env, EC, WARPS, false, false, true> : k_rollout_gru_generic<Env, EC, WARPS, false>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    int per_sm = 0;
    if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, WARPS * 32, smem);
    if (e != cudaSuccess || per_sm < 1) {
        snprintf(err, errlen, "generic GRU rollout kernel cannot be launched (smem %zu B): %s", smem, cudaGetErrorString(e));
        return -1;
    }
    if (ctas_per_sm > 0 && ctas_per_sm < per_sm) per_sm = ctas_per_sm;
    int grid = per_sm * num_sms;
    const int need = (rp.shard.n_local + WARPS - 1) / WARPS;
    if (grid > need) grid = need;
    kern<<<grid, WARPS * 32, smem, st>>>(rp);
    e = cudaGetLastError();
    if (e != cudaSuccess) { snprintf(err, errlen, "generic GRU rollout launch failed: %s", cudaGetErrorString(e)); return -1; }
    *launches += 1;
    return 0;
}

}  // namespace ses

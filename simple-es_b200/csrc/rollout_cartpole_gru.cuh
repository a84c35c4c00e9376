// rollout_cartpole_gru.cuh -- K1, CartPole-v1 (optionally POMDP) with the GRU policy (D = 6562).
//
// Replaces the same reference code as rollout_cartpole_mlp.cuh, with GymEnvModel's GRU branch
// (networks/neural_network.py:15-16,25-27,38-40; torch nn.GRU cell, SURVEY.md Appendix A.3).
//
// Mapping (DESIGN.md section 5.2): 26 kB of weights per offspring do not fit per lane, so a WARP owns
// one offspring: its weights live in shared memory, lane j owns hidden unit j, and the warp steps up
// to EC episodes of that offspring in lockstep so that every weight read from shared memory feeds EC
// FMAs.  The six gate rows of lane j are stored as PAIRS so that the GEMV runs on packed FFMA2
// (two IEEE fmas per issue slot, same bits as two FFMA):
//     wrz_i[k/2][j] = { W_ir[j][k], W_iz[j][k], W_ir[j][k+1], W_iz[j][k+1] }     x[k] is the broadcast scalar
//     wrz_h[k/2][j] = { W_hr[j][k], W_hz[j][k], W_hr[j][k+1], W_hz[j][k+1] }     h[k] is the broadcast scalar
//     wn   [k/2][j] = { W_in[j][k], W_hn[j][k], W_in[j][k+1], W_hn[j][k+1] }     times the pair { x[k], h[k] }
// (conflict-free LDS.128 per lane); x and h live interleaved in xh[e][k] = { x[k], h[k] } and come back as
// broadcast LDS.128.  Every accumulator still sees its products in ascending k, one rounding per fma, as the
// contract states.  Lane e (e < EC) additionally owns the float64 cart-pole state of episode e and evaluates
// the two logits (packed as { z0, z1 }) in the contract's sequential order, then the physics.  8 warps
// (offspring) are resident per SM -- shared-memory capacity is what bounds this variant.
#pragma once
#include <cstdio>
#include <cstdlib>
#include "rollout_cartpole_mlp.cuh"

namespace ses {

constexpr int GRU_D = param_count(4, 2, 1);            // 6562
constexpr int G3 = 3 * HID;                            // 96 gate rows
// flat parameter offsets (nn.Module.parameters() order, networks/neural_network.py:12-17)
constexpr int GO_W1 = 0, GO_B1 = 128, GO_WIH = 160, GO_WHH = GO_WIH + G3 * HID, GO_BIH = GO_WHH + G3 * HID,
              GO_BHH = GO_BIH + G3, GO_W2 = GO_BHH + G3, GO_B2 = GO_W2 + 2 * HID;
static_assert(GO_B2 + 2 == GRU_D, "GRU layout");
constexpr int GRU_NQ = (GRU_D + 3) / 4;                // 1641 quads (flat order)

template <int EC>
struct __align__(16) GruWarpSmem {
    float4 wrz_i[HID / 2][HID];    // see the header comment
    float4 wrz_h[HID / 2][HID];
    float4 wn[HID / 2][HID];
    float4 small[(GRU_D - 2 * G3 * HID + 3) / 4 + 1];   // W1, b1 | b_ih, b_hh, W2, b2 in flat order (gap removed)
    float2 w2p[HID];               // { W2[0][j], W2[1][j] }
    float2 xh[EC][HID];            // { tanh(fc1)[k], h[k] } per episode
    float obuf[EC][HID + 4];       // tanh(h') per episode; rows 16 B aligned and 4 banks apart: lane e walks row e
};

// place flat quad (4 consecutive columns c0..c0+3 of gate row `row`) of W_ih (hh = 0) or W_hh (hh = 1)
template <class Smem>
__device__ __forceinline__ void gru_store_gate_quad(Smem &sm, int hh, int row, int c0, const float4 w)
{
    const int g = row >> 5, j = row & 31;                      // torch gate order r, z, n
    float *base;
    int comp;
    if (g == 2) { base = reinterpret_cast<float *>(&sm.wn[0][0]); comp = hh; }
    else { base = reinterpret_cast<float *>(hh ? &sm.wrz_h[0][0] : &sm.wrz_i[0][0]); comp = g; }
    // element (k, j) of a [HID/2][HID] float4 table: quad (k/2, j), component 2*(k&1) + comp
    const int kp = c0 >> 1;                                    // c0 is a multiple of 4
    float *q0 = base + ((size_t)kp * HID + j) * 4, *q1 = base + ((size_t)(kp + 1) * HID + j) * 4;
    q0[comp] = w.x; q0[2 + comp] = w.y; q1[comp] = w.z; q1[2 + comp] = w.w;
}

// index into `small` (floats) of flat parameter d outside the two big matrices
__device__ __forceinline__ int gru_small_index(int d) { return d < GO_WIH ? d : d - 2 * G3 * HID; }

// weights of one offspring: flat quad q -> shared memory (big matrices tiled, the rest in flat order); the calling threads
// take quads first, first + stride, ...
template <class Smem>
__device__ __forceinline__ void gru_load_weights(Smem &sm, const RolloutParams &p, int id, int local_idx, int first, int stride)
{
    const float *prow = p.w_override ? p.w_override + (size_t)local_idx * GRU_D
                                     : p.parents + (size_t)p.layout.parent(id) * GRU_D;
    const bool pert = p.w_override ? false : p.layout.perturbed(id);
    float sg;
    const uint32_t nid = p.layout.noise_id(id, sg);
    for (int q = first; q < GRU_NQ; q += stride) {
        // 6562 = 4*1640 + 2 and every block boundary is a multiple of 4 except the very end
        const float4 w = offspring_quad(prow, GRU_D, q, pert, __fmul_rn(p.sigma, sg), p.seed, nid, p.gen);
        const int d = 4 * q;
        if (d >= GO_WIH && d < GO_WHH) {
            const int o = d - GO_WIH; gru_store_gate_quad(sm, 0, o >> 5, o & 31, w);
        } else if (d >= GO_WHH && d < GO_BIH) {
            const int o = d - GO_WHH; gru_store_gate_quad(sm, 1, o >> 5, o & 31, w);
        } else {
            sm.small[gru_small_index(d) >> 2] = w;
            if (d >= GO_W2 && d < GO_B2) {             // fc2 rows also as { W2[0][j], W2[1][j] } pairs
                const int r = (d - GO_W2) >> 5, j = (d - GO_W2) & 31;
                float *wp = reinterpret_cast<float *>(&sm.w2p[0]);
                wp[2 * j + r] = w.x; wp[2 * (j + 1) + r] = w.y; wp[2 * (j + 2) + r] = w.z; wp[2 * (j + 3) + r] = w.w;
            }
        }
    }
}

// per-lane constants of an offspring: fc1 row j, biases of gate rows j, 32+j, 64+j, fc2 bias
struct GruLaneConsts { float4 w1; float b1, bir, biz, bin, bhr, bhz, bhn, b20, b21; };

__device__ __forceinline__ GruLaneConsts gru_lane_consts(const float4 *small, int lane)
{
    const float *smallf = reinterpret_cast<const float *>(small);
    GruLaneConsts c;
    c.w1 = small[lane];                                            // W1[j][0..3]
    c.b1 = smallf[GO_B1 + lane];
    c.bir = smallf[gru_small_index(GO_BIH) + lane]; c.biz = smallf[gru_small_index(GO_BIH) + HID + lane];
    c.bin = smallf[gru_small_index(GO_BIH) + 2 * HID + lane];
    c.bhr = smallf[gru_small_index(GO_BHH) + lane]; c.bhz = smallf[gru_small_index(GO_BHH) + HID + lane];
    c.bhn = smallf[gru_small_index(GO_BHH) + 2 * HID + lane];
    c.b20 = smallf[gru_small_index(GO_B2)]; c.b21 = smallf[gru_small_index(GO_B2) + 1];
    return c;
}

// recording (ses_record): state, action and return (the step count) after step nstep of episode m of policy j
__device__ __forceinline__ void gru_record_step(const RolloutParams &p, int j, int m, int nstep, double x, double xd, double th, double thd,
                                                int action)
{
    const size_t r = record_row(p, j, m, nstep - 1);
    double *t = p.trace + r * 4;
    t[0] = x; t[1] = xd; t[2] = th; t[3] = thd;
    p.trace_actions[r] = action;
    p.trace_returns[r] = (double)nstep;
}

// SPEC (the default since round 2: 4.38 ms against 4.62 ms at P = 4097 converged on a B200; SES_GRU_VARIANT=0 selects the
// plain kernel in the test build): the
// float64 physics leaves the serial tail of the step.  In the default kernel the <= 5 lanes that own an episode run, after
// the cell, 32 dependent FFMA2 (logits) and then the whole cart-pole chain while 27 lanes idle.  Here lanes [EC, 2 EC) mirror
// the episode states of lanes [0, EC), and at the START of the step lanes [0, EC) advance their copy assuming action 0 and
// lanes [EC, 2 EC) assuming action 1 -- the same warp instructions the owners would issue anyway, on lanes that were idle --
// with the branch-free division (cartpole_step_fastdiv).  The physics therefore depends on nothing the policy computes and
// sits in the same basic block as the (fully unrolled) GEMV, so the scheduler can fill the FFMA2 stream's issue gaps with
// it; after the argmax each lane takes the two velocities from the candidate of the chosen action (4 SHFL) -- position,
// angle and `done` do not depend on the action at all.
//
// One chunk of up to EC episodes (e0 .. e0 + ne - 1 of offspring `id`) stepped in lockstep by the calling warp; xh / obuf are
// the warp's EC staging rows.  Returns the sum of the episode lengths (on every lane).
// EVAL (ses_evaluate): `id` is the virtual offspring (policy * layout.group + chunk), e0 the chunk's first episode of the policy;
// initial states from STREAM_EVAL, and every episode stores its return and length.  TRACE && EVAL (ses_record): every step of
// every episode is recorded as well, by the owner lanes only (never the SPEC mirrors).  FINAL (training, ses_set_final_states):
// the owner lanes store each episode's final state.
template <int EC, bool SPEC, bool TRACE, int WREG = 0, bool EVAL = false, bool FINAL = false, class Smem>
__device__ __forceinline__ int gru_run_chunk(Smem &sm, float2 (*xh)[HID], float (*obuf)[HID + 4], const GruLaneConsts &c,
                                             const RolloutParams &p, int id, int local_idx, int e0, int ne, int lane)
{
    const unsigned FULL = 0xffffffffu;
    const float4 w1 = c.w1;
    const float b1 = c.b1, bir = c.bir, biz = c.biz, bin = c.bin, bhr = c.bhr, bhz = c.bhz, bhn = c.bhn, b20 = c.b20, b21 = c.b21;
    // ------------------------------------------------------------ a chunk of up to EC episodes
    double x = 0.0, xd = 0.0, th = 0.0, thd = 0.0;             // lane e: state of episode e0 + e
    int nstep = 0;
    // SPEC: lanes [EC, 2 EC) hold a mirror of the states of lanes [0, EC) (the action-1 candidates)
    const int ei = SPEC ? (lane >= EC ? lane - EC : lane) : lane;
    bool alive = SPEC ? (lane < 2 * EC && ei < ne) : (lane < ne);
    if (alive) {
        if (p.init_states) {
            const double *s0 = p.init_states + 4 * (e0 + ei);
            x = s0[0]; xd = s0[1]; th = s0[2]; thd = s0[3];
        } else {
            if constexpr (EVAL) cartpole_init(p.seed, 1, p.gen, 0u, (uint32_t)(e0 + ei), x, xd, th, thd, STREAM_EVAL);
            else cartpole_init(p.seed, p.init_mode, p.gen, (uint32_t)id, (uint32_t)(e0 + ei), x, xd, th, thd);
        }
    }
    if constexpr (EVAL && TRACE) {                             // recording: the chunks of policy 0 store the initial states
        if (alive && lane < EC && id < p.layout.group) {
            double *t = p.trace_initial + (size_t)4 * (e0 + lane);
            t[0] = x; t[1] = xd; t[2] = th; t[3] = thd;
        }
    }
    float h[EC];
#pragma unroll
    for (int e = 0; e < EC; ++e) { h[e] = 0.0f; xh[e][lane] = make_float2(0.0f, 0.0f); }      // model.reset() (neural_network.py:38-40)
    unsigned alive_mask = __ballot_sync(FULL, alive);
    // WREG: lane j keeps its quads of the n-gate table (WREG >= 1) and of W_hh's r/z table (WREG >= 2) in registers
    [[maybe_unused]] float4 wn_r[WREG >= 1 ? HID / 2 : 1], wh_r[WREG >= 2 ? HID / 2 : 1];
    if constexpr (WREG >= 1) {
#pragma unroll
        for (int kp = 0; kp < HID / 2; ++kp) wn_r[kp] = sm.wn[kp][lane];
    }
    if constexpr (WREG >= 2) {
#pragma unroll
        for (int kp = 0; kp < HID / 2; ++kp) wh_r[kp] = sm.wrz_h[kp][lane];
    }
    constexpr int NP = EC / 2;                                 // episode pairs for the packed tanh

    while (alive_mask) {
        // fc1 for every live episode: obs of episode e lives in lane e
        const float o0 = (float)x, o2 = (float)th;
        const float o1 = p.pomdp ? 0.0f : (float)xd;
        const float o3 = p.pomdp ? 0.0f : (float)thd;
        {
            float a[EC];
#pragma unroll
            for (int e = 0; e < EC; ++e) {
                const float q0 = __shfl_sync(FULL, o0, e), q1 = __shfl_sync(FULL, o1, e),
                            q2 = __shfl_sync(FULL, o2, e), q3 = __shfl_sync(FULL, o3, e);
                a[e] = b1;
                a[e] = fmaf(w1.x, q0, a[e]); a[e] = fmaf(w1.y, q1, a[e]); a[e] = fmaf(w1.z, q2, a[e]); a[e] = fmaf(w1.w, q3, a[e]);
            }
#pragma unroll
            for (int pe = 0; pe < NP; ++pe) {
                const float2 t = tanh32x2<false>(make_float2(a[2 * pe], a[2 * pe + 1]));
                xh[2 * pe][lane].x = t.x; xh[2 * pe + 1][lane].x = t.y;
            }
            if constexpr (EC & 1) xh[EC - 1][lane].x = tanh32_fast_t<false>(a[EC - 1]);
        }
        __syncwarp();
        // SPEC: this lane's candidate next state (action 0 on lanes < EC, action 1 on the mirror lanes); independent of
        // everything below up to the argmax
        [[maybe_unused]] double cx = x, cxd = xd, cth = th, cthd = thd;
        [[maybe_unused]] bool cdone = false;
        if constexpr (SPEC) cdone = cartpole_step_fastdiv(cx, cxd, cth, cthd, lane >= EC ? 1 : 0);
        // gate pre-activations of lane j, as pairs: { r_i, z_i } (W_ih x), { r_h, z_h } (W_hh h), { n_i, n_h }
        float2 grz_i[EC], grz_h[EC], gn[EC];
#pragma unroll
        for (int e = 0; e < EC; ++e) { grz_i[e] = make_float2(bir, biz); grz_h[e] = make_float2(bhr, bhz); gn[e] = make_float2(bin, bhn); }
#pragma unroll(SPEC ? HID / 2 : 2)
        for (int kp = 0; kp < HID / 2; ++kp) {
            float4 a = sm.wrz_i[kp][lane], c, n;
            if constexpr (WREG >= 2) c = wh_r[kp]; else c = sm.wrz_h[kp][lane];
            if constexpr (WREG >= 1) n = wn_r[kp]; else n = sm.wn[kp][lane];
#pragma unroll
            for (int e = 0; e < EC; ++e) {
                const float4 v = *reinterpret_cast<const float4 *>(&xh[e][2 * kp]);      // { x[k], h[k], x[k+1], h[k+1] }
                grz_i[e] = __ffma2_rn(make_float2(a.x, a.y), make_float2(v.x, v.x), grz_i[e]);
                grz_h[e] = __ffma2_rn(make_float2(c.x, c.y), make_float2(v.y, v.y), grz_h[e]);
                gn[e] = __ffma2_rn(make_float2(n.x, n.y), make_float2(v.x, v.y), gn[e]);
                grz_i[e] = __ffma2_rn(make_float2(a.z, a.w), make_float2(v.z, v.z), grz_i[e]);
                grz_h[e] = __ffma2_rn(make_float2(c.z, c.w), make_float2(v.w, v.w), grz_h[e]);
                gn[e] = __ffma2_rn(make_float2(n.z, n.w), make_float2(v.z, v.w), gn[e]);
            }
        }
        __syncwarp();                                          // everyone has read xh before h is rewritten
        // GRU cell (torch gate order r, z, n) and the output non-linearity
        float npre[EC], zg[EC];
#pragma unroll
        for (int e = 0; e < EC; ++e) {
            // { r, z } = sigm32({ r_i + r_h, z_i + z_h }) = 0.5 * tanh32(0.5 * s) + 0.5
            const float2 sres = __fadd2_rn(grz_i[e], grz_h[e]);
            const float2 t = tanh32x2<false>(__fmul2_rn(make_float2(0.5f, 0.5f), sres));
            const float2 rz = __ffma2_rn(make_float2(0.5f, 0.5f), t, make_float2(0.5f, 0.5f));
            npre[e] = fmaf(rz.x, gn[e].y, gn[e].x);
            zg[e] = rz.y;
        }
        float ng[EC];
#pragma unroll
        for (int pe = 0; pe < NP; ++pe) {
            const float2 t = tanh32x2<false>(make_float2(npre[2 * pe], npre[2 * pe + 1]));
            ng[2 * pe] = t.x; ng[2 * pe + 1] = t.y;
        }
        if constexpr (EC & 1) ng[EC - 1] = tanh32_fast_t<false>(npre[EC - 1]);
#pragma unroll
        for (int e = 0; e < EC; ++e) {
            // a finished episode keeps its (unused) state; the values are simply never read again
            h[e] = fmaf(zg[e], h[e], __fmul_rn(__fsub_rn(1.0f, zg[e]), ng[e]));
            xh[e][lane].y = h[e];
        }
#pragma unroll
        for (int pe = 0; pe < NP; ++pe) {
            const float2 t = tanh32x2<false>(make_float2(h[2 * pe], h[2 * pe + 1]));
            obuf[2 * pe][lane] = t.x; obuf[2 * pe + 1][lane] = t.y;
        }
        if constexpr (EC & 1) obuf[EC - 1][lane] = tanh32_fast_t<false>(h[EC - 1]);
        __syncwarp();
        // lane e: logits in the contract's sequential order (as the pair { z0, z1 }), action, physics
        bool done = false;
        int action = 0;
        if (alive && (!SPEC || lane < EC)) {
            float2 z = make_float2(b20, b21);
            const float4 *orow = reinterpret_cast<const float4 *>(obuf[lane]);
            const float4 *wp = reinterpret_cast<const float4 *>(sm.w2p);
            float2 sblk = make_float2(0.0f, 0.0f);                 // contract 4.4: four blocks of eight hidden units
#pragma unroll
            for (int jq = 0; jq < HID / 4; ++jq) {
                const float4 o = orow[jq], wa = wp[2 * jq], wb = wp[2 * jq + 1];
                sblk = __ffma2_rn(make_float2(wa.x, wa.y), make_float2(o.x, o.x), sblk);
                sblk = __ffma2_rn(make_float2(wa.z, wa.w), make_float2(o.y, o.y), sblk);
                sblk = __ffma2_rn(make_float2(wb.x, wb.y), make_float2(o.z, o.z), sblk);
                sblk = __ffma2_rn(make_float2(wb.z, wb.w), make_float2(o.w, o.w), sblk);
                if (jq & 1) { z = __fadd2_rn(z, sblk); sblk = make_float2(0.0f, 0.0f); }
            }
            const float z0 = z.x, z1 = z.y;
            action = argmax_softmax2(z0, z1);
            if constexpr (!SPEC) {
                done = cartpole_step(x, xd, th, thd, action);
                ++nstep;
                if (nstep >= p.max_step) done = true;
                if constexpr (TRACE && EVAL) {
                    gru_record_step(p, id / p.layout.group, e0 + lane, nstep, x, xd, th, thd, action);
                } else if constexpr (TRACE) {
                    const int local = local_idx;
                    if (e0 + lane == 0 && local < p.n_trace && nstep <= 200) {
                        double *t = p.trace + ((size_t)local * 200 + (nstep - 1)) * 4;
                        t[0] = x; t[1] = xd; t[2] = th; t[3] = thd;
                        p.trace_actions[(size_t)local * 200 + (nstep - 1)] = action;
                    }
                }
                if (done) alive = false;
            }
        }
        if constexpr (SPEC) {
            // owner and mirror of episode ei both continue from the candidate of the chosen action
            const int act = __shfl_sync(FULL, action, ei);
            const int src = ei + (act ? EC : 0);
            const double sxd = __shfl_sync(FULL, cxd, src), sthd = __shfl_sync(FULL, cthd, src);
            if (alive) {
                x = cx; th = cth; xd = sxd; thd = sthd;            // x, theta, done: the same in both candidates
                done = cdone;
                ++nstep;
                if (nstep >= p.max_step) done = true;
                if constexpr (TRACE && EVAL) {
                    if (lane < EC) gru_record_step(p, id / p.layout.group, e0 + lane, nstep, x, xd, th, thd, act);
                } else if constexpr (TRACE) {
                    const int local = local_idx;
                    if (lane < EC && e0 + lane == 0 && local < p.n_trace && nstep <= 200) {
                        double *t = p.trace + ((size_t)local * 200 + (nstep - 1)) * 4;
                        t[0] = x; t[1] = xd; t[2] = th; t[3] = thd;
                        p.trace_actions[(size_t)local * 200 + (nstep - 1)] = act;
                    }
                }
                if (done) alive = false;
            }
        }
        alive_mask = __ballot_sync(FULL, alive);
    }
    if constexpr (FINAL) {
        if (lane < ne) {                                       // lanes < ne <= EC: the owners, never a SPEC mirror
            double *row = final_row(p, id, e0 + lane, 4);
            row[0] = x; row[1] = xd; row[2] = th; row[3] = thd;
        }
    }
    // chunk total: lanes 0..ne-1 hold their episode lengths
    if constexpr (EVAL) {
        if (lane < ne) {
            const size_t at = (size_t)(id / p.layout.group) * p.eval_episodes + e0 + lane;
            if constexpr (!TRACE) p.eval_returns[at] = (double)nstep;   // (recording stored the returns step by step)
            p.eval_lengths[at] = nstep;
        }
    }
    int n = lane < ne ? nstep : 0;
#pragma unroll
    for (int o = 16; o; o >>= 1) n += __shfl_xor_sync(FULL, n, o);
    return n;
}

template <int EC, int WARPS, bool TRACE, bool SPEC = false, int WREG = 0, bool EVAL = false, bool FINAL = false>
__global__ void __launch_bounds__(WARPS * 32, 2) k_rollout_cartpole_gru(const RolloutParams p)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    GruWarpSmem<EC> &sm = reinterpret_cast<GruWarpSmem<EC> *>(smem_raw)[threadIdx.x >> 5];
    const int lane = threadIdx.x & 31;
    const unsigned FULL = 0xffffffffu;

    unsigned long long warp_steps = 0;
    for (;;) {
        // ---------------------------------------------------------------- next offspring
        int id = 0;
        if (lane == 0) id = atomicAdd(p.work_counter, 1);
        id = __shfl_sync(FULL, id, 0);
        if (id >= p.shard.n_local) break;
        const int local_idx = id;
        id = p.shard.local_to_id(local_idx);
        __syncwarp();
        gru_load_weights(sm, p, id, local_idx, lane, 32);
        __syncwarp();
        const GruLaneConsts c = gru_lane_consts(sm.small, lane);
        if constexpr (EVAL) {                                      // one chunk of p.E == EC episodes, the policy's last one partial
            const int e0 = (id % p.layout.group) * p.E;
            warp_steps += (unsigned long long)gru_run_chunk<EC, SPEC, TRACE, WREG, true>(sm, sm.xh, sm.obuf, c, p, id, local_idx, e0,
                                                                                          min(p.E, p.eval_episodes - e0), lane);
            continue;
        }
        long long total_steps = 0;
        for (int e0 = 0; e0 < p.E; e0 += EC)
            total_steps += gru_run_chunk<EC, SPEC, TRACE, WREG, false, FINAL>(sm, sm.xh, sm.obuf, c, p, id, local_idx, e0, min(EC, p.E - e0), lane);
        warp_steps += (unsigned long long)total_steps;
        if (lane == 0) {
            p.steps[id] = total_steps;
            publish_fitness(p, id, __ddiv_rn((double)total_steps, (double)p.E));
        }
    }
    if (p.total_steps && lane == 0 && warp_steps) atomicAdd(p.total_steps, warp_steps);
}

#ifdef SES_BUILD_TESTS
// ---------------------------------------------------------------------------------------------------------------------
// PAIR kernel (test build only, SES_GRU_VARIANT=2; an experiment that lost).  Shared memory holds 8 offspring per SM and that is all the single-warp mapping
// above can keep resident: 2 warps per sub-partition, which leaves the FFMA2 stream's latencies (the five tanh chains of a
// step, the 32-long logit chain, LDS) half exposed (issue utilisation 49 % in profiles/r01_gru_final_conv.txt).  Here TWO warps
// share one offspring's weights: warp A steps ECA of its episodes, warp B the other ECB (3 + 2 for E = 5), each with its own
// staging rows -- the same instruction stream per episode, 4 warps per sub-partition to hide it behind, and both warps
// regenerate the weights together (half the quads each).  The pair meets at a named barrier (bar.sync id, 64) three times per
// offspring: offspring index handed over, weights complete, step counts merged (which also frees the weights).
// Register budget 128 (16 warps per SM).
template <int ECA, int ECB>
struct __align__(16) GruPairSmem {
    float4 wrz_i[HID / 2][HID];    // as GruWarpSmem
    float4 wrz_h[HID / 2][HID];
    float4 wn[HID / 2][HID];
    float4 small[(GRU_D - 2 * G3 * HID + 3) / 4 + 1];
    float2 w2p[HID];
    float2 xh[ECA + ECB][HID];     // rows [0, ECA) warp A, [ECA, ECA + ECB) warp B
    float obuf[ECA + ECB][HID + 4];
    int ctl[4];                    // [0] offspring handed to the pair; [2..3] warp B's step count (64 bit)
};

__device__ __forceinline__ void pair_barrier(int pair)
{
    asm volatile("bar.sync %0, 64;" :: "r"(pair + 1) : "memory");
}

template <int ECA, int ECB, int PAIRS, bool TRACE>
__global__ void __launch_bounds__(PAIRS * 64, 2) k_rollout_cartpole_gru_pair(const RolloutParams p)
{
    static_assert(ECA >= ECB && ECB >= 1, "warp A takes the larger share");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int warp = threadIdx.x >> 5, pair = warp >> 1, half = warp & 1, lane = threadIdx.x & 31;
    GruPairSmem<ECA, ECB> &sm = reinterpret_cast<GruPairSmem<ECA, ECB> *>(smem_raw)[pair];
    volatile int *ctl = sm.ctl;

    unsigned long long warp_steps = 0;
    for (;;) {
        // ---------------------------------------------------------------- next offspring of the pair
        if (half == 0 && lane == 0) ctl[0] = atomicAdd(p.work_counter, 1);
        pair_barrier(pair);
        const int local_idx = ctl[0];
        if (local_idx >= p.shard.n_local) break;                       // both warps leave together
        const int id = p.shard.local_to_id(local_idx);
        gru_load_weights(sm, p, id, local_idx, half * 32 + lane, 64);
        pair_barrier(pair);
        const GruLaneConsts c = gru_lane_consts(sm.small, lane);
        long long total_steps = 0;
        for (int e0 = 0; e0 < p.E; e0 += ECA + ECB) {
            const int ne = min(ECA + ECB, p.E - e0);
            const int ne_a = max((ne + 1) >> 1, ne - ECB);             // a partial chunk is shared evenly
            if (half == 0) total_steps += gru_run_chunk<ECA, true, TRACE>(sm, sm.xh, sm.obuf, c, p, id, local_idx, e0, ne_a, lane);
            else total_steps += gru_run_chunk<ECB, true, TRACE>(sm, sm.xh + ECA, sm.obuf + ECA, c, p, id, local_idx, e0 + ne_a, ne - ne_a, lane);
        }
        warp_steps += (unsigned long long)total_steps;
        if (half == 1 && lane == 0) { ctl[2] = (int)(total_steps & 0xffffffffll); ctl[3] = (int)(total_steps >> 32); }
        pair_barrier(pair);
        if (half == 0 && lane == 0) {
            total_steps += (long long)(((unsigned long long)(unsigned)ctl[3] << 32) | (unsigned)ctl[2]);
            p.steps[id] = total_steps;
            publish_fitness(p, id, __ddiv_rn((double)total_steps, (double)p.E));
        }
    }
    if (p.total_steps && lane == 0 && warp_steps) atomicAdd(p.total_steps, warp_steps);
}

template <int ECA, int ECB>
static int launch_rollout_cartpole_gru_pair(int num_sms, int ctas_per_sm, const RolloutParams &rp, bool trace, cudaStream_t st,
                                            int64_t *launches, char *err, size_t errlen)
{
    constexpr int PAIRS = 4;
    const size_t smem = PAIRS * sizeof(GruPairSmem<ECA, ECB>);
    auto kern = trace ? k_rollout_cartpole_gru_pair<ECA, ECB, PAIRS, true> : k_rollout_cartpole_gru_pair<ECA, ECB, PAIRS, false>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    int per_sm = 0;
    if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, PAIRS * 64, smem);
    if (e != cudaSuccess || per_sm < 1) {
        snprintf(err, errlen, "GRU pair rollout kernel cannot be launched (smem %zu B): %s", smem, cudaGetErrorString(e));
        return -1;
    }
    if (ctas_per_sm > 0 && ctas_per_sm < per_sm) per_sm = ctas_per_sm;
    int grid = per_sm * num_sms;
    const int need = (rp.shard.n_local + PAIRS - 1) / PAIRS;
    if (grid > need) grid = need;
    kern<<<grid, PAIRS * 64, smem, st>>>(rp);
    e = cudaGetLastError();
    if (e != cudaSuccess) { snprintf(err, errlen, "GRU pair rollout launch failed: %s", cudaGetErrorString(e)); return -1; }
    *launches += 1;
    return 0;
}
#endif  // SES_BUILD_TESTS

template <int EC, bool EVAL = false>
static int launch_rollout_cartpole_gru_ec(int num_sms, int ctas_per_sm, const RolloutParams &rp, bool trace, cudaStream_t st,
                                          int64_t *launches, char *err, size_t errlen, bool final_states = false)
{
    constexpr int WARPS = 4;
    const size_t smem = WARPS * sizeof(GruWarpSmem<EC>);
    void (*kern)(const RolloutParams);
    // the product's kernel: speculative physics (SPEC, -5 %) with the n-gate table in registers (WREG = 1, another -3.7 %:
    // 4.14 ms at P = 4097 converged); the test build keeps the others selectable: SES_GRU_VARIANT 0 plain, 1 SPEC with every
    // table in shared memory, 3 the default, 4 SPEC with W_hh's r/z table in registers as well (255 registers, slower)
#ifdef SES_BUILD_TESTS
    const char *ev = getenv("SES_GRU_VARIANT");                       // read per launch: tests switch it inside one process
    const int spec = ev && *ev ? atoi(ev) : 3;
    kern = spec == 1 ? (trace ? k_rollout_cartpole_gru<EC, WARPS, true, true> : k_rollout_cartpole_gru<EC, WARPS, false, true>)
              : spec == 4 ? (trace ? k_rollout_cartpole_gru<EC, WARPS, true, true, 2> : k_rollout_cartpole_gru<EC, WARPS, false, true, 2>)
              : spec == 0 ? (trace ? k_rollout_cartpole_gru<EC, WARPS, true, false> : k_rollout_cartpole_gru<EC, WARPS, false, false>)
                          : (trace ? k_rollout_cartpole_gru<EC, WARPS, true, true, 1> : k_rollout_cartpole_gru<EC, WARPS, false, true, 1>);
#else
    kern = trace ? k_rollout_cartpole_gru<EC, WARPS, true, true, 1> : k_rollout_cartpole_gru<EC, WARPS, false, true, 1>;
#endif
    if constexpr (EVAL)                                                // the product's kernel, evaluation / recording instance
        kern = trace ? k_rollout_cartpole_gru<EC, WARPS, true, true, 1, true> : k_rollout_cartpole_gru<EC, WARPS, false, true, 1, true>;
    else if (final_states)                                             // the product's kernel, final-state instance
        kern = k_rollout_cartpole_gru<EC, WARPS, false, true, 1, false, true>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    int per_sm = 0;
    if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, WARPS * 32, smem);
    if (e != cudaSuccess || per_sm < 1) {
        snprintf(err, errlen, "GRU rollout kernel cannot be launched (smem %zu B): %s", smem, cudaGetErrorString(e));
        return -1;
    }
    if (ctas_per_sm > 0 && ctas_per_sm < per_sm) per_sm = ctas_per_sm;
    const int n_local = rp.shard.n_local;
    int grid = per_sm * num_sms;
    const int need = (n_local + WARPS - 1) / WARPS;
    if (grid > need) grid = need;
    kern<<<grid, WARPS * 32, smem, st>>>(rp);
    e = cudaGetLastError();
    if (e != cudaSuccess) { snprintf(err, errlen, "GRU rollout launch failed: %s", cudaGetErrorString(e)); return -1; }
    *launches += 1;
    return 0;
}

static int launch_rollout_cartpole_gru(int num_sms, int ctas_per_sm, const RolloutParams &rp, bool trace, cudaStream_t st,
                                       int64_t *launches, char *err, size_t errlen)
{
    if (rp.final_states) {                                             // the product's kernel with the final-state output
        switch (rp.E >= 5 ? 5 : rp.E) {
        case 1: return launch_rollout_cartpole_gru_ec<1>(num_sms, ctas_per_sm, rp, false, st, launches, err, errlen, true);
        case 2: return launch_rollout_cartpole_gru_ec<2>(num_sms, ctas_per_sm, rp, false, st, launches, err, errlen, true);
        case 3: return launch_rollout_cartpole_gru_ec<3>(num_sms, ctas_per_sm, rp, false, st, launches, err, errlen, true);
        case 4: return launch_rollout_cartpole_gru_ec<4>(num_sms, ctas_per_sm, rp, false, st, launches, err, errlen, true);
        default: return launch_rollout_cartpole_gru_ec<5>(num_sms, ctas_per_sm, rp, false, st, launches, err, errlen, true);
        }
    }
    // episodes of one offspring step in lockstep, EC at a time (E > 5: chunks of 5, the last one partial)
#ifdef SES_BUILD_TESTS
    {   // SES_GRU_VARIANT=2: the warp-pair kernel (rejected: 5.48 ms against 4.30 ms, profiles/r02_k1_experiments.md)
        const char *ev = getenv("SES_GRU_VARIANT");
        if (ev && *ev && atoi(ev) == 2 && rp.E >= 2) {
            switch (rp.E >= 5 ? 5 : rp.E) {
            case 2: return launch_rollout_cartpole_gru_pair<1, 1>(num_sms, ctas_per_sm, rp, trace, st, launches, err, errlen);
            case 3: return launch_rollout_cartpole_gru_pair<2, 1>(num_sms, ctas_per_sm, rp, trace, st, launches, err, errlen);
            case 4: return launch_rollout_cartpole_gru_pair<2, 2>(num_sms, ctas_per_sm, rp, trace, st, launches, err, errlen);
            default: return launch_rollout_cartpole_gru_pair<3, 2>(num_sms, ctas_per_sm, rp, trace, st, launches, err, errlen);
            }
        }
    }
#endif
    switch (rp.E >= 5 ? 5 : rp.E) {
    case 1: return launch_rollout_cartpole_gru_ec<1>(num_sms, ctas_per_sm, rp, trace, st, launches, err, errlen);
    case 2: return launch_rollout_cartpole_gru_ec<2>(num_sms, ctas_per_sm, rp, trace, st, launches, err, errlen);
    case 3: return launch_rollout_cartpole_gru_ec<3>(num_sms, ctas_per_sm, rp, trace, st, launches, err, errlen);
    case 4: return launch_rollout_cartpole_gru_ec<4>(num_sms, ctas_per_sm, rp, trace, st, launches, err, errlen);
    default: return launch_rollout_cartpole_gru_ec<5>(num_sms, ctas_per_sm, rp, trace, st, launches, err, errlen);
    }
}

}  // namespace ses

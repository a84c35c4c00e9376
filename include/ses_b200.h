/*
 * ses_b200.h -- C ABI of the B200 population-rollout engine for simple-es.
 *
 * The reference (jinPrelude/simple-es) is pure Python and has no FFI: its extension points
 * are three ABCs wired by builder.build_loop (builder.py:27-86).  This header is therefore the
 * NEW boundary a maintainer binds with ctypes (see INTEGRATION.md); every entry point names the
 * reference code it replaces (paths relative to the reference repo).
 *
 * Conventions
 *   - plain C types only; every *_dev pointer is caller-owned DEVICE memory (e.g. a torch
 *     tensor's data_ptr()); the library allocates only its own scratch inside the handle.
 *   - `stream` is a cudaStream_t passed as void*; every call is stream-ordered and does not
 *     synchronise the host unless documented (the *_host entry points do).
 *   - return value 0 = ok, < 0 = error; ses_last_error() gives the message (thread local).
 *   - offspring ids are GLOBAL population indices; a handle owns the slice [id_begin, id_end).
 *   - there is NO CPU fallback: without a CUDA device every compute entry point fails.
 */
#ifndef SES_B200_H
#define SES_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SES_ABI_VERSION 1

/* env.name -> SES_ENV_*: "CartPole-v1" / "CartPole-v0" (same physics, TimeLimit 500 / 200: pass max_step), "simple_spread",
 * "MountainCar-v0", "Acrobot-v1" (discrete classic control any reference config can name, envs/gym_wrapper.py:8-9),
 * "Pendulum-v0" (continuous action: the policy's tanh head, networks/neural_network.py:32-33, `discrete_action: False`) */
enum { SES_ENV_CARTPOLE = 0, SES_ENV_SIMPLE_SPREAD = 1, SES_ENV_MOUNTAINCAR = 2, SES_ENV_ACROBOT = 3, SES_ENV_PENDULUM = 4 };
enum { SES_INIT_SHARED = 0, SES_INIT_FRESH = 1 };

/* Static description of one engine instance (one per process / GPU).
 * Mirrors what builder.build_env / build_network / the strategy constructors read from the
 * YAML (builder.py:10-75, conf/cartpole.yaml, conf/simplespread.yaml). */
typedef struct ses_config {
    int32_t env;          /* SES_ENV_*                                   (env.name)                */
    int32_t obs_dim;      /* network.num_state   4 | 12 (N=2) | 18 (N=3) | 2 (MountainCar) | 6 (Acrobot) | 3 (Pendulum) */
    int32_t act_dim;      /* network.num_action  2 | 5 | 3 | 3 | 1                                 */
    int32_t gru;          /* network.gru                                                           */
    int32_t pomdp;        /* env.pomdp: CartPole obs[1], obs[3] zeroed   (envs/gym_wrapper.py:69-77) */
    int32_t n_agents;     /* simple_spread N (reference hard-codes 2, envs/pettingzoo_wrapper.py:9) */
    int32_t max_step;     /* env.max_step; 0 encodes the YAML string "None"                        */
    int32_t eval_ep_num;  /* --eval-ep-num                               (run_es.py:36-41)         */
    int32_t population;   /* P: n+1 | k*(n//k) | n                       (SURVEY.md section 8)     */
    int32_t group;        /* index layout: parent(i) = i / group                                   */
    int32_t n_head;       /* offspring with (i % group) < n_head are unperturbed copies            */
    int32_t n_parents;    /* rows of the parent table (1, or elite_num for simple_genetic)         */
    uint32_t seed;        /* --seed; keys every Philox stream                                      */
    int32_t init_mode;    /* SES_INIT_SHARED: one [E] table of initial states for everybody (the   */
                          /* reference's mp.Pool behaviour, loop.py:66-74); SES_INIT_FRESH: per    */
                          /* (generation, offspring, episode)                                      */
    int32_t id_begin;     /* this handle's slice of the population (multi-GPU sharding)            */
    int32_t id_end;
    int32_t device;       /* CUDA device ordinal                                                   */
    int32_t antithetic;   /* opt-in, not in the reference: perturbed offspring of a group come in  */
                          /* mirrored pairs (+eps, -eps) sharing one Philox counter; 0 = off       */
    int32_t shard_block;  /* 0: this handle owns the contiguous ids [id_begin, id_end); B > 0: block-cyclic   */
    int32_t shard_rank;   /* sharding -- blocks of B consecutive ids are dealt round robin to shard_world    */
    int32_t shard_world;  /* handles, this one owns blocks b with b % shard_world == shard_rank (id_begin = 0, */
                          /* id_end = population); w_override rows / traces are in local order               */
    int32_t continuous_action; /* network.discrete_action == False: action = tanh(fc2(...)) (networks/neural_network.py:32-33); */
                          /* required for (and only valid with) SES_ENV_PENDULUM                   */
    int32_t reserved[2];
} ses_config;

typedef struct ses_handle ses_handle;

int ses_abi_version(void);
const char *ses_last_error(void);

/* D = number of policy parameters (networks/neural_network.py:12-17): 226 / 6562 / 581 / 773 / 195 / 323. */
int ses_param_count(int32_t obs_dim, int32_t act_dim, int32_t gru);

int ses_create(const ses_config *cfg, ses_handle **out);
int ses_destroy(ses_handle *h);

/* K1 -- replaces the per-generation fan-out `p.map(RolloutWorker, ...)` (loop.py:66-78),
 * RolloutWorker (loop.py:108-125), GymEnvModel.forward (networks/neural_network.py:20-36), the
 * env wrappers' reset/step (envs/gym_wrapper.py:23-45, envs/pettingzoo_wrapper.py:22-58) and the
 * perturbation half of _gen_offsprings (offspring_strategies.py:53-60,169-176,312-326).
 *   parents_dev      [n_parents][D] f32
 *   w_override_dev   optional [n_local][D] f32 in local order: explicit offspring weights instead of Philox perturbation
 *                    (sigma is then unused): sep_cma_es's samples (ses_cma_sample), or the reference's own perturbed arrays
 *                    in verification mode
 *   init_states_dev  optional [E][state_dim] f64 explicit initial states (verification mode);
 *                    NULL -> Philox stream per cfg.init_mode
 *   fitness_dev      [P] f64, written at [id_begin, id_end): total reward / eval_ep_num (loop.py:124)
 *   steps_dev        [P] i64, written at [id_begin, id_end): env steps simulated for that offspring
 *   trace_dev        optional [n_trace][200][state_dim] f64: state after each of the first 200 steps
 *                    of episode 0 for the first n_trace offspring of the slice; trace_actions_dev
 *                    [n_trace][200][n_agents] i32 likewise */
int ses_rollout(ses_handle *h, uint32_t generation, float sigma, const float *parents_dev,
                const float *w_override_dev, const double *init_states_dev, double *fitness_dev,
                int64_t *steps_dev, double *trace_dev, int32_t *trace_actions_dev, int32_t n_trace,
                void *stream);

/* Policy evaluation -- the GPU half of the reference's test.py (test.py:31-68; no rendering):
 * n_pol policies x n_episodes episodes of this handle's env / network, common initial states.
 *   policies_dev     [n_pol][D] f32, used as given (no noise, no antithetic pairing)
 *   init_states_dev  optional [n_episodes][state_dim] f64 explicit initial states (verification mode);
 *                    NULL -> episode m starts from Philox stream 2 at counter (m, 0, round, block), keyed
 *                    by cfg.seed: every policy of the call sees the same episodes (DESIGN.md section 4.9)
 *   returns_dev      [n_pol][n_episodes] f64: the episode's return (sequential sum of its step rewards)
 *   lengths_dev      [n_pol][n_episodes] i32: its env steps (truncated at max_step as in training)
 * Runs on this handle's device only; its strategy layout, shard and peers play no part. */
int ses_evaluate(ses_handle *h, uint32_t round, const float *policies_dev, int32_t n_pol, int32_t n_episodes,
                 const double *init_states_dev, double *returns_dev, int32_t *lengths_dev, void *stream);

/* Episode recording -- what the reference's test.py shows on screen, as data (pixels stay out of scope): the same episodes
 * as ses_evaluate (episode m does not depend on n_episodes: recording K episodes reproduces episodes 0 .. K-1 of any
 * ses_evaluate call of the same round / init_states), with every step stored.  T = the handle's effective max_step.
 *   initial_dev      [n_episodes][state_dim] f64: each episode's initial state in the layout of init_states rows (simple_spread:
 *                    agent positions, then landmark positions)
 *   states_dev       [n_pol][n_episodes][T][state_dim] f64: the state after step t + 1, laid out as ses_rollout's trace (the
 *                    gym envs: their env.unwrapped.state; simple_spread: agent positions, then agent velocities)
 *   actions_dev      [n_pol][n_episodes][T][n_agents] i32: the action of step t + 1 (Pendulum: the float32's bit pattern)
 *   returns_dev      [n_pol][n_episodes][T] f64: the return after step t + 1; at t + 1 = lengths it equals ses_evaluate's return
 *   lengths_dev      [n_pol][n_episodes] i32
 * Rows past an episode's end are not written.  Every buffer is required; the other arguments are ses_evaluate's. */
int ses_record(ses_handle *h, uint32_t round, const float *policies_dev, int32_t n_pol, int32_t n_episodes,
               const double *init_states_dev, double *initial_dev, double *states_dev, int32_t *actions_dev,
               double *returns_dev, int32_t *lengths_dev, void *stream);

/* K2-- replaces np.flip(np.argsort(rewards)) (offspring_strategies.py:112,234,380) with the tie
 * order pinned to descending fitness, then DESCENDING index (== kind="stable"), and the centered
 * rank shaping (offspring_strategies.py:392-398).
 *   fitness_dev [n] f64 -> order_dev [n] i32 (order[0] = best); shaped_dev optional [n] f64.
 *   key_bits: 0 = sort the full float64 key; k>0 = caller guarantees fitness*key_scale is an
 *   integer of magnitude < 2^k (CartPole: total steps; MountainCar / Acrobot: minus the total steps),
 *   which needs ceil((k+1)/8) radix passes instead of 8. */
int ses_rank_desc(ses_handle *h, const double *fitness_dev, int32_t n, int32_t key_bits, double key_scale,
                  int32_t *order_dev, double *shaped_dev, void *stream);

/* K3a -- replaces the openai_es gradient loop + Adam (offspring_strategies.py:401-416,
 * learning_strategies/optimizers.py:13-57).  Noise is re-derived from Philox(generation, id);
 * eps_override_dev optional [P][D] f32 materialised noise (verification mode).
 *   shaped_dev [P] f64; mu/m/v [D] f32 updated in place; update_factor = -lr/(P*sigma);
 *   adam_a = lr*sqrt(1-beta2^t)/(1-beta1^t) (float64, computed by the caller as optimizers.py:43-47);
 *   grad_out_dev optional [D] f32 (the scaled gradient handed to Adam). */
int ses_update_openai(ses_handle *h, uint32_t generation, const double *shaped_dev,
                      const float *eps_override_dev, double update_factor, double adam_a, double beta1,
                      double beta2, double adam_eps, float *mu_dev, float *m_dev, float *v_dev,
                      float *grad_out_dev, void *stream);

/* K3a' -- the same gradient followed by SGD with momentum instead of Adam.  Opt-in (engine.optimizer: sgd): the reference's
 * optimizers.py ships Adam only; this is the SGD of the file it names as its source (OpenAI es_distributed/optimizers.py):
 * v = momentum*v + (1-momentum)*g; theta += -stepsize*v, all float32 (numpy >= 2 dtypes of the reference's list-of-arrays idiom).
 *   mu/v [D] f32 updated in place; update_factor = -lr/(P*sigma); stepsize = learning_rate; momentum in [0, 1). */
int ses_update_openai_sgd(ses_handle *h, uint32_t generation, const double *shaped_dev,
                          const float *eps_override_dev, double update_factor, double stepsize, double momentum,
                          float *mu_dev, float *v_dev, float *grad_out_dev, void *stream);

/* K3b -- replaces _gen_offsprings' materialisation for selected ids: rows of out_dev [n][D] are the
 * weights offspring ids_dev[j] had in `generation` (parent + sigma*Philox noise).  Used for the
 * simple_genetic elite carry-over (offspring_strategies.py:114-116) and for checkpoints. */
int ses_materialize(ses_handle *h, uint32_t generation, float sigma, const float *parents_dev,
                    const float *w_override_dev, const int32_t *ids_dev, int32_t n, float *out_dev, void *stream);

/* K3c -- replaces the simple_evolution elite mean (offspring_strategies.py:241-250): float32 running
 * sum of the k best offspring in rank order, divided by k. order_dev from ses_rank_desc. */
int ses_update_elite_mean(ses_handle *h, uint32_t generation, float sigma, const float *parents_dev,
                          const float *w_override_dev, const int32_t *order_dev, int32_t k, float *mu_out_dev,
                          void *stream);

/* Multi-GPU fitness exchange fused into K1 (replaces the result half of Pool.map, loop.py:74: floats coming
 * back from the workers).  Each handle owns an exchange buffer ([2][P] f64, double buffered by generation
 * parity, + flags) allocated with cudaMalloc.  ses_peer_export writes its 64-byte CUDA IPC handle; after the
 * ranks have exchanged those (any host channel), ses_peer_attach maps every peer's buffer over NVLink.  From
 * then on a ses_rollout whose fitness_dev is ses_peer_fitness_ptr(parity) also stores each fitness value
 * straight into every peer's buffer from inside the kernel, and ses_peer_barrier (a flag barrier over peer
 * memory, stream ordered) makes the full vector visible on every rank -- no collective moves data.
 * ses_peer_check reports a barrier that timed out (a dead peer). */
int ses_peer_export(ses_handle *h, void *ipc_handle_out /* 64 bytes */);
int ses_peer_attach(ses_handle *h, const void *ipc_handles /* [world][64] */, int32_t rank, int32_t world);
int ses_peer_fitness_ptr(ses_handle *h, int32_t parity, double **out);
int ses_peer_barrier(ses_handle *h, void *stream);
int ses_peer_check(ses_handle *h);

/* Whole generation with HOST buffers (the e2e path of bench.py): H2D of the strategy state,
 * K1+K2+K3 for openai_es, D2H of fitness [P] and the updated state; synchronises `stream`.
 * Requires a single-slice handle (id_begin = 0, id_end = P). */
int ses_generation_openai_host(ses_handle *h, uint32_t generation, float sigma, double learning_rate,
                               int64_t adam_t, float *mu_host, float *m_host, float *v_host,
                               double *fitness_host, int64_t *total_steps_host, void *stream);

/* The same for the two elite strategies (one whole ESLoop.run iteration each, loop.py:61-84, with host buffers; single-slice
 * handle; synchronises `stream`):
 *   simple_evolution (offspring_strategies.py:213-258): mu_host [D] in -> K1, K2, elite mean of the elite_num best -> mu_host out.
 *     The caller applies `sigma *= sigma_decay` afterwards (:251), as for ses_update_elite_mean.
 *   simple_genetic (:94-124): elites_host [n_parents][D] in -> K1, K2, the n_parents best offspring's weights -> elites_host out.
 * fitness_host [P] f64 and total_steps_host (env steps simulated) as in ses_generation_openai_host. */
int ses_generation_evolution_host(ses_handle *h, uint32_t generation, float sigma, int32_t elite_num, float *mu_host,
                                  double *fitness_host, int64_t *total_steps_host, void *stream);
int ses_generation_genetic_host(ses_handle *h, uint32_t generation, float sigma, float *elites_host,
                                double *fitness_host, int64_t *total_steps_host, void *stream);

/* Measurement hook: FP32 (non-tensor) FFMA peak of `device` in TFLOP/s from a dependent-free FFMA
 * microbenchmark -- the denominator of the rollout kernel's roofline in bench.py. */
int ses_measure_fp32_peak(int32_t device, double *tflops_out);
/* The same with packed FFMA2 (fma.rn.f32x2): two FMAs per issue slot. */
int ses_measure_fp32x2_peak(int32_t device, double *tflops_out);

/* Optional device counter (uint64): every ses_rollout adds the env steps it simulated (bench.py's numerator). */
int ses_set_step_counter(ses_handle *h, uint64_t *counter_dev);

/* Optional device buffer [population][eval_ep_num][state_dim] f64 (NULL: off, the default).  While set, every ses_rollout also
 * stores the state after each episode's last step at row (global offspring id) * eval_ep_num + episode, in the layout of
 * ses_record's states (the gym envs: env.unwrapped.state; simple_spread: agent positions, then agent velocities).  Only the
 * rows of the ids this handle owns are written; fitness and steps are the same as without it.  ses_rollout then refuses
 * n_trace > 0.  ses_evaluate and ses_record ignore it. */
int ses_set_final_states(ses_handle *h, double *final_states_dev);

/* Novelty search with reward (the nsr_es strategy, DESIGN.md section 4.10).  float64 throughout, each operation separately
 * rounded; every call is stream-ordered and runs on the handle's device.  1 <= n <= population.
 * ses_behavior:     bc_dev[i][d] = (sum over e in episode order of final_states_dev[i][e][d]) / eval_ep_num, i < n
 * ses_novelty:      novelty_dev[i] = mean of the Euclidean distances sqrt(sum_d (bc[i][d] - archive[a][d])^2) from bc_dev[i] to
 *                   its min(k, n_archive) nearest rows of archive_dev [n_archive][state_dim], added in ascending order;
 *                   1 <= k <= 32, n_archive >= 1
 * ses_blend_shaped: out_dev[i] = (1 - w) shaped_f_dev[i] + w shaped_n_dev[i], 0 <= w <= 1 (w = 0 returns shaped_f_dev's
 *                   values, w = 1 shaped_n_dev's, for any shaping without -0.0 entries such as ses_rank_desc's) */
int ses_behavior(ses_handle *h, const double *final_states_dev, int32_t n, double *bc_dev, void *stream);
int ses_novelty(ses_handle *h, const double *bc_dev, int32_t n, const double *archive_dev, int32_t n_archive, int32_t k,
                double *novelty_dev, void *stream);
int ses_blend_shaped(ses_handle *h, const double *shaped_f_dev, const double *shaped_n_dev, int32_t n, double w, double *out_dev,
                     void *stream);

/* Separable CMA-ES (the sep_cma_es strategy, DESIGN.md section 4.11; Ros & Hansen 2008).  Needs the layout group = population,
 * n_head = 0, antithetic = 0: every offspring is sampled.  State, all [D] f64 device vectors unless noted: mean m, diagonal
 * covariance c, evolution paths p_sigma and p_c, and sigma ([1] f64, on the device because it depends on |p_sigma|).  float64
 * with each operation separately rounded; sigma goes through the device exp (<= 1 ulp), everything else is defined bit for bit.
 * ses_cma_sample: out_dev [n_local][D] f32, row l = (float)(m + sigma (sqrt(c) z)) for the id this handle holds at local index l
 *                 (ses_rollout's w_override order), z[d] = the Philox normal of (generation, id) that K3 re-derives.
 * ses_cma_update: one generation's update from order_dev [population] (ses_rank_desc of the full fitness vector):
 *                 s_dev [population] f64 := weights_dev[r] at order[r] for r < mu, else 0 (weights_dev [mu] f64);
 *                 <z> = sum_j s_j z_j and Q = sum_j s_j z_j^2 by the reduction tree of ses_update_openai (rows sharded over the
 *                 attached peers likewise); then p_sigma, h_sigma = (|p_sigma| < threshold), m (old sigma, old c), p_c, c and sigma
 *                 as section 4.11 writes them; parent_dev [D] f32 := (float)m.  1 <= mu <= population. */
typedef struct ses_cma_params {
    double one_m_cs;   /* 1 - c_sigma                          */
    double k_sigma;    /* sqrt(c_sigma (2 - c_sigma) mu_eff)   */
    double one_m_cc;   /* 1 - c_c                              */
    double k_c;        /* sqrt(c_c (2 - c_c) mu_eff)           */
    double cc2;        /* c_c (2 - c_c)                        */
    double c_keep;     /* 1 - c_1 - c_mu                       */
    double c1;         /* c_1 (separable rescaling applied)    */
    double cmu;        /* c_mu (separable rescaling applied)   */
    double damp;       /* c_sigma / d_sigma                    */
    double chi;        /* E|N(0, I_D)|: chi_D                  */
} ses_cma_params;
int ses_cma_sample(ses_handle *h, uint32_t generation, const double *mean_dev, const double *c_dev, const double *sigma_dev,
                   float *out_dev, void *stream);
int ses_cma_update(ses_handle *h, uint32_t generation, const int32_t *order_dev, const double *weights_dev, int32_t mu,
                   const ses_cma_params *params, double threshold, double *s_dev, double *mean_dev, double *c_dev,
                   double *p_sigma_dev, double *p_c_dev, double *sigma_dev, float *parent_dev, void *stream);

/* MAP-Elites (the map_elites strategy, DESIGN.md section 4.12; Mouret & Clune 2015).  Needs the layout group = 1, n_head = 0,
 * antithetic = 0 (n_parents = population): offspring i is parent row i + sigma * its Philox noise.  The archive has
 * n_cells = prod cells[j] cells, every buffer a caller-owned device array indexed by cell c:
 *   F_dev [n_cells] f64 the elite's fitness; NaN marks an empty cell (fill with NaN before the first call)
 *   B_dev [n_cells][state_dim] f64 its behaviour;  born_dev [n_cells][2] i32 its (generation, offspring id);  W_dev [n_cells][D] f32
 *   its weights.
 * The spec picks n_dims in [1, 4] distinct final-state coordinates dims[j] in [0, state_dim) with finite low[j], finite
 * width[j] = high - low > 0 (computed by the caller in float64) and cells[j] >= 1; n_cells <= 2^20 and n_cells * D * 4 bytes
 * <= 4 GiB.  Cell of a behaviour row b: per dimension s = ((b[dims[j]] - low) / width) * cells (float64, each operation
 * rounded), k = 0 if s < 1, cells - 1 if s >= cells - 1, floor(s) otherwise; c is row-major over the dimensions.
 * ses_map_insert: reads parents_dev [population][D] f32 (the table the generation was rolled out with), order_dev [population]
 *                 (ses_rank_desc of the full fitness vector), fitness_dev [population] f64 and bc_dev [population][state_dim]
 *                 f64 (ses_behavior).  An offspring whose fitness or a descriptor coordinate is NaN is unplaced; each cell's
 *                 placed offspring of smallest rank enters iff the cell is empty or its fitness > F (a tie keeps the incumbent),
 *                 writing F, B, born = (generation, id) and W = its weights (those of ses_materialize(generation, sigma)).
 * ses_map_select: from F_dev and W_dev: stats_dev [4] f64 := (n_occ, best cell c* (largest F, ties to the lowest index; -1
 *                 when empty), F[c*] (NaN when empty), the QD score sum of F over occupied cells in section 4.12's order); then
 *                 parent row i of parents_dev [population][D] := W[L[(r_i * n_occ) >> 32]], L the occupied cells ascending and
 *                 r_i word 0 of Philox(i, generation, 0, 0; seed, 3), or seed_row_dev [D] f32 when the archive is empty.
 * Both refuse null buffers, a bad spec and another layout.  Only the first call, and one with more cells than any before,
 * waits for the stream: it allocates the handle's scratch (per-cell claims, zero between calls, and the occupied-cell list). */
typedef struct ses_map_spec {
    int32_t n_dims;
    int32_t dims[4];
    double low[4];
    double width[4];
    int32_t cells[4];
} ses_map_spec;
int ses_map_insert(ses_handle *h, uint32_t generation, float sigma, const float *parents_dev, const int32_t *order_dev,
                   const double *fitness_dev, const double *bc_dev, const ses_map_spec *spec, double *F_dev, double *B_dev,
                   int32_t *born_dev, float *W_dev, void *stream);
int ses_map_select(ses_handle *h, uint32_t generation, const ses_map_spec *spec, const double *F_dev, const float *W_dev,
                   const float *seed_row_dev, double *stats_dev, float *parents_dev, void *stream);

/* Number of kernels this library has launched on behalf of the handle (bench.py "gpu_launches"). */
int64_t ses_launch_count(ses_handle *h);

#ifdef __cplusplus
}
#endif
#endif /* SES_B200_H */

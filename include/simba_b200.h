/*
 * simba_b200.h — C-ABI of the B200-native CEM-MPC planner (libsimba_b200.so).
 *
 * The reference (yardenas/ethz-safe-learning, "simba") has no FFI: its boundary for this path is
 * duck-typed Python (`policy.generate_action(state)`, simba/agents/agent.py:120). Each entry point
 * below names the reference code it replaces (file:line relative to the reference root). The
 * Python mirror of the reference interface (ethz-safe-learning_b200/simba_b200) binds these with
 * ctypes; INTEGRATION.md shows the stub a reference maintainer would add.
 *
 * Conventions
 *   - plain C types only; every pointer documented as HOST or DEVICE. The caller owns all arrays
 *     it passes; the library owns only what lives inside a handle.
 *   - every function returns 0 (SIMBA_OK) or a negative simba_status; simba_last_error() gives
 *     the message of the calling thread's last failure. Nothing throws or aborts across the ABI.
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream). All launches are
 *     asynchronous on it unless the function name ends in _host.
 *   - a handle is bound to the CUDA device that was current when it was created; it is not
 *     re-entrant. Different handles are independent.
 *   - there is NO CPU fallback: on a machine without an sm_100 GPU every compute entry point
 *     returns SIMBA_ERR_ARCH / SIMBA_ERR_CUDA.
 *   - all floating-point arrays are fp32, row-major, innermost index last.
 */
#ifndef SIMBA_B200_H_
#define SIMBA_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SIMBA_MAX_ACT 16          /* action dims                                    */
#define SIMBA_MAX_CONSTRAINTS 4   /* vases, hazards, pillars, gremlins (safety_gym.py:148-163) */
#define SIMBA_MAX_HORIZON 64      /* per-row cost history is a 64-bit mask          */
#define SIMBA_MAX_MEMBERS 64

typedef enum simba_status {
  SIMBA_OK = 0,
  SIMBA_ERR_BAD_CONFIG = -1,   /* a field is out of range                              */
  SIMBA_ERR_SHAPE = -2,        /* divisibility (tf.split needs B % E == 0), sizes      */
  SIMBA_ERR_CUDA = -3,         /* a CUDA runtime call failed                           */
  SIMBA_ERR_NCCL = -4,         /* NCCL missing or a collective failed                  */
  SIMBA_ERR_ARCH = -5,         /* device is not sm_100                                 */
  SIMBA_ERR_UNSUPPORTED = -6,  /* valid in the reference, not offered on the fused path */
  SIMBA_ERR_NOT_READY = -7,    /* weights / scaler / comm not set                      */
  SIMBA_ERR_NONFINITE = -8     /* scaler bounds not finite (transition_model.py:28-29 NaN case) */
} simba_status;

/* objective = how a candidate's particles become one score (SURVEY.md section 8, a10-a12) */
typedef enum simba_objective {
  SIMBA_OBJ_REWARD = 0,          /* MpcPolicy.compute_objective   simba/policies/mpc_policy.py:26-39   */
  SIMBA_OBJ_SAFE_PENALTY = 1,    /* SafeCemMpc.compute_objective  simba/policies/safe_cem_mpc.py:76-96 */
  SIMBA_OBJ_LEAST_COST = 2,      /* optimize_for_safety (dead code in the reference) safe_cem_mpc.py:40-74,98-108 */
  SIMBA_OBJ_FEASIBLE_FIRST = 3   /* feasible ranked by return, then fewest violations (north-star mode) */
} simba_objective;

typedef enum simba_precision {
  SIMBA_PREC_FP32 = 0,           /* fp32 SIMT rollout: the 1e-4 parity contract                    */
  SIMBA_PREC_BF16_TC = 1         /* bf16 tcgen05 rollout, fp32 accumulate: separately stated tolerance */
} simba_precision;

typedef enum simba_member_map {
  SIMBA_MAP_SPLIT = 0,           /* tf.split: member(r) = r / (P*N/E), r = p*N + i (mlp_ensemble.py:123) */
  SIMBA_MAP_PARTICLE = 1         /* member(p) = floor(p*E/P); equals SPLIT whenever E divides P      */
} simba_member_map;

/* ---- ensemble model: replaces the live Keras variables of MlpEnsemble.ensemble[e]
 *      (simba/models/mlp_ensemble.py:111-112) and TransitionModel.inputs_min/max
 *      (simba/models/transition_model.py:28-29,47-50) ---------------------------------------- */
typedef struct simba_model simba_model_t;

typedef struct simba_model_config {
  int32_t obs_dim;        /* O  (transition_model.py:26) */
  int32_t act_dim;        /* A  (transition_model.py:27) */
  int32_t ensemble_size;  /* E  (mlp_ensemble.py:107)    */
  int32_t n_layers;       /* L  hidden BaseLayers (mlp_ensemble.py:46-49) */
  int32_t units;          /* U  (mlp_ensemble.py:13)     */
} simba_model_config_t;

int simba_model_create(const simba_model_config_t* cfg, simba_model_t** out);
int simba_model_destroy(simba_model_t* m);
/* layer in [0, L): hidden Dense l; L: mu head; L+1: var head. kernel is the Keras layout
 * [in, out]; bias [out]. HOST pointers. (mlp_ensemble.py:13,28-30) */
int simba_model_set_layer(simba_model_t* m, int32_t member, int32_t layer,
                          const float* kernel_in_out, const float* bias);
/* inputs_min / inputs_max: HOST [O + A]. scale_features = 0 makes scale() the identity.
 * Non-finite bounds return SIMBA_ERR_NONFINITE (the reference would produce NaN before its
 * first fit, transition_model.py:85-87). */
int simba_model_set_scaler(simba_model_t* m, const float* inputs_min, const float* inputs_max,
                           int32_t scale_features);
/* pack + upload the fp32 and bf16 weight images; must follow set_layer / set_scaler changes */
int simba_model_commit(simba_model_t* m);

/* ---- reward / cost scorer: replaces SafetyGymStateScorer (simba/environment_utils/safety_gym.py
 *      :104-192, goal task) as a parameter struct ------------------------------------------- */
typedef struct simba_scorer {
  int32_t goal_begin, goal_end;      /* goal_lidar slice (safety_gym.py:170); ignored if goal_dist_index >= 0 */
  int32_t goal_dist_index;           /* observe_goal_dist: relu(obs[idx]) (safety_gym.py:172-174); -1 otherwise */
  int32_t n_constraints;             /* constrained lidar slices, in the reference's order     */
  int32_t con_begin[SIMBA_MAX_CONSTRAINTS];
  int32_t con_end[SIMBA_MAX_CONSTRAINTS];
  float con_size[SIMBA_MAX_CONSTRAINTS];   /* vases_size / hazards_size / ... (safety_gym.py:151,155,159,163) */
  float lidar_max_dist;              /* safety_gym_registery.py:14 */
  float goal_threshold;              /* goal_size * 0.8 (safety_gym.py:117) */
  float reward_distance, reward_goal;
  float reward_clip;                 /* 0 = no clip (safety_gym.py:141-142) */
  int32_t constrain_indicator;       /* safety_gym.py:164-165 */
} simba_scorer_t;

/* ---- planner: replaces CemMpc / SafeCemMpc objects (simba/policies/cem_mpc.py:7-29,
 *      safe_cem_mpc.py:8-34). Immutable after creation (the reference bakes these ints into its
 *      tf.function trace, tune_cem_policy.py:108-115); weights are shared through the model. --- */
typedef struct simba_planner simba_planner_t;

typedef struct simba_planner_config {
  int32_t horizon;         /* H */
  int32_t iterations;      /* I */
  int32_t n_samples;       /* N (global population) */
  int32_t n_elite;         /* K */
  int32_t particles;       /* P */
  int32_t n_states;        /* S independent states planned per call (1 = the reference) */
  float smoothing, stddev_threshold, noise_stddev;            /* cem_mpc.py:26-29 */
  float posterior_mean_threshold;                             /* safe_cem_mpc.py:33 [sic threashold] */
  float prior_mu, prior_sigma;                                /* safe_cem_mpc.py:81 (0.5, 0.27) */
  int32_t objective;             /* simba_objective  */
  int32_t sampling_propagation;  /* transition_model.py:75 */
  int32_t precision;             /* simba_precision  */
  int32_t member_map;            /* simba_member_map */
  int32_t rank, world_size;      /* population shard: this rank rolls out candidates
                                    [rank*N/world, (rank+1)*N/world)           */
  float act_low[SIMBA_MAX_ACT], act_high[SIMBA_MAX_ACT];      /* clip bounds  (mpc_policy.py:45-57) */
  float init_mean[SIMBA_MAX_ACT], init_stddev[SIMBA_MAX_ACT]; /* initial mu, sigma                  */
  simba_scorer_t scorer;
} simba_planner_config_t;

int simba_planner_create(simba_model_t* model, const simba_planner_config_t* cfg,
                         simba_planner_t** out);
int simba_planner_destroy(simba_planner_t* p);

/* External normal draws (parity mode). DEVICE pointers or NULL (NULL = Philox4x32-10, see
 * csrc/philox.cuh and oracle/philox.py for the counter map):
 *   z_actions [I, S, N, H, A]   (cem_mpc.py:44)
 *   eps       [I, S, H, P*N, O] (mlp_ensemble.py:193), rows are global r = p*N + i
 *   z_final   [S, A]            (cem_mpc.py:68)                                          */
int simba_planner_set_external_draws(simba_planner_t* p, const float* z_actions, const float* eps,
                                     const float* z_final);

/* k1  action sampling — cem_mpc.py:44-48.  a = clip(z*sigma + mu, lb, ub) for ALL N candidates.
 * mu, sigma [S, H, A]; z_or_null [S, N, H, A]; out_actions [S, N, H, A]. DEVICE. */
int simba_sample_actions(simba_planner_t* p, const float* mu, const float* sigma,
                         const float* z_or_null, uint64_t seed, int32_t iteration,
                         const int32_t* active_or_null, float* out_actions, void* stream);

/* k2-k7  fused ensemble rollout + scoring — cem_mpc.py:49-55, transition_model.py:64-87,
 * mlp_ensemble.py:122-132,189-193, safety_gym.py:110-166, the per-row part of
 * mpc_policy.py:26-37 / safe_cem_mpc.py:82-93. One launch per CEM iteration; trajectories
 * never reach HBM. states [S, O]; actions [S, N, H, A]; eps_or_null [S, H, P*N, O];
 * outputs per local row [S, P, N_local]: cumulative masked reward, bit t = cost(s_t)*(1-done_t)
 * (done order per objective), and the unmasked cost sum. DEVICE. */
int simba_rollout_score(simba_planner_t* p, const float* states, const float* actions,
                        const float* eps_or_null, uint64_t seed, int32_t iteration,
                        const int32_t* active_or_null, float* out_row_return,
                        uint64_t* out_row_costmask, float* out_row_costsum, void* stream);

/* k8  cross-particle reduction — mpc_policy.py:38-39, safe_cem_mpc.py:94-96,110-120,98-108.
 * -> per local candidate (return, cost) pairs [S, N_local, 2]: return = mean over particles;
 * cost = max_t count_t (SAFE_PENALTY / FEASIBLE_FIRST), mean cost sum (LEAST_COST), 0 (REWARD). */
int simba_score_reduce(simba_planner_t* p, const float* row_return, const uint64_t* row_costmask,
                       const float* row_costsum, const int32_t* active_or_null,
                       float* out_pairs_local, void* stream);

/* the one collective: NCCL all-gather of the (return, cost) pairs over NVLink.
 * pairs_local [S, N_local, 2] -> out_pairs_all [world, S, N_local, 2]. world_size 1 = device copy. */
int simba_allgather_scores(simba_planner_t* p, const float* pairs_local, float* out_pairs_all,
                           void* stream);

/* k9  elite selection — cem_mpc.py:56-60. Top-K of the score implied by `objective`
 * (ties -> lower index), ascending index order; best-so-far update with strict '>'.
 * pairs_all [world, S, N_local, 2]; actions [S, N, H, A]; out_elite [S, K] int32;
 * best_action [S, A] and best_score [S] are read-modify-write. DEVICE. */
int simba_select_elites(simba_planner_t* p, const float* pairs_all, const float* actions,
                        const int32_t* active_or_null, int32_t* out_elite, float* out_scores_or_null,
                        float* best_action, float* best_score, void* stream);

/* k10  refit — cem_mpc.py:61-67. Population moments of the elites, smoothing, and the
 * early-exit test mean(sigma) <= stddev_threshold which clears active[s]. mu/sigma [S, H, A]
 * are updated in place; iterations_run[S] counts iterations executed. DEVICE. */
int simba_refit(simba_planner_t* p, const float* actions, const int32_t* elite, float* mu,
                float* sigma, int32_t* active_or_null, int32_t* iterations_run_or_null,
                void* stream);

/* k11  final exploration noise — cem_mpc.py:68 (not re-clipped). */
int simba_finalize_action(simba_planner_t* p, const float* best_action, const float* z_or_null,
                          uint64_t seed, float* out_action, void* stream);

/* The planning call — CemMpc.do_generate_action, cem_mpc.py:35-68 (SafeCemMpc: safe_cem_mpc.py
 * :36-38). DEVICE pointers, asynchronous: states [S, O] -> out_action [S, A], out_score [S],
 * out_iterations [S] (may be NULL). Runs as one CUDA graph of the kernels above. */
int simba_plan(simba_planner_t* p, const float* states, uint64_t seed, float* out_action,
               float* out_score, int32_t* out_iterations, void* stream);

/* Same with HOST buffers (pageable or pinned), synchronous: what generate_action() calls —
 * cem_mpc.py:31-33. Includes the host<->device copies. */
int simba_plan_host(simba_planner_t* p, const float* states_host, uint64_t seed,
                    float* out_action_host, float* out_score_host, int32_t* out_iterations_host);

/* workspace access for tests / diagnostics: DEVICE pointer + byte size of an internal buffer */
typedef enum simba_buffer {
  SIMBA_BUF_ACTIONS = 0, SIMBA_BUF_ROW_RETURN = 1, SIMBA_BUF_ROW_COSTMASK = 2,
  SIMBA_BUF_ROW_COSTSUM = 3, SIMBA_BUF_PAIRS_LOCAL = 4, SIMBA_BUF_PAIRS_ALL = 5,
  SIMBA_BUF_ELITE = 6, SIMBA_BUF_MU = 7, SIMBA_BUF_SIGMA = 8, SIMBA_BUF_BEST_ACTION = 9,
  SIMBA_BUF_BEST_SCORE = 10, SIMBA_BUF_ACTIVE = 11, SIMBA_BUF_SCORES = 12
} simba_buffer;
int simba_planner_buffer(simba_planner_t* p, int32_t which, void** out_ptr, uint64_t* out_bytes);
/* copy an internal buffer to caller-owned DEVICE memory (dst must hold out_bytes of the query above) */
int simba_planner_copy_buffer(simba_planner_t* p, int32_t which, void* dst_device, void* stream);
/* number of kernel launches one simba_plan() enqueues (graph nodes that are kernels) */
int simba_planner_launches_per_plan(simba_planner_t* p, int32_t* out);
/* Beta-posterior count threshold c_max used for the safety test (safe_cem_mpc.py:110-120) */
int simba_planner_count_threshold(simba_planner_t* p, int32_t* out);
/* the rollout kernel a planner launches, chosen at creation from the shapes, the precision and the
 * device's SM count */
typedef enum simba_rollout_kernel {
  SIMBA_ROLLOUT_FP32 = 0,          /* fp32 SIMT, 32-row tiles                                        */
  SIMBA_ROLLOUT_TC_ONE_CTA = 1,    /* bf16 tcgen05, one CTA per 128-row tile                         */
  SIMBA_ROLLOUT_TC_PAIR = 2,       /* bf16 tcgen05, a cluster of two CTAs per tile (at most SMs / 2 tiles) */
  SIMBA_ROLLOUT_TC_TWO_TILE = 3,   /* bf16 tcgen05, persistent CTAs, two tiles per work item (more tiles than SMs) */
  SIMBA_ROLLOUT_TC_WIDE = 4,       /* bf16 tcgen05 weight-streaming kernel, 128 < units <= ~416      */
  SIMBA_ROLLOUT_TC_WIDE_OBS = 5    /* the same with 128 state columns: obs_dim + act_dim + 2 <= 128, obs_dim <= 124,
                                      units <= 384, for bf16 shapes the kernels above reject           */
} simba_rollout_kernel;
/* -> *kernel (simba_rollout_kernel) and *work_items, the number of work items one launch walks */
int simba_planner_rollout_kernel(simba_planner_t* p, int32_t* kernel, int32_t* work_items);

/* multi-GPU plumbing: the communicator for simba_allgather_scores. unique_id is NCCL's
 * 128-byte ncclUniqueId, produced on rank 0 and broadcast by the caller (torch.distributed). */
int simba_nccl_unique_id(void* out_128_bytes_host);
int simba_planner_init_nccl(simba_planner_t* p, const void* unique_id_128_bytes_host);

/* ---- model-level entry points (the other public methods of the reference's model interface) -- */
/* TransitionModel.unfold_sequences — transition_model.py:64-77. s0 [B, O]; actions [B, H, A];
 * eps_or_null [H, B, O]; out_traj [B, H+1, O] (s_0, then s_1 .. s_H). member map = tf.split (B % E == 0).
 * fp32 SIMT kernel (rollout_f32_kernel), 1 <= H <= 65535. Noise: eps_or_null, else Philox NOISE stream with
 * row = batch index, iteration 0, state 0. DEVICE pointers, asynchronous on stream. */
int simba_unfold(simba_model_t* m, const float* s0, const float* actions, const float* eps_or_null,
                 uint64_t seed, int32_t batch, int32_t horizon, int32_t sampling_propagation,
                 float* out_traj, void* stream);
/* The same on the bf16 tcgen05 rollout kernels of a bf16 planner (the trajectory form of the kernel
 * simba_unfold_tc_kernel reports): same arguments, layouts and noise contract, with weights, activations and
 * normal draws rounded to bf16 as the planner's rollouts are; states stay fp32. s_0 is copied bit for bit.
 * SIMBA_ERR_UNSUPPORTED for shapes no tcgen05 kernel covers (no fp32 fall-back). */
int simba_unfold_tc(simba_model_t* m, const float* s0, const float* actions, const float* eps_or_null,
                    uint64_t seed, int32_t batch, int32_t horizon, int32_t sampling_propagation,
                    float* out_traj, void* stream);
/* -> *kernel (simba_rollout_kernel) and *work_items that simba_unfold_tc would launch for this batch and
 * horizon on the current device */
int simba_unfold_tc_kernel(simba_model_t* m, int32_t batch, int32_t horizon, int32_t* kernel,
                           int32_t* work_items);
/* MlpEnsemble.forward / __call__ — mlp_ensemble.py:122-132,189-193. x [B, O+A] is used as given
 * (already scaled); out_mu, out_var [B, O]; out_sample_or_null = mu + sqrt(var) * eps. */
int simba_ensemble_forward(simba_model_t* m, const float* x, const float* eps_or_null,
                           int32_t batch, float* out_mu, float* out_var, float* out_sample_or_null,
                           void* stream);
/* The same on the bf16 tcgen05 kernels of a bf16 planner (the forward form of the kernel
 * simba_ensemble_forward_tc_kernel reports): same arguments, layouts and errors, with x, weights and activations
 * rounded to bf16 as the planner's rollouts are, fp32 accumulators and eps rounded to bf16 in the sample. mu is the
 * head's fp32 accumulator; var = softplus(raw) + 1e-4 on the MUFU path. SIMBA_ERR_UNSUPPORTED for shapes no
 * tcgen05 kernel covers (no fp32 fall-back). */
int simba_ensemble_forward_tc(simba_model_t* m, const float* x, const float* eps_or_null, int32_t batch,
                              float* out_mu, float* out_var, float* out_sample_or_null, void* stream);
/* -> *kernel (simba_rollout_kernel) and *work_items that simba_ensemble_forward_tc would launch for this batch on
 * the current device: those of simba_unfold_tc_kernel at horizon 1 */
int simba_ensemble_forward_tc_kernel(simba_model_t* m, int32_t batch, int32_t* kernel, int32_t* work_items);
/* TransitionModel.scale — transition_model.py:79-87. x [B, O+A] -> out [B, O+A]. */
int simba_scale(simba_model_t* m, const float* x, int32_t batch, float* out, void* stream);
/* compute_objective on materialised trajectories — mpc_policy.py:26-39 / safe_cem_mpc.py:76-96.
 * traj [P*N, H+1, O] -> out_scores [N] (and out_pairs [N, 2] if not NULL). */
int simba_score_trajectories(simba_planner_t* p, const float* traj, float* out_scores,
                             float* out_pairs_or_null, void* stream);
/* SafetyGymStateScorer.reward / .cost on batches — safety_gym.py:110-166. obs, next_obs [B, O]. */
int simba_scorer_eval(const simba_scorer_t* sc, const float* obs, const float* next_obs,
                      int32_t batch, int32_t obs_dim, float* out_reward, int32_t* out_done,
                      float* out_cost, void* stream);

/* ---- ensemble training step (SURVEY.md section 8 f1) ----------------------------------------
 * Replaces MlpEnsemble.training_step / validation_step / fit (simba/models/mlp_ensemble.py:134-187):
 * forward (training=True, dropout 0), negative_log_likelihood (:64-67) summed over members / E,
 * backward, and tf.keras.optimizers.Adam(clipvalue, epsilon) with EpochLearningRateSchedule
 * (:70-88, :113-117) — CUDA kernels on fp32 master weights that stay on the device. The GEMMs run
 * in fp32 (default) or, with precision = SIMBA_PREC_BF16_TC, on bf16 tcgen05 tensor cores. */
typedef struct simba_trainer simba_trainer_t;
typedef struct simba_trainer_config {
  int32_t batch_size;        /* models.yaml:4 — the largest training batch (rows per member)     */
  int32_t max_eval_rows;     /* row capacity of validation_step chunks (>= batch_size)          */
  float learning_rate;       /* models.yaml:6                                                   */
  int32_t lr_schedule;       /* models.yaml:7: 1 = EpochLearningRateSchedule                    */
  int32_t steps_per_epoch;   /* mlp_ensemble.py:114 (training_steps)                            */
  int32_t train_epochs;      /* agent_factory.py:22                                             */
  float beta1, beta2;        /* Keras defaults 0.9, 0.999                                       */
  float epsilon;             /* mlp_ensemble.py:117 (1e-5)                                      */
  float clipvalue;           /* mlp_ensemble.py:116 (1.0); <= 0 disables clipping               */
  float dropout_rate;        /* models.yaml:13 (0.0): Dropout after every hidden ReLU in training */
  uint64_t dropout_seed;     /* Philox key of the dropout masks (stream 4, see oracle/philox.py)  */
  int32_t precision;         /* simba_precision. SIMBA_PREC_FP32 (0): the fp32 SIMT kernels, parity
                                with the oracle. SIMBA_PREC_BF16_TC: bf16 tcgen05 GEMMs with fp32
                                accumulation, NLL and Adam on fp32 master weights (DESIGN.md section 5,
                                "bf16 training"); covers units <= 416, obs_dim + act_dim <= 126,
                                obs_dim <= 124, n_layers <= 6 and returns SIMBA_ERR_UNSUPPORTED for
                                any other shape (no fp32 fall-back)                               */
} simba_trainer_config_t;

/* Copies the model's current (set_layer) weights as fp32 master weights; Adam state zeroed. The
 * model handle must outlive the trainer (simba_trainer_sync_model writes back into it). */
int simba_trainer_create(simba_model_t* m, const simba_trainer_config_t* cfg, simba_trainer_t** out);
int simba_trainer_destroy(simba_trainer_t* t);
/* MlpEnsemble.training_step — mlp_ensemble.py:134-146. x DEVICE [E, rows, O+A] (already scaled),
 * y DEVICE [E, rows, O], rows <= batch_size; out_loss DEVICE [1] (may be NULL). Async on stream. */
int simba_trainer_step(simba_trainer_t* t, const float* x, const float* y, int32_t rows,
                       float* out_loss, void* stream);
/* The inner loop of MlpEnsemble.fit — mlp_ensemble.py:172-186: `steps` training steps, step s on
 * rows batch_index[s, e, 0:batch_rows[s]] of inputs/targets for member e. inputs DEVICE [n, O+A],
 * targets DEVICE [n, O], batch_index DEVICE int32 [steps, E, batch_size], batch_rows DEVICE int32
 * [steps] or NULL (= batch_size everywhere), out_losses DEVICE [steps]. One CUDA graph per step. */
int simba_trainer_fit(simba_trainer_t* t, const float* inputs, const float* targets, int64_t n,
                      const int32_t* batch_index, const int32_t* batch_rows, int32_t steps,
                      float* out_losses, void* stream);
/* MlpEnsemble.validation_step — mlp_ensemble.py:148-156: every member on the same rows.
 * x DEVICE [rows, O+A], y DEVICE [rows, O]; out_loss DEVICE [1]. */
int simba_trainer_validation(simba_trainer_t* t, const float* x, const float* y, int64_t rows,
                             float* out_loss, void* stream);
/* Hands the trained weights to the model handle (set_layer + commit, bumps its generation so
 * planners re-capture). Synchronises the stream. */
int simba_trainer_sync_model(simba_trainer_t* t, void* stream);
/* which: 0 weights, 1 last gradients (before clipping), 2 Adam m, 3 Adam v. Keras layout
 * (kernel [in, out], bias [out]) of `layer` in [0, L+2) as in simba_model_set_layer. HOST out. */
int simba_trainer_get(simba_trainer_t* t, int32_t which, int32_t member, int32_t layer,
                      float* kernel_out, float* bias_out);
/* optimizer.iterations */
int64_t simba_trainer_iterations(simba_trainer_t* t);
/* kernels launched by one training step (for bench.py's gpu_launches) */
int simba_trainer_launches_per_step(simba_trainer_t* t);
/* read back the weights given to simba_model_set_layer. HOST out. */
int simba_model_get_layer(simba_model_t* m, int32_t member, int32_t layer, float* kernel_out,
                          float* bias_out);

/* ---- RNG contract probes (tests) --------------------------------------------------------- */
/* raw Philox4x32-10 block: HOST in/out, computed ON THE DEVICE (no CPU path). */
int simba_philox_raw(const uint32_t counter[4], const uint32_t key[2], uint32_t out[4]);
/* the normals a kernel draws: stream 1 = ACTION (rows = candidates, elems = H*A),
 * 2 = NOISE (rows = global rows, elems = O; t = step), 3 = FINAL. out DEVICE [n_rows, n_elems]. */
int simba_philox_normals(uint64_t seed, int32_t rng_stream, int32_t iteration, int32_t t,
                         int32_t state_index, int32_t first_row, int32_t n_rows, int32_t n_elems,
                         int32_t fast_math, float* out, void* stream);

const char* simba_last_error(void);
const char* simba_version(void);
/* 0 if the current device is an sm_100 GPU, else SIMBA_ERR_ARCH / SIMBA_ERR_CUDA */
int simba_device_check(void);

#ifdef __cplusplus
}
#endif
#endif /* SIMBA_B200_H_ */

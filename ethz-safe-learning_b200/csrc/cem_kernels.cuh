// Parameter blocks + launchers of the small CEM kernels (cem_kernels.cu).
#pragma once
#include "common.cuh"

namespace simba {

struct SampleParams {                 // cem_mpc.py:44-48
  int32_t S, N, H, A;
  const float* mu;                    // [S, H, A]
  const float* sigma;                 // [S, H, A]
  const float* z;                     // [S, N, H, A] or null
  float lb[SIMBA_MAX_ACT], ub[SIMBA_MAX_ACT];
  uint64_t seed;
  const uint64_t* seed_ptr;   // if not null the seed is read from device memory (graph replay)
  int32_t iteration;
  const int32_t* active;
  float* out;                         // [S, N, H, A]
  // Population sharding: a rank samples only the candidates it rolls out, [cand0, cand0 + n_cand)
  // (n_cand = 0 means all N). Any rank can regenerate any candidate's row from (seed, iteration, i):
  // selection and refit do that for the elite rows other ranks sampled (regen below).
  int32_t cand0, n_cand;
};

struct ReduceParams {                 // mpc_policy.py:38-39, safe_cem_mpc.py:94-120
  int32_t S, P, N_local, H, objective;
  const float* row_return;            // [S, P, N_local]
  const uint64_t* row_costmask;
  const float* row_costsum;
  const int32_t* active;
  float* out_pairs;                   // [S, N_local, 2]
};

struct SelectParams {                 // cem_mpc.py:56-60
  int32_t S, N, N_local, K, H, A, objective;
  float c_max;
  const float* pairs_all;             // [world, S, N_local, 2]
  const float* actions;               // [S, N, H, A]
  const int32_t* active;
  unsigned long long* key_scratch;    // [S, N] staged order keys (planner workspace)
  int32_t* out_elite;                 // [S, K]
  float* out_scores;                  // [S, N] or null
  float* best_action;                 // [S, A]
  float* best_score;                  // [S]
  int32_t regen;                      // the best candidate's row may not be in `actions`: recompute it
  SampleParams sample;                // ... with this iteration's sampling parameters
};

struct RefitParams {                  // cem_mpc.py:61-67
  int32_t S, N, K, H, A;
  float smoothing, one_minus_smoothing, stddev_threshold;
  float* actions;
  const int32_t* elite;
  float* mu;
  float* sigma;
  int32_t* active;
  int32_t* iterations_run;
  int32_t groups;                     // set by the launch functions: max(1, threads / (H * A)) row groups of the gather
  int32_t regen;                      // elite rows sampled by other ranks are recomputed into `actions` first
  SampleParams sample;                // (same counters => bit-identical to the owner rank's rows)
};

struct FinalizeParams {               // cem_mpc.py:68
  int32_t S, A;
  float noise_stddev;
  const float* best;
  const float* z;
  uint64_t seed;
  const uint64_t* seed_ptr;   // if not null the seed is read from device memory (graph replay)
  float* out;
};

struct PlanInitParams {               // cem_mpc.py:36-42
  int32_t S, H, A;
  float init_mean[SIMBA_MAX_ACT], init_stddev[SIMBA_MAX_ACT];
  float* mu;
  float* sigma;
  float* best_action;
  float* best_score;
  int32_t* active;
  int32_t* iterations_run;
};

struct UpdateParams {                 // fused k8 + k9 + k10 (+ next k1 | k11): one rank, N <= 1024
  ReduceParams reduce;
  SelectParams select;
  RefitParams refit;
  SampleParams sample;                // next iteration's sampling (ignored when last)
  FinalizeParams finalize;            // used when last
  int32_t last;
  int32_t pdl;                        // launch with programmatic stream serialization
  int32_t stage;                      // set by launch_cem_update: rows, actions and draws of a state fit in shared memory
  int32_t chunks, per;                // set by launch_cem_update: threads / N key chunks per candidate, keys per chunk
  float inv_N, inv_JB;                // set by launch_cem_update: reciprocals for div_small
  float* out_score;
  int32_t* out_iters;
  long long* timeline;                // -DSIMBA_TC_TIMELINE builds: clock64 stamps of the phases (tools/tc_timeline.py)
};

// MPPI update (Williams et al., "Information theoretic MPC for model-based reinforcement learning", ICRA 2017):
// w_i = exp((score_i - max score) / temperature), 0 for a NaN score; mu <- smoothing mu + (1 - smoothing) sum w a / sum w;
// sigma stays fixed. One rank: pairs hold all N candidates.
struct MppiParams {
  int32_t S, N, H, A, objective;
  float c_max, temperature, smoothing, one_minus_smoothing;
  const float* pairs;                 // [S, N, 2]
  const float* actions;               // [S, N, H, A]
  const int32_t* active;
  float* mu;                          // [S, H, A], updated in place
  float* best_action;                 // [S, A]   best-so-far (strict '>'), as CEM's selection keeps it
  float* best_score;                  // [S]
  int32_t* iterations_run;            // [S] or null
};

struct MppiUpdateParams {             // fused k8 + MPPI update (+ next k1 | k11): one rank, N <= 1024
  ReduceParams reduce;
  MppiParams mppi;
  SampleParams sample;                // next iteration's sampling (ignored when last)
  FinalizeParams finalize;            // used when last, on mu[s, 0, :]
  int32_t last;
  int32_t pdl;
  int32_t stage;                      // set by launch_mppi_update: rows and actions of a state fit in shared memory
  float* out_score;
  int32_t* out_iters;
};

cudaError_t launch_cem_update(const UpdateParams& u, cudaStream_t st);
cudaError_t launch_mppi_refit(const MppiParams& p, cudaStream_t st);
cudaError_t launch_mppi_update(const MppiUpdateParams& u, cudaStream_t st);
cudaError_t launch_mppi_finalize(const FinalizeParams& p, int HA, cudaStream_t st);   // p.best = mu [S, H, A]
// Dynamic shared memory of the MPPI kernels: the fused update without its optional staging area (P particles, N <= 1024
// candidates), and the separate refit at any N. A plan whose refit does not fit the device is rejected.
size_t mppi_update_smem_bytes(int P, int N, int H, int A, bool* staged);
size_t mppi_refit_smem_bytes(int N, int H, int A);
// Dynamic shared memory of the fused update kernel at these sizes (P particles, N candidates, K elites, horizon H,
// A action dims): the refit scratch and selection keys, plus the staging area of per-row outputs, actions and draws
// when that fits under 200 KB (*staged)
size_t cem_update_smem_bytes(int P, int N, int K, int H, int A, bool* staged);
cudaError_t launch_plan_begin(const PlanInitParams& ip, const SampleParams& sp, cudaStream_t st);
cudaError_t launch_sample_actions(const SampleParams& p, cudaStream_t st);
cudaError_t launch_score_reduce(const ReduceParams& p, cudaStream_t st);
cudaError_t launch_select_elites(const SelectParams& p, cudaStream_t st);
cudaError_t launch_refit(const RefitParams& p, cudaStream_t st);
cudaError_t launch_finalize(const FinalizeParams& p, cudaStream_t st);
cudaError_t launch_plan_init(const PlanInitParams& p, cudaStream_t st);
cudaError_t launch_plan_output(const float* best_score, const int32_t* iterations_run,
                               float* out_score, int32_t* out_iters, int S, cudaStream_t st);
cudaError_t launch_scale(const float* x, const float* smin, const float* sdelta, int scale_on,
                         long batch, int IN, float* out, cudaStream_t st);
cudaError_t launch_scorer_eval(const simba_scorer_t& sc, const float* obs, const float* next_obs,
                               int batch, int O, float* out_reward, int32_t* out_done,
                               float* out_cost, cudaStream_t st);
cudaError_t launch_score_traj_rows(const simba_scorer_t& sc, const float* traj, int rows, int H,
                                   int O, int objective, float* row_return, uint64_t* row_costmask,
                                   float* row_costsum, cudaStream_t st);
cudaError_t launch_pairs_to_scores(const float* pairs, int n, int objective, float c_max,
                                   float* out_scores, cudaStream_t st);
cudaError_t launch_philox_raw(const uint32_t ctr[4], const uint32_t key[2], uint32_t* out_dev,
                              cudaStream_t st);
cudaError_t launch_philox_normals(uint64_t seed, int stream, int iteration, int t, int s,
                                  int first_row, int n_rows, int n_elems, int fast, float* out,
                                  cudaStream_t st);

}  // namespace simba

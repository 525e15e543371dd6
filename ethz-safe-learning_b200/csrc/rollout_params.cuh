// Launch parameters shared by the fp32 and bf16-tcgen05 rollout kernels.
#pragma once
#include <vector>

#include "common.cuh"

namespace simba {

constexpr int kF32TileRows = 32;     // rows per CTA of the fp32 kernel
constexpr int kTcTileRows = 128;     // rows per tile of the tcgen05 kernel (UMMA_M)

// The rollout kernel a planner launches; simba_planner_rollout_kernel reports it with these values.
enum class RolloutKernel : int32_t {
  kF32 = SIMBA_ROLLOUT_FP32,                // rollout_f32.cu, 32-row tiles
  kTcOneCta = SIMBA_ROLLOUT_TC_ONE_CTA,     // rollout_tc.cu <1,4>: one CTA per 128-row tile
  kTcPair = SIMBA_ROLLOUT_TC_PAIR,          // <1,4,pair>: a cluster of two CTAs per tile splits the head pass
  kTcTwoTile = SIMBA_ROLLOUT_TC_TWO_TILE,   // <2,2>: persistent CTAs, two tiles per work item (MMA / epilogue ping-pong)
  kTcWide = SIMBA_ROLLOUT_TC_WIDE,          // rollout_tc_wide.cu <64>: 128 < units <= ~416
  kTcWideObs = SIMBA_ROLLOUT_TC_WIDE_OBS,   // rollout_tc_wide.cu <128>: obs_dim + act_dim + 2 <= 128, obs_dim <= 124, units <= 384
};

struct RolloutParams {
  RowGeom g;
  simba_scorer_t scorer;
  const Tile* tiles;
  int32_t n_tiles;
  int32_t L, U;
  // fp32 image: per member, chunks [n_chunks][16][128] in consumption order; biases padded per layer
  // (rollout_f32_pack)
  const float* w_f32;
  const float* bias_f32;
  int32_t n_chunks, bias_stride, act_rows;
  // bf16 image of the tcgen05 family that runs the model, w_tc_member_bytes per member, in the layout of that
  // family's kernel file (rollout_tc_pack, rollout_tc_wide_pack)
  const void* w_tc;
  int64_t w_tc_member_bytes;
  RolloutKernel kernel;       // the kernel launch_rollout runs
  int32_t n_sms;              // SMs of the planner's device (grid of the persistent tcgen05 kernels)
  int32_t pdl;                // launch with programmatic stream serialization (fused plan path)
  float tc_scale_a[128];      // bf16 path: x_scaled[k] = fma(x[k], a[k], b[k]); zero beyond O + A
  float tc_scale_b[128];
  // scaler (transition_model.py:79-87): x_scaled = (x - smin) / sdelta, sdelta already holds 1.01
  // where max - min < 1e-5
  const float* smin;
  const float* sdelta;
  int32_t scale_on;
  // inputs
  const float* states;        // [S, O] (or per row when state_per_row)
  int64_t state_stride;
  int32_t state_per_row;
  const float* actions;       // [S, N, H, A] : offset = (s * N + i) * action_stride + t * A + a
  int64_t action_stride;
  const float* eps;           // [S, H, P*N, O] or null -> Philox
  uint64_t seed;
  const uint64_t* seed_ptr;   // if not null the seed is read from device memory (graph replay)
  int32_t iteration;
  int32_t sampling_propagation;
  int32_t objective;
  const int32_t* active;      // [S] or null
  // outputs
  float* row_return;
  uint64_t* row_costmask;
  float* row_costsum;
  float* traj_out;            // [rows, H+1, O] or null
  float* mu_out;              // [rows, O] or null (with var_out; sample_out optional)
  float* var_out;
  float* sample_out;
  long long* timeline;        // clock64 stamps of CTA 0 (-DSIMBA_TC_TIMELINE builds only, else null)
};

// Launches the kernel prm.kernel names over prm.tiles: the forward form of a tcgen05 kernel when prm.mu_out is set,
// its trajectory form when prm.traj_out is, its planning form otherwise (the fp32 kernel takes all three from prm at
// run time). Defined in api.cu, next to choose_rollout, which picks prm.kernel and the tile list.
cudaError_t launch_rollout(const RolloutParams& prm, cudaStream_t stream);
// the branches of launch_rollout, one per kernel file
cudaError_t launch_rollout_f32(const RolloutParams& prm, cudaStream_t stream);
cudaError_t launch_rollout_tc(const RolloutParams& prm, cudaStream_t stream);        // kTc{OneCta,Pair,TwoTile}
cudaError_t launch_rollout_tc_wide(const RolloutParams& prm, cudaStream_t stream);   // kTcWide{,Obs}; prm.U: the model's units

// Shape rules of the tcgen05 kernels, from the model alone (api.cu's tc_family combines them). rollout_tc.cu:
bool rollout_tc_supported(int O, int A, int L, int U);
bool rollout_tc_two_tiles_fit(int L, int n_constraints);
bool rollout_tc_pair_fits(int L, int n_constraints);
// The weight-streaming kernel comes in two state widths `sw`: 64 (prm.kernel kTcWide) and 128 (kTcWideObs).
bool rollout_tc_wide_supported(int sw, int O, int A, int L, int U);
bool rollout_tc_wide_fits(int sw, int L, int U, int n_constraints);

// What the weight packers read: the model's config and its Keras layers. Layer l of member e has the kernel
// [K][N] (row-major) and the bias [N] at index e * (n_layers + 2) + l; layers n_layers and n_layers + 1 are the
// mu and raw-variance heads.
struct ModelWeights {
  const simba_model_config_t& cfg;
  const std::vector<std::vector<float>>& kernels;
  const std::vector<std::vector<float>>& biases;
  const float* kernel(int e, int l) const { return kernels[(size_t)e * (cfg.n_layers + 2) + l].data(); }
  const float* bias(int e, int l) const { return biases[(size_t)e * (cfg.n_layers + 2) + l].data(); }
};
// Each kernel file packs the weight image its kernels read. The fp32 packer fills the image and its geometry
// (RolloutParams::n_chunks, bias_stride, act_rows), or returns SIMBA_ERR_UNSUPPORTED for units the fp32 kernel's
// shared memory cannot hold. The tcgen05 packers fill the image of all members and return a member's bytes
// (RolloutParams::w_tc_member_bytes); they run only for shapes that rollout_tc_supported / rollout_tc_wide_supported
// accept.
int rollout_f32_pack(const ModelWeights& mw, std::vector<float>& w, std::vector<float>& b, int& n_chunks,
                     int& bias_stride, int& act_rows);
int64_t rollout_tc_pack(const ModelWeights& mw, std::vector<uint16_t>& img);
int64_t rollout_tc_wide_pack(int sw, const ModelWeights& mw, std::vector<uint16_t>& img);

}  // namespace simba

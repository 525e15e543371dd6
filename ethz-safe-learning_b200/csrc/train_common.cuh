// Device pieces shared by the two ensemble trainers: the fp32 SIMT kernels (trainer_f32.cu) and the bf16
// tcgen05 kernels (trainer_tc.cu). Both run the same step contract — batch gather through the fit
// descriptor, Philox stream-4 dropout masks, the Gaussian negative log-likelihood with its gradient,
// the fixed-order loss reduction and clip + Adam on the fp32 master weights — so these are written once,
// with the description of a training launch (TrainDesc) that the handle in trainer.cu passes to either.
#pragma once
#include <cstdint>

#include "common.cuh"

namespace simba {

struct TrainState {
  int iterations;        // optimizer.iterations
  int fit_step;          // step index inside the running fit()
  float lr_t;            // lr(iterations) * sqrt(1 - beta2^t) / (1 - beta1^t) of the current step
  float loss;
  unsigned nll_ticket;
};

struct FitDesc {
  const float* inputs;
  const float* targets;
  const int* batch_index;   // [steps, E, bmax]
  const int* batch_rows;    // [steps] or null
  float* losses;            // [steps] or null
  int bmax;
};

struct OptParams {
  float lr0, beta1, beta2, epsilon, clipvalue;
  int schedule, steps_per_epoch, train_epochs;
};

constexpr int kMaxTrainLayers = 18;   // train layers: up to 16 hidden layers + the merged Gaussian head

// Train layer l: the Keras kernel [K x N] and its bias as one [(K + 1) x N] row-major block of a member's theta, at
// float offset `off` (the bias is the row that multiplies the constant 1). The Gaussian head's two Dense layers are
// one block with N = 2 * O whose columns interleave (mu_0, var_0, mu_1, var_1, ...).
struct TrainLayer {
  int K, N;
  int64_t off;
};

// Swish training (SIMBA_ACT_SWISH): the backward pass cannot recover swish'(Z) from H, so the training forward pass
// stores, per hidden layer, the multiplier M_l = keep * swish'(Z_l) of dZ_{l-1} = M_l * (dZ_l . theta_l^T). m[l],
// 1 <= l <= L: [E][estride][N_{l-1}], the layout of dz[l - 1].
struct SwishMult {
  float* m[kMaxTrainLayers];
  int64_t estride;                    // rows per member (batch)
};

// What the trainer handle (trainer.cu) owns, and the inputs of one call, in a form both precisions launch from. Each
// launcher below translates it into its own kernels' arguments.
struct TrainDesc {
  int L;                              // hidden layers; layer L is the head
  TrainLayer layer[kMaxTrainLayers];
  float* act[kMaxTrainLayers];        // act[l], l >= 1: input of layer l [E][act_estride][K_l] (H_l after dropout)
  int64_t act_estride;                // rows per member (cap)
  float* dz[kMaxTrainLayers];         // dz[l]: gradient w.r.t. the pre-activation of layer l [E][dz_estride][N_l]
  int64_t dz_estride;                 // rows per member (batch)
  const float* x;                     // [E][rows][K_0] (estride may be 0: validation shares its rows)
  int64_t x_estride;
  int gather;                         // 1: batch rows follow the fit descriptor's index
  const float* y;                     // [E][rows][O]
  int64_t y_estride;
  float *theta, *m, *v, *grad;        // fp32 master weights, Adam slots and last gradient, [E][pn]
  int64_t pn;
  uint8_t* img;                       // derived from theta, img_member_bytes per member, rewritten by every update:
  int64_t img_member_bytes;           // theta^T for fp32, the UMMA images for bf16
  int out_dim, ensemble;
  float* partial;                     // [E][tiles_cap][2]: NLL partials of the chain's row tiles
  int tiles_cap;
  int train;                          // 0: forward and likelihood only (validation)
  float* out_loss;
  float dropout_rate, dropout_scale;
  uint64_t dropout_seed;
  int activation;                     // simba_activation of the hidden layers
  SwishMult mult;                     // swish models only (else null)
};

// The host side of each precision: train_f32_* (trainer_f32.cu) and train_tc_* (trainer_tc.cu, bf16 tcgen05).
//   check        SIMBA_OK, or SIMBA_ERR_UNSUPPORTED with its message for a shape the kernels cannot train
//   image_bytes  a member's image
//   pack         one member's image from its host theta; `img` must be zeroed
//   chain        forward + likelihood (+ back-propagation of the activations when d.train) over `grid_rows` rows;
//                `row_tiles` receives the CTAs per member, i.e. the partials it writes
//   update       weight gradients, clip and Adam for every layer, and the image of the new weights
int train_f32_check(const TrainDesc& d);
int train_tc_check(const simba_model_config_t& mc);
int64_t train_f32_image_bytes(const TrainDesc& d);
int64_t train_tc_image_bytes(const TrainDesc& d);
void train_f32_pack(const TrainDesc& d, const float* theta, uint8_t* img);
void train_tc_pack(const TrainDesc& d, const float* theta, uint8_t* img);
cudaError_t train_f32_chain(const TrainDesc& d, const OptParams& opt, const FitDesc* desc, TrainState* st,
                            int grid_rows, int rows_fixed, int step_off, cudaStream_t s, int& row_tiles);
cudaError_t train_tc_chain(const TrainDesc& d, const OptParams& opt, const FitDesc* desc, TrainState* st,
                           int grid_rows, int rows_fixed, int step_off, cudaStream_t s, int& row_tiles);
cudaError_t train_f32_update(const TrainDesc& d, const OptParams& opt, const FitDesc* desc, const TrainState* st,
                             int rows_fixed, int step_off, cudaStream_t s);
cudaError_t train_tc_update(const TrainDesc& d, const OptParams& opt, const FitDesc* desc, const TrainState* st,
                            int rows_fixed, int step_off, cudaStream_t s);

}  // namespace simba

namespace {
// using-declarations, not `using namespace simba`: the directive would put simba's unnamed namespace (tc_ptx.cuh)
// beside this one, and nvcc's host stubs for kernels kept in this one (trainer_f32.cu) would then be ambiguous
using simba::FitDesc;
using simba::OptParams;
using simba::TrainState;
using simba::philox4x32_10;
using simba::philox_key;
using simba::softplus_tf;
using simba::u01;
using simba::SwishMult;
using simba::kActSwish;
using simba::swish_f32;
using simba::swish_grad_f32;

// A captured graph holds several consecutive steps: step i of the graph works at
// (st->fit_step + i, st->iterations + i) and one single-thread kernel advances the counters at
// the end of the graph, so no kernel of the step needs a grid-wide "last CTA" handshake for it.
__device__ __forceinline__ int resolve_rows(const FitDesc* desc, const TrainState* st, int rows_fixed,
                                            int step_off) {
  if (desc != nullptr && desc->batch_rows != nullptr) return desc->batch_rows[st->fit_step + step_off];
  return rows_fixed;
}

// fit(): `train_inputs[shuffles_per_mlp]` (mlp_ensemble.py:175-176) is never materialised — the
// kernels that read the batch follow the index
__device__ __forceinline__ const int* batch_rows_of(const FitDesc* desc, const TrainState* st, int e,
                                                    int ensemble, int step_off) {
  return desc->batch_index + ((int64_t)(st->fit_step + step_off) * ensemble + e) * desc->bmax;
}

__device__ __forceinline__ float block_sum(float v, float* scratch) {
  // fixed-order tree: shuffles inside the warp, then thread 0 adds the warp sums in order
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  __syncthreads();
  if (l == 0) scratch[w] = v;
  __syncthreads();
  float s = 0.0f;
  if (threadIdx.x == 0)
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) s += scratch[i];
  return s;   // valid in thread 0
}

__device__ float schedule_lr(const OptParams& o, int iterations) {
  if (!o.schedule) return o.lr0;
  const float epochs = floorf((float)(iterations / o.steps_per_epoch));
  return fmaxf(o.lr0 * (1.0f - epochs / (float)o.train_epochs), 0.0f);
}

// Dropout after every hidden activation in training (mlp_ensemble.py:17-22): keep = u01(philox) >= rate,
// kept activations scaled by 1 / (1 - rate). One Philox block covers columns col .. col + 3 (col a
// multiple of 4). Counter (column block, batch row, iteration, member | layer << 8 | stream 4 << 28),
// key = dropout_seed — restated in oracle/philox.py.
__device__ __forceinline__ void dropout_keep4(int col, int row, uint32_t iteration, int member, int layer,
                                              float rate, float scale, uint64_t seed, float (&keep)[4]) {
  const uint4 bits = philox4x32_10(
      make_uint4((uint32_t)(col >> 2), (uint32_t)row, iteration,
                 (uint32_t)member | ((uint32_t)layer << 8) | (4u << 28)),
      philox_key(seed));
  keep[0] = u01(bits.x) >= rate ? scale : 0.0f;
  keep[1] = u01(bits.y) >= rate ? scale : 0.0f;
  keep[2] = u01(bits.z) >= rate ? scale : 0.0f;
  keep[3] = u01(bits.w) >= rate ? scale : 0.0f;
}

// negative_log_likelihood (mlp_ensemble.py:64-67) of one output: accumulates log(2 pi var) and
// (mu - y)^2 / var, and returns d(loss)/d(mu) and d(loss)/d(raw var) for the loss scale c =
// 1 / (rows * O * E). var = softplus(raw) + 1e-4 (mlp_ensemble.py:30), accurate libm math.
__device__ __forceinline__ void nll_terms(float mu, float pre, float y, float c, float& s_log, float& s_sq,
                                          float& d_mu, float& d_pre) {
  const float var = softplus_tf(pre) + 1e-4f;
  const float diff = mu - y;
  const float inv = 1.0f / var;
  s_log += logf(6.28318530717958647692f * var);
  s_sq += diff * diff * inv;
  d_mu = c * diff * inv;
  d_pre = 0.5f * c * (inv - diff * diff * inv * inv) * (1.0f / (1.0f + expf(-pre)));
}

// clip + tf.keras.optimizers.Adam (non-amsgrad) of one variable, in two halves so that callers can store
// the slots before the weight: adam_slots (mo, ve) -> (m, v), then adam_weight -> the new weight
__device__ __forceinline__ void adam_slots(float g, float mo, float ve, const OptParams& o, float& m, float& v) {
  if (o.clipvalue > 0.0f) g = fminf(fmaxf(g, -o.clipvalue), o.clipvalue);
  m = mo + (1.0f - o.beta1) * (g - mo);
  v = ve + (1.0f - o.beta2) * (g * g - ve);
}
__device__ __forceinline__ float adam_weight(float w, float m, float v, const OptParams& o, float lr_t) {
  return w - lr_t * m / (sqrtf(v) + o.epsilon);
}

// End of the bf16 chain kernel, every CTA: its NLL partials (s_log, s_sq summed over the block) go to
// partial[e][tile]. In training, the last CTA to arrive adds every member's partials in a fixed order,
// stores the loss and the step's lr_t, and re-arms the ticket. `tiles` row tiles cover the batch. The
// fp32 chain kernel keeps the same sequence inline: called from there, this function changes that
// kernel's register allocation.
__device__ __forceinline__ void finish_chain_loss(float s_log, float s_sq, float* scratch, bool& last,
                                                  float* partial, int tiles_cap, int tiles, int rows,
                                                  int out_dim, int ensemble, int train, float* out_loss,
                                                  const OptParams& opt, const FitDesc* desc, TrainState* st,
                                                  int step_off) {
  const int tid = threadIdx.x, e = blockIdx.y;
  const float t_log = block_sum(s_log, scratch);
  const float t_sq = block_sum(s_sq, scratch);
  if (tid == 0) {
    partial[((int64_t)e * tiles_cap + blockIdx.x) * 2 + 0] = t_log;
    partial[((int64_t)e * tiles_cap + blockIdx.x) * 2 + 1] = t_sq;
  }
  if (!train) return;
  if (tid == 0) {
    __threadfence();
    last = (atomicAdd(&st->nll_ticket, 1u) == gridDim.x * gridDim.y - 1);
  }
  __syncthreads();
  if (!last || tid >= 32) return;
  __threadfence();
  const float denom = (float)rows * (float)out_dim;
  float loss = 0.0f;
  for (int m = 0; m < ensemble; ++m) {
    float sl = 0.0f, sq = 0.0f;
    for (int t = tid; t < tiles; t += 32) {
      sl += __ldcg(&partial[((int64_t)m * tiles_cap + t) * 2 + 0]);
      sq += __ldcg(&partial[((int64_t)m * tiles_cap + t) * 2 + 1]);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      sl += __shfl_down_sync(0xffffffffu, sl, o);
      sq += __shfl_down_sync(0xffffffffu, sq, o);
    }
    loss += (0.5f * (sl / denom) + 0.5f * (sq / denom)) / (float)ensemble;
  }
  if (tid != 0) return;
  const int it = st->iterations + step_off;
  const float t = (float)(it + 1);
  st->lr_t = schedule_lr(opt, it) * sqrtf(1.0f - powf(opt.beta2, t)) / (1.0f - powf(opt.beta1, t));
  st->loss = loss;
  if (out_loss) *out_loss = loss;
  if (desc != nullptr && desc->losses != nullptr) desc->losses[st->fit_step + step_off] = loss;
  st->nll_ticket = 0;
}

}  // namespace

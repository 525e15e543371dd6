// Ensemble training step on the device (include/simba_b200.h "ensemble training step"):
// replaces MlpEnsemble.training_step / validation_step / fit's inner loop
// (simba/models/mlp_ensemble.py:134-187). This file is the handle: the fp32 master weights, Adam state,
// activation and gradient buffers, the loss accumulators and the captured fit graphs, the same for both
// precisions. The kernels of a step are the chosen precision's: trainer_f32.cu's fp32 SIMT kernels
// (SIMBA_PREC_FP32) or trainer_tc.cu's tcgen05 kernels (SIMBA_PREC_BF16_TC), two launches per step either way.
// Each also reads one image derived from the master weights, which the handle allocates and packs for the
// chosen precision only.
#include <cstdint>
#include <cstring>
#include <vector>

#include "common.cuh"
#include "internal.h"
#include "train_common.cuh"

using namespace simba;

// simba_model_create allows up to 16 hidden layers; the merged head is one more train layer
static_assert(16 + 1 <= kMaxTrainLayers, "train layers of the largest model");

namespace {

constexpr int kGraphSteps = 16;  // fit(): steps per CUDA-graph launch

__global__ void advance_kernel(TrainState* st, int n) {
  st->iterations += n;
  st->fit_step += n;
}

__global__ void set_fit_desc_kernel(FitDesc d, FitDesc* out, TrainState* st) {
  *out = d;
  st->fit_step = 0;
}

// validation_step (mlp_ensemble.py:148-156): chunk partials -> running sums -> loss
__global__ void val_accumulate_kernel(const float* partial, int tiles_cap, int tiles, int ensemble,
                                      double* acc, int reset) {
  const int e = threadIdx.x;
  if (e >= ensemble) return;
  double sl = reset ? 0.0 : acc[e * 2], sq = reset ? 0.0 : acc[e * 2 + 1];
  for (int t = 0; t < tiles; ++t) {
    sl += partial[((int64_t)e * tiles_cap + t) * 2 + 0];
    sq += partial[((int64_t)e * tiles_cap + t) * 2 + 1];
  }
  acc[e * 2] = sl;
  acc[e * 2 + 1] = sq;
}

__global__ void val_finalize_kernel(const double* acc, int ensemble, double denom, float* out_loss) {
  double loss = 0.0;
  for (int e = 0; e < ensemble; ++e)
    loss += (0.5 * acc[e * 2] / denom + 0.5 * acc[e * 2 + 1] / denom) / ensemble;
  *out_loss = (float)loss;
}

}   // namespace

// ---------------------------------------------------------------------------------------------
// handle
// ---------------------------------------------------------------------------------------------
struct simba_trainer {
  simba_model_t* model = nullptr;
  simba_trainer_config_t cfg{};
  int E = 0, L = 0, U = 0, O = 0, IN = 0;
  int cap_rows = 0;
  TrainDesc d{};                     // layers and device buffers; the call inputs (x .. out_loss) stay zero here
  double* val_acc = nullptr;
  TrainState* state = nullptr;
  FitDesc* desc = nullptr;
  cudaGraphExec_t fit_graph = nullptr;      // one training step
  cudaGraphExec_t fit_graph_n = nullptr;    // kGraphSteps consecutive steps (amortises the launch gap)
  cudaStream_t graph_stream = nullptr;
};

static bool bf16(const simba_trainer_t* t) { return t->cfg.precision == SIMBA_PREC_BF16_TC; }

static OptParams opt_params(const simba_trainer_t* t) {
  OptParams o;
  o.lr0 = t->cfg.learning_rate;
  o.beta1 = t->cfg.beta1;
  o.beta2 = t->cfg.beta2;
  o.epsilon = t->cfg.epsilon;
  o.clipvalue = t->cfg.clipvalue;
  o.schedule = t->cfg.lr_schedule;
  o.steps_per_epoch = t->cfg.steps_per_epoch;
  o.train_epochs = t->cfg.train_epochs;
  return o;
}

// Keras arrays of one member -> the [(K+1) x N] blocks of theta (host)
static int pull_member(simba_trainer_t* t, int e, float* theta_e) {
  std::vector<float> kern, bias, kern2, bias2;
  for (int l = 0; l < t->L; ++l) {
    const TrainLayer& ly = t->d.layer[l];
    kern.resize((size_t)ly.K * ly.N);
    bias.resize(ly.N);
    int rc = simba_model_get_layer(t->model, e, l, kern.data(), bias.data());
    if (rc) return rc;
    float* dst = theta_e + ly.off;
    memcpy(dst, kern.data(), kern.size() * sizeof(float));
    memcpy(dst + kern.size(), bias.data(), bias.size() * sizeof(float));
  }
  const int U = t->U, O = t->O;
  kern.resize((size_t)U * O); bias.resize(O); kern2.resize((size_t)U * O); bias2.resize(O);
  int rc = simba_model_get_layer(t->model, e, t->L, kern.data(), bias.data());
  if (rc) return rc;
  rc = simba_model_get_layer(t->model, e, t->L + 1, kern2.data(), bias2.data());
  if (rc) return rc;
  float* dst = theta_e + t->d.layer[t->L].off;
  for (int k = 0; k < U; ++k)
    for (int o = 0; o < O; ++o) {
      dst[(size_t)k * 2 * O + 2 * o] = kern[(size_t)k * O + o];
      dst[(size_t)k * 2 * O + 2 * o + 1] = kern2[(size_t)k * O + o];
    }
  for (int o = 0; o < O; ++o) {
    dst[(size_t)U * 2 * O + 2 * o] = bias[o];
    dst[(size_t)U * 2 * O + 2 * o + 1] = bias2[o];
  }
  return SIMBA_OK;
}

// one block of theta (host) -> Keras kernel / bias of `layer` in [0, L + 2)
static void split_layer(const simba_trainer_t* t, const float* theta_e, int layer, float* kernel,
                        float* bias) {
  if (layer < t->L) {
    const TrainLayer& ly = t->d.layer[layer];
    const float* src = theta_e + ly.off;
    const size_t nk = (size_t)ly.K * ly.N;
    memcpy(kernel, src, nk * sizeof(float));
    memcpy(bias, src + nk, ly.N * sizeof(float));
    return;
  }
  const int U = t->U, O = t->O, c0 = layer == t->L ? 0 : 1;
  const float* src = theta_e + t->d.layer[t->L].off;
  for (int k = 0; k < U; ++k)
    for (int o = 0; o < O; ++o) kernel[(size_t)k * O + o] = src[(size_t)k * 2 * O + 2 * o + c0];
  for (int o = 0; o < O; ++o) bias[o] = src[(size_t)U * 2 * O + 2 * o + c0];
}

extern "C" int simba_trainer_destroy(simba_trainer_t* t) {
  if (!t) return SIMBA_OK;
  if (t->fit_graph) cudaGraphExecDestroy(t->fit_graph);
  if (t->fit_graph_n) cudaGraphExecDestroy(t->fit_graph_n);
  if (t->graph_stream) cudaStreamDestroy(t->graph_stream);
  TrainDesc& d = t->d;
  cudaFree(d.theta); cudaFree(d.img); cudaFree(d.m); cudaFree(d.v); cudaFree(d.grad);
  for (int l = 0; l <= t->L; ++l) {
    cudaFree(d.act[l]);
    cudaFree(d.dz[l]);
    cudaFree(d.mult.m[l]);
  }
  cudaFree(d.partial); cudaFree(t->val_acc);
  cudaFree(t->state); cudaFree(t->desc);
  delete t;
  return SIMBA_OK;
}

extern "C" int simba_trainer_create(simba_model_t* model, const simba_trainer_config_t* cfg,
                                    simba_trainer_t** out) {
  if (!model || !cfg || !out) return set_error(SIMBA_ERR_BAD_CONFIG, "null argument");
  if (cfg->batch_size < 1 || cfg->batch_size > (1 << 20))
    return set_error(SIMBA_ERR_BAD_CONFIG, "batch_size %d out of range", cfg->batch_size);
  if (cfg->lr_schedule && (cfg->steps_per_epoch < 1 || cfg->train_epochs < 1))
    return set_error(SIMBA_ERR_BAD_CONFIG, "lr_schedule needs steps_per_epoch >= 1 and train_epochs >= 1");
  if (!(cfg->beta1 >= 0.0f && cfg->beta1 < 1.0f && cfg->beta2 >= 0.0f && cfg->beta2 < 1.0f) ||
      !(cfg->epsilon > 0.0f) || !(cfg->learning_rate >= 0.0f))
    return set_error(SIMBA_ERR_BAD_CONFIG, "Adam hyper-parameters out of range");
  if (!(cfg->dropout_rate >= 0.0f && cfg->dropout_rate < 1.0f))
    return set_error(SIMBA_ERR_BAD_CONFIG, "dropout_rate %g outside [0, 1)", cfg->dropout_rate);
  if (cfg->precision != SIMBA_PREC_FP32 && cfg->precision != SIMBA_PREC_BF16_TC)
    return set_error(SIMBA_ERR_BAD_CONFIG, "precision %d is neither SIMBA_PREC_FP32 nor SIMBA_PREC_BF16_TC",
                     cfg->precision);
  const simba_model_config_t* mc = model_config(model);
  const bool tc = cfg->precision == SIMBA_PREC_BF16_TC;
  int rc = tc ? train_tc_check(*mc) : SIMBA_OK;
  if (rc) return rc;
  rc = simba_device_check();
  if (rc) return rc;
  auto* t = new simba_trainer();
  t->model = model;
  t->cfg = *cfg;
  t->E = mc->ensemble_size; t->L = mc->n_layers; t->U = mc->units; t->O = mc->obs_dim;
  t->IN = mc->obs_dim + mc->act_dim;
  t->cap_rows = cfg->max_eval_rows > cfg->batch_size ? cfg->max_eval_rows : cfg->batch_size;
  TrainDesc& d = t->d;
  d.L = t->L;
  int64_t off = 0;
  for (int l = 0; l <= t->L; ++l) {
    const int K = l == 0 ? t->IN : t->U;
    const int N = l < t->L ? t->U : 2 * t->O;
    d.layer[l] = TrainLayer{K, N, off};
    off += (int64_t)(K + 1) * N;
  }
  d.pn = off;
  rc = tc ? SIMBA_OK : train_f32_check(d);
  if (rc) { delete t; return rc; }
  const int E = t->E;
  std::vector<float> host((size_t)E * d.pn);
  for (int e = 0; e < E; ++e) {
    rc = pull_member(t, e, host.data() + (size_t)e * d.pn);
    if (rc) { delete t; return rc; }
  }
#define TRY_OR_FREE(expr)                                                                       \
  do {                                                                                          \
    cudaError_t _e = (expr);                                                                    \
    if (_e != cudaSuccess) {                                                                    \
      simba_trainer_destroy(t);                                                                 \
      return set_error(SIMBA_ERR_CUDA, "%s failed: %s", #expr, cudaGetErrorString(_e));         \
    }                                                                                           \
  } while (0)
  const size_t pbytes = (size_t)E * d.pn * sizeof(float);
  TRY_OR_FREE(cudaMalloc(&d.theta, pbytes));
  TRY_OR_FREE(cudaMalloc(&d.m, pbytes));
  TRY_OR_FREE(cudaMalloc(&d.v, pbytes));
  TRY_OR_FREE(cudaMalloc(&d.grad, pbytes));
  TRY_OR_FREE(cudaMemcpy(d.theta, host.data(), pbytes, cudaMemcpyHostToDevice));
  {
    d.img_member_bytes = tc ? train_tc_image_bytes(d) : train_f32_image_bytes(d);
    std::vector<uint8_t> img((size_t)E * d.img_member_bytes, 0);
    for (int e = 0; e < E; ++e)
      (tc ? train_tc_pack : train_f32_pack)(d, host.data() + (size_t)e * d.pn,
                                            img.data() + (size_t)e * d.img_member_bytes);
    TRY_OR_FREE(cudaMalloc(&d.img, img.size()));
    TRY_OR_FREE(cudaMemcpy(d.img, img.data(), img.size(), cudaMemcpyHostToDevice));
  }
  TRY_OR_FREE(cudaMemset(d.m, 0, pbytes));
  TRY_OR_FREE(cudaMemset(d.v, 0, pbytes));
  TRY_OR_FREE(cudaMemset(d.grad, 0, pbytes));
  const size_t R = t->cap_rows;
  d.act_estride = t->cap_rows;
  d.dz_estride = cfg->batch_size;
  for (int l = 0; l <= t->L; ++l) {
    TRY_OR_FREE(cudaMalloc(&d.act[l], (size_t)E * R * d.layer[l].K * sizeof(float)));
    TRY_OR_FREE(cudaMalloc(&d.dz[l], (size_t)E * cfg->batch_size * d.layer[l].N * sizeof(float)));
  }
  d.activation = model_activation(model);
  if (d.activation == SIMBA_ACT_SWISH) {             // the backward multipliers of the hidden layers
    d.mult.estride = cfg->batch_size;
    for (int l = 1; l <= t->L; ++l)
      TRY_OR_FREE(cudaMalloc(&d.mult.m[l], (size_t)E * cfg->batch_size * d.layer[l].K * sizeof(float)));
  }
  d.tiles_cap = (int)((R + 3) / 4);                    // the smallest row tile of either chain kernel
  TRY_OR_FREE(cudaMalloc(&d.partial, (size_t)E * d.tiles_cap * 2 * sizeof(float)));
  TRY_OR_FREE(cudaMalloc(&t->val_acc, (size_t)E * 2 * sizeof(double)));
  TRY_OR_FREE(cudaMalloc(&t->state, sizeof(TrainState)));
  TRY_OR_FREE(cudaMemset(t->state, 0, sizeof(TrainState)));
  TRY_OR_FREE(cudaMalloc(&t->desc, sizeof(FitDesc)));
  TRY_OR_FREE(cudaMemset(t->desc, 0, sizeof(FitDesc)));
#undef TRY_OR_FREE
  d.out_dim = t->O; d.ensemble = E;
  d.dropout_rate = cfg->dropout_rate;
  d.dropout_scale = 1.0f / (1.0f - cfg->dropout_rate);
  d.dropout_seed = cfg->dropout_seed;
  *out = t;
  return SIMBA_OK;
}

static int enqueue_step(simba_trainer_t* t, const float* x, int64_t x_estride, const float* y,
                        int64_t y_estride, int rows_fixed, const FitDesc* desc, float* out_loss,
                        int step_off, cudaStream_t s) {
  TrainDesc d = t->d;
  d.x = x; d.x_estride = x_estride; d.gather = desc ? 1 : 0;
  d.y = y; d.y_estride = y_estride;
  d.train = 1; d.out_loss = out_loss;
  const int grid_rows = desc ? t->cfg.batch_size : rows_fixed;
  const OptParams opt = opt_params(t);
  int row_tiles;
  SIMBA_CUDA_TRY((bf16(t) ? train_tc_chain : train_f32_chain)(d, opt, desc, t->state, grid_rows, rows_fixed,
                                                             step_off, s, row_tiles));
  SIMBA_CUDA_TRY((bf16(t) ? train_tc_update : train_f32_update)(d, opt, desc, t->state, rows_fixed, step_off, s));
  return SIMBA_OK;
}

extern "C" int simba_trainer_step(simba_trainer_t* t, const float* x, const float* y, int32_t rows,
                                  float* out_loss, void* stream) {
  if (!t || !x || !y) return set_error(SIMBA_ERR_BAD_CONFIG, "null argument");
  if (rows < 1 || rows > t->cfg.batch_size)
    return set_error(SIMBA_ERR_SHAPE, "rows %d outside [1, batch_size %d]", rows, t->cfg.batch_size);
  int rc = enqueue_step(t, x, (int64_t)rows * t->IN, y, (int64_t)rows * t->O, rows, nullptr, out_loss,
                        0, (cudaStream_t)stream);
  if (rc) return rc;
  advance_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(t->state, 1);
  SIMBA_CUDA_TRY(cudaGetLastError());
  return SIMBA_OK;
}

extern "C" int simba_trainer_fit(simba_trainer_t* t, const float* inputs, const float* targets,
                                 int64_t n, const int32_t* batch_index, const int32_t* batch_rows,
                                 int32_t steps, float* out_losses, void* stream) {
  if (!t || !inputs || !targets || !batch_index)
    return set_error(SIMBA_ERR_BAD_CONFIG, "null argument");
  if (n < 1 || steps < 0) return set_error(SIMBA_ERR_SHAPE, "n %lld / steps %d", (long long)n, steps);
  cudaStream_t s = (cudaStream_t)stream;
  const int B = t->cfg.batch_size;
  FitDesc d{inputs, targets, batch_index, batch_rows, out_losses, B};
  set_fit_desc_kernel<<<1, 1, 0, s>>>(d, t->desc, t->state);
  SIMBA_CUDA_TRY(cudaGetLastError());
  if (!t->fit_graph) {
    // every pointer the step reads is either owned by the handle or reached through *desc, and the
    // step index lives in device memory, so the captured steps serve every fit() call
    if (!t->graph_stream) SIMBA_CUDA_TRY(cudaStreamCreateWithFlags(&t->graph_stream, cudaStreamNonBlocking));
    for (int which = 0; which < 2; ++which) {
      cudaGraph_t graph = nullptr;
      SIMBA_CUDA_TRY(cudaStreamBeginCapture(t->graph_stream, cudaStreamCaptureModeThreadLocal));
      int rc = SIMBA_OK;
      const int n = which ? kGraphSteps : 1;
      for (int i = 0; i < n && rc == SIMBA_OK; ++i)
        rc = enqueue_step(t, nullptr, 0, nullptr, 0, B, t->desc, nullptr, i, t->graph_stream);
      advance_kernel<<<1, 1, 0, t->graph_stream>>>(t->state, n);
      cudaError_t ce = cudaStreamEndCapture(t->graph_stream, &graph);
      if (rc) { if (graph) cudaGraphDestroy(graph); return rc; }
      SIMBA_CUDA_TRY(ce);
      ce = cudaGraphInstantiate(which ? &t->fit_graph_n : &t->fit_graph, graph, 0);
      cudaGraphDestroy(graph);
      SIMBA_CUDA_TRY(ce);
    }
  }
  int i = 0;
  for (; i + kGraphSteps <= steps; i += kGraphSteps) SIMBA_CUDA_TRY(cudaGraphLaunch(t->fit_graph_n, s));
  for (; i < steps; ++i) SIMBA_CUDA_TRY(cudaGraphLaunch(t->fit_graph, s));
  return SIMBA_OK;
}

extern "C" int simba_trainer_validation(simba_trainer_t* t, const float* x, const float* y,
                                        int64_t rows, float* out_loss, void* stream) {
  if (!t || !x || !y || !out_loss) return set_error(SIMBA_ERR_BAD_CONFIG, "null argument");
  if (rows < 1) return set_error(SIMBA_ERR_SHAPE, "rows %lld", (long long)rows);
  cudaStream_t s = (cudaStream_t)stream;
  for (int64_t r0 = 0; r0 < rows; r0 += t->cap_rows) {
    const int nr = (int)((rows - r0) < t->cap_rows ? (rows - r0) : t->cap_rows);
    TrainDesc d = t->d;                                 // every member reads these rows: estrides 0, no gather
    d.x = x + r0 * t->IN;
    d.y = y + r0 * t->O;
    int tiles;
    SIMBA_CUDA_TRY((bf16(t) ? train_tc_chain : train_f32_chain)(d, opt_params(t), nullptr, t->state, nr, nr, 0, s,
                                                               tiles));
    val_accumulate_kernel<<<1, 32, 0, s>>>(t->d.partial, t->d.tiles_cap, tiles, t->E, t->val_acc,
                                           r0 == 0 ? 1 : 0);
  }
  val_finalize_kernel<<<1, 1, 0, s>>>(t->val_acc, t->E, (double)rows * t->O, out_loss);
  SIMBA_CUDA_TRY(cudaGetLastError());
  return SIMBA_OK;
}

extern "C" int simba_trainer_sync_model(simba_trainer_t* t, void* stream) {
  if (!t) return set_error(SIMBA_ERR_BAD_CONFIG, "null argument");
  std::vector<float> host((size_t)t->E * t->d.pn);
  SIMBA_CUDA_TRY(cudaMemcpyAsync(host.data(), t->d.theta, host.size() * sizeof(float),
                                 cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  SIMBA_CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));
  std::vector<float> kern, bias;
  for (int e = 0; e < t->E; ++e)
    for (int layer = 0; layer < t->L + 2; ++layer) {
      const int K = layer == 0 ? t->IN : t->U, N = layer < t->L ? t->U : t->O;
      kern.resize((size_t)K * N);
      bias.resize(N);
      split_layer(t, host.data() + (size_t)e * t->d.pn, layer, kern.data(), bias.data());
      int rc = simba_model_set_layer(t->model, e, layer, kern.data(), bias.data());
      if (rc) return rc;
    }
  return simba_model_commit(t->model);
}

extern "C" int simba_trainer_get(simba_trainer_t* t, int32_t which, int32_t member, int32_t layer,
                                 float* kernel_out, float* bias_out) {
  if (!t || !kernel_out || !bias_out) return set_error(SIMBA_ERR_BAD_CONFIG, "null argument");
  if (which < 0 || which > 3 || member < 0 || member >= t->E || layer < 0 || layer >= t->L + 2)
    return set_error(SIMBA_ERR_BAD_CONFIG, "which %d / member %d / layer %d out of range", which,
                     member, layer);
  const TrainDesc& d = t->d;
  const float* src = which == 0 ? d.theta : which == 1 ? d.grad : which == 2 ? d.m : d.v;
  std::vector<float> host(d.pn);
  SIMBA_CUDA_TRY(cudaDeviceSynchronize());
  SIMBA_CUDA_TRY(cudaMemcpy(host.data(), src + (size_t)member * d.pn, d.pn * sizeof(float),
                            cudaMemcpyDeviceToHost));
  split_layer(t, host.data(), layer, kernel_out, bias_out);
  return SIMBA_OK;
}

extern "C" int64_t simba_trainer_iterations(simba_trainer_t* t) {
  if (!t) return -1;
  TrainState st;
  if (cudaDeviceSynchronize() != cudaSuccess) return -1;
  if (cudaMemcpy(&st, t->state, sizeof(st), cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
  return st.iterations;
}

// chain + update
extern "C" int simba_trainer_launches_per_step(simba_trainer_t* t) {
  return t ? 2 : 0;
}

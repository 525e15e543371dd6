// C-ABI of libsimba_b200.so (include/simba_b200.h): handles, device weight images (each packed by the
// kernel file that reads it), work lists, the CUDA-graph planning call and the NCCL all-gather.
// Host-side C++; every compute step is a CUDA kernel from rollout_f32.cu / rollout_tc.cu /
// cem_kernels.cu — there is no CPU path.
#include <dlfcn.h>

#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "cem_kernels.cuh"
#include "internal.h"
#include "rollout_params.cuh"

using namespace simba;

// ---------------------------------------------------------------------------------------------
// errors
// ---------------------------------------------------------------------------------------------
static thread_local std::string g_last_error;

int simba::set_error(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_last_error = buf;
  return code;
}

extern "C" const char* simba_last_error(void) { return g_last_error.c_str(); }
extern "C" const char* simba_version(void) { return "simba_b200 0.1 (sm_100a)"; }

extern "C" int simba_device_check(void) {
  int dev = 0;
  SIMBA_CUDA_TRY(cudaGetDevice(&dev));
  cudaDeviceProp prop;
  SIMBA_CUDA_TRY(cudaGetDeviceProperties(&prop, dev));
  if (prop.major != 10)
    return set_error(SIMBA_ERR_ARCH, "device %d is sm_%d%d; this library is built for sm_100a only", dev,
                     prop.major, prop.minor);
  return SIMBA_OK;
}

// ---------------------------------------------------------------------------------------------
// model
// ---------------------------------------------------------------------------------------------
struct simba_model {
  simba_model_config_t cfg{};
  int device = 0;
  std::vector<std::vector<float>> kernels, biases;   // [E * (L + 2)]
  std::vector<char> layer_set;
  std::vector<float> smin, smax;
  int scale_on = 1;
  bool scaler_set = false, committed = false;
  uint64_t generation = 0;     // bumped by every commit; planners re-capture their graph when it changes
  // device images
  float* d_w_f32 = nullptr;
  float* d_bias_f32 = nullptr;
  void* d_w_tc = nullptr;       // bf16 image of the tcgen05 family that runs the model (tc_family), if any
  int64_t w_tc_member_bytes = 0;
  float tc_scale_a[128] = {0}, tc_scale_b[128] = {0};
  float* d_smin = nullptr;
  float* d_sdelta = nullptr;
  int n_chunks = 0, bias_stride = 0, act_rows = 0;
  // scratch for the model-level entry points (tile lists are rebuilt per call size)
  Tile* d_tiles = nullptr;
  int tiles_cap = 0;

  int layer_in(int l) const { return l == 0 ? cfg.obs_dim + cfg.act_dim : cfg.units; }
  int layer_out(int l) const { return l < cfg.n_layers ? cfg.units : cfg.obs_dim; }
};

extern "C" int simba_model_create(const simba_model_config_t* cfg, simba_model_t** out) {
  if (!cfg || !out) return set_error(SIMBA_ERR_BAD_CONFIG, "null argument");
  if (cfg->obs_dim < 1 || cfg->act_dim < 1 || cfg->act_dim > SIMBA_MAX_ACT)
    return set_error(SIMBA_ERR_BAD_CONFIG, "obs_dim %d / act_dim %d out of range (act_dim <= %d)",
                     cfg->obs_dim, cfg->act_dim, SIMBA_MAX_ACT);
  if (cfg->ensemble_size < 1 || cfg->ensemble_size > SIMBA_MAX_MEMBERS)
    return set_error(SIMBA_ERR_BAD_CONFIG, "ensemble_size %d out of range [1, %d]", cfg->ensemble_size,
                     SIMBA_MAX_MEMBERS);
  if (cfg->n_layers < 1 || cfg->n_layers > 16 || cfg->units < 1 || cfg->units > 4096)
    return set_error(SIMBA_ERR_BAD_CONFIG, "n_layers %d / units %d out of range", cfg->n_layers,
                     cfg->units);
  int rc = simba_device_check();
  if (rc != SIMBA_OK) return rc;
  simba_model* m = new simba_model();
  m->cfg = *cfg;
  cudaGetDevice(&m->device);
  const int nl = cfg->ensemble_size * (cfg->n_layers + 2);
  m->kernels.resize(nl);
  m->biases.resize(nl);
  m->layer_set.assign(nl, 0);
  *out = m;
  return SIMBA_OK;
}

static void model_free_device(simba_model* m) {
  cudaFree(m->d_w_f32); cudaFree(m->d_bias_f32); cudaFree(m->d_w_tc);
  cudaFree(m->d_smin); cudaFree(m->d_sdelta);
  m->d_w_f32 = m->d_bias_f32 = m->d_smin = m->d_sdelta = nullptr;
  m->d_w_tc = nullptr;
}

extern "C" int simba_model_destroy(simba_model_t* m) {
  if (!m) return SIMBA_OK;
  cudaSetDevice(m->device);
  model_free_device(m);
  cudaFree(m->d_tiles);
  delete m;
  return SIMBA_OK;
}

extern "C" int simba_model_set_layer(simba_model_t* m, int32_t member, int32_t layer,
                                     const float* kernel, const float* bias) {
  if (!m || !kernel || !bias) return set_error(SIMBA_ERR_BAD_CONFIG, "null argument");
  const int L = m->cfg.n_layers;
  if (member < 0 || member >= m->cfg.ensemble_size || layer < 0 || layer >= L + 2)
    return set_error(SIMBA_ERR_BAD_CONFIG, "member %d / layer %d out of range", member, layer);
  const int K = m->layer_in(layer), N = m->layer_out(layer);
  const int idx = member * (L + 2) + layer;
  m->kernels[idx].assign(kernel, kernel + (size_t)K * N);
  m->biases[idx].assign(bias, bias + N);
  m->layer_set[idx] = 1;
  m->committed = false;
  return SIMBA_OK;
}

extern "C" int simba_model_get_layer(simba_model_t* m, int32_t member, int32_t layer,
                                     float* kernel_out, float* bias_out) {
  if (!m || !kernel_out || !bias_out) return set_error(SIMBA_ERR_BAD_CONFIG, "null argument");
  const int L = m->cfg.n_layers;
  if (member < 0 || member >= m->cfg.ensemble_size || layer < 0 || layer >= L + 2)
    return set_error(SIMBA_ERR_BAD_CONFIG, "member %d / layer %d out of range", member, layer);
  const int idx = member * (L + 2) + layer;
  if (!m->layer_set[idx])
    return set_error(SIMBA_ERR_NOT_READY, "member %d layer %d has no weights", member, layer);
  memcpy(kernel_out, m->kernels[idx].data(), m->kernels[idx].size() * sizeof(float));
  memcpy(bias_out, m->biases[idx].data(), m->biases[idx].size() * sizeof(float));
  return SIMBA_OK;
}

const simba_model_config_t* simba::model_config(const simba_model_t* m) { return &m->cfg; }

extern "C" int simba_model_set_scaler(simba_model_t* m, const float* mn, const float* mx,
                                      int32_t scale_features) {
  if (!m) return set_error(SIMBA_ERR_BAD_CONFIG, "null argument");
  const int IN = m->cfg.obs_dim + m->cfg.act_dim;
  m->scale_on = scale_features ? 1 : 0;
  if (m->scale_on) {
    if (!mn || !mx) return set_error(SIMBA_ERR_BAD_CONFIG, "scale_features set but bounds are null");
    for (int k = 0; k < IN; ++k)
      if (!std::isfinite(mn[k]) || !std::isfinite(mx[k]))
        return set_error(SIMBA_ERR_NONFINITE,
                         "inputs_min/max[%d] is not finite: the reference's scale() would produce NaN "
                         "(transition_model.py:85-87); fit statistics first", k);
    m->smin.assign(mn, mn + IN);
    m->smax.assign(mx, mx + IN);
  } else {
    m->smin.assign(IN, 0.0f);
    m->smax.assign(IN, 1.0f);
  }
  m->scaler_set = true;
  m->committed = false;
  return SIMBA_OK;
}

// first commit: allocate; later commits overwrite in place (the sizes are fixed by the model config)
template <class D, class T>
static cudaError_t upload(D*& dst, const std::vector<T>& host) {
  const size_t bytes = host.size() * sizeof(T);
  const cudaError_t e = dst ? cudaSuccess : cudaMalloc(&dst, bytes);
  return e != cudaSuccess ? e : cudaMemcpy(dst, host.data(), bytes, cudaMemcpyHostToDevice);
}

// scaler: delta = max - min, 1.01 where delta < 1e-5 (transition_model.py:85-86), for the fp32 kernel and
// simba_scale; the bf16 kernels take it as x_scaled = fma(x, a, b) (m->tc_scale_a, m->tc_scale_b)
static std::vector<float> pack_scaler(simba_model* m) {
  const int IN = m->cfg.obs_dim + m->cfg.act_dim;
  std::vector<float> delta(IN), inv(IN);
  for (int k = 0; k < IN; ++k) {
    volatile float d = m->smax[k] - m->smin[k];
    if (d < 1e-5f) d = 1.01f;
    delta[k] = d;
    inv[k] = 1.0f / d;
  }
  for (int k = 0; k < 128; ++k) {
    m->tc_scale_a[k] = k < IN ? (m->scale_on ? inv[k] : 1.0f) : 0.0f;
    m->tc_scale_b[k] = k < IN ? (m->scale_on ? -m->smin[k] * inv[k] : 0.0f) : 0.0f;
  }
  return delta;
}

// The one shape rule of the tcgen05 kernels: the family that runs a model, from its config alone. kTcOneCta stands
// for rollout_tc.cu (whose variant choose_rollout picks), kTcWide and kTcWideObs for rollout_tc_wide.cu <64> and
// <128>, kF32 for none. Each family runs every shape an earlier one rejects, and none other. simba_model_commit packs
// the weight image of this family alone, so the kernel choose_rollout picks always finds its image.
static RolloutKernel tc_family(const simba_model_config_t& c) {
  const int O = c.obs_dim, A = c.act_dim, L = c.n_layers, U = c.units;
  if (rollout_tc_supported(O, A, L, U)) return RolloutKernel::kTcOneCta;
  if (rollout_tc_wide_supported(64, O, A, L, U)) return RolloutKernel::kTcWide;
  if (rollout_tc_wide_supported(128, O, A, L, U)) return RolloutKernel::kTcWideObs;
  return RolloutKernel::kF32;
}

extern "C" int simba_model_commit(simba_model_t* m) {
  if (!m) return set_error(SIMBA_ERR_BAD_CONFIG, "null argument");
  const auto& c = m->cfg;
  const int L = c.n_layers;
  for (size_t i = 0; i < m->layer_set.size(); ++i)
    if (!m->layer_set[i])
      return set_error(SIMBA_ERR_NOT_READY, "member %zu layer %zu has no weights", i / (L + 2),
                       i % (L + 2));
  if (!m->scaler_set) return set_error(SIMBA_ERR_NOT_READY, "scaler not set");
  SIMBA_CUDA_TRY(cudaSetDevice(m->device));
  // Device images are allocated on the first commit and updated IN PLACE afterwards (their sizes
  // are fixed by the immutable model config): planners that captured a CUDA graph keep valid
  // pointers when the weights or the scaler change (e.g. after every model.fit of the agent loop).
  // The copies below are synchronous, so they are ordered after earlier launches on any stream
  // only by the caller's own synchronisation (generate_action is synchronous).
  const ModelWeights mw{c, m->kernels, m->biases};
  std::vector<float> w, b;
  const int rc = rollout_f32_pack(mw, w, b, m->n_chunks, m->bias_stride, m->act_rows);
  if (rc != SIMBA_OK) return rc;
  SIMBA_CUDA_TRY(cudaDeviceSynchronize());
  SIMBA_CUDA_TRY(upload(m->d_w_f32, w));
  SIMBA_CUDA_TRY(upload(m->d_bias_f32, b));
  // the bf16 image of the tcgen05 family that runs this shape, if any
  const RolloutKernel family = tc_family(c);
  std::vector<uint16_t> img;
  m->w_tc_member_bytes = 0;
  if (family == RolloutKernel::kTcOneCta) m->w_tc_member_bytes = rollout_tc_pack(mw, img);
  if (family == RolloutKernel::kTcWide) m->w_tc_member_bytes = rollout_tc_wide_pack(64, mw, img);
  if (family == RolloutKernel::kTcWideObs) m->w_tc_member_bytes = rollout_tc_wide_pack(128, mw, img);
  if (family != RolloutKernel::kF32) SIMBA_CUDA_TRY(upload(m->d_w_tc, img));
  SIMBA_CUDA_TRY(upload(m->d_smin, m->smin));
  SIMBA_CUDA_TRY(upload(m->d_sdelta, pack_scaler(m)));
  m->committed = true;
  ++m->generation;
  return SIMBA_OK;
}

static void fill_model_params(const simba_model* m, RolloutParams& prm) {
  prm.L = m->cfg.n_layers;
  prm.U = m->cfg.units;
  prm.w_f32 = m->d_w_f32;
  prm.bias_f32 = m->d_bias_f32;
  prm.n_chunks = m->n_chunks;
  prm.bias_stride = m->bias_stride;
  prm.act_rows = m->act_rows;
  prm.w_tc = m->d_w_tc;
  prm.w_tc_member_bytes = m->w_tc_member_bytes;
  memcpy(prm.tc_scale_a, m->tc_scale_a, sizeof(prm.tc_scale_a));
  memcpy(prm.tc_scale_b, m->tc_scale_b, sizeof(prm.tc_scale_b));
  prm.smin = m->d_smin;
  prm.sdelta = m->d_sdelta;
  prm.scale_on = m->scale_on;
}

// ---------------------------------------------------------------------------------------------
// row geometry + tile lists
// ---------------------------------------------------------------------------------------------
static int build_geom(int S, int P, int N, int world, int rank, int H, int O, int A, int E,
                      int member_map, RowGeom& g) {
  if (N % world) return set_error(SIMBA_ERR_SHAPE, "n_samples %d not divisible by world_size %d", N, world);
  memset(&g, 0, sizeof(g));
  g.S = S; g.P = P; g.N = N; g.N_local = N / world; g.cand0 = rank * g.N_local;
  g.H = H; g.O = O; g.A = A; g.E = E;
  const long B = (long)P * N;
  if (member_map == SIMBA_MAP_SPLIT) {
    if (B % E)
      return set_error(SIMBA_ERR_SHAPE,
                       "tf.split needs particles*n_samples (%ld) divisible by ensemble_size (%d) "
                       "(mlp_ensemble.py:123); use member_map=PARTICLE", B, E);
    if (world > 1 && P % E)
      return set_error(SIMBA_ERR_SHAPE,
                       "member_map=SPLIT with world_size > 1 needs ensemble_size (%d) to divide "
                       "particles (%d)", E, P);
    if (world == 1) {
      for (int e = 0; e < E; ++e) { g.lr_lo[e] = (int)(e * (B / E)); g.rows_per_state[e] = (int)(B / E); }
      return SIMBA_OK;
    }
  }
  for (int e = 0; e < E; ++e) {
    const int p_lo = (int)(((long)e * P + E - 1) / E), p_hi = (int)(((long)(e + 1) * P + E - 1) / E);
    g.lr_lo[e] = p_lo * g.N_local;
    g.rows_per_state[e] = (p_hi - p_lo) * g.N_local;
  }
  return SIMBA_OK;
}

// `group` > 1 pads every member's tile run with empty tiles to a multiple of `group`, so that a CTA
// that takes `group` consecutive tiles never mixes members (its weights are one member's).
static void build_tiles(const RowGeom& g, int tile_rows, std::vector<Tile>& tiles, int group = 1) {
  tiles.clear();
  for (int e = 0; e < g.E; ++e) {
    const long total = (long)g.S * g.rows_per_state[e];
    for (long k0 = 0; k0 < total; k0 += tile_rows) {
      Tile t;
      t.member = e; t.k0 = (int)k0; t.count = (int)std::min<long>(tile_rows, total - k0); t.pad = 0;
      tiles.push_back(t);
    }
    while (tiles.size() % group) {
      Tile t;
      t.member = e; t.k0 = 0; t.count = 0; t.pad = 0;
      tiles.push_back(t);
    }
  }
}

// Two tiles per work item, persistent CTAs (one per SM): the items of the last, partly filled round are split into
// single-tile items when that still fits in one round. A lone tile takes ~0.6 of a pair's time (no ping-pong
// partner, but nothing to share the SM with either), so the launch ends ~0.4 item earlier — 0.5 % at 82 rounds.
static void split_tail_items(std::vector<Tile>& tiles, int sms) {
  const size_t n_items = tiles.size() / 2;
  if (sms <= 0 || n_items <= (size_t)sms) return;
  const size_t rounds = (n_items + sms - 1) / sms;
  const size_t last = n_items - (size_t)sms * (rounds - 1);
  if (2 * last > (size_t)sms) return;
  std::vector<Tile> tail(tiles.end() - 2 * last, tiles.end());
  tiles.resize(tiles.size() - 2 * last);
  for (size_t i = 0; i < tail.size(); i += 2) {
    for (int h = 0; h < 2; ++h) {
      if (tail[i + h].count == 0) continue;
      Tile empty = tail[i + h];
      empty.k0 = 0; empty.count = 0;
      tiles.push_back(tail[i + h]);
      tiles.push_back(empty);
    }
  }
}

// The rollout kernel and the tile list it walks, for a planner (nc constraints) or a trajectory call (traj, nc = 0),
// from the precision, the row geometry and the SM count. fp32 runs rollout_f32_kernel on 32-row tiles; bf16 runs the
// tcgen05 family tc_family names on 128-row tiles, or fails. The diagnostic switches SIMBA_B200_NO_TAIL_SPLIT and
// SIMBA_B200_NO_PAIR are read here and nowhere else.
static int choose_rollout(const simba_model_config_t& mc, int precision, const RowGeom& g, int nc, bool traj, int sms,
                          RolloutKernel& kernel, std::vector<Tile>& tiles) {
  const int L = mc.n_layers, U = mc.units;
  kernel = RolloutKernel::kF32;
  build_tiles(g, precision == SIMBA_PREC_FP32 ? kF32TileRows : kTcTileRows, tiles);
  if (precision == SIMBA_PREC_FP32) return SIMBA_OK;
  kernel = tc_family(mc);
  if (kernel == RolloutKernel::kTcOneCta) {
    if ((int)tiles.size() > sms && rollout_tc_two_tiles_fit(L, nc)) {
      // more tiles than SMs: two tiles per CTA so one tile's MMAs overlap the other's epilogue
      kernel = RolloutKernel::kTcTwoTile;
      build_tiles(g, kTcTileRows, tiles, 2);
      if (getenv("SIMBA_B200_NO_TAIL_SPLIT") == nullptr) split_tail_items(tiles, sms);
    } else if (!traj && (int)tiles.size() * 2 <= sms && rollout_tc_pair_fits(L, nc) &&
               getenv("SIMBA_B200_NO_PAIR") == nullptr) {
      // few tiles (a single plan): two SMs per tile, the head pass split between them
      kernel = RolloutKernel::kTcPair;
    }
    return SIMBA_OK;
  }
  if (kernel == RolloutKernel::kTcWide && rollout_tc_wide_fits(64, L, U, nc)) return SIMBA_OK;
  if (kernel == RolloutKernel::kTcWideObs && rollout_tc_wide_fits(128, L, U, nc)) return SIMBA_OK;
  return set_error(SIMBA_ERR_UNSUPPORTED,
                   "no bf16 tcgen05 kernel covers obs_dim %d, act_dim %d, %d x %d units with %d constraints: they "
                   "cover units <= 128 (obs_dim <= 60, obs_dim+act_dim <= 64, <= 5 layers), 128 < units <= ~416 (less "
                   "with several constrained lidars; obs_dim+act_dim <= 62) and, for other shapes, obs_dim+act_dim <= "
                   "126 with obs_dim <= 124, act_dim <= 4, units <= 384 and <= 6 layers; use fp32 for this shape",
                   mc.obs_dim, mc.act_dim, L, U, nc);
}

// the work items of a launch: the two-tile kernel's item i is tiles [2i, 2i + 1]
static int32_t n_work_items(RolloutKernel kernel, const std::vector<Tile>& tiles) {
  return (int32_t)tiles.size() / (kernel == RolloutKernel::kTcTwoTile ? 2 : 1);
}

cudaError_t simba::launch_rollout(const RolloutParams& prm, cudaStream_t stream) {
  if (prm.n_tiles == 0) return cudaSuccess;
  switch (prm.kernel) {
    case RolloutKernel::kF32: return launch_rollout_f32(prm, stream);
    case RolloutKernel::kTcWide:
    case RolloutKernel::kTcWideObs: return launch_rollout_tc_wide(prm, stream);
    default: return launch_rollout_tc(prm, stream);
  }
}

// ---------------------------------------------------------------------------------------------
// NCCL, loaded lazily so that a process that already holds torch's bundled libnccl reuses it
// ---------------------------------------------------------------------------------------------
namespace {
struct NcclUniqueId { char internal[128]; };
typedef void* NcclComm;
typedef int (*nccl_get_unique_id_t)(NcclUniqueId*);
typedef int (*nccl_comm_init_rank_t)(NcclComm*, int, NcclUniqueId, int);
typedef int (*nccl_all_gather_t)(const void*, void*, size_t, int, NcclComm, cudaStream_t);
typedef int (*nccl_comm_destroy_t)(NcclComm);
typedef const char* (*nccl_get_error_string_t)(int);
struct NcclApi {
  void* lib = nullptr;
  nccl_get_unique_id_t get_unique_id = nullptr;
  nccl_comm_init_rank_t comm_init_rank = nullptr;
  nccl_all_gather_t all_gather = nullptr;
  nccl_comm_destroy_t comm_destroy = nullptr;
  nccl_get_error_string_t get_error_string = nullptr;
} g_nccl;
constexpr int kNcclFloat = 7;

int nccl_load() {
  if (g_nccl.lib) return SIMBA_OK;
  const char* names[] = {"libnccl.so.2", "libnccl.so"};
  for (const char* n : names) {
    g_nccl.lib = dlopen(n, RTLD_NOW | RTLD_NOLOAD);
    if (g_nccl.lib) break;
  }
  for (const char* n : names) {
    if (g_nccl.lib) break;
    g_nccl.lib = dlopen(n, RTLD_NOW);
  }
  if (!g_nccl.lib) return set_error(SIMBA_ERR_NCCL, "cannot load libnccl.so.2: %s", dlerror());
  g_nccl.get_unique_id = (nccl_get_unique_id_t)dlsym(g_nccl.lib, "ncclGetUniqueId");
  g_nccl.comm_init_rank = (nccl_comm_init_rank_t)dlsym(g_nccl.lib, "ncclCommInitRank");
  g_nccl.all_gather = (nccl_all_gather_t)dlsym(g_nccl.lib, "ncclAllGather");
  g_nccl.comm_destroy = (nccl_comm_destroy_t)dlsym(g_nccl.lib, "ncclCommDestroy");
  g_nccl.get_error_string = (nccl_get_error_string_t)dlsym(g_nccl.lib, "ncclGetErrorString");
  if (!g_nccl.get_unique_id || !g_nccl.comm_init_rank || !g_nccl.all_gather || !g_nccl.comm_destroy)
    return set_error(SIMBA_ERR_NCCL, "libnccl is missing a required symbol");
  return SIMBA_OK;
}
}  // namespace

#define NCCL_TRY(expr)                                                                     \
  do {                                                                                     \
    int _r = (expr);                                                                       \
    if (_r != 0)                                                                           \
      return set_error(SIMBA_ERR_NCCL, "%s failed: %s", #expr,                             \
                       g_nccl.get_error_string ? g_nccl.get_error_string(_r) : "nccl error");\
  } while (0)

// ---------------------------------------------------------------------------------------------
// planner
// ---------------------------------------------------------------------------------------------
struct simba_planner {
  simba_model* model = nullptr;
  simba_planner_config_t cfg{};
  int device = 0;
  RowGeom geom{};
  RolloutKernel kernel = RolloutKernel::kF32;
  std::vector<Tile> tiles;     // the two-tile kernel's work item i is tiles [2i, 2i + 1]
  Tile* d_tiles = nullptr;
  int n_sms = 0;

  bool use_pdl = false;        // programmatic dependent launch between rollout and fused update kernels
  bool fused_update = false;   // one rank, N <= 1024: reduce+select+refit(+next sample | finalize) in one kernel
  int c_max = -1;
  // workspace
  float *actions = nullptr, *row_ret = nullptr, *row_csum = nullptr, *pairs_local = nullptr,
        *pairs_all = nullptr, *mu = nullptr, *sigma = nullptr, *best_action = nullptr,
        *best_score = nullptr, *scores = nullptr;
  uint64_t* row_cmask = nullptr;
  unsigned long long* key_scratch = nullptr;
  int32_t *elite = nullptr, *active = nullptr, *iters = nullptr;
  // planning-call staging
  float *d_states = nullptr, *d_out_action = nullptr, *d_out_score = nullptr;
  int32_t* d_out_iters = nullptr;
  uint64_t* d_seed = nullptr;
  uint64_t* h_seed_ring = nullptr;     // pinned
  int seed_slot = 0;
  float* h_out = nullptr;              // pinned: [S*A action][S score][S iters(int)]
  uint8_t* h_in = nullptr;             // pinned: [seed (16 bytes)][S*O states] of a plan_host() call
  uint8_t* d_in = nullptr;             // device: the same block; d_seed and d_states point into it
  float* d_out = nullptr;              // device: [S*A action][S score][S iters(int)]; the d_out_* pointers point into it
  const float *ext_z_actions = nullptr, *ext_eps = nullptr, *ext_z_final = nullptr;
  cudaStream_t own_stream = nullptr;
  cudaEvent_t plan_done = nullptr;   // recorded after every plan: the next plan (any stream) waits on it
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t graph_exec = nullptr;
  int launches_per_plan = 0;
  uint64_t graph_generation = 0;   // model generation the graph was captured against
  NcclComm comm = nullptr;
};

static int beta_count_threshold(int P, float thr, float mu, float sigma) {
  // fp32 restatement of safe_cem_mpc.py:116-120, evaluated for every possible integer count
  volatile float one_minus = 1.0f - mu;
  volatile float s2 = sigma * sigma;
  volatile float q = one_minus / s2;
  volatile float inv_mu = 1.0f / mu;
  volatile float d = q - inv_mu;
  volatile float mu2 = mu * mu;
  volatile float alpha = d * mu2;
  volatile float f = inv_mu - 1.0f;
  volatile float beta = alpha * f;
  volatile float ab = alpha + beta;
  volatile float denom = ab + (float)P;
  int c_max = -1;
  for (int c = 0; c <= P; ++c) {
    volatile float num = alpha + (float)c;
    volatile float post = num / denom;
    if (post <= thr) c_max = c;
  }
  return c_max;
}

static int validate_scorer(const simba_scorer_t& s, int O) {
  if (s.goal_dist_index >= O) return set_error(SIMBA_ERR_BAD_CONFIG, "goal_dist_index out of range");
  if (s.goal_dist_index < 0 &&
      (s.goal_begin < 0 || s.goal_end > O || s.goal_begin >= s.goal_end))
    return set_error(SIMBA_ERR_BAD_CONFIG, "goal lidar slice [%d, %d) invalid for obs_dim %d",
                     s.goal_begin, s.goal_end, O);
  if (s.n_constraints < 0 || s.n_constraints > SIMBA_MAX_CONSTRAINTS)
    return set_error(SIMBA_ERR_BAD_CONFIG, "n_constraints %d out of range", s.n_constraints);
  for (int j = 0; j < s.n_constraints; ++j)
    if (s.con_begin[j] < 0 || s.con_end[j] > O || s.con_begin[j] >= s.con_end[j])
      return set_error(SIMBA_ERR_BAD_CONFIG, "constraint slice %d invalid", j);
  if (!s.constrain_indicator && s.n_constraints > 1)
    return set_error(SIMBA_ERR_UNSUPPORTED,
                     "constrain_indicator=False with more than one constrained object class is not "
                     "offered on the fused path (per-step cost must fit one bit)");
  return SIMBA_OK;
}

static void planner_free(simba_planner* p) {
  if (p->graph_exec) cudaGraphExecDestroy(p->graph_exec);
  if (p->graph) cudaGraphDestroy(p->graph);
  if (p->comm && g_nccl.comm_destroy) g_nccl.comm_destroy(p->comm);
  if (p->own_stream) cudaStreamDestroy(p->own_stream);
  if (p->plan_done) cudaEventDestroy(p->plan_done);
  cudaFree(p->d_tiles); cudaFree(p->actions); cudaFree(p->row_ret); cudaFree(p->row_csum);
  cudaFree(p->pairs_local); cudaFree(p->pairs_all); cudaFree(p->mu); cudaFree(p->sigma);
  cudaFree(p->best_action); cudaFree(p->best_score); cudaFree(p->scores); cudaFree(p->row_cmask); cudaFree(p->key_scratch);
  cudaFree(p->elite); cudaFree(p->active); cudaFree(p->iters);
  cudaFree(p->d_in); cudaFree(p->d_out);           // d_seed / d_states and d_out_* are interior pointers
  cudaFreeHost(p->h_seed_ring); cudaFreeHost(p->h_out); cudaFreeHost(p->h_in);
}

extern "C" int simba_planner_destroy(simba_planner_t* p) {
  if (!p) return SIMBA_OK;
  cudaSetDevice(p->device);
  planner_free(p);
  delete p;
  return SIMBA_OK;
}

extern "C" int simba_planner_create(simba_model_t* model, const simba_planner_config_t* cfg,
                                    simba_planner_t** out) {
  if (!model || !cfg || !out) return set_error(SIMBA_ERR_BAD_CONFIG, "null argument");
  if (!model->committed) return set_error(SIMBA_ERR_NOT_READY, "model not committed");
  const auto& mc = model->cfg;
  if (cfg->horizon < 1 || cfg->horizon > SIMBA_MAX_HORIZON)
    return set_error(SIMBA_ERR_BAD_CONFIG, "horizon %d out of range [1, %d]", cfg->horizon,
                     SIMBA_MAX_HORIZON);
  if (cfg->horizon * mc.act_dim > 1024)
    return set_error(SIMBA_ERR_BAD_CONFIG, "horizon*act_dim %d > 1024", cfg->horizon * mc.act_dim);
  if (cfg->iterations < 1 || cfg->iterations > 65535)
    return set_error(SIMBA_ERR_BAD_CONFIG, "iterations %d out of range", cfg->iterations);
  if (cfg->n_samples < 1 || cfg->n_elite < 1 || cfg->n_elite > cfg->n_samples)
    return set_error(SIMBA_ERR_BAD_CONFIG, "need 1 <= n_elite (%d) <= n_samples (%d)", cfg->n_elite,
                     cfg->n_samples);
  if (cfg->particles < 1 || cfg->particles > 255)
    return set_error(SIMBA_ERR_BAD_CONFIG, "particles %d out of range [1, 255]", cfg->particles);
  if (cfg->n_states < 1) return set_error(SIMBA_ERR_BAD_CONFIG, "n_states %d < 1", cfg->n_states);
  if (cfg->world_size < 1 || cfg->rank < 0 || cfg->rank >= cfg->world_size)
    return set_error(SIMBA_ERR_BAD_CONFIG, "rank %d / world_size %d invalid", cfg->rank, cfg->world_size);
  if (cfg->objective < 0 || cfg->objective > 3)
    return set_error(SIMBA_ERR_BAD_CONFIG, "objective %d unknown", cfg->objective);
  if (cfg->precision != SIMBA_PREC_FP32 && cfg->precision != SIMBA_PREC_BF16_TC)
    return set_error(SIMBA_ERR_BAD_CONFIG, "precision %d unknown", cfg->precision);
  int rc = validate_scorer(cfg->scorer, mc.obs_dim);
  if (rc != SIMBA_OK) return rc;
  if ((long)cfg->n_states * cfg->particles * cfg->n_samples > 0x7fffffffL / 2)
    return set_error(SIMBA_ERR_BAD_CONFIG, "n_states*particles*n_samples too large");

  simba_planner* p = new simba_planner();
  p->model = model;
  p->cfg = *cfg;
  p->device = model->device;
  cudaError_t ce = cudaSetDevice(p->device);
  if (ce != cudaSuccess) { delete p; return set_error(SIMBA_ERR_CUDA, "cudaSetDevice: %s", cudaGetErrorString(ce)); }
  rc = build_geom(cfg->n_states, cfg->particles, cfg->n_samples, cfg->world_size, cfg->rank,
                  cfg->horizon, mc.obs_dim, mc.act_dim, mc.ensemble_size, cfg->member_map, p->geom);
  if (rc != SIMBA_OK) { delete p; return rc; }
  ce = cudaDeviceGetAttribute(&p->n_sms, cudaDevAttrMultiProcessorCount, p->device);
  if (ce != cudaSuccess) { delete p; return set_error(SIMBA_ERR_CUDA, "SM count: %s", cudaGetErrorString(ce)); }
  rc = choose_rollout(mc, cfg->precision, p->geom, cfg->scorer.n_constraints, false, p->n_sms, p->kernel, p->tiles);
  if (rc != SIMBA_OK) { delete p; return rc; }

  p->fused_update = cfg->world_size == 1 && cfg->n_samples <= 1024 && getenv("SIMBA_B200_NO_FUSE") == nullptr;
  p->use_pdl = p->fused_update && cfg->precision == SIMBA_PREC_BF16_TC && getenv("SIMBA_B200_NO_PDL") == nullptr;
  p->c_max = beta_count_threshold(cfg->particles, cfg->posterior_mean_threshold, cfg->prior_mu,
                                  cfg->prior_sigma);

  const size_t S = cfg->n_states, N = cfg->n_samples, Nl = p->geom.N_local, P = cfg->particles;
  const size_t HA = (size_t)cfg->horizon * mc.act_dim, A = mc.act_dim, O = mc.obs_dim;
  const size_t W = cfg->world_size;
#define PL_ALLOC(ptr, bytes)                                                              \
  do {                                                                                    \
    cudaError_t _e = cudaMalloc((void**)&(ptr), (bytes));                                 \
    if (_e != cudaSuccess) {                                                              \
      planner_free(p); delete p;                                                          \
      return set_error(SIMBA_ERR_CUDA, "cudaMalloc(%zu) failed: %s", (size_t)(bytes),     \
                       cudaGetErrorString(_e));                                           \
    }                                                                                     \
  } while (0)
  PL_ALLOC(p->d_tiles, std::max<size_t>(1, p->tiles.size()) * sizeof(Tile));
  PL_ALLOC(p->actions, S * N * HA * 4);
  PL_ALLOC(p->row_ret, S * P * Nl * 4);
  PL_ALLOC(p->row_csum, S * P * Nl * 4);
  PL_ALLOC(p->row_cmask, S * P * Nl * 8);
  PL_ALLOC(p->pairs_local, S * Nl * 8);
  PL_ALLOC(p->pairs_all, W * S * Nl * 8);
  PL_ALLOC(p->mu, S * HA * 4);
  PL_ALLOC(p->sigma, S * HA * 4);
  PL_ALLOC(p->best_action, S * A * 4);
  PL_ALLOC(p->best_score, S * 4);
  PL_ALLOC(p->scores, S * N * 4);
  PL_ALLOC(p->key_scratch, S * N * 8);
  PL_ALLOC(p->elite, S * (size_t)cfg->n_elite * 4);
  PL_ALLOC(p->active, S * 4);
  PL_ALLOC(p->iters, S * 4);
  // one input block (seed + states) and one output block (action, score, iterations): a host-buffer plan is one
  // copy in and one copy out around the graph
  PL_ALLOC(p->d_in, 16 + S * O * 4);
  p->d_seed = reinterpret_cast<uint64_t*>(p->d_in);
  p->d_states = reinterpret_cast<float*>(p->d_in + 16);
  PL_ALLOC(p->d_out, S * (A + 2) * 4);
  p->d_out_action = p->d_out;
  p->d_out_score = p->d_out + S * A;
  p->d_out_iters = reinterpret_cast<int32_t*>(p->d_out + S * A + S);
#undef PL_ALLOC
  if (cudaMemcpy(p->d_tiles, p->tiles.data(), p->tiles.size() * sizeof(Tile),
                 cudaMemcpyHostToDevice) != cudaSuccess ||
      cudaMallocHost((void**)&p->h_seed_ring, 64 * sizeof(uint64_t)) != cudaSuccess ||
      cudaMallocHost((void**)&p->h_out, S * (A + 2) * 4) != cudaSuccess ||
      cudaMallocHost((void**)&p->h_in, 16 + S * O * 4) != cudaSuccess ||
      cudaStreamCreateWithFlags(&p->own_stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreateWithFlags(&p->plan_done, cudaEventDisableTiming) != cudaSuccess) {
    planner_free(p); delete p;
    return set_error(SIMBA_ERR_CUDA, "planner staging allocation failed: %s",
                     cudaGetErrorString(cudaGetLastError()));
  }
  *out = p;
  return SIMBA_OK;
}

extern "C" int simba_planner_set_external_draws(simba_planner_t* p, const float* z_actions,
                                                const float* eps, const float* z_final) {
  if (!p) return set_error(SIMBA_ERR_BAD_CONFIG, "null argument");
  p->ext_z_actions = z_actions; p->ext_eps = eps; p->ext_z_final = z_final;
  if (p->graph_exec) { cudaGraphExecDestroy(p->graph_exec); p->graph_exec = nullptr; }
  if (p->graph) { cudaGraphDestroy(p->graph); p->graph = nullptr; }
  return SIMBA_OK;
}

extern "C" int simba_planner_count_threshold(simba_planner_t* p, int32_t* out) {
  if (!p || !out) return set_error(SIMBA_ERR_BAD_CONFIG, "null argument");
  *out = p->c_max;
  return SIMBA_OK;
}

extern "C" int simba_planner_rollout_kernel(simba_planner_t* p, int32_t* kernel, int32_t* work_items) {
  if (!p || !kernel || !work_items) return set_error(SIMBA_ERR_BAD_CONFIG, "null argument");
  *kernel = (int32_t)p->kernel;
  *work_items = n_work_items(p->kernel, p->tiles);
  return SIMBA_OK;
}

extern "C" int simba_planner_buffer(simba_planner_t* p, int32_t which, void** out_ptr,
                                    uint64_t* out_bytes) {
  if (!p || !out_ptr || !out_bytes) return set_error(SIMBA_ERR_BAD_CONFIG, "null argument");
  const auto& c = p->cfg; const auto& mc = p->model->cfg;
  const uint64_t S = c.n_states, N = c.n_samples, Nl = p->geom.N_local, P = c.particles;
  const uint64_t HA = (uint64_t)c.horizon * mc.act_dim, A = mc.act_dim, W = c.world_size;
  switch (which) {
    case SIMBA_BUF_ACTIONS: *out_ptr = p->actions; *out_bytes = S * N * HA * 4; break;
    case SIMBA_BUF_ROW_RETURN: *out_ptr = p->row_ret; *out_bytes = S * P * Nl * 4; break;
    case SIMBA_BUF_ROW_COSTMASK: *out_ptr = p->row_cmask; *out_bytes = S * P * Nl * 8; break;
    case SIMBA_BUF_ROW_COSTSUM: *out_ptr = p->row_csum; *out_bytes = S * P * Nl * 4; break;
    case SIMBA_BUF_PAIRS_LOCAL: *out_ptr = p->pairs_local; *out_bytes = S * Nl * 8; break;
    case SIMBA_BUF_PAIRS_ALL: *out_ptr = p->pairs_all; *out_bytes = W * S * Nl * 8; break;
    case SIMBA_BUF_ELITE: *out_ptr = p->elite; *out_bytes = S * (uint64_t)c.n_elite * 4; break;
    case SIMBA_BUF_MU: *out_ptr = p->mu; *out_bytes = S * HA * 4; break;
    case SIMBA_BUF_SIGMA: *out_ptr = p->sigma; *out_bytes = S * HA * 4; break;
    case SIMBA_BUF_BEST_ACTION: *out_ptr = p->best_action; *out_bytes = S * A * 4; break;
    case SIMBA_BUF_BEST_SCORE: *out_ptr = p->best_score; *out_bytes = S * 4; break;
    case SIMBA_BUF_ACTIVE: *out_ptr = p->active; *out_bytes = S * 4; break;
    case SIMBA_BUF_SCORES: *out_ptr = p->scores; *out_bytes = S * N * 4; break;
    default: return set_error(SIMBA_ERR_BAD_CONFIG, "unknown buffer %d", which);
  }
  return SIMBA_OK;
}

extern "C" int simba_planner_copy_buffer(simba_planner_t* p, int32_t which, void* dst, void* stream) {
  void* src = nullptr;
  uint64_t bytes = 0;
  int rc = simba_planner_buffer(p, which, &src, &bytes);
  if (rc != SIMBA_OK) return rc;
  if (!dst) return set_error(SIMBA_ERR_BAD_CONFIG, "null argument");
  SIMBA_CUDA_TRY(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return SIMBA_OK;
}

// ---- per-kernel entry points -------------------------------------------------------------------
static SampleParams make_sample_params(simba_planner_t* p, const float* mu, const float* sigma,
                                       const float* z, uint64_t seed, const uint64_t* seed_ptr,
                                       int32_t iteration, const int32_t* active, float* out) {
  SampleParams sp{};
  sp.seed_ptr = seed_ptr;
  sp.S = p->cfg.n_states; sp.N = p->cfg.n_samples; sp.H = p->cfg.horizon; sp.A = p->model->cfg.act_dim;
  sp.mu = mu; sp.sigma = sigma; sp.z = z; sp.seed = seed; sp.iteration = iteration;
  sp.active = active; sp.out = out;
  memcpy(sp.lb, p->cfg.act_low, sizeof(sp.lb));
  memcpy(sp.ub, p->cfg.act_high, sizeof(sp.ub));
  return sp;
}

static int do_sample_actions(simba_planner_t* p, const float* mu, const float* sigma,
                             const float* z, uint64_t seed, const uint64_t* seed_ptr,
                             int32_t iteration, const int32_t* active, float* out, void* stream) {
  if (!p || !mu || !sigma || !out) return set_error(SIMBA_ERR_BAD_CONFIG, "null argument");
  const SampleParams sp = make_sample_params(p, mu, sigma, z, seed, seed_ptr, iteration, active, out);
  SIMBA_CUDA_TRY(launch_sample_actions(sp, (cudaStream_t)stream));
  return SIMBA_OK;
}

extern "C" int simba_sample_actions(simba_planner_t* p, const float* mu, const float* sigma,
                                    const float* z, uint64_t seed, int32_t iteration,
                                    const int32_t* active, float* out, void* stream) {
  return do_sample_actions(p, mu, sigma, z, seed, nullptr, iteration, active, out, stream);
}

static int do_rollout_score(simba_planner_t* p, const float* states, const float* actions,
                            const float* eps, uint64_t seed, const uint64_t* seed_ptr,
                            int32_t iteration, const int32_t* active, float* row_return,
                            uint64_t* row_costmask, float* row_costsum, void* stream, bool pdl = false) {
  if (!p || !states || !actions || !row_return || !row_costmask || !row_costsum)
    return set_error(SIMBA_ERR_BAD_CONFIG, "null argument");
  RolloutParams prm{};
  prm.seed_ptr = seed_ptr;
  prm.g = p->geom;
  prm.scorer = p->cfg.scorer;
  prm.tiles = p->d_tiles;
  prm.n_tiles = (int)p->tiles.size();
  fill_model_params(p->model, prm);
  prm.states = states; prm.state_stride = p->geom.O; prm.state_per_row = 0;
  prm.actions = actions; prm.action_stride = (int64_t)p->geom.H * p->geom.A;
  prm.eps = eps; prm.seed = seed; prm.iteration = iteration;
  prm.sampling_propagation = p->cfg.sampling_propagation;
  prm.objective = p->cfg.objective;
  prm.active = active;
  prm.row_return = row_return; prm.row_costmask = row_costmask; prm.row_costsum = row_costsum;
  prm.kernel = p->kernel;
  prm.n_sms = p->n_sms;
  prm.pdl = pdl ? 1 : 0;
#ifdef SIMBA_TC_TIMELINE
  // debug builds only (tools/tc_timeline.py): a scratch buffer for the kernels' clock64 stamps
  if (const char* tlp = getenv("SIMBA_TC_TIMELINE_PTR"))
    prm.timeline = reinterpret_cast<long long*>(strtoull(tlp, nullptr, 10));
#endif
  SIMBA_CUDA_TRY(launch_rollout(prm, (cudaStream_t)stream));
  return SIMBA_OK;
}

extern "C" int simba_rollout_score(simba_planner_t* p, const float* states, const float* actions,
                                   const float* eps, uint64_t seed, int32_t iteration,
                                   const int32_t* active, float* row_return, uint64_t* row_costmask,
                                   float* row_costsum, void* stream) {
  return do_rollout_score(p, states, actions, eps, seed, nullptr, iteration, active, row_return,
                          row_costmask, row_costsum, stream);
}

static ReduceParams make_reduce_params(simba_planner_t* p, const float* row_return,
                                       const uint64_t* row_costmask, const float* row_costsum,
                                       const int32_t* active, float* out_pairs_local) {
  ReduceParams rp{};
  rp.S = p->cfg.n_states; rp.P = p->cfg.particles; rp.N_local = p->geom.N_local;
  rp.H = p->cfg.horizon; rp.objective = p->cfg.objective;
  rp.row_return = row_return; rp.row_costmask = row_costmask; rp.row_costsum = row_costsum;
  rp.active = active; rp.out_pairs = out_pairs_local;
  return rp;
}

static SelectParams make_select_params(simba_planner_t* p, const float* pairs_all, const float* actions,
                                       const int32_t* active, int32_t* out_elite, float* out_scores,
                                       float* best_action, float* best_score) {
  SelectParams sp{};
  sp.S = p->cfg.n_states; sp.N = p->cfg.n_samples; sp.N_local = p->geom.N_local;
  sp.K = p->cfg.n_elite; sp.H = p->cfg.horizon; sp.A = p->model->cfg.act_dim;
  sp.objective = p->cfg.objective; sp.c_max = (float)p->c_max;
  sp.key_scratch = p->key_scratch;
  sp.pairs_all = pairs_all; sp.actions = actions; sp.active = active; sp.out_elite = out_elite;
  sp.out_scores = out_scores; sp.best_action = best_action; sp.best_score = best_score;
  return sp;
}

static RefitParams make_refit_params(simba_planner_t* p, const float* actions, const int32_t* elite,
                                     float* mu, float* sigma, int32_t* active, int32_t* iterations_run) {
  RefitParams rp{};
  rp.S = p->cfg.n_states; rp.N = p->cfg.n_samples; rp.K = p->cfg.n_elite; rp.H = p->cfg.horizon;
  rp.A = p->model->cfg.act_dim;
  rp.smoothing = p->cfg.smoothing;
  rp.one_minus_smoothing = (float)(1.0 - (double)p->cfg.smoothing);
  rp.stddev_threshold = p->cfg.stddev_threshold;
  rp.actions = const_cast<float*>(actions); rp.elite = elite; rp.mu = mu; rp.sigma = sigma; rp.active = active;
  rp.iterations_run = iterations_run;
  return rp;
}

static FinalizeParams make_finalize_params(simba_planner_t* p, const float* best_action, const float* z,
                                           uint64_t seed, const uint64_t* seed_ptr, float* out_action) {
  FinalizeParams fp{};
  fp.seed_ptr = seed_ptr;
  fp.S = p->cfg.n_states; fp.A = p->model->cfg.act_dim; fp.noise_stddev = p->cfg.noise_stddev;
  fp.best = best_action; fp.z = z; fp.seed = seed; fp.out = out_action;
  return fp;
}

extern "C" int simba_score_reduce(simba_planner_t* p, const float* row_return,
                                  const uint64_t* row_costmask, const float* row_costsum,
                                  const int32_t* active, float* out_pairs_local, void* stream) {
  if (!p || !row_return || !row_costmask || !row_costsum || !out_pairs_local)
    return set_error(SIMBA_ERR_BAD_CONFIG, "null argument");
  const ReduceParams rp = make_reduce_params(p, row_return, row_costmask, row_costsum, active, out_pairs_local);
  SIMBA_CUDA_TRY(launch_score_reduce(rp, (cudaStream_t)stream));
  return SIMBA_OK;
}

extern "C" int simba_allgather_scores(simba_planner_t* p, const float* pairs_local,
                                      float* out_pairs_all, void* stream) {
  if (!p || !pairs_local || !out_pairs_all) return set_error(SIMBA_ERR_BAD_CONFIG, "null argument");
  const size_t count = (size_t)p->cfg.n_states * p->geom.N_local * 2;
  if (p->cfg.world_size == 1) {
    if (pairs_local != out_pairs_all)
      SIMBA_CUDA_TRY(cudaMemcpyAsync(out_pairs_all, pairs_local, count * 4, cudaMemcpyDeviceToDevice,
                               (cudaStream_t)stream));
    return SIMBA_OK;
  }
  if (!p->comm) return set_error(SIMBA_ERR_NOT_READY, "world_size > 1 but simba_planner_init_nccl was not called");
  NCCL_TRY(g_nccl.all_gather(pairs_local, out_pairs_all, count, kNcclFloat, p->comm,
                             (cudaStream_t)stream));
  return SIMBA_OK;
}

extern "C" int simba_select_elites(simba_planner_t* p, const float* pairs_all, const float* actions,
                                   const int32_t* active, int32_t* out_elite, float* out_scores,
                                   float* best_action, float* best_score, void* stream) {
  if (!p || !pairs_all || !actions || !out_elite || !best_action || !best_score)
    return set_error(SIMBA_ERR_BAD_CONFIG, "null argument");
  const SelectParams sp = make_select_params(p, pairs_all, actions, active, out_elite, out_scores,
                                             best_action, best_score);
  SIMBA_CUDA_TRY(launch_select_elites(sp, (cudaStream_t)stream));
  return SIMBA_OK;
}

extern "C" int simba_refit(simba_planner_t* p, const float* actions, const int32_t* elite, float* mu,
                           float* sigma, int32_t* active, int32_t* iterations_run, void* stream) {
  if (!p || !actions || !elite || !mu || !sigma) return set_error(SIMBA_ERR_BAD_CONFIG, "null argument");
  const RefitParams rp = make_refit_params(p, actions, elite, mu, sigma, active, iterations_run);
  SIMBA_CUDA_TRY(launch_refit(rp, (cudaStream_t)stream));
  return SIMBA_OK;
}

static int do_finalize_action(simba_planner_t* p, const float* best_action, const float* z,
                              uint64_t seed, const uint64_t* seed_ptr, float* out_action,
                              void* stream) {
  if (!p || !best_action || !out_action) return set_error(SIMBA_ERR_BAD_CONFIG, "null argument");
  const FinalizeParams fp = make_finalize_params(p, best_action, z, seed, seed_ptr, out_action);
  SIMBA_CUDA_TRY(launch_finalize(fp, (cudaStream_t)stream));
  return SIMBA_OK;
}

extern "C" int simba_finalize_action(simba_planner_t* p, const float* best_action, const float* z,
                                     uint64_t seed, float* out_action, void* stream) {
  return do_finalize_action(p, best_action, z, seed, nullptr, out_action, stream);
}

// ---- the planning call ---------------------------------------------------------------------------
// One plan = init + I x (sample, rollout, reduce, [all-gather], select, refit) + finalize + output,
// captured once as a CUDA graph. The graph reads the states from p->d_states and the Philox seed from
// p->d_seed (device memory), so neither a new state nor a new seed needs a re-capture; the early
// exit of cem_mpc.py:66-67 is the device-side active[] flag that turns later nodes into no-ops.
static int enqueue_plan(simba_planner* p, cudaStream_t st, int* n_launches) {
  const uint64_t* sp = p->d_seed;
  const auto& c = p->cfg;
  const auto& mc = p->model->cfg;
  const size_t S = c.n_states, N = c.n_samples, HA = (size_t)c.horizon * mc.act_dim;
  const size_t B = (size_t)c.particles * N, O = mc.obs_dim;
  int launches = 0;
  PlanInitParams ip{};
  ip.S = c.n_states; ip.H = c.horizon; ip.A = mc.act_dim;
  memcpy(ip.init_mean, c.init_mean, sizeof(ip.init_mean));
  memcpy(ip.init_stddev, c.init_stddev, sizeof(ip.init_stddev));
  ip.mu = p->mu; ip.sigma = p->sigma; ip.best_action = p->best_action; ip.best_score = p->best_score;
  ip.active = p->active; ip.iterations_run = p->iters;
  const bool multi = c.world_size > 1;
  float* pairs_all = multi ? p->pairs_all : p->pairs_local;
  if (!p->fused_update) { SIMBA_CUDA_TRY(launch_plan_init(ip, st)); ++launches; }
  if (p->fused_update) {
    // small population on one rank: init + sample(0) in one launch, then per iteration rollout + one fused update kernel
    const float* z0 = p->ext_z_actions;
    const SampleParams sp0 = make_sample_params(p, p->mu, p->sigma, z0, 0, sp, 0, p->active, p->actions);
    SIMBA_CUDA_TRY(launch_plan_begin(ip, sp0, st)); ++launches;
    int rc = SIMBA_OK;
    for (int it = 0; it < c.iterations; ++it) {
      const float* eps = p->ext_eps ? p->ext_eps + (size_t)it * S * c.horizon * B * O : nullptr;
      // every rollout is a programmatic dependent launch: the first one's prologue (barriers, TMEM, the weight
      // copies, tables) overlaps the sample kernel, which triggers its dependents at once; later ones overlap the
      // update kernel. The rollout's dependency wait covers the full completion of the kernel before it.
      rc = do_rollout_score(p, p->d_states, p->actions, eps, 0, sp, it, p->active, p->row_ret,
                            p->row_cmask, p->row_csum, st, p->use_pdl);
      if (rc) return rc; ++launches;
      UpdateParams u{};
      u.pdl = p->use_pdl ? 1 : 0;
      u.reduce = make_reduce_params(p, p->row_ret, p->row_cmask, p->row_csum, p->active, p->pairs_local);
      u.select = make_select_params(p, p->pairs_local, p->actions, p->active, p->elite, nullptr,
                                    p->best_action, p->best_score);
      u.refit = make_refit_params(p, p->actions, p->elite, p->mu, p->sigma, p->active, p->iters);
      const float* zn = (p->ext_z_actions && it + 1 < c.iterations)
                            ? p->ext_z_actions + (size_t)(it + 1) * S * N * HA : nullptr;
      u.sample = make_sample_params(p, p->mu, p->sigma, zn, 0, sp, it + 1, p->active, p->actions);
      u.finalize = make_finalize_params(p, p->best_action, p->ext_z_final, 0, sp, p->d_out_action);
      u.last = (it + 1 == c.iterations) ? 1 : 0;
      u.out_score = p->d_out_score;
      u.out_iters = p->d_out_iters;
#ifdef SIMBA_TC_TIMELINE
      if (const char* tlp = getenv("SIMBA_TC_TIMELINE_PTR"))
        u.timeline = reinterpret_cast<long long*>(strtoull(tlp, nullptr, 10)) + (3 * 64 + 1 + it) * 64;
#endif
      SIMBA_CUDA_TRY(launch_cem_update(u, st)); ++launches;
    }
    if (n_launches) *n_launches = launches;
    return SIMBA_OK;
  }
  for (int it = 0; it < c.iterations; ++it) {
    const float* z = p->ext_z_actions ? p->ext_z_actions + (size_t)it * S * N * HA : nullptr;
    const float* eps = p->ext_eps ? p->ext_eps + (size_t)it * S * c.horizon * B * O : nullptr;
    // population sharding: this rank samples only the candidates it rolls out; selection and refit
    // recompute the elite rows the other ranks sampled (SURVEY.md section 8 e)
    SampleParams smp = make_sample_params(p, p->mu, p->sigma, z, 0, sp, it, p->active, p->actions);
    if (multi) { smp.cand0 = p->geom.cand0; smp.n_cand = p->geom.N_local; }
    SIMBA_CUDA_TRY(launch_sample_actions(smp, st)); ++launches;
    int rc = do_rollout_score(p, p->d_states, p->actions, eps, 0, sp, it, p->active, p->row_ret,
                              p->row_cmask, p->row_csum, st);
    if (rc) return rc; ++launches;
    rc = simba_score_reduce(p, p->row_ret, p->row_cmask, p->row_csum, p->active, p->pairs_local, st);
    if (rc) return rc; ++launches;
    if (multi) {
      rc = simba_allgather_scores(p, p->pairs_local, p->pairs_all, st);
      if (rc) return rc; ++launches;
    }
    SelectParams slp = make_select_params(p, pairs_all, p->actions, p->active, p->elite, nullptr,
                                          p->best_action, p->best_score);
    RefitParams rfp = make_refit_params(p, p->actions, p->elite, p->mu, p->sigma, p->active, p->iters);
    if (multi) { slp.regen = 1; slp.sample = smp; rfp.regen = 1; rfp.sample = smp; }
    SIMBA_CUDA_TRY(launch_select_elites(slp, st)); ++launches;
    SIMBA_CUDA_TRY(launch_refit(rfp, st)); ++launches;
  }
  int rc = do_finalize_action(p, p->best_action, p->ext_z_final, 0, sp, p->d_out_action, st);
  if (rc) return rc; ++launches;
  SIMBA_CUDA_TRY(launch_plan_output(p->best_score, p->iters, p->d_out_score, p->d_out_iters, c.n_states, st));
  ++launches;
  if (n_launches) *n_launches = launches;
  return SIMBA_OK;
}

static int ensure_graph(simba_planner* p) {
  if (!p->model->committed) return set_error(SIMBA_ERR_NOT_READY, "model has uncommitted changes");
  if (p->graph_exec && p->graph_generation == p->model->generation) return SIMBA_OK;
  // kernel parameters (scaler constants, flags) are baked into the graph nodes: a re-committed
  // model needs a fresh capture (weights themselves are updated in place and would not)
  if (p->graph_exec) { cudaGraphExecDestroy(p->graph_exec); p->graph_exec = nullptr; }
  if (p->graph) { cudaGraphDestroy(p->graph); p->graph = nullptr; }
  SIMBA_CUDA_TRY(cudaStreamBeginCapture(p->own_stream, cudaStreamCaptureModeThreadLocal));
  int launches = 0;
  int rc = enqueue_plan(p, p->own_stream, &launches);
  cudaGraph_t g = nullptr;
  cudaError_t ce = cudaStreamEndCapture(p->own_stream, &g);
  if (rc != SIMBA_OK) { if (g) cudaGraphDestroy(g); return rc; }
  if (ce != cudaSuccess) return set_error(SIMBA_ERR_CUDA, "graph capture failed: %s", cudaGetErrorString(ce));
  p->graph = g;
  SIMBA_CUDA_TRY(cudaGraphInstantiate(&p->graph_exec, p->graph, 0));
  p->launches_per_plan = launches;
  p->graph_generation = p->model->generation;
  return SIMBA_OK;
}

// stage the seed in a pinned ring slot and copy it to the device ahead of the graph (up to 64
// un-synchronised plans may be queued per planner; they execute one after the other: the plan entry
// points chain them with an event even across streams)
static int upload_seed(simba_planner* p, uint64_t seed, cudaStream_t st) {
  uint64_t* slot = p->h_seed_ring + (p->seed_slot++ & 63);
  *slot = seed;
  SIMBA_CUDA_TRY(cudaMemcpyAsync(p->d_seed, slot, 8, cudaMemcpyHostToDevice, st));
  return SIMBA_OK;
}

extern "C" int simba_planner_launches_per_plan(simba_planner_t* p, int32_t* out) {
  if (!p || !out) return set_error(SIMBA_ERR_BAD_CONFIG, "null argument");
  const int per_iter = 5 + (p->cfg.world_size > 1 ? 1 : 0);
  *out = p->fused_update ? 1 + 2 * p->cfg.iterations : 1 + per_iter * p->cfg.iterations + 2;
  return SIMBA_OK;
}

extern "C" int simba_plan(simba_planner_t* p, const float* states, uint64_t seed, float* out_action,
                          float* out_score, int32_t* out_iterations, void* stream) {
  if (!p || !states || !out_action || !out_score) return set_error(SIMBA_ERR_BAD_CONFIG, "null argument");
  SIMBA_CUDA_TRY(cudaSetDevice(p->device));
  cudaStream_t st = (cudaStream_t)stream;
  const size_t S = p->cfg.n_states, O = p->model->cfg.obs_dim, A = p->model->cfg.act_dim;
  int rc = ensure_graph(p);
  if (rc != SIMBA_OK) return rc;
  // a planner owns ONE workspace (seed, states, mu / sigma, actions, outputs): plans issued on different
  // streams are serialised behind each other here (a no-op when the caller keeps to one stream)
  if (p->plan_done) SIMBA_CUDA_TRY(cudaStreamWaitEvent(st, p->plan_done, 0));
  rc = upload_seed(p, seed, st);
  if (rc != SIMBA_OK) return rc;
  if (states != p->d_states)
    SIMBA_CUDA_TRY(cudaMemcpyAsync(p->d_states, states, S * O * 4, cudaMemcpyDeviceToDevice, st));
  SIMBA_CUDA_TRY(cudaGraphLaunch(p->graph_exec, st));
  if (out_action != p->d_out_action)
    SIMBA_CUDA_TRY(cudaMemcpyAsync(out_action, p->d_out_action, S * A * 4, cudaMemcpyDeviceToDevice, st));
  if (out_score != p->d_out_score)
    SIMBA_CUDA_TRY(cudaMemcpyAsync(out_score, p->d_out_score, S * 4, cudaMemcpyDeviceToDevice, st));
  if (out_iterations && out_iterations != p->d_out_iters)
    SIMBA_CUDA_TRY(cudaMemcpyAsync(out_iterations, p->d_out_iters, S * 4, cudaMemcpyDeviceToDevice, st));
  if (p->plan_done) SIMBA_CUDA_TRY(cudaEventRecord(p->plan_done, st));
  return SIMBA_OK;
}

extern "C" int simba_plan_host(simba_planner_t* p, const float* states_host, uint64_t seed,
                               float* out_action_host, float* out_score_host,
                               int32_t* out_iterations_host) {
  if (!p || !states_host || !out_action_host) return set_error(SIMBA_ERR_BAD_CONFIG, "null argument");
  SIMBA_CUDA_TRY(cudaSetDevice(p->device));
  const size_t S = p->cfg.n_states, O = p->model->cfg.obs_dim, A = p->model->cfg.act_dim;
  cudaStream_t st = p->own_stream;
  int rc = ensure_graph(p);
  if (rc != SIMBA_OK) return rc;
  if (p->plan_done) SIMBA_CUDA_TRY(cudaStreamWaitEvent(st, p->plan_done, 0));    // behind a plan_device() on another stream
  // seed + states staged in pinned memory: one host-to-device copy (the call is synchronous, so one staging
  // block is enough), the graph, one device-to-host copy of the three results
  memcpy(p->h_in, &seed, sizeof(seed));
  memcpy(p->h_in + 16, states_host, S * O * 4);
  SIMBA_CUDA_TRY(cudaMemcpyAsync(p->d_in, p->h_in, 16 + S * O * 4, cudaMemcpyHostToDevice, st));
  SIMBA_CUDA_TRY(cudaGraphLaunch(p->graph_exec, st));
  float* h_act = p->h_out;
  float* h_score = p->h_out + S * A;
  int32_t* h_iters = reinterpret_cast<int32_t*>(p->h_out + S * A + S);
  SIMBA_CUDA_TRY(cudaMemcpyAsync(p->h_out, p->d_out, S * (A + 2) * 4, cudaMemcpyDeviceToHost, st));
  SIMBA_CUDA_TRY(cudaStreamSynchronize(st));
  memcpy(out_action_host, h_act, S * A * 4);
  if (out_score_host) memcpy(out_score_host, h_score, S * 4);
  if (out_iterations_host) memcpy(out_iterations_host, h_iters, S * 4);
  return SIMBA_OK;
}

// ---- NCCL plumbing ---------------------------------------------------------------------------------
extern "C" int simba_nccl_unique_id(void* out) {
  if (!out) return set_error(SIMBA_ERR_BAD_CONFIG, "null argument");
  int rc = nccl_load();
  if (rc != SIMBA_OK) return rc;
  NcclUniqueId id;
  NCCL_TRY(g_nccl.get_unique_id(&id));
  memcpy(out, &id, sizeof(id));
  return SIMBA_OK;
}

extern "C" int simba_planner_init_nccl(simba_planner_t* p, const void* uid) {
  if (!p || !uid) return set_error(SIMBA_ERR_BAD_CONFIG, "null argument");
  int rc = nccl_load();
  if (rc != SIMBA_OK) return rc;
  SIMBA_CUDA_TRY(cudaSetDevice(p->device));
  NcclUniqueId id;
  memcpy(&id, uid, sizeof(id));
  NCCL_TRY(g_nccl.comm_init_rank(&p->comm, p->cfg.world_size, id, p->cfg.rank));
  return SIMBA_OK;
}

// ---- model-level entry points -----------------------------------------------------------------------
// The model keeps one device tile list for its entry points. It is overwritten only after a device-wide
// synchronise, so a launch of any entry point still in flight on another stream never sees it change.
static int model_upload_tiles(simba_model* m, const std::vector<Tile>& tiles) {
  if ((int)tiles.size() > m->tiles_cap) {
    cudaFree(m->d_tiles);
    m->d_tiles = nullptr;
    m->tiles_cap = 0;
    SIMBA_CUDA_TRY(cudaMalloc((void**)&m->d_tiles, tiles.size() * sizeof(Tile)));
    m->tiles_cap = (int)tiles.size();
  }
  // synchronous copy: orders after any earlier kernel that still reads the old list
  SIMBA_CUDA_TRY(cudaDeviceSynchronize());
  SIMBA_CUDA_TRY(cudaMemcpy(m->d_tiles, tiles.data(), tiles.size() * sizeof(Tile), cudaMemcpyHostToDevice));
  return SIMBA_OK;
}

// the device check of the bf16 unfold entry points, per call: one attribute query (cudaGetDeviceProperties, which
// simba_device_check uses, costs milliseconds)
static int unfold_tc_device_check(const simba_model* m) {
  int dev = 0;
  if (m) dev = m->device;
  else SIMBA_CUDA_TRY(cudaGetDevice(&dev));
  int major = 0;
  SIMBA_CUDA_TRY(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
  if (major != 10) return set_error(SIMBA_ERR_ARCH, "device %d is sm_%d*; the tcgen05 kernels need sm_100a", dev, major);
  return SIMBA_OK;
}

// The rows of the model's own entry points: `batch` rows of one state under the tf.split member map, each from its
// own s_0, scored by nothing. Checks the call and sets prm.g, prm.kernel and prm.n_sms; `tiles` is the kernel's list.
// The trajectory forms have no per-row cost mask, so the horizon is bounded by the Philox step counter alone.
static int model_rollout_choice(simba_model* m, int precision, int32_t batch, int32_t horizon, RolloutParams& prm,
                                std::vector<Tile>& tiles) {
  if (!m->committed) return set_error(SIMBA_ERR_NOT_READY, "model not committed");
  if (horizon < 1 || horizon > 65535 || batch < 1)
    return set_error(SIMBA_ERR_BAD_CONFIG, "batch %d / horizon %d out of range", batch, horizon);
  SIMBA_CUDA_TRY(cudaSetDevice(m->device));
  int rc = build_geom(1, 1, batch, 1, 0, horizon, m->cfg.obs_dim, m->cfg.act_dim, m->cfg.ensemble_size,
                      SIMBA_MAP_SPLIT, prm.g);
  if (rc != SIMBA_OK) return rc;
  SIMBA_CUDA_TRY(cudaDeviceGetAttribute(&prm.n_sms, cudaDevAttrMultiProcessorCount, m->device));
  return choose_rollout(m->cfg, precision, prm.g, 0, true, prm.n_sms, prm.kernel, tiles);
}

// model_rollout_choice, the tile upload and the model side of prm
static int model_rollout_params(simba_model* m, int precision, int32_t batch, int32_t horizon, RolloutParams& prm) {
  std::vector<Tile> tiles;
  int rc = model_rollout_choice(m, precision, batch, horizon, prm, tiles);
  if (rc != SIMBA_OK) return rc;
  rc = model_upload_tiles(m, tiles);
  if (rc != SIMBA_OK) return rc;
  memset(&prm.scorer, 0, sizeof(prm.scorer));
  prm.scorer.goal_dist_index = 0;      // any in-range read; results are discarded
  prm.scorer.lidar_max_dist = 1.0f;
  prm.tiles = m->d_tiles;
  prm.n_tiles = (int)tiles.size();
  fill_model_params(m, prm);
  prm.objective = SIMBA_OBJ_REWARD;
  return SIMBA_OK;
}

static int unfold(int precision, simba_model_t* m, const float* s0, const float* actions, const float* eps,
                  uint64_t seed, int32_t batch, int32_t horizon, int32_t sampling_propagation, float* out_traj,
                  void* stream) {
  if (precision != SIMBA_PREC_FP32) {
    int rc = unfold_tc_device_check(m);
    if (rc != SIMBA_OK) return rc;
  }
  if (!m || !s0 || !actions || !out_traj) return set_error(SIMBA_ERR_BAD_CONFIG, "null argument");
  RolloutParams prm{};
  int rc = model_rollout_params(m, precision, batch, horizon, prm);
  if (rc != SIMBA_OK) return rc;
  prm.states = s0; prm.state_stride = m->cfg.obs_dim; prm.state_per_row = 1;
  prm.actions = actions; prm.action_stride = (int64_t)horizon * m->cfg.act_dim;
  prm.eps = eps; prm.seed = seed;
  prm.sampling_propagation = sampling_propagation;
  prm.traj_out = out_traj;
  SIMBA_CUDA_TRY(launch_rollout(prm, (cudaStream_t)stream));
  return SIMBA_OK;
}

extern "C" int simba_unfold(simba_model_t* m, const float* s0, const float* actions,
                            const float* eps, uint64_t seed, int32_t batch, int32_t horizon,
                            int32_t sampling_propagation, float* out_traj, void* stream) {
  return unfold(SIMBA_PREC_FP32, m, s0, actions, eps, seed, batch, horizon, sampling_propagation, out_traj, stream);
}

extern "C" int simba_unfold_tc(simba_model_t* m, const float* s0, const float* actions,
                               const float* eps, uint64_t seed, int32_t batch, int32_t horizon,
                               int32_t sampling_propagation, float* out_traj, void* stream) {
  return unfold(SIMBA_PREC_BF16_TC, m, s0, actions, eps, seed, batch, horizon, sampling_propagation, out_traj,
                stream);
}

extern "C" int simba_unfold_tc_kernel(simba_model_t* m, int32_t batch, int32_t horizon, int32_t* kernel,
                                      int32_t* work_items) {
  int rc = unfold_tc_device_check(m);
  if (rc != SIMBA_OK) return rc;
  if (!m || !kernel || !work_items) return set_error(SIMBA_ERR_BAD_CONFIG, "null argument");
  RolloutParams prm{};
  std::vector<Tile> tiles;
  rc = model_rollout_choice(m, SIMBA_PREC_BF16_TC, batch, horizon, prm, tiles);
  if (rc != SIMBA_OK) return rc;
  *kernel = (int32_t)prm.kernel;
  *work_items = n_work_items(prm.kernel, tiles);
  return SIMBA_OK;
}

// The forward pass of the model's rows (mlp_ensemble.py:122-132, :189-193) as a one-step rollout whose state is x's
// first O columns and whose action is the rest: a set prm.mu_out selects the forward form of the kernel.
static int ensemble_forward(int precision, simba_model_t* m, const float* x, const float* eps, int32_t batch,
                            float* out_mu, float* out_var, float* out_sample, void* stream) {
  if (precision != SIMBA_PREC_FP32) {
    int rc = unfold_tc_device_check(m);
    if (rc != SIMBA_OK) return rc;
  }
  if (!m || !x || !out_mu || !out_var) return set_error(SIMBA_ERR_BAD_CONFIG, "null argument");
  RolloutParams prm{};
  int rc = model_rollout_params(m, precision, batch, 1, prm);
  if (rc != SIMBA_OK) return rc;
  const int O = m->cfg.obs_dim, IN = O + m->cfg.act_dim;
  prm.scale_on = 0;                               // x is used as given (mlp_ensemble.py:190)
  if (precision != SIMBA_PREC_FP32) {
    // the tcgen05 kernels scale through these tables alone: the identity of scale_on = 0 (pack_scaler), not the
    // model's own
    for (int k = 0; k < 128; ++k) {
      prm.tc_scale_a[k] = k < IN ? 1.0f : 0.0f;
      prm.tc_scale_b[k] = 0.0f;
    }
    prm.sampling_propagation = out_sample != nullptr;   // the draws enter the head pass only for a sample
  }
  prm.states = x; prm.state_stride = IN; prm.state_per_row = 1;
  prm.actions = x + O; prm.action_stride = IN;
  prm.eps = eps;
  prm.mu_out = out_mu; prm.var_out = out_var; prm.sample_out = out_sample;
  if (out_sample && !eps) return set_error(SIMBA_ERR_BAD_CONFIG, "out_sample needs eps");
  SIMBA_CUDA_TRY(launch_rollout(prm, (cudaStream_t)stream));
  return SIMBA_OK;
}

extern "C" int simba_ensemble_forward(simba_model_t* m, const float* x, const float* eps,
                                      int32_t batch, float* out_mu, float* out_var,
                                      float* out_sample, void* stream) {
  return ensemble_forward(SIMBA_PREC_FP32, m, x, eps, batch, out_mu, out_var, out_sample, stream);
}

extern "C" int simba_ensemble_forward_tc(simba_model_t* m, const float* x, const float* eps, int32_t batch,
                                         float* out_mu, float* out_var, float* out_sample, void* stream) {
  return ensemble_forward(SIMBA_PREC_BF16_TC, m, x, eps, batch, out_mu, out_var, out_sample, stream);
}

// the forward form runs the variant of the trajectory form at H = 1
extern "C" int simba_ensemble_forward_tc_kernel(simba_model_t* m, int32_t batch, int32_t* kernel,
                                                int32_t* work_items) {
  return simba_unfold_tc_kernel(m, batch, 1, kernel, work_items);
}

extern "C" int simba_scale(simba_model_t* m, const float* x, int32_t batch, float* out, void* stream) {
  if (!m || !x || !out) return set_error(SIMBA_ERR_BAD_CONFIG, "null argument");
  if (!m->committed) return set_error(SIMBA_ERR_NOT_READY, "model not committed");
  SIMBA_CUDA_TRY(cudaSetDevice(m->device));
  SIMBA_CUDA_TRY(launch_scale(x, m->d_smin, m->d_sdelta, m->scale_on, batch,
                        m->cfg.obs_dim + m->cfg.act_dim, out, (cudaStream_t)stream));
  return SIMBA_OK;
}

extern "C" int simba_score_trajectories(simba_planner_t* p, const float* traj, float* out_scores,
                                        float* out_pairs, void* stream) {
  if (!p || !traj || !out_scores) return set_error(SIMBA_ERR_BAD_CONFIG, "null argument");
  if (p->cfg.n_states != 1 || p->cfg.world_size != 1)
    return set_error(SIMBA_ERR_UNSUPPORTED, "score_trajectories needs n_states == 1 and world_size == 1");
  SIMBA_CUDA_TRY(cudaSetDevice(p->device));
  cudaStream_t st = (cudaStream_t)stream;
  const int rows = p->cfg.particles * p->cfg.n_samples;
  SIMBA_CUDA_TRY(launch_score_traj_rows(p->cfg.scorer, traj, rows, p->cfg.horizon, p->model->cfg.obs_dim,
                                  p->cfg.objective, p->row_ret, p->row_cmask, p->row_csum, st));
  int rc = simba_score_reduce(p, p->row_ret, p->row_cmask, p->row_csum, nullptr, p->pairs_local, st);
  if (rc != SIMBA_OK) return rc;
  SIMBA_CUDA_TRY(launch_pairs_to_scores(p->pairs_local, p->cfg.n_samples, p->cfg.objective,
                                  (float)p->c_max, out_scores, st));
  if (out_pairs)
    SIMBA_CUDA_TRY(cudaMemcpyAsync(out_pairs, p->pairs_local, (size_t)p->cfg.n_samples * 8,
                             cudaMemcpyDeviceToDevice, st));
  return SIMBA_OK;
}

extern "C" int simba_scorer_eval(const simba_scorer_t* sc, const float* obs, const float* next_obs,
                                 int32_t batch, int32_t obs_dim, float* out_reward,
                                 int32_t* out_done, float* out_cost, void* stream) {
  if (!sc || !obs) return set_error(SIMBA_ERR_BAD_CONFIG, "null argument");
  int rc = validate_scorer(*sc, obs_dim);
  if (rc != SIMBA_OK) return rc;
  SIMBA_CUDA_TRY(launch_scorer_eval(*sc, obs, next_obs, batch, obs_dim, out_reward, out_done, out_cost,
                              (cudaStream_t)stream));
  return SIMBA_OK;
}

// ---- RNG probes ----------------------------------------------------------------------------------------
extern "C" int simba_philox_raw(const uint32_t counter[4], const uint32_t key[2], uint32_t out[4]) {
  if (!counter || !key || !out) return set_error(SIMBA_ERR_BAD_CONFIG, "null argument");
  uint32_t* d = nullptr;
  SIMBA_CUDA_TRY(cudaMalloc((void**)&d, 16));
  cudaError_t e = launch_philox_raw(counter, key, d, nullptr);
  if (e == cudaSuccess) e = cudaMemcpy(out, d, 16, cudaMemcpyDeviceToHost);
  cudaFree(d);
  SIMBA_CUDA_TRY(e);
  return SIMBA_OK;
}

extern "C" int simba_philox_normals(uint64_t seed, int32_t rng_stream, int32_t iteration, int32_t t,
                                    int32_t state_index, int32_t first_row, int32_t n_rows,
                                    int32_t n_elems, int32_t fast_math, float* out, void* stream) {
  if (!out || n_rows < 1 || n_elems < 1) return set_error(SIMBA_ERR_BAD_CONFIG, "bad argument");
  SIMBA_CUDA_TRY(launch_philox_normals(seed, rng_stream, iteration, t, state_index, first_row, n_rows,
                                 n_elems, fast_math, out, (cudaStream_t)stream));
  return SIMBA_OK;
}

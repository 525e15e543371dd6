// fp32 SIMT kernels of the ensemble training step (simba_trainer_config_t.precision = SIMBA_PREC_FP32, the
// default): replace MlpEnsemble.training_step / validation_step / fit's inner loop
// (simba/models/mlp_ensemble.py:134-187) in fp32 throughout, as the reference trains. trainer.cu owns the buffers and
// launches these through train_f32_chain / train_f32_update (train_common.cuh).
//
// Shape of the work: E members x batch 64 x a 4x128 MLP is 28 MFLOP per member-step — nothing a
// launch can hide — so the step is latency-bound and the design minimises dependent launches and
// dependent memory round trips. Forward and back-propagation of the activations are ROW-LOCAL
// (row r of every H_l and dZ_l depends only on row r of the batch), so one CTA walks an 8-row
// tile through the whole chain without any inter-CTA dependency:
//   chain   1 launch   H_{l+1} = relu([H_l, 1] . theta_l), l < L; head -> (mu, var) -> likelihood,
//                      d(mu), d(raw var), lr_t; then dZ_{l-1} = relu'(H_l) * (dZ_l . theta_l^T),
//                      l = L..1. Weights stream from L2 as TMA bulk copies (cp.async.bulk +
//                      mbarrier) into a two-chunk ring — chunk q + 1 lands while chunk q is
//                      multiplied; activations stay in shared memory between layers and are
//                      written out once for the update kernel.
//   update  1 launch   dtheta_l = [H_l, 1]^T . dZ_l for EVERY layer, clip, Adam — one grid
// i.e. 2 launches per step (one CUDA graph), and fit()'s batch gather is folded into the loads.
// Parameters of train layer l are one [(K_l + 1) x N_l] row-major block (Keras kernel [in, out]
// followed by the bias row): "bias" is the row that multiplies the constant 1, and the
// weight-gradient GEMM yields the bias gradient as its last row. The Gaussian head's two Dense
// layers (mlp_ensemble.py:28-30) are one block with N = 2 * O whose columns interleave
// (mu_0, var_0, mu_1, var_1, ...), so a thread's accumulators hold complete (mu, var) pairs and
// mu / var never go to memory. The update kernel also maintains theta_l^T, so back-propagation
// reads its weights with the same unit-stride tile pattern as the forward pass.
// Reductions are in a fixed order: results are bit-reproducible run to run.
#include <algorithm>
#include <cstdint>

#include "common.cuh"
#include "internal.h"
#include "tc_ptx.cuh"
#include "train_common.cuh"

namespace {

// simba's names come in by using-declarations: with `using namespace simba`, this unnamed namespace and tc_ptx.cuh's
// (inside simba) would be ambiguous in the host stubs nvcc generates for these kernels
using simba::kMaxTrainLayers;
// PTX wrappers (tc_ptx.cuh)
using simba::bulk_g2s;
using simba::fence_barrier_init;
using simba::fence_proxy_async;
using simba::mbar_expect_tx;
using simba::mbar_init;
using simba::smem_u32;

// batch rows per chain CTA: template parameter R of the chain kernel (4, 8 or 16; the host picks
// the smallest that keeps the grid near one wave: 64-row batch x 5 members -> R = 4, 80 CTAs)
constexpr int kChunkK = 128;     // weight chunk: [128 k] x [128 n] fp32 = 64 KB, two in flight
constexpr int kChunkN = 128;
constexpr int kChainThreads = 256;
constexpr int kChainWarps = 8;
__host__ __device__ constexpr int chain_row_groups(int rows) { return rows > 8 ? 2 : 1; }   // 16 rows: 2 row groups x 4 k-slices
constexpr int kTileU = 32;       // update kernel: [32 k] x [32 n] tile of dtheta
constexpr int kRowsU = 64;       // update kernel: batch rows per staged chunk
constexpr int kThreadsU = 256;

// The chain kernel's own mbarrier wait: try_wait without the suspend-time hint, bounded at 2^26 polls (a protocol
// bug must fault the kernel, never hang the GPU). tc_ptx.cuh's hinted mbar_wait would change this kernel's code.
__device__ __forceinline__ void chain_mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t spins = 0;
  while (true) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    if (ok != 0) return;
    if (++spins > (1u << 26)) __trap();
  }
}

// ---------------------------------------------------------------------------------------------
// chain kernel: forward (BaseLayer.call / GaussianHead.call, mlp_ensemble.py:17-22, :28-34),
// negative_log_likelihood (:64-67) with its gradient, and the activation back-propagation
// ---------------------------------------------------------------------------------------------
#ifdef SIMBA_TRAIN_TIMELINE
__device__ long long g_train_tl[512];
#define TL(slot) do { if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) g_train_tl[(slot)] = clock64(); } while (0)
#else
#define TL(slot) do { } while (0)
#endif

enum PassKind { kPassHidden = 0, kPassHead = 1, kPassBackward = 2 };

// one GEMM of the chain: out[16 x n_dim] = in[16 x k_dim] . W[k_dim x n_dim]   (W row-major, ld = n_dim)
struct ChainPass {
  int64_t w_off;          // into theta (forward / head) or theta^T (backward), per member
  int64_t bias_off;       // forward / head: the bias row inside theta
  int k_dim, n_dim;
  int kind;
  float* out;             // hidden: H_{l+1} [E][cap][n]; head: dZ_L [E][B][n]; backward: dZ_{l-1}
  int64_t out_estride;
  const float* mask;      // backward: H_l [E][cap][n_dim of this pass]; > 0 <=> the unit was active
  int64_t mask_estride;
};

struct ChainArgs {
  ChainPass pass[2 * kMaxTrainLayers];
  int n_forward;          // hidden layers + head
  int n_pass;             // n_forward (+ backward passes when training)
  const float* x;         // [E][rows][K_0] (estride may be 0: validation shares its rows)
  int64_t x_estride;
  int gather;             // 1: batch rows follow the fit descriptor's index
  const float* y;         // [E][rows][O]
  int64_t y_estride;
  const float* theta;     // [E][pn]
  const float* thetaT;    // [E][pnT]
  int64_t pn, pnT;
  int ld_act;             // row stride of the shared activation tiles (widest layer)
  int out_dim, ensemble;
  int aligned;            // every chunk row is 16-byte aligned -> 16-byte cp.async
  float* partial;         // [E][tiles_cap][2]
  int tiles_cap;
  int train;
  float* out_loss;
  // Dropout after every hidden ReLU in training (mlp_ensemble.py:17-22): keep = u01(philox) >= rate,
  // kept activations scaled by 1 / (1 - rate). Counter (column block, batch row, iteration,
  // member | layer << 8 | stream 4 << 28), key = dropout_seed — restated in oracle/philox.py.
  float dropout_rate, dropout_scale;
  uint64_t dropout_seed;
};

struct ChunkCursor {      // walks the chunks of the chain in execution order
  int pass, n0, k0;
};

__device__ __forceinline__ bool next_chunk(const ChainArgs& a, ChunkCursor& c) {
  const ChainPass& p = a.pass[c.pass];
  c.k0 += kChunkK;
  if (c.k0 < p.k_dim) return true;
  c.k0 = 0;
  c.n0 += kChunkN;
  if (c.n0 < p.n_dim) return true;
  c.n0 = 0;
  c.pass += 1;
  return c.pass < a.n_pass;
}

// row stride of a weight chunk in shared memory: a layer no wider than one chunk is one contiguous
// block of theta, copied by a single bulk instruction and kept at its own row stride
__device__ __forceinline__ int chunk_stride(const ChainArgs& a, const ChainPass& p) {
  return (a.aligned && p.n_dim <= kChunkN) ? p.n_dim : kChunkN;
}

// Requests chunk `c` into `buf`. Aligned shapes: TMA bulk copies issued by warp 0 (ONE instruction
// when the layer is no wider than a chunk), completion on `bar`. Other shapes (tests with odd
// widths): plain loads by every thread, visible after the caller's next __syncthreads. Rows
// [kc, roundup4(kc)) are zeroed: the multiply consumes k in groups of 4.
__device__ __forceinline__ void issue_chunk(const ChainArgs& a, const ChunkCursor& c, int e, float* buf,
                                            uint32_t bar) {
  const ChainPass& p = a.pass[c.pass];
  const float* base = (p.kind == kPassBackward ? a.thetaT + e * a.pnT : a.theta + e * a.pn) + p.w_off;
  const float* src = base + (int64_t)c.k0 * p.n_dim + c.n0;
  const int kc = min(kChunkK, p.k_dim - c.k0), nc = min(kChunkN, p.n_dim - c.n0);
  const int S = chunk_stride(a, p);
  const int kc4 = (kc + 3) & ~3;
  const int tid = threadIdx.x;
  for (int i = kc * S + tid; i < kc4 * S; i += kChainThreads) buf[i] = 0.0f;
  if (a.aligned) {
    if (kc4 != kc) fence_proxy_async();
    if (tid < 32) {
      if (tid == 0) mbar_expect_tx(bar, (uint32_t)(kc * nc * sizeof(float)));
      __syncwarp();
      if (p.n_dim <= kChunkN) {
        if (tid == 0) bulk_g2s(smem_u32(buf), src, (uint32_t)(kc * nc * sizeof(float)), bar);
      } else {
        for (int k = tid; k < kc; k += 32)
          bulk_g2s(smem_u32(buf + k * S), src + (int64_t)k * p.n_dim, (uint32_t)(nc * sizeof(float)), bar);
      }
    }
  } else {
    for (int i = tid; i < kc * nc; i += kChainThreads) {
      const int k = i / nc, n = i - k * nc;
      buf[k * S + n] = __ldcg(src + (int64_t)k * p.n_dim + n);
    }
  }
}

// The multiply: the 8 warps form kRowGroups row groups x kSplitK k-slices (R <= 8: 1 x 8, i.e.
// every warp covers all rows of the tile and one eighth of K, so each weight element is read
// from shared memory exactly once per CTA; R = 16: 2 x 4 to bound the register tile). Warp slice s takes k-groups s, s + kSplitK, ... A
// lane owns 4 columns, so a thread accumulates a [kGroupRows x 4] register tile of independent
// FMA chains, and the operands of a k-group (4 weight float4s + kGroupRows broadcast activation
// float4s) sit in registers ahead of their use. The partial tiles are added in a fixed order
// through shared memory when the layer's last chunk is done.
template <int kRows>
__global__ void __launch_bounds__(kChainThreads)
train_chain_kernel(ChainArgs a, OptParams opt, const FitDesc* desc, TrainState* st, int rows_fixed,
                   int step_off) {
  constexpr int kRowGroups = chain_row_groups(kRows);   // the 8 warps: kRowGroups row groups x kSplitK k-slices
  constexpr int kSplitK = kChainWarps / kRowGroups;
  constexpr int kGroupRows = kRows / kRowGroups;
  constexpr int kEpiWarps = kRows < kChainWarps ? kRows : kChainWarps;   // warps that own rows in the epilogue
  constexpr int kEpiRows = kRows / kEpiWarps;                            // rows per such warp
  extern __shared__ __align__(16) float smem[];
  float* red = smem + 2 * kChunkK * kChunkN;                 // [2 halves][4 k-slices][8][128]
  float* act0 = red + kRowGroups * kSplitK * kGroupRows * kChunkN;
  float* act1 = act0 + kRows * a.ld_act;
  __shared__ float scratch[kChainThreads / 32];
  __shared__ __align__(8) unsigned long long bars[2];
  __shared__ bool last;

  const int rows = resolve_rows(desc, st, rows_fixed, step_off);
  const int e = blockIdx.y, r0 = blockIdx.x * kRows;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int rgroup = warp / kSplitK, kslice = warp % kSplitK;   // multiply: rows kGroupRows * rgroup ..
  const int cl = 4 * lane;                          // chunk-local columns cl .. cl + 3 (both phases)
  // epilogue: warp w finishes rows kEpiRows * w .. of the tile
  const int ld = a.ld_act;
  float s_log = 0.0f, s_sq = 0.0f;
  TL(0);

  if (r0 < rows) {
    if (tid == 0) {
      mbar_init(smem_u32(&bars[0]), 1);
      mbar_init(smem_u32(&bars[1]), 1);
      fence_barrier_init();
    }
    __syncthreads();
    ChunkCursor cur{0, 0, 0}, nxt{0, 0, 0};
    issue_chunk(a, cur, e, smem, smem_u32(&bars[0]));
    bool more = next_chunk(a, nxt);
    // the batch tile (layer 0 input), zero-padded to a multiple of 4 columns
    {
      const int K0 = a.pass[0].k_dim, K0r = (K0 + 3) & ~3;
      const int* gidx = a.gather ? batch_rows_of(desc, st, e, a.ensemble, step_off) : nullptr;
      const float* X = a.x + e * a.x_estride;
      for (int i = tid; i < kRows * K0r; i += kChainThreads) {
        const int r = i / K0r, k = i - r * K0r;
        float v = 0.0f;
        if (r0 + r < rows && k < K0) {
          const float* row = gidx ? desc->inputs + (int64_t)gidx[r0 + r] * K0 : X + (int64_t)(r0 + r) * K0;
          v = __ldg(row + k);
        }
        act0[r * ld + k] = v;
      }
    }
    __syncthreads();
    float* in = act0;
    float* out = act1;
    float acc[kGroupRows][4] = {};
    int q = 0;
    TL(1);
    while (true) {
      const ChainPass& p = a.pass[cur.pass];
      const float* wb = smem + (q & 1) * kChunkK * kChunkN;
      TL(8 + q * 8 + 0);
      if (more)
        issue_chunk(a, nxt, e, smem + ((q + 1) & 1) * kChunkK * kChunkN, smem_u32(&bars[(q + 1) & 1]));
      TL(8 + q * 8 + 1);
      const int kc = min(kChunkK, p.k_dim - cur.k0);
      const int kc4 = (kc + 3) & ~3;
      const bool last_k = cur.k0 + kChunkK >= p.k_dim;
      const int c0 = cur.n0 + cl;
      // epilogue operands are requested before the multiply so their latency hides behind it
      float pb[4] = {};                              // bias (forward / head)
      float pm[kEpiRows][4] = {};                    // backward: H_l (mask); head: targets at even j
      if (last_k) {
        if (p.kind != kPassBackward) {
          const float* bias = a.theta + e * a.pn + p.bias_off;
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (c0 + j < p.n_dim) pb[j] = __ldcg(bias + c0 + j);
        }
#pragma unroll
        for (int i = 0; i < kEpiRows; ++i) {
          const int r = r0 + kEpiRows * warp + i;
          if (warp >= kEpiWarps || r >= rows) continue;
          if (p.kind == kPassBackward) {
            const float* h = p.mask + e * p.mask_estride + (int64_t)r * p.n_dim;
#pragma unroll
            for (int j = 0; j < 4; ++j)
              if (c0 + j < p.n_dim) pm[i][j] = __ldcg(h + c0 + j);
          } else if (p.kind == kPassHead) {
            const float* y = a.gather
                ? desc->targets + (int64_t)batch_rows_of(desc, st, e, a.ensemble, step_off)[r] * a.out_dim
                : a.y + e * a.y_estride + (int64_t)r * a.out_dim;
#pragma unroll
            for (int j = 0; j < 4; j += 2)
              if (c0 + j < p.n_dim) pm[i][j] = __ldg(y + ((c0 + j) >> 1));
          }
        }
      }
      if (a.aligned) chain_mbar_wait(smem_u32(&bars[q & 1]), (q >> 1) & 1);
      TL(8 + q * 8 + 2);
      {
        const int S = chunk_stride(a, p);
        const float* w = wb + cl;
        const float* xin = in + (rgroup * kGroupRows) * ld + cur.k0;
        for (int kk = 4 * kslice; kk < kc4; kk += 4 * kSplitK) {
          const float4 w0 = *reinterpret_cast<const float4*>(w + (kk + 0) * S);
          const float4 w1 = *reinterpret_cast<const float4*>(w + (kk + 1) * S);
          const float4 w2 = *reinterpret_cast<const float4*>(w + (kk + 2) * S);
          const float4 w3 = *reinterpret_cast<const float4*>(w + (kk + 3) * S);
          float4 x[kGroupRows];
#pragma unroll
          for (int i = 0; i < kGroupRows; ++i) x[i] = *reinterpret_cast<const float4*>(xin + i * ld + kk);
#pragma unroll
          for (int i = 0; i < kGroupRows; ++i) {
            acc[i][0] = fmaf(x[i].x, w0.x, acc[i][0]); acc[i][1] = fmaf(x[i].x, w0.y, acc[i][1]);
            acc[i][2] = fmaf(x[i].x, w0.z, acc[i][2]); acc[i][3] = fmaf(x[i].x, w0.w, acc[i][3]);
          }
#pragma unroll
          for (int i = 0; i < kGroupRows; ++i) {
            acc[i][0] = fmaf(x[i].y, w1.x, acc[i][0]); acc[i][1] = fmaf(x[i].y, w1.y, acc[i][1]);
            acc[i][2] = fmaf(x[i].y, w1.z, acc[i][2]); acc[i][3] = fmaf(x[i].y, w1.w, acc[i][3]);
          }
#pragma unroll
          for (int i = 0; i < kGroupRows; ++i) {
            acc[i][0] = fmaf(x[i].z, w2.x, acc[i][0]); acc[i][1] = fmaf(x[i].z, w2.y, acc[i][1]);
            acc[i][2] = fmaf(x[i].z, w2.z, acc[i][2]); acc[i][3] = fmaf(x[i].z, w2.w, acc[i][3]);
          }
#pragma unroll
          for (int i = 0; i < kGroupRows; ++i) {
            acc[i][0] = fmaf(x[i].w, w3.x, acc[i][0]); acc[i][1] = fmaf(x[i].w, w3.y, acc[i][1]);
            acc[i][2] = fmaf(x[i].w, w3.z, acc[i][2]); acc[i][3] = fmaf(x[i].w, w3.w, acc[i][3]);
          }
        }
      }
      TL(8 + q * 8 + 3);
      if (last_k) {
        // add the k-slices of each row group in slice order, then the epilogue of this warp's rows,
        // columns c0 .. c0 + 3
#pragma unroll
        for (int i = 0; i < kGroupRows; ++i) {
          *reinterpret_cast<float4*>(red + ((rgroup * kSplitK + kslice) * kGroupRows + i) * kChunkN + cl) =
              make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
          acc[i][0] = acc[i][1] = acc[i][2] = acc[i][3] = 0.0f;
        }
        __syncthreads();
#pragma unroll
        for (int i = 0; i < kEpiRows; ++i) {
          if (warp >= kEpiWarps) continue;
          const int rl = kEpiRows * warp + i, r = r0 + rl;
          const bool row_ok = r < rows;
          float v[4] = {};
#pragma unroll
          for (int sl = 0; sl < kSplitK; ++sl) {
            const float4 pv = *reinterpret_cast<const float4*>(
                red + (((rl / kGroupRows) * kSplitK + sl) * kGroupRows + (rl % kGroupRows)) * kChunkN + cl);
            v[0] += pv.x; v[1] += pv.y; v[2] += pv.z; v[3] += pv.w;
          }
          if (p.kind == kPassHead) {
            const float c = 1.0f / ((float)rows * (float)a.out_dim * (float)a.ensemble);
#pragma unroll
            for (int j = 0; j < 4; j += 2) {
              float d_mu = 0.0f, d_pre = 0.0f;
              if (c0 + j < p.n_dim && row_ok)
                nll_terms(v[j] + pb[j], v[j + 1] + pb[j + 1], pm[i][j], c, s_log, s_sq, d_mu, d_pre);
              v[j] = d_mu;
              v[j + 1] = d_pre;
            }
          } else {
            float keep[4] = {1.0f, 1.0f, 1.0f, 1.0f};          // forward: dropout mask / (1 - rate)
            float back = 1.0f;                                   // backward: the same 1 / (1 - rate)
            if (a.train && a.dropout_rate > 0.0f) {
              if (p.kind == kPassHidden) {
                dropout_keep4(c0, r, (uint32_t)(st->iterations + step_off), e, cur.pass, a.dropout_rate,
                              a.dropout_scale, a.dropout_seed, keep);
              } else {
                back = a.dropout_scale;       // H > 0 <=> unit active AND kept (H is stored after dropout)
              }
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const bool ok = c0 + j < p.n_dim;
              if (p.kind == kPassHidden) v[j] = ok ? fmaxf(v[j] + pb[j], 0.0f) * keep[j] : 0.0f;
              else v[j] = (ok && row_ok && pm[i][j] > 0.0f) ? v[j] * back : 0.0f;
            }
          }
          // columns past n_dim are written as zeros so that the next pass can consume k in groups of 4
          if (c0 + 3 < ld) {
            *reinterpret_cast<float4*>(out + rl * ld + c0) = make_float4(v[0], v[1], v[2], v[3]);
          } else {
#pragma unroll
            for (int j = 0; j < 4; ++j)
              if (c0 + j < ld) out[rl * ld + c0 + j] = v[j];
          }
          if (row_ok && (p.kind != kPassHead || a.train)) {
            float* gout = p.out + e * p.out_estride + (int64_t)r * p.n_dim + c0;
            if (a.aligned && c0 + 3 < p.n_dim) {
              *reinterpret_cast<float4*>(gout) = make_float4(v[0], v[1], v[2], v[3]);
            } else {
#pragma unroll
              for (int j = 0; j < 4; ++j)
                if (c0 + j < p.n_dim) gout[j] = v[j];
            }
          }
        }
      }
      TL(8 + q * 8 + 4);
      const int done_pass = cur.pass;
      if (!more) break;
      cur = nxt;
      more = next_chunk(a, nxt);
      ++q;
      if (cur.pass != done_pass) { float* t = in; in = out; out = t; }
      __syncthreads();       // the old chunk buffer and activation tile are free; the new tile is visible
    }
  }

  TL(2);
  const float t_log = block_sum(s_log, scratch);
  const float t_sq = block_sum(s_sq, scratch);
  if (tid == 0) {
    a.partial[((int64_t)e * a.tiles_cap + blockIdx.x) * 2 + 0] = t_log;
    a.partial[((int64_t)e * a.tiles_cap + blockIdx.x) * 2 + 1] = t_sq;
  }
  if (!a.train) return;
  // the last CTA to arrive adds the partials in a fixed order and prepares the update
  if (tid == 0) {
    __threadfence();
    last = (atomicAdd(&st->nll_ticket, 1u) == gridDim.x * gridDim.y - 1);
  }
  __syncthreads();
  if (!last || tid >= 32) return;
  __threadfence();
  const int tiles = (rows + kRows - 1) / kRows;
  const float denom = (float)rows * (float)a.out_dim;
  float loss = 0.0f;
  for (int m = 0; m < a.ensemble; ++m) {
    float sl = 0.0f, sq = 0.0f;
    for (int t = tid; t < tiles; t += 32) {
      sl += __ldcg(&a.partial[((int64_t)m * a.tiles_cap + t) * 2 + 0]);
      sq += __ldcg(&a.partial[((int64_t)m * a.tiles_cap + t) * 2 + 1]);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      sl += __shfl_down_sync(0xffffffffu, sl, o);
      sq += __shfl_down_sync(0xffffffffu, sq, o);
    }
    loss += (0.5f * (sl / denom) + 0.5f * (sq / denom)) / (float)a.ensemble;
  }
  if (tid != 0) return;
  const int it = st->iterations + step_off;
  const float t = (float)(it + 1);
  st->lr_t = schedule_lr(opt, it) * sqrtf(1.0f - powf(opt.beta2, t)) / (1.0f - powf(opt.beta1, t));
  st->loss = loss;
  if (a.out_loss) *a.out_loss = loss;
  if (desc != nullptr && desc->losses != nullptr) desc->losses[st->fit_step + step_off] = loss;
  st->nll_ticket = 0;
}

// ---------------------------------------------------------------------------------------------
// weight gradient + clip + Adam for every layer in one grid; also refreshes theta^T
// ---------------------------------------------------------------------------------------------
struct UpdLayer {
  const float* h;       // input of the layer [E][rows][K]
  int64_t h_estride;
  const float* dz;      // [E][rows][N]
  int64_t dz_estride;
  int64_t off, offT;    // offT < 0: no transposed copy (layer 0 is never back-propagated through)
  int K, N;
  int gather_h;         // layer 0 inside fit: rows follow the batch index
  int tile_begin;       // first tile index of this layer in the grid
  int n_tiles_n;
};
struct UpdArgs {
  UpdLayer layers[kMaxTrainLayers];
  int n_layers;
  float* theta;
  float* thetaT;
  float* m;
  float* v;
  float* grad;
  int64_t pn, pnT;
  int ensemble;
};

__global__ void __launch_bounds__(kThreadsU)
train_update_kernel(UpdArgs a, OptParams opt, const FitDesc* desc, const TrainState* st, int rows_fixed,
                    int step_off) {
  const int rows = resolve_rows(desc, st, rows_fixed, step_off);
  int li = 0;
#pragma unroll 1
  while (li + 1 < a.n_layers && (int)blockIdx.x >= a.layers[li + 1].tile_begin) ++li;
  const UpdLayer& L = a.layers[li];
  const int t_in = blockIdx.x - L.tile_begin;
  const int tk0 = (t_in / L.n_tiles_n) * kTileU, tn0 = (t_in % L.n_tiles_n) * kTileU;
  const int e = blockIdx.y;
  __shared__ float Hs[kRowsU][kTileU + 1];
  __shared__ __align__(16) float Zs[kRowsU][kTileU];
  const float* H = L.h + e * L.h_estride;
  const float* dZ = L.dz + e * L.dz_estride;
  const int* gidx = L.gather_h ? batch_rows_of(desc, st, e, a.ensemble, step_off) : nullptr;
  const int tid = threadIdx.x, tx = tid & 7, ty = tid >> 3;
  // the Adam operands are fetched while the gradient tile is being computed
  const int k = tk0 + ty;
  float th[4], mo[4], ve[4];
  const int64_t p0 = e * a.pn + L.off + (int64_t)k * L.N + tn0 + tx * 4;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const bool ok = k <= L.K && tn0 + tx * 4 + j < L.N;
    th[j] = ok ? a.theta[p0 + j] : 0.0f;
    mo[j] = ok ? a.m[p0 + j] : 0.0f;
    ve[j] = ok ? a.v[p0 + j] : 0.0f;
  }
  float acc[4] = {};
  for (int r0 = 0; r0 < rows; r0 += kRowsU) {
    if (r0) __syncthreads();
    // every global load of the chunk is in flight before the first shared store
    float hv[kRowsU * kTileU / kThreadsU], zv[kRowsU * kTileU / kThreadsU];
#pragma unroll
    for (int j = 0; j < kRowsU * kTileU / kThreadsU; ++j) {
      const int i = tid + j * kThreadsU, r = i >> 5, kk = i & 31;
      float h = 0.0f, z = 0.0f;
      if (r0 + r < rows) {
        if (tk0 + kk < L.K) {
          const float* row = gidx ? desc->inputs + (int64_t)gidx[r0 + r] * L.K : H + (int64_t)(r0 + r) * L.K;
          h = __ldcg(row + tk0 + kk);
        } else if (tk0 + kk == L.K) {
          h = 1.0f;                                   // the bias row
        }
        if (tn0 + kk < L.N) z = __ldcg(dZ + (int64_t)(r0 + r) * L.N + tn0 + kk);
      }
      hv[j] = h;
      zv[j] = z;
    }
#pragma unroll
    for (int j = 0; j < kRowsU * kTileU / kThreadsU; ++j) {
      const int i = tid + j * kThreadsU;
      Hs[i >> 5][i & 31] = hv[j];
      Zs[i >> 5][i & 31] = zv[j];
    }
    __syncthreads();
#pragma unroll 8
    for (int r = 0; r < kRowsU; ++r) {
      const float h = Hs[r][ty];
      const float4 z = *reinterpret_cast<const float4*>(&Zs[r][tx * 4]);
      acc[0] = fmaf(h, z.x, acc[0]); acc[1] = fmaf(h, z.y, acc[1]);
      acc[2] = fmaf(h, z.z, acc[2]); acc[3] = fmaf(h, z.w, acc[3]);
    }
  }
  const float lr_t = st->lr_t;
  float nw[4] = {0.0f, 0.0f, 0.0f, 0.0f};
  if (k <= L.K) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (tn0 + tx * 4 + j >= L.N) continue;
      float m, v;
      a.grad[p0 + j] = acc[j];
      adam_slots(acc[j], mo[j], ve[j], opt, m, v);
      a.m[p0 + j] = m;
      a.v[p0 + j] = v;
      nw[j] = adam_weight(th[j], m, v, opt, lr_t);
      a.theta[p0 + j] = nw[j];
    }
  }
  if (L.offT >= 0) {
    // theta_l^T [N][K] for the chain kernel's back-propagation, written with unit stride along k
    __syncthreads();
#pragma unroll
    for (int j = 0; j < 4; ++j) Hs[tx * 4 + j][ty] = nw[j];          // Hs[n][k]
    __syncthreads();
    float* T = a.thetaT + e * a.pnT + L.offT;
    for (int i = tid; i < kTileU * kTileU; i += kThreadsU) {
      const int n = i >> 5, kk = i & 31;
      if (tn0 + n < L.N && tk0 + kk < L.K) T[(int64_t)(tn0 + n) * L.K + tk0 + kk] = Hs[n][kk];
    }
  }
}

}   // namespace

namespace simba {

static size_t chain_smem_bytes(int tile_rows, int ld_act) {
  // weight ring + partial tiles [8 warps worth of (rows / groups) x 128] + two activation tiles
  return (size_t)(2 * kChunkK * kChunkN + kChainWarps * (tile_rows / chain_row_groups(tile_rows)) * kChunkN +
                  2 * tile_rows * ld_act) * sizeof(float);
}

// row stride of the chain's shared activation tiles: the widest layer, in whole float4s
static int act_stride(const TrainDesc& d) {
  int ld = 0;
  for (int l = 0; l <= d.L; ++l) ld = std::max(ld, (std::max(d.layer[l].K, d.layer[l].N) + 3) & ~3);
  return ld;
}

// the smallest row tile that keeps the grid within about one wave of SMs
static int chain_tile_rows(int ensemble, int grid_rows) {
  for (int R : {4, 8})
    if ((int64_t)ensemble * ((grid_rows + R - 1) / R) <= 160) return R;
  return 16;
}

// The image is theta^T: per member, layers 1..L as [N][K] row-major blocks, in layer order (layer 0 is never
// back-propagated through). Float offset of layer l's block; l = L + 1 gives a member's size.
static int64_t theta_t_offset(const TrainDesc& d, int l) {
  int64_t off = 0;
  for (int j = 1; j < l; ++j) off += (int64_t)d.layer[j].N * d.layer[j].K;
  return off;
}

int train_f32_check(const TrainDesc& d) {
  // largest variant (16-row tiles): weight ring + partial tiles + two activation tiles
  if (chain_smem_bytes(16, act_stride(d)) > 220 * 1024)
    return set_error(SIMBA_ERR_UNSUPPORTED, "units %d: activation tiles do not fit shared memory", d.layer[0].N);
  return SIMBA_OK;
}

int64_t train_f32_image_bytes(const TrainDesc& d) { return theta_t_offset(d, d.L + 1) * (int64_t)sizeof(float); }

void train_f32_pack(const TrainDesc& d, const float* theta, uint8_t* img) {
  for (int l = 1; l <= d.L; ++l) {
    const TrainLayer& ly = d.layer[l];
    const float* W = theta + ly.off;
    float* T = reinterpret_cast<float*>(img) + theta_t_offset(d, l);
    for (int k = 0; k < ly.K; ++k)
      for (int n = 0; n < ly.N; ++n) T[(size_t)n * ly.K + k] = W[(size_t)k * ly.N + n];
  }
}

cudaError_t train_f32_chain(const TrainDesc& d, const OptParams& opt, const FitDesc* desc, TrainState* st,
                            int grid_rows, int rows_fixed, int step_off, cudaStream_t s, int& row_tiles) {
  ChainArgs a{};
  int np = 0;
  for (int l = 0; l <= d.L; ++l) {
    const TrainLayer& ly = d.layer[l];
    ChainPass& p = a.pass[np++];
    p.w_off = ly.off;
    p.bias_off = ly.off + (int64_t)ly.K * ly.N;
    p.k_dim = ly.K; p.n_dim = ly.N;
    p.kind = l < d.L ? kPassHidden : kPassHead;
    p.out = l < d.L ? d.act[l + 1] : d.dz[l];
    p.out_estride = (l < d.L ? d.act_estride : d.dz_estride) * ly.N;
  }
  a.n_forward = np;
  if (d.train)
    for (int l = d.L; l >= 1; --l) {
      const TrainLayer& ly = d.layer[l];
      ChainPass& p = a.pass[np++];
      p.w_off = theta_t_offset(d, l);
      p.k_dim = ly.N; p.n_dim = ly.K;
      p.kind = kPassBackward;
      p.out = d.dz[l - 1]; p.out_estride = d.dz_estride * ly.K;      // K_l == N_{l-1}
      p.mask = d.act[l]; p.mask_estride = d.act_estride * ly.K;
    }
  a.n_pass = np;
  a.x = d.x; a.x_estride = d.x_estride; a.gather = d.gather;
  a.y = d.y; a.y_estride = d.y_estride;
  a.theta = d.theta; a.thetaT = reinterpret_cast<const float*>(d.img);
  a.pn = d.pn; a.pnT = d.img_member_bytes / (int64_t)sizeof(float);
  a.ld_act = act_stride(d); a.out_dim = d.out_dim; a.ensemble = d.ensemble;
  // forward chunk rows are N_l floats long, backward ones K_l = N_{l-1}
  a.aligned = 1;
  for (int l = 0; l <= d.L; ++l)
    if (d.layer[l].N % 4) a.aligned = 0;
  a.partial = d.partial; a.tiles_cap = d.tiles_cap; a.train = d.train; a.out_loss = d.out_loss;
  a.dropout_rate = d.dropout_rate; a.dropout_scale = d.dropout_scale; a.dropout_seed = d.dropout_seed;
  const int TR = chain_tile_rows(d.ensemble, grid_rows);
  auto kernel = TR == 4 ? train_chain_kernel<4> : TR == 8 ? train_chain_kernel<8> : train_chain_kernel<16>;
  const size_t smem = chain_smem_bytes(TR, a.ld_act);
  const cudaError_t err = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (err != cudaSuccess) return err;
  row_tiles = (grid_rows + TR - 1) / TR;
  kernel<<<dim3(row_tiles, d.ensemble), kChainThreads, smem, s>>>(a, opt, desc, st, rows_fixed, step_off);
  return cudaGetLastError();
}

cudaError_t train_f32_update(const TrainDesc& d, const OptParams& opt, const FitDesc* desc, const TrainState* st,
                             int rows_fixed, int step_off, cudaStream_t s) {
  UpdArgs u{};
  int tiles = 0;
  for (int l = 0; l <= d.L; ++l) {
    const TrainLayer& ly = d.layer[l];
    UpdLayer& U = u.layers[l];
    U.h = l == 0 ? d.x : d.act[l];
    U.h_estride = l == 0 ? d.x_estride : d.act_estride * ly.K;
    U.gather_h = l == 0 ? d.gather : 0;
    U.dz = d.dz[l];
    U.dz_estride = d.dz_estride * ly.N;
    U.off = ly.off; U.offT = l == 0 ? -1 : theta_t_offset(d, l); U.K = ly.K; U.N = ly.N;
    U.tile_begin = tiles;
    U.n_tiles_n = (ly.N + kTileU - 1) / kTileU;
    tiles += ((ly.K + 1 + kTileU - 1) / kTileU) * U.n_tiles_n;
  }
  u.n_layers = d.L + 1;
  u.theta = d.theta; u.thetaT = reinterpret_cast<float*>(d.img); u.m = d.m; u.v = d.v; u.grad = d.grad;
  u.pn = d.pn; u.pnT = d.img_member_bytes / (int64_t)sizeof(float); u.ensemble = d.ensemble;
  train_update_kernel<<<dim3(tiles, d.ensemble), kThreadsU, 0, s>>>(u, opt, desc, st, rows_fixed, step_off);
  return cudaGetLastError();
}

}  // namespace simba

#ifdef SIMBA_TRAIN_TIMELINE
extern "C" int simba_debug_train_timeline(long long* out) {
  SIMBA_CUDA_TRY(cudaDeviceSynchronize());
  SIMBA_CUDA_TRY(cudaMemcpyFromSymbol(out, g_train_tl, sizeof(long long) * 512));
  return SIMBA_OK;
}
#endif

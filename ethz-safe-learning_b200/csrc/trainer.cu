// Ensemble training step on the device (include/simba_b200.h "ensemble training step"):
// replaces MlpEnsemble.training_step / validation_step / fit's inner loop
// (simba/models/mlp_ensemble.py:134-187). fp32 throughout — the reference trains in fp32 and the
// planner's fp32 and bf16 weight images are both derived from these master weights. With
// precision = SIMBA_PREC_BF16_TC the handle below runs trainer_tc.cu's tcgen05 kernels instead, on the
// same master weights, Adam state, buffers and graphs.
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
#include <cstring>
#include <vector>

#include "common.cuh"
#include "internal.h"
#include "train_common.cuh"

using namespace simba;

namespace {

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
constexpr int kMaxTrainLayers = 18;
constexpr int kGraphSteps = 16;  // fit(): steps per CUDA-graph launch

__global__ void advance_kernel(TrainState* st, int n) {
  st->iterations += n;
  st->fit_step += n;
}

__global__ void set_fit_desc_kernel(FitDesc d, FitDesc* out, TrainState* st) {
  *out = d;
  st->fit_step = 0;
}

// ---- PTX wrappers: mbarrier + TMA bulk copy (cp.async.bulk) -----------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// bounded: a protocol bug must fault the kernel, never hang the GPU
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > (1u << 26)) __trap();
  }
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
      "l"(src), "r"(bytes), "r"(bar)
      : "memory");
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
      if (a.aligned) mbar_wait(smem_u32(&bars[q & 1]), (q >> 1) & 1);
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

static size_t chain_smem_bytes(int tile_rows, int ld_act) {
  // weight ring + partial tiles [8 warps worth of (rows / groups) x 128] + two activation tiles
  return (size_t)(2 * kChunkK * kChunkN + kChainWarps * (tile_rows / chain_row_groups(tile_rows)) * kChunkN +
                  2 * tile_rows * ld_act) * sizeof(float);
}


// ---------------------------------------------------------------------------------------------
// handle
// ---------------------------------------------------------------------------------------------
struct simba_trainer {
  simba_model_t* model = nullptr;
  simba_trainer_config_t cfg{};
  int E = 0, L = 0, U = 0, O = 0, IN = 0;
  int cap_rows = 0;
  int64_t pn = 0;
  int64_t pnT = 0;
  std::vector<int> off, offT, K, N;  // train layers 0..L (L = merged head); offT[0] = -1
  float *theta = nullptr, *thetaT = nullptr, *m = nullptr, *v = nullptr, *grad = nullptr;
  int ld_act = 0, aligned = 0;
  size_t chain_smem = 0;
  std::vector<float*> act;           // act[l]: input of train layer l (act[0] = gathered x)
  std::vector<float*> dz;            // dz[l]: gradient w.r.t. the pre-activation of train layer l
  float* partial = nullptr;
  int tiles_cap = 0;
  double* val_acc = nullptr;
  TrainState* state = nullptr;
  FitDesc* desc = nullptr;
  std::vector<int> tile_begin;       // update grid: first tile of each layer
  int n_upd_tiles = 0;
  // bf16 tcgen05 path (trainer_tc.cu): per member the layers' UMMA weight images, rebuilt by every update
  uint8_t* img = nullptr;
  int64_t img_member_bytes = 0;
  std::vector<TcLayer> tc;
  std::vector<int> tc_tile_begin;
  int tc_tiles = 0;
  cudaGraphExec_t fit_graph = nullptr;      // one training step
  cudaGraphExec_t fit_graph_n = nullptr;    // kGraphSteps consecutive steps (amortises the launch gap)
  cudaStream_t graph_stream = nullptr;
  int launches_per_step = 0;
};

static int chain_tile_rows(const simba_trainer_t* t, int grid_rows) {
  for (int R : {4, 8})
    if ((int64_t)t->E * ((grid_rows + R - 1) / R) <= 160) return R;
  return 16;
}

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
    kern.resize((size_t)t->K[l] * t->N[l]);
    bias.resize(t->N[l]);
    int rc = simba_model_get_layer(t->model, e, l, kern.data(), bias.data());
    if (rc) return rc;
    float* dst = theta_e + t->off[l];
    memcpy(dst, kern.data(), kern.size() * sizeof(float));
    memcpy(dst + kern.size(), bias.data(), bias.size() * sizeof(float));
  }
  const int U = t->U, O = t->O;
  kern.resize((size_t)U * O); bias.resize(O); kern2.resize((size_t)U * O); bias2.resize(O);
  int rc = simba_model_get_layer(t->model, e, t->L, kern.data(), bias.data());
  if (rc) return rc;
  rc = simba_model_get_layer(t->model, e, t->L + 1, kern2.data(), bias2.data());
  if (rc) return rc;
  float* dst = theta_e + t->off[t->L];
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
    const float* src = theta_e + t->off[layer];
    const size_t nk = (size_t)t->K[layer] * t->N[layer];
    memcpy(kernel, src, nk * sizeof(float));
    memcpy(bias, src + nk, t->N[layer] * sizeof(float));
    return;
  }
  const int U = t->U, O = t->O, c0 = layer == t->L ? 0 : 1;
  const float* src = theta_e + t->off[t->L];
  for (int k = 0; k < U; ++k)
    for (int o = 0; o < O; ++o) kernel[(size_t)k * O + o] = src[(size_t)k * 2 * O + 2 * o + c0];
  for (int o = 0; o < O; ++o) bias[o] = src[(size_t)U * 2 * O + 2 * o + c0];
}

extern "C" int simba_trainer_destroy(simba_trainer_t* t) {
  if (!t) return SIMBA_OK;
  if (t->fit_graph) cudaGraphExecDestroy(t->fit_graph);
  if (t->fit_graph_n) cudaGraphExecDestroy(t->fit_graph_n);
  if (t->graph_stream) cudaStreamDestroy(t->graph_stream);
  cudaFree(t->theta); cudaFree(t->thetaT); cudaFree(t->img); cudaFree(t->m); cudaFree(t->v); cudaFree(t->grad);
  for (float* p : t->act) cudaFree(p);
  for (float* p : t->dz) cudaFree(p);
  cudaFree(t->partial); cudaFree(t->val_acc);
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
  if (cfg->precision == SIMBA_PREC_BF16_TC &&
      !train_tc_supported(mc->obs_dim + mc->act_dim, mc->obs_dim, mc->n_layers, mc->units))
    return set_error(SIMBA_ERR_UNSUPPORTED,
                     "bf16 tcgen05 training covers units <= 416, obs_dim + act_dim <= 126, obs_dim <= 124 and "
                     "n_layers <= 6 (got units %d, obs_dim %d, act_dim %d, n_layers %d); precision fp32 trains "
                     "this shape",
                     mc->units, mc->obs_dim, mc->act_dim, mc->n_layers);
  int rc = simba_device_check();
  if (rc) return rc;
  if (mc->n_layers + 1 > kMaxTrainLayers)
    return set_error(SIMBA_ERR_UNSUPPORTED, "n_layers %d > %d", mc->n_layers, kMaxTrainLayers - 1);
  auto* t = new simba_trainer();
  t->model = model;
  t->cfg = *cfg;
  t->E = mc->ensemble_size; t->L = mc->n_layers; t->U = mc->units; t->O = mc->obs_dim;
  t->IN = mc->obs_dim + mc->act_dim;
  t->cap_rows = cfg->max_eval_rows > cfg->batch_size ? cfg->max_eval_rows : cfg->batch_size;
  int64_t off = 0;
  for (int l = 0; l <= t->L; ++l) {
    const int K = l == 0 ? t->IN : t->U;
    const int N = l < t->L ? t->U : 2 * t->O;
    t->K.push_back(K); t->N.push_back(N); t->off.push_back((int)off);
    off += (int64_t)(K + 1) * N;
    t->offT.push_back(l == 0 ? -1 : (int)t->pnT);
    if (l > 0) t->pnT += (int64_t)N * K;
    t->ld_act = std::max(t->ld_act, (std::max(K, N) + 3) & ~3);
  }
  t->pn = off;
  t->aligned = (t->U % 4 == 0 && (2 * t->O) % 4 == 0) ? 1 : 0;
  // largest variant (16-row tiles): weight ring + partial tiles + two activation tiles
  t->chain_smem = chain_smem_bytes(16, t->ld_act);
  if (t->chain_smem > 220 * 1024) {
    const int units = t->U;
    delete t;
    return set_error(SIMBA_ERR_UNSUPPORTED, "units %d: activation tiles do not fit shared memory", units);
  }
  const int E = t->E;
  std::vector<float> host((size_t)E * t->pn);
  for (int e = 0; e < E; ++e) {
    rc = pull_member(t, e, host.data() + (size_t)e * t->pn);
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
  const size_t pbytes = (size_t)E * t->pn * sizeof(float);
  TRY_OR_FREE(cudaMalloc(&t->theta, pbytes));
  TRY_OR_FREE(cudaMalloc(&t->m, pbytes));
  TRY_OR_FREE(cudaMalloc(&t->v, pbytes));
  TRY_OR_FREE(cudaMalloc(&t->grad, pbytes));
  TRY_OR_FREE(cudaMemcpy(t->theta, host.data(), pbytes, cudaMemcpyHostToDevice));
  {
    std::vector<float> hostT((size_t)E * std::max<int64_t>(t->pnT, 1));
    for (int e = 0; e < E; ++e)
      for (int l = 1; l <= t->L; ++l) {
        const float* W = host.data() + (size_t)e * t->pn + t->off[l];
        float* T = hostT.data() + (size_t)e * t->pnT + t->offT[l];
        for (int k = 0; k < t->K[l]; ++k)
          for (int n = 0; n < t->N[l]; ++n) T[(size_t)n * t->K[l] + k] = W[(size_t)k * t->N[l] + n];
      }
    TRY_OR_FREE(cudaMalloc(&t->thetaT, hostT.size() * sizeof(float)));
    TRY_OR_FREE(cudaMemcpy(t->thetaT, hostT.data(), hostT.size() * sizeof(float), cudaMemcpyHostToDevice));
  }
  if (cfg->precision == SIMBA_PREC_BF16_TC) {
    for (int l = 0; l <= t->L; ++l) t->tc.push_back(TcLayer{t->K[l], t->N[l], t->off[l], 0, 0});
    t->img_member_bytes = train_tc_layout(t->tc.data(), t->L + 1);
    std::vector<uint8_t> img((size_t)E * t->img_member_bytes, 0);
    for (int e = 0; e < E; ++e)
      train_tc_pack(t->tc.data(), t->L + 1, host.data() + (size_t)e * t->pn, img.data() + (size_t)e * t->img_member_bytes);
    TRY_OR_FREE(cudaMalloc(&t->img, img.size()));
    TRY_OR_FREE(cudaMemcpy(t->img, img.data(), img.size(), cudaMemcpyHostToDevice));
    for (int l = 0; l <= t->L; ++l) {
      t->tc_tile_begin.push_back(t->tc_tiles);
      t->tc_tiles += train_tc_update_tiles(t->tc[l]);
    }
  }
  TRY_OR_FREE(cudaFuncSetAttribute(train_chain_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   (int)chain_smem_bytes(4, t->ld_act)));
  TRY_OR_FREE(cudaFuncSetAttribute(train_chain_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   (int)chain_smem_bytes(8, t->ld_act)));
  TRY_OR_FREE(cudaFuncSetAttribute(train_chain_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   (int)chain_smem_bytes(16, t->ld_act)));
  TRY_OR_FREE(cudaMemset(t->m, 0, pbytes));
  TRY_OR_FREE(cudaMemset(t->v, 0, pbytes));
  TRY_OR_FREE(cudaMemset(t->grad, 0, pbytes));
  const size_t R = t->cap_rows;
  t->act.assign(t->L + 1, nullptr);
  t->dz.assign(t->L + 1, nullptr);
  for (int l = 0; l <= t->L; ++l) {
    TRY_OR_FREE(cudaMalloc(&t->act[l], (size_t)E * R * t->K[l] * sizeof(float)));
    TRY_OR_FREE(cudaMalloc(&t->dz[l], (size_t)E * cfg->batch_size * t->N[l] * sizeof(float)));
  }
  t->tiles_cap = (int)((R + 3) / 4);                    // smallest row tile
  TRY_OR_FREE(cudaMalloc(&t->partial, (size_t)E * t->tiles_cap * 2 * sizeof(float)));
  TRY_OR_FREE(cudaMalloc(&t->val_acc, (size_t)E * 2 * sizeof(double)));
  TRY_OR_FREE(cudaMalloc(&t->state, sizeof(TrainState)));
  TRY_OR_FREE(cudaMemset(t->state, 0, sizeof(TrainState)));
  TRY_OR_FREE(cudaMalloc(&t->desc, sizeof(FitDesc)));
  TRY_OR_FREE(cudaMemset(t->desc, 0, sizeof(FitDesc)));
  for (int l = 0; l <= t->L; ++l) {
    t->tile_begin.push_back(t->n_upd_tiles);
    t->n_upd_tiles += ((t->K[l] + 1 + kTileU - 1) / kTileU) * ((t->N[l] + kTileU - 1) / kTileU);
  }
#undef TRY_OR_FREE
  t->launches_per_step = 2;
  *out = t;
  return SIMBA_OK;
}

// the chain kernel: forward + likelihood (+ back-propagation of the activations when `train`).
// x may be shared by the members (estride 0, validation) or gathered through the fit descriptor.
static int enqueue_chain(simba_trainer_t* t, const float* x, int64_t x_estride, const float* y,
                         int64_t y_estride, int gather, int grid_rows, int rows_fixed,
                         const FitDesc* desc, int train, float* out_loss, int step_off,
                         cudaStream_t s) {
  const int64_t R = t->cap_rows, B = t->cfg.batch_size;
  if (t->cfg.precision == SIMBA_PREC_BF16_TC) {
    TcChainArgs a{};
    for (int l = 0; l <= t->L; ++l) {
      a.layer[l] = t->tc[l];
      a.act[l] = t->act[l];
      a.dz[l] = t->dz[l];
    }
    a.L = t->L;
    a.act_estride = R; a.dz_estride = B;
    a.x = x; a.x_estride = x_estride; a.gather = gather;
    a.y = y; a.y_estride = y_estride;
    a.img = t->img; a.img_member_bytes = t->img_member_bytes;
    a.out_dim = t->O; a.ensemble = t->E;
    a.partial = t->partial; a.tiles_cap = t->tiles_cap; a.train = train; a.out_loss = out_loss;
    a.dropout_rate = t->cfg.dropout_rate;
    a.dropout_scale = 1.0f / (1.0f - t->cfg.dropout_rate);
    a.dropout_seed = t->cfg.dropout_seed;
    SIMBA_CUDA_TRY(train_tc_chain(a, opt_params(t), desc, t->state, grid_rows, rows_fixed, step_off, s));
    return SIMBA_OK;
  }
  ChainArgs a{};
  int np = 0;
  for (int l = 0; l <= t->L; ++l) {
    ChainPass& p = a.pass[np++];
    p.w_off = t->off[l];
    p.bias_off = t->off[l] + (int64_t)t->K[l] * t->N[l];
    p.k_dim = t->K[l]; p.n_dim = t->N[l];
    p.kind = l < t->L ? kPassHidden : kPassHead;
    p.out = l < t->L ? t->act[l + 1] : t->dz[l];
    p.out_estride = l < t->L ? R * t->N[l] : B * t->N[l];
  }
  a.n_forward = np;
  if (train)
    for (int l = t->L; l >= 1; --l) {
      ChainPass& p = a.pass[np++];
      p.w_off = t->offT[l];
      p.k_dim = t->N[l]; p.n_dim = t->K[l];
      p.kind = kPassBackward;
      p.out = t->dz[l - 1]; p.out_estride = B * t->K[l];      // K_l == N_{l-1}
      p.mask = t->act[l]; p.mask_estride = R * t->K[l];
    }
  a.n_pass = np;
  a.x = x; a.x_estride = x_estride; a.gather = gather;
  a.y = y; a.y_estride = y_estride;
  a.theta = t->theta; a.thetaT = t->thetaT; a.pn = t->pn; a.pnT = t->pnT;
  a.ld_act = t->ld_act; a.out_dim = t->O; a.ensemble = t->E; a.aligned = t->aligned;
  a.partial = t->partial; a.tiles_cap = t->tiles_cap; a.train = train; a.out_loss = out_loss;
  a.dropout_rate = t->cfg.dropout_rate;
  a.dropout_scale = 1.0f / (1.0f - t->cfg.dropout_rate);
  a.dropout_seed = t->cfg.dropout_seed;
  // the smallest row tile that keeps the grid within about one wave of SMs
  const int TR = chain_tile_rows(t, grid_rows);
  dim3 grid((grid_rows + TR - 1) / TR, t->E);
  const size_t smem = chain_smem_bytes(TR, t->ld_act);
  const OptParams opt = opt_params(t);
  if (TR == 4)
    train_chain_kernel<4><<<grid, kChainThreads, smem, s>>>(a, opt, desc, t->state, rows_fixed, step_off);
  else if (TR == 8)
    train_chain_kernel<8><<<grid, kChainThreads, smem, s>>>(a, opt, desc, t->state, rows_fixed, step_off);
  else
    train_chain_kernel<16><<<grid, kChainThreads, smem, s>>>(a, opt, desc, t->state, rows_fixed, step_off);
  SIMBA_CUDA_TRY(cudaGetLastError());
  return SIMBA_OK;
}

static int enqueue_step(simba_trainer_t* t, const float* x, int64_t x_estride, const float* y,
                        int64_t y_estride, int rows_fixed, const FitDesc* desc, float* out_loss,
                        int step_off, cudaStream_t s) {
  const int64_t R = t->cap_rows, B = t->cfg.batch_size;
  const int gather = desc ? 1 : 0;
  const int grid_rows = desc ? t->cfg.batch_size : rows_fixed;
  int rc = enqueue_chain(t, x, x_estride, y, y_estride, gather, grid_rows, rows_fixed, desc, 1,
                         out_loss, step_off, s);
  if (rc) return rc;
  if (t->cfg.precision == SIMBA_PREC_BF16_TC) {
    TcUpdArgs u{};
    for (int l = 0; l <= t->L; ++l) {
      u.layer[l] = t->tc[l];
      u.tile_begin[l] = t->tc_tile_begin[l];
      u.n_tiles_n[l] = (t->N[l] + 127) / 128;
      u.h[l] = l == 0 ? x : t->act[l];
      u.h_estride[l] = l == 0 ? x_estride : R * t->K[l];
      u.dz[l] = t->dz[l];
    }
    u.n_layers = t->L + 1;
    u.gather0 = gather;
    u.dz_estride = B;
    u.theta = t->theta; u.m = t->m; u.v = t->v; u.grad = t->grad; u.pn = t->pn;
    u.img = t->img; u.img_member_bytes = t->img_member_bytes; u.ensemble = t->E;
    SIMBA_CUDA_TRY(train_tc_update(u, opt_params(t), desc, t->state, t->tc_tiles, rows_fixed, step_off, s));
    return SIMBA_OK;
  }
  UpdArgs u{};
  for (int l = 0; l <= t->L; ++l) {
    UpdLayer& U = u.layers[l];
    U.h = l == 0 ? x : t->act[l];
    U.h_estride = l == 0 ? x_estride : R * t->K[l];
    U.gather_h = l == 0 ? gather : 0;
    U.dz = t->dz[l];
    U.dz_estride = B * t->N[l];
    U.off = t->off[l]; U.offT = t->offT[l]; U.K = t->K[l]; U.N = t->N[l];
    U.tile_begin = t->tile_begin[l];
    U.n_tiles_n = (t->N[l] + kTileU - 1) / kTileU;
  }
  u.n_layers = t->L + 1;
  u.theta = t->theta; u.thetaT = t->thetaT; u.m = t->m; u.v = t->v; u.grad = t->grad;
  u.pn = t->pn; u.pnT = t->pnT; u.ensemble = t->E;
  train_update_kernel<<<dim3(t->n_upd_tiles, t->E), kThreadsU, 0, s>>>(u, opt_params(t), desc,
                                                                        t->state, rows_fixed, step_off);
  SIMBA_CUDA_TRY(cudaGetLastError());
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
    int rc = enqueue_chain(t, x + r0 * t->IN, 0, y + r0 * t->O, 0, 0, nr, nr, nullptr, 0, nullptr, 0, s);
    if (rc) return rc;
    const int R = t->cfg.precision == SIMBA_PREC_BF16_TC ? kTcRows : chain_tile_rows(t, nr);
    const int tiles = (nr + R - 1) / R;
    val_accumulate_kernel<<<1, 32, 0, s>>>(t->partial, t->tiles_cap, tiles, t->E, t->val_acc,
                                           r0 == 0 ? 1 : 0);
  }
  val_finalize_kernel<<<1, 1, 0, s>>>(t->val_acc, t->E, (double)rows * t->O, out_loss);
  SIMBA_CUDA_TRY(cudaGetLastError());
  return SIMBA_OK;
}

extern "C" int simba_trainer_sync_model(simba_trainer_t* t, void* stream) {
  if (!t) return set_error(SIMBA_ERR_BAD_CONFIG, "null argument");
  std::vector<float> host((size_t)t->E * t->pn);
  SIMBA_CUDA_TRY(cudaMemcpyAsync(host.data(), t->theta, host.size() * sizeof(float),
                                 cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  SIMBA_CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));
  std::vector<float> kern, bias;
  for (int e = 0; e < t->E; ++e)
    for (int layer = 0; layer < t->L + 2; ++layer) {
      const int K = layer == 0 ? t->IN : t->U, N = layer < t->L ? t->U : t->O;
      kern.resize((size_t)K * N);
      bias.resize(N);
      split_layer(t, host.data() + (size_t)e * t->pn, layer, kern.data(), bias.data());
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
  const float* src = which == 0 ? t->theta : which == 1 ? t->grad : which == 2 ? t->m : t->v;
  std::vector<float> host(t->pn);
  SIMBA_CUDA_TRY(cudaDeviceSynchronize());
  SIMBA_CUDA_TRY(cudaMemcpy(host.data(), src + (size_t)member * t->pn, t->pn * sizeof(float),
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

#ifdef SIMBA_TRAIN_TIMELINE
extern "C" int simba_debug_train_timeline(long long* out) {
  SIMBA_CUDA_TRY(cudaDeviceSynchronize());
  SIMBA_CUDA_TRY(cudaMemcpyFromSymbol(out, g_train_tl, sizeof(long long) * 512));
  return SIMBA_OK;
}
#endif

extern "C" int simba_trainer_launches_per_step(simba_trainer_t* t) {
  return t ? t->launches_per_step : 0;
}

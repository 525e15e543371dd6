// bf16 tcgen05 ensemble training step (simba_trainer_config_t.precision = SIMBA_PREC_BF16_TC): the same
// contract as trainer.cu's fp32 kernels — forward with dropout, Gaussian NLL and its gradient, activation
// back-propagation, weight gradients, clip and Adam on fp32 master weights — with every GEMM on the tensor
// cores (bf16 operands, fp32 accumulation in tensor memory). Two launches per step, captured in the same
// 16-step graphs as the fp32 path.
//
//   chain   one CTA per (member, 128-row batch tile), 4 warps; thread r owns batch row r = TMEM lane r.
//           Passes: layers 0..L-1 (hidden), L (head), then back-propagation L..1. Each pass is one GEMM
//           D[128 x N] = A[128 x K] . B[N x K]^T: A (the activations, bf16) sits in shared memory, B (the
//           layer's bf16 image) streams from L2 in 64-wide K chunks through a two-stage cp.async.bulk ring
//           (full / empty mbarriers). One elected lane issues the copies and the tcgen05.mma's (N > 256 is
//           two MMAs of N/2) and commits the accumulator onto an mbarrier; all four warps then drain their
//           rows from TMEM and run the pass's epilogue in fp32:
//             hidden    relu, dropout (trainer Philox stream 4, train_common.cuh), H_{l+1} -> global for the
//                       update kernel, bf16 into the A tile with the constant ones of the bias columns
//             head      NLL partials, d(mu), d(raw var) (accurate libm math, train_common.cuh) -> dZ_L
//             backward  dZ_{l-1} = relu'(H_l) * (dZ_l . theta_l^T), the mask read back from H_l
//           The next pass's A operand overwrites the tile in place: its MMAs have all retired.
//   update  one CTA per (member, layer, 128-row tile of theta, 128-column tile): dtheta = [H, 1]^T . dZ on
//           tcgen05 with the batch as the MMA's K, accumulated over every batch row in order (no atomics:
//           bit-reproducible), then clip + Adam in fp32 (train_common.cuh) and the two bf16 images.
//
// Operand majorness: every operand here is K-major SWIZZLE_NONE. The weight-gradient GEMM reduces over
// the batch, so its operands are H^T and dZ^T; rather than set the instruction descriptor's transpose bits
// (MN-major operands) the update kernel's staging threads, which already convert fp32 -> bf16, insert the
// bias row of ones and follow fit()'s gather, write the transposed core matrices directly. Every MMA of
// the trainer therefore uses the one descriptor form (`desc_kmajor`), and no kernel writes a second global
// layout of the activations.
#include <algorithm>

#include "common.cuh"
#include "internal.h"
#include "tc_ptx.cuh"
#include "train_common.cuh"

namespace {

constexpr int kThreads = 128;
constexpr int kChunkK = 64;           // K elements per streamed weight chunk
constexpr int kGroupBytes = 2048;     // one 8-wide K group of the 128-row A tile
constexpr int kUpdRows = 64;          // batch rows per staged chunk of the update kernel
constexpr int kUpdTile = 128;         // update tile: [128 k] x [128 n]
constexpr int kGStride = kUpdTile + 1;
constexpr int kAdamBatch = 8;        // update epilogue: elements per thread in flight together

__host__ __device__ inline int r16(int x) { return (x + 15) & ~15; }

// K-major SWIZZLE_NONE descriptor: core matrices 128 B, `lbo` between K groups, `sbo` between 8-row groups
__device__ __forceinline__ uint64_t desc_kmajor(uint32_t addr, uint32_t lbo, uint32_t sbo) {
  uint64_t d = 0;
  d |= (uint64_t)((addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)((lbo >> 4) & 0x3FFFu) << 16;
  d |= (uint64_t)((sbo >> 4) & 0x3FFFu) << 32;
  d |= (uint64_t)1 << 46;
  return d;
}

// pass p of the chain: forward layers 0..L (L = head), then backward layers L..1
struct PassGeom {
  int layer, kind;          // kind 0 hidden, 1 head, 2 backward
  int np, kp;               // MMA N (rows of the image), MMA K (columns)
  int64_t img_off;
};
__device__ __forceinline__ PassGeom pass_geom(const TcChainArgs& a, int p) {
  PassGeom g;
  if (p <= a.L) {
    const TcLayer& l = a.layer[p];
    g.layer = p; g.kind = p < a.L ? 0 : 1;
    g.np = r16(l.N); g.kp = r16(l.K + 2); g.img_off = l.fwd_off;
  } else {
    const int li = 2 * a.L + 1 - p;
    const TcLayer& l = a.layer[li];
    g.layer = li; g.kind = 2;
    g.np = r16(l.K); g.kp = r16(l.N); g.img_off = l.bwd_off;
  }
  return g;
}

__device__ __forceinline__ uint32_t pack2(float lo, float hi) { return pack_bf16(lo, hi); }

// 8 bf16 of the A tile: K group `kg` of row r
__device__ __forceinline__ void store_a8(uint32_t a_base, int kg, int r, const float* v) {
  st_shared_v4(a_base + (uint32_t)kg * kGroupBytes + (uint32_t)(r >> 3) * 128u + (uint32_t)(r & 7) * 16u,
               pack2(v[0], v[1]), pack2(v[2], v[3]), pack2(v[4], v[5]), pack2(v[6], v[7]));
}

}  // namespace

namespace simba {
namespace {

__global__ void __launch_bounds__(kThreads, 1)
train_tc_chain_kernel(const TcChainArgs a, const OptParams opt, const FitDesc* desc, TrainState* st,
                      int rows_fixed, int step_off, int n_pass, uint32_t stage_bytes, uint32_t a_bytes,
                      uint32_t tmem_cols) {
  extern __shared__ __align__(1024) uint8_t smem[];
  __shared__ __align__(8) uint64_t bars[5];      // full[2], empty[2], accumulator
  __shared__ uint32_t tmem_slot;
  __shared__ float scratch[kThreads / 32];
  __shared__ bool last;
  const int rows = resolve_rows(desc, st, rows_fixed, step_off);
  const int e = blockIdx.y, r0 = blockIdx.x * kTcRows;
  const int tid = threadIdx.x, warp = tid >> 5;
  const int r = tid, rg = r0 + r;
  const bool row_ok = rg < rows;
  float s_log = 0.0f, s_sq = 0.0f;

  if (r0 < rows) {
    const uint32_t a_base = smem_u32(smem);
    const uint32_t stage0 = a_base + a_bytes;
    const uint32_t full0 = smem_u32(&bars[0]), empty0 = smem_u32(&bars[2]);   // stage s: + 8 s
    const uint32_t acc_bar = smem_u32(&bars[4]);
    if (tid == 0) {
      for (int i = 0; i < 5; ++i) mbar_init(smem_u32(&bars[i]), 1);
      fence_barrier_init();
    }
    if (warp == 0) tmem_alloc(smem_u32(&tmem_slot), tmem_cols);
    const uint8_t* img = a.img + (int64_t)e * a.img_member_bytes;
    const int* gidx = a.gather ? batch_rows_of(desc, st, e, a.ensemble, step_off) : nullptr;

    // layer-0 input: this row of the batch, ones at k = K_0, K_0 + 1, zeros up to the padded K
    {
      const int K0 = a.layer[0].K, kp0 = r16(K0 + 2);
      const float* xr = nullptr;
      if (row_ok) xr = gidx ? desc->inputs + (int64_t)gidx[rg] * K0 : a.x + e * a.x_estride + (int64_t)rg * K0;
      for (int kg = 0; kg < kp0 / 8; ++kg) {
        float v[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int k = kg * 8 + i;
          v[i] = k < K0 ? (row_ok ? __ldg(xr + k) : 0.0f) : (k < K0 + 2 ? 1.0f : 0.0f);
        }
        store_a8(a_base, kg, r, v);
      }
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_slot;
    const uint32_t t_row = tmem_base + ((uint32_t)(warp * 32) << 16);

    // chunk g of the whole chain -> stage g % 2 (issued by the elected lane of warp 0)
    auto issue = [&](int g, const PassGeom& pg, int c) {
      const int s = g & 1;
      if (g >= 2) mbar_wait(empty0 + 8u * s, ((g >> 1) - 1) & 1);
      const int kc = min(kChunkK, pg.kp - c * kChunkK);
      const uint32_t bytes = (uint32_t)kc * (uint32_t)pg.np * 2u;
      mbar_expect_tx(full0 + 8u * s, bytes);
      bulk_g2s(stage0 + (uint32_t)s * stage_bytes, img + pg.img_off + (int64_t)c * kChunkK * pg.np * 2, bytes,
               full0 + 8u * s);
    };
    if (warp == 0) {
      if (elect_one()) issue(0, pass_geom(a, 0), 0);
      __syncwarp();
    }
    const float c_nll = 1.0f / ((float)rows * (float)a.out_dim * (float)a.ensemble);
    const bool dropout = a.train && a.dropout_rate > 0.0f;
    const uint32_t iteration = (uint32_t)(st->iterations + step_off);
    int g0 = 0;                                   // first chunk of the current pass
    for (int p = 0; p < n_pass; ++p) {
      const PassGeom pg = pass_geom(a, p);
      const int nch = (pg.kp + kChunkK - 1) / kChunkK;
      if (warp == 0) {
        if (elect_one()) {
          const int N1 = pg.np <= 256 ? pg.np : r16(pg.np / 2), N2 = pg.np - N1;
          const uint32_t idesc1 = umma_idesc_n((uint32_t)N1), idesc2 = N2 > 0 ? umma_idesc_n((uint32_t)N2) : 0u;
          const uint32_t lbo_b = (uint32_t)pg.np * 16u;
          for (int c = 0; c < nch; ++c) {
            const int g = g0 + c, s = g & 1;
            mbar_wait(full0 + 8u * s, (g >> 1) & 1);
            tc_fence_after();
            const int ksteps = min(kChunkK, pg.kp - c * kChunkK) / 16;
            const uint32_t b0 = stage0 + (uint32_t)s * stage_bytes;
            for (int t = 0; t < ksteps; ++t) {
              const int kg = (c * kChunkK + t * 16) / 8;
              const uint64_t ad = desc_kmajor(a_base + (uint32_t)kg * kGroupBytes, kGroupBytes, 128u);
              const uint32_t bt = b0 + (uint32_t)t * 2u * lbo_b;
              const uint32_t acc = (c > 0 || t > 0) ? 1u : 0u;
              umma_bf16(tmem_base, ad, desc_kmajor(bt, lbo_b, 128u), idesc1, acc);
              if (N2 > 0)
                umma_bf16(tmem_base + (uint32_t)N1, ad, desc_kmajor(bt + (uint32_t)N1 * 16u, lbo_b, 128u), idesc2,
                          acc);
            }
            umma_commit(empty0 + 8u * s);
            // the next chunk of the chain (this pass or the first of the next) lands while these MMAs run
            if (c + 1 < nch) issue(g + 1, pg, c + 1);
            else if (p + 1 < n_pass) issue(g + 1, pass_geom(a, p + 1), 0);
          }
          umma_commit(acc_bar);
        }
        __syncwarp();
      }
      g0 += nch;
      mbar_wait(acc_bar, (uint32_t)p & 1u);
      tc_fence_after();

      const TcLayer& ly = a.layer[pg.layer];
      if (pg.kind == 0) {
        // ---- hidden layer: relu, dropout, H_{l+1} out, bf16 A tile (ones at N, N + 1) ----
        const int N = ly.N, kp_next = r16(N + 2);
        float* hout = a.act[pg.layer + 1] + ((int64_t)e * a.act_estride + rg) * N;
        for (int c0 = 0; c0 < kp_next; c0 += 16) {
          uint32_t v[16];
          if (c0 < pg.np) {
            tmem_ld<16>(t_row + (uint32_t)c0, v);
            tmem_ld_wait();
          }
          float h[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) h[j] = (c0 + j < N) ? fmaxf(__uint_as_float(v[j]), 0.0f) : 0.0f;
          if (dropout) {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              if (c0 + 4 * q >= N) continue;
              float keep[4];
              dropout_keep4(c0 + 4 * q, rg, iteration, e, pg.layer, a.dropout_rate, a.dropout_scale,
                            a.dropout_seed, keep);
#pragma unroll
              for (int i = 0; i < 4; ++i) h[4 * q + i] *= keep[i];
            }
          }
          if (a.train && row_ok) {
#pragma unroll
            for (int j = 0; j < 16; ++j)
              if (c0 + j < N) hout[c0 + j] = h[j];
          }
#pragma unroll
          for (int j = 0; j < 16; ++j)
            if (c0 + j == N || c0 + j == N + 1) h[j] = 1.0f;
          store_a8(a_base, c0 / 8, r, h);
          store_a8(a_base, c0 / 8 + 1, r, h + 8);
        }
      } else if (pg.kind == 1) {
        // ---- Gaussian head: columns interleave (mu_o, raw var_o); NLL partials and dZ_L ----
        const int N = ly.N;
        const float* yr = nullptr;
        if (row_ok)
          yr = gidx ? desc->targets + (int64_t)gidx[rg] * a.out_dim : a.y + e * a.y_estride + (int64_t)rg * a.out_dim;
        float* dzo = a.dz[a.L] + ((int64_t)e * a.dz_estride + rg) * N;
        for (int c0 = 0; c0 < pg.np; c0 += 16) {
          uint32_t v[16];
          tmem_ld<16>(t_row + (uint32_t)c0, v);
          tmem_ld_wait();
          float d[16];
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            float d_mu = 0.0f, d_pre = 0.0f;
            if (c0 + 2 * i < N && row_ok)
              nll_terms(__uint_as_float(v[2 * i]), __uint_as_float(v[2 * i + 1]), __ldg(yr + (c0 / 2 + i)), c_nll,
                        s_log, s_sq, d_mu, d_pre);
            d[2 * i] = d_mu;
            d[2 * i + 1] = d_pre;
          }
          if (a.train) {
            if (row_ok) {
#pragma unroll
              for (int j = 0; j < 16; ++j)
                if (c0 + j < N) dzo[c0 + j] = d[j];
            }
            store_a8(a_base, c0 / 8, r, d);
            store_a8(a_base, c0 / 8 + 1, r, d + 8);
          }
        }
      } else {
        // ---- back-propagation through layer l >= 1: dZ_{l-1} = relu'(H_l) * (dZ_l . theta_l^T) ----
        const int K = ly.K, l = pg.layer;
        const float back = dropout ? a.dropout_scale : 1.0f;  // H > 0 <=> active AND kept (stored after dropout)
        const float* hm = a.act[l] + ((int64_t)e * a.act_estride + rg) * K;
        float* dzo = a.dz[l - 1] + ((int64_t)e * a.dz_estride + rg) * K;
        for (int c0 = 0; c0 < pg.np; c0 += 16) {
          uint32_t v[16];
          tmem_ld<16>(t_row + (uint32_t)c0, v);
          tmem_ld_wait();
          float d[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const int k = c0 + j;
            d[j] = (k < K && row_ok && hm[k] > 0.0f) ? __uint_as_float(v[j]) * back : 0.0f;
          }
          if (row_ok) {
#pragma unroll
            for (int j = 0; j < 16; ++j)
              if (c0 + j < K) dzo[c0 + j] = d[j];
          }
          if (l > 1) {
            store_a8(a_base, c0 / 8, r, d);
            store_a8(a_base, c0 / 8 + 1, r, d + 8);
          }
        }
      }
      fence_proxy_async();                        // the new A tile -> visible to the next pass's MMAs
      tc_fence_before();
      __syncthreads();
      tc_fence_after();
    }
    if (warp == 0) tmem_dealloc(tmem_base, tmem_cols);
  }
  finish_chain_loss(s_log, s_sq, scratch, last, a.partial, a.tiles_cap, (rows + kTcRows - 1) / kTcRows, rows,
                    a.out_dim, a.ensemble, a.train, a.out_loss, opt, desc, st, step_off);
}

// dtheta tile [128 k] x [128 n] of one layer = [H, 1]^T . dZ over every batch row, then clip + Adam and the
// bf16 images of the new weights
__global__ void __launch_bounds__(kThreads)
train_tc_update_kernel(const TcUpdArgs a, const OptParams opt, const FitDesc* desc, const TrainState* st,
                       int rows_fixed, int step_off) {
  extern __shared__ __align__(1024) uint8_t smem[];
  __shared__ __align__(8) uint64_t mma_bar;
  __shared__ uint32_t tmem_slot;
  const int rows = resolve_rows(desc, st, rows_fixed, step_off);
  int li = 0;
#pragma unroll 1
  while (li + 1 < a.n_layers && (int)blockIdx.x >= a.tile_begin[li + 1]) ++li;
  const TcLayer& L = a.layer[li];
  const int t_in = blockIdx.x - a.tile_begin[li];
  const int m0 = (t_in / a.n_tiles_n[li]) * kUpdTile, n0 = (t_in % a.n_tiles_n[li]) * kUpdTile;
  const int K = L.K, N = L.N;
  const int nn = min(kUpdTile, N - n0), nnp = r16(nn);
  const int mrows = min(kUpdTile, K + 1 - m0);
  const int e = blockIdx.y;
  const int tid = threadIdx.x, warp = tid >> 5;
  uint8_t* a_sm = smem;                                    // [128 m] x [64 rows] bf16
  uint8_t* b_sm = smem + kUpdTile * kUpdRows * 2;          // [nnp n] x [64 rows] bf16
  float* G = reinterpret_cast<float*>(b_sm + kUpdTile * kUpdRows * 2);   // [128][129] fp32
  const uint32_t a_base = smem_u32(a_sm), b_base = smem_u32(b_sm), bar = smem_u32(&mma_bar);
  if (tid == 0) {
    mbar_init(bar, 1);
    fence_barrier_init();
  }
  if (warp == 0) tmem_alloc(smem_u32(&tmem_slot), kUpdTile);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_slot;
  const float* H = a.h[li] + e * a.h_estride[li];
  const float* dZ = a.dz[li] + (int64_t)e * a.dz_estride * N;
  const int* gidx = (li == 0 && a.gather0) ? batch_rows_of(desc, st, e, a.ensemble, step_off) : nullptr;
  const int k = m0 + tid;                                  // staging: this thread's row of theta / column of dZ
  const int nc = n0 + tid;
  int chunk = 0;
  for (int rb = 0; rb < rows; rb += kUpdRows, ++chunk) {
    const int nr = min(kUpdRows, rows - rb);
    for (int j = 0; j < kUpdRows / 8; ++j) {
      float hv[8], zv[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int row = rb + j * 8 + i;
        float h = 0.0f, z = 0.0f;
        if (j * 8 + i < nr) {
          if (k < K) {
            const float* hr = gidx ? desc->inputs + (int64_t)gidx[row] * K : H + (int64_t)row * K;
            h = __ldcg(hr + k);
          } else if (k == K) {
            h = 1.0f;                                       // the bias row
          }
          if (tid < nn) z = __ldcg(dZ + (int64_t)row * N + nc);
        }
        hv[i] = h;
        zv[i] = z;
      }
      st_shared_v4(a_base + (uint32_t)j * kGroupBytes + (uint32_t)(tid >> 3) * 128u + (uint32_t)(tid & 7) * 16u,
                   pack2(hv[0], hv[1]), pack2(hv[2], hv[3]), pack2(hv[4], hv[5]), pack2(hv[6], hv[7]));
      if (tid < nnp)
        st_shared_v4(b_base + (uint32_t)j * (uint32_t)nnp * 16u + (uint32_t)(tid >> 3) * 128u + (uint32_t)(tid & 7) * 16u,
                     pack2(zv[0], zv[1]), pack2(zv[2], zv[3]), pack2(zv[4], zv[5]), pack2(zv[6], zv[7]));
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (warp == 0) {
      if (elect_one()) {
        const uint32_t idesc = umma_idesc_n((uint32_t)nnp);
        const int ksteps = (nr + 15) / 16;
        for (int t = 0; t < ksteps; ++t)
          umma_bf16(tmem_base, desc_kmajor(a_base + (uint32_t)t * 2u * kGroupBytes, kGroupBytes, 128u),
                    desc_kmajor(b_base + (uint32_t)t * 2u * (uint32_t)nnp * 16u, (uint32_t)nnp * 16u, 128u), idesc,
                    (rb > 0 || t > 0) ? 1u : 0u);
        umma_commit(bar);
      }
      __syncwarp();
    }
    mbar_wait(bar, (uint32_t)chunk & 1u);                  // MMAs retired: the staging tiles are free
    tc_fence_after();
  }
  // accumulator row tid (theta row m0 + tid) -> G
  {
    const uint32_t t_row = tmem_base + ((uint32_t)(warp * 32) << 16);
    for (int c0 = 0; c0 < nnp; c0 += 16) {
      uint32_t v[16];
      tmem_ld<16>(t_row + (uint32_t)c0, v);
      tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 16; ++j) G[tid * kGStride + c0 + j] = rows > 0 ? __uint_as_float(v[j]) : 0.0f;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, kUpdTile);
  // clip + Adam, coalesced along n; G takes the new weights. kAdamBatch elements per thread have their
  // master weight and slots in flight together (one memory latency per batch, not per element).
  const float lr_t = st->lr_t;
  const int total = mrows * nn;
  for (int i0 = tid; i0 < total; i0 += kAdamBatch * kThreads) {
    int64_t p[kAdamBatch];
    float w[kAdamBatch], mo[kAdamBatch], vo[kAdamBatch];
#pragma unroll
    for (int b = 0; b < kAdamBatch; ++b) {
      const int i = i0 + b * kThreads, ml = i / nn, nl = i - ml * nn;
      p[b] = i < total ? e * a.pn + L.off + (int64_t)(m0 + ml) * N + n0 + nl : -1;
      w[b] = p[b] >= 0 ? a.theta[p[b]] : 0.0f;
      mo[b] = p[b] >= 0 ? a.m[p[b]] : 0.0f;
      vo[b] = p[b] >= 0 ? a.v[p[b]] : 0.0f;
    }
#pragma unroll
    for (int b = 0; b < kAdamBatch; ++b) {
      if (p[b] < 0) continue;
      const int i = i0 + b * kThreads, ml = i / nn, nl = i - ml * nn;
      const float g = G[ml * kGStride + nl];
      float m, v;
      a.grad[p[b]] = g;
      adam_slots(g, mo[b], vo[b], opt, m, v);
      a.m[p[b]] = m;
      a.v[p[b]] = v;
      const float nw = adam_weight(w[b], m, v, opt, lr_t);
      a.theta[p[b]] = nw;
      G[ml * kGStride + nl] = nw;
    }
  }
  __syncthreads();
  uint8_t* img = a.img + (int64_t)e * a.img_member_bytes;
  // forward image: 16 bytes = 8 consecutive k of one n; the tile holding the bias row adds k = K (bf16 of the
  // bias) and K + 1 (its residual)
  {
    const int npf = r16(N);
    const bool has_bias = m0 + mrows == K + 1;
    const int nq = has_bias ? (mrows + 1 + 7) / 8 : mrows / 8;
    uint8_t* fwd = img + L.fwd_off;
    for (int i = tid; i < nq * nn; i += kThreads) {
      const int q = i / nn, nl = i - q * nn, n = n0 + nl;
      float v[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int kl = q * 8 + j, kk = m0 + kl;
        float x = 0.0f;
        if (kk < K) {
          x = G[kl * kGStride + nl];
        } else if (kk == K) {
          x = __bfloat162float(__float2bfloat16_rn(G[kl * kGStride + nl]));
        } else if (kk == K + 1) {
          const float b = G[(K - m0) * kGStride + nl];
          x = b - __bfloat162float(__float2bfloat16_rn(b));
        }
        v[j] = x;
      }
      *reinterpret_cast<uint4*>(fwd + (int64_t)(m0 / 8 + q) * npf * 16 + (n >> 3) * 128 + (n & 7) * 16) =
          make_uint4(pack2(v[0], v[1]), pack2(v[2], v[3]), pack2(v[4], v[5]), pack2(v[6], v[7]));
    }
  }
  // backward image (layers >= 1): 16 bytes = 8 consecutive n of one k < K
  if (L.bwd_off >= 0) {
    const int npb = r16(K);
    const int krows = min(kUpdTile, K - m0), ng = (nn + 7) / 8;
    uint8_t* bwd = img + L.bwd_off;
    for (int i = tid; i < krows * ng; i += kThreads) {
      const int kl = i % krows, q = i / krows, kk = m0 + kl;
      float v[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = (q * 8 + j < nn) ? G[kl * kGStride + q * 8 + j] : 0.0f;
      *reinterpret_cast<uint4*>(bwd + (int64_t)(n0 / 8 + q) * npb * 16 + (kk >> 3) * 128 + (kk & 7) * 16) =
          make_uint4(pack2(v[0], v[1]), pack2(v[2], v[3]), pack2(v[4], v[5]), pack2(v[6], v[7]));
    }
  }
}

}  // namespace

// ---- host side ----------------------------------------------------------------------------------------
// Coverage: the shapes of both bf16 planner families. The chain kernel keeps a [128 x (units + 2)] bf16
// A tile and two [units x 64] weight chunks in shared memory (217 KB at 416 units) and up to 416 fp32
// accumulator columns in tensor memory; the heads (N = 2 obs_dim <= 248) are one MMA.
bool train_tc_supported(int in_dim, int obs_dim, int n_layers, int units) {
  return units >= 1 && units <= 416 && in_dim <= 126 && obs_dim >= 1 && obs_dim <= 124 && n_layers >= 1 &&
         n_layers <= 6;
}

int64_t train_tc_layout(TcLayer* layers, int n) {
  int64_t off = 0;
  for (int l = 0; l < n; ++l) {
    layers[l].fwd_off = off;
    off += (int64_t)r16(layers[l].N) * r16(layers[l].K + 2) * 2;
    layers[l].bwd_off = -1;
    if (l > 0) {
      layers[l].bwd_off = off;
      off += (int64_t)r16(layers[l].K) * r16(layers[l].N) * 2;
    }
  }
  return off;
}

// element (row, col) of a K-major SWIZZLE_NONE image with `rows_p` padded rows, in bf16 units
static size_t img_index(int row, int col, int rows_p) {
  return (size_t)(col >> 3) * rows_p * 8 + (size_t)(row >> 3) * 64 + (size_t)(row & 7) * 8 + (col & 7);
}

void train_tc_pack(const TcLayer* layers, int n, const float* theta, uint8_t* img) {
  for (int l = 0; l < n; ++l) {
    const TcLayer& L = layers[l];
    const float* W = theta + L.off;
    uint16_t* fwd = reinterpret_cast<uint16_t*>(img + L.fwd_off);
    const int npf = r16(L.N);
    for (int k = 0; k <= L.K; ++k)
      for (int c = 0; c < L.N; ++c) {
        const float w = W[(size_t)k * L.N + c];
        if (k < L.K) fwd[img_index(c, k, npf)] = bf16_bits(w);
        else bf16_split(w, fwd[img_index(c, k, npf)], fwd[img_index(c, k + 1, npf)]);
      }
    if (L.bwd_off < 0) continue;
    uint16_t* bwd = reinterpret_cast<uint16_t*>(img + L.bwd_off);
    const int npb = r16(L.K);
    for (int k = 0; k < L.K; ++k)
      for (int c = 0; c < L.N; ++c) bwd[img_index(k, c, npb)] = bf16_bits(W[(size_t)k * L.N + c]);
  }
}

int train_tc_update_tiles(const TcLayer& l) {
  return ((l.K + 1 + kUpdTile - 1) / kUpdTile) * ((l.N + kUpdTile - 1) / kUpdTile);
}

// Each CTA allocates a power of two of TMEM columns (>= 32) and nothing else on the SM may then be short of
// them: the dynamic shared memory request is raised until no more CTAs fit the SM than its 512 columns allow.
static size_t smem_for_tmem(size_t smem, uint32_t tmem_cols) {
  const size_t per_sm = 233472;                            // 228 KB, of which 1 KB is reserved per CTA
  const size_t max_ctas = 512 / tmem_cols;
  const size_t floor_bytes = per_sm / (max_ctas + 1) - 1024 + 16;
  return std::max(smem, floor_bytes);
}

cudaError_t train_tc_chain(const TcChainArgs& a, const OptParams& opt, const FitDesc* desc, TrainState* st,
                           int grid_rows, int rows_fixed, int step_off, cudaStream_t s) {
  const int n_pass = a.train ? 2 * a.L + 1 : a.L + 1;
  int ka = r16(a.layer[0].K + 2), np_max = 0;
  for (int l = 0; l <= a.L; ++l) {
    const TcLayer& L = a.layer[l];
    ka = std::max(ka, std::max(r16(L.N + 2), r16(L.N)));
    np_max = std::max(np_max, r16(L.N));
    if (l > 0 && a.train) np_max = std::max(np_max, r16(L.K));
  }
  const uint32_t a_bytes = (uint32_t)ka * 256u;
  const uint32_t stage_bytes = (uint32_t)np_max * kChunkK * 2u;
  uint32_t tmem_cols = 32;
  while ((int)tmem_cols < np_max) tmem_cols <<= 1;
  const size_t smem = smem_for_tmem((size_t)a_bytes + 2 * stage_bytes, tmem_cols);
  cudaError_t err = cudaFuncSetAttribute(train_tc_chain_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)smem);
  if (err != cudaSuccess) return err;
  dim3 grid((grid_rows + kTcRows - 1) / kTcRows, a.ensemble);
  train_tc_chain_kernel<<<grid, kThreads, smem, s>>>(a, opt, desc, st, rows_fixed, step_off, n_pass, stage_bytes,
                                                     a_bytes, tmem_cols);
  return cudaGetLastError();
}

cudaError_t train_tc_update(const TcUpdArgs& a, const OptParams& opt, const FitDesc* desc, const TrainState* st,
                            int n_tiles, int rows_fixed, int step_off, cudaStream_t s) {
  const size_t smem = smem_for_tmem((size_t)2 * kUpdTile * kUpdRows * 2 + (size_t)kUpdTile * kGStride * 4, kUpdTile);
  cudaError_t err = cudaFuncSetAttribute(train_tc_update_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)smem);
  if (err != cudaSuccess) return err;
  train_tc_update_kernel<<<dim3(n_tiles, a.ensemble), kThreads, smem, s>>>(a, opt, desc, st, rows_fixed, step_off);
  return cudaGetLastError();
}

}  // namespace simba

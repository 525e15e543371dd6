// fp32 SIMT fused rollout + scoring kernel — the 1e-4 parity contract of the planner.
//
// Replaces, per CEM iteration and in ONE launch, the reference's
//   tf.tile / broadcast_to                     simba/policies/cem_mpc.py:49-54        (index math)
//   TransitionModel.unfold_sequences / scale   simba/models/transition_model.py:64-87
//   MlpEnsemble.forward / __call__             simba/models/mlp_ensemble.py:122-132,189-193
//   SafetyGymStateScorer.reward / .cost        simba/environment_utils/safety_gym.py:110-166
//   per-row part of compute_objective          simba/policies/mpc_policy.py:30-37,
//                                              simba/policies/safe_cem_mpc.py:82-93
// Trajectories stay on chip; only (return, cost mask, cost sum) per row reach HBM.
//
// One CTA = one ensemble member x TM rows, 256 threads. Activations live in shared memory
// transposed ([k][row]); the member's fp32 weights (283 KB for 4x128 — more than one SM's shared
// memory) are streamed from L2 as [16 x 128] chunks through a 3-stage cp.async ring in exactly
// the order they are consumed, so the ring never drains across layers or steps. Each thread owns a
// 4(row) x 4(col) register tile: per k one broadcast LDS.128 of activations and one LDS.128 of
// weights feed 16 FFMAs (FMA-pipe bound, not LDS bound).
#include <algorithm>

#include "common.cuh"
#include "internal.h"
#include "rollout_params.cuh"

namespace simba {

namespace {
constexpr int TM = kF32TileRows;      // rows per CTA
constexpr int NB = 128;               // output columns per pass: weight chunk = [KC k rows][NB cols] fp32
constexpr int KC = 16;                // k rows per weight chunk
constexpr int NT = 256;
constexpr int WSTAGES = 3;
constexpr int CHUNK = KC * NB;        // floats

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
  const uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(d), "l"(gmem_src));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;\n" ::"n"(N));
}
}  // namespace

__global__ void __launch_bounds__(NT) rollout_f32_kernel(const RolloutParams prm) {
  extern __shared__ float4 smem_f4[];
  float* smem = reinterpret_cast<float*>(smem_f4);
  const RowGeom& g = prm.g;
  const int tid = threadIdx.x;
  const int O = g.O, A = g.A, H = g.H, IN = O + A;
  const int OS = O | 1;                       // odd row stride: conflict-free column walks
  const int rows_buf = prm.act_rows;          // rows of each activation buffer ([k][TM])

  float* wbuf = smem;                                   // [WSTAGES][CHUNK]
  float* buf0 = wbuf + WSTAGES * CHUNK;                 // [rows_buf][TM]
  float* buf1 = buf0 + rows_buf * TM;
  float* state = buf1 + rows_buf * TM;                  // [TM][OS]
  float* smin = state + TM * OS;                        // [IN]
  float* sdel = smin + IN;                              // [IN]
  int64_t* row_meta = reinterpret_cast<int64_t*>(sdel + IN + ((2 * IN) & 1));   // 8B aligned below

  const Tile tile = prm.tiles[blockIdx.x];
  const int member = tile.member;

  // ---- early exit: every state this tile touches has stopped iterating (cem_mpc.py:66-67) ----
  if (prm.active != nullptr) {
    const int m = g.rows_per_state[member];
    const int s_first = tile.k0 / m, s_last = (tile.k0 + tile.count - 1) / m;
    bool any = false;
    for (int s = s_first; s <= s_last; ++s) any = any || (prm.active[s] != 0);
    if (!any) return;
  }

  // ---- per-row metadata --------------------------------------------------------------------
  // row_meta[0*TM + r] = action base offset, [1*TM + r] = eps row (global), [2*TM+r] = out index,
  // [3*TM + r] = state index (source of s_0)
  RowId my{};
  const bool my_valid = tid < tile.count;
  if (tid < TM) {
    RowId id = decode_row(g, member, tile.k0 + (tid < tile.count ? tid : 0));
    my = id;
    row_meta[0 * TM + tid] = ((int64_t)id.s * g.N + id.i_global) * prm.action_stride;
    row_meta[1 * TM + tid] = id.r_global;
    row_meta[2 * TM + tid] = id.out;
    row_meta[3 * TM + tid] = prm.state_per_row ? id.r_global : (int64_t)id.s;
    row_meta[4 * TM + tid] = id.s;
  }
  for (int k = tid; k < IN; k += NT) {
    smin[k] = prm.scale_on ? prm.smin[k] : 0.0f;
    sdel[k] = prm.scale_on ? prm.sdelta[k] : 1.0f;
  }
  __syncthreads();
  for (int idx = tid; idx < TM * O; idx += NT) {
    const int row = idx / O, o = idx - row * O;
    float v = 0.0f;
    if (row < tile.count) v = prm.states[row_meta[3 * TM + row] * prm.state_stride + o];
    state[row * OS + o] = v;
    if (prm.traj_out != nullptr && row < tile.count)
      prm.traj_out[(row_meta[2 * TM + row] * (H + 1)) * O + o] = v;
  }
  __syncthreads();

  RowScore rs{};
  const bool done_first = objective_done_first(prm.objective);
  if (tid < TM) {
    const float* srow = state + tid * OS;
    row_score_init(rs, prm.scorer, [&](int b) { return srow[b]; });
  }

  // ---- weight chunk ring ---------------------------------------------------------------------
  const float* wsrc = prm.w_f32 + (size_t)member * prm.n_chunks * CHUNK;
  const float* bias = prm.bias_f32 + (size_t)member * prm.bias_stride;
  const int G = prm.n_chunks;
  const long total_chunks = (long)G * H;
  auto prefetch = [&](long a) {
    if (a < total_chunks) {
      const float* src = wsrc + (size_t)(a % G) * CHUNK;
      float* dst = wbuf + (a % WSTAGES) * CHUNK;
#pragma unroll
      for (int i = 0; i < CHUNK / 4 / NT; ++i) {
        const int f4 = tid + i * NT;
        cp_async16(dst + f4 * 4, src + f4 * 4);
      }
    }
    cp_async_commit();
  };
  prefetch(0);
  prefetch(1);
  long a = 0;   // absolute chunk counter

  const int rg = tid & 7, cg = tid >> 3;
  const uint64_t seed = prm.seed_ptr ? *prm.seed_ptr : prm.seed;
  const int L = prm.L, U = prm.U;

  for (int t = 0; t < H; ++t) {
    // ---- x = scale([s_t, a_t]) -> buf0[k][row]   (transition_model.py:72, :79-87) -------------
    const int in_rows = (IN + KC - 1) / KC * KC;
    for (int idx = tid; idx < in_rows * TM; idx += NT) {
      const int k = idx / TM, row = idx - k * TM;
      float v = 0.0f;
      if (k < O) {
        v = __fdiv_rn(__fsub_rn(state[row * OS + k], smin[k]), sdel[k]);
      } else if (k < IN) {
        const float av = (row < tile.count)
                             ? prm.actions[row_meta[0 * TM + row] + (int64_t)t * A + (k - O)] : 0.0f;
        v = __fdiv_rn(__fsub_rn(av, smin[k]), sdel[k]);
      }
      buf0[idx] = v;
    }
    // (visibility of buf0 is ensured by the __syncthreads at the top of the first chunk below)

    float* in = buf0;
    float* out = buf1;
    int bias_off = 0;
    for (int l = 0; l <= L; ++l) {              // l == L: the two Gaussian heads as one N = 2*O GEMM
      const int K = (l == 0) ? IN : U;
      const int N = (l == L) ? 2 * O : U;
      const int Kp = (K + KC - 1) / KC * KC;
      const int Np = (N + NB - 1) / NB * NB;
      for (int nb = 0; nb < Np; nb += NB) {
        float acc[4][4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[i][j] = 0.0f;
        for (int kc = 0; kc < Kp; kc += KC) {
          cp_async_wait<1>();
          __syncthreads();
          prefetch(a + 2);
          const float* wb = wbuf + (a % WSTAGES) * CHUNK + 4 * cg;
          const float* ib = in + kc * TM + 4 * rg;
#pragma unroll
          for (int kk = 0; kk < KC; ++kk) {
            const float4 av = *reinterpret_cast<const float4*>(ib + kk * TM);
            const float4 wv = *reinterpret_cast<const float4*>(wb + kk * NB);
            const float ar[4] = {av.x, av.y, av.z, av.w};
            const float wr[4] = {wv.x, wv.y, wv.z, wv.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
              for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(ar[i], wr[j], acc[i][j]);
          }
          ++a;
        }
        // epilogue: bias (+ ReLU for hidden layers, mlp_ensemble.py:19-20) -> out[n][row]
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int n = nb + 4 * cg + j;
          const float b = bias[bias_off + n];
          float4 v;
          v.x = acc[0][j] + b; v.y = acc[1][j] + b; v.z = acc[2][j] + b; v.w = acc[3][j] + b;
          if (l < L) {
            v.x = fmaxf(v.x, 0.0f); v.y = fmaxf(v.y, 0.0f);
            v.z = fmaxf(v.z, 0.0f); v.w = fmaxf(v.w, 0.0f);
          }
          *reinterpret_cast<float4*>(out + n * TM + 4 * rg) = v;
        }
      }
      bias_off += Np;
      float* tmp = in; in = out; out = tmp;
    }
    __syncthreads();
    // `in` now holds the head outputs transposed: rows [0, O) = mu, rows [O, 2O) = pre-softplus var

    // ---- s_{t+1} = s_t + (mu + sqrt(var) * eps | mu)   (mlp_ensemble.py:192-193,
    //      transition_model.py:75) -------------------------------------------------------------
    const int JB = (O + 7) / 8;                 // one Philox NOISE block = 8 consecutive outputs
    for (int item = tid; item < TM * JB; item += NT) {
      const int j = item / TM, row = item - j * TM;
      if (row >= tile.count) continue;
      const int64_t rgl = row_meta[1 * TM + row];
      const int s = (int)row_meta[4 * TM + row];
      float e8[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      const bool need_eps = prm.sampling_propagation || prm.sample_out != nullptr;
      if (need_eps) {
        if (prm.eps != nullptr) {
          const float* ep = prm.eps + (((int64_t)s * H + t) * ((int64_t)g.P * g.N) + rgl) * O;
#pragma unroll
          for (int q = 0; q < 8; ++q)
            if (8 * j + q < O) e8[q] = ep[8 * j + q];
        } else {
          philox_noise8<false>(seed, (uint32_t)s, (uint32_t)prm.iteration, (uint32_t)t, (uint32_t)rgl,
                               (uint32_t)j, e8);
        }
      }
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        const int o = 8 * j + q;
        if (o >= O) break;
        const float mu = in[o * TM + row];
        const float var = __fadd_rn(softplus_tf(in[(O + o) * TM + row]), 1e-4f);
        const float sd = sqrtf(var);
        const float smp = __fadd_rn(mu, __fmul_rn(sd, e8[q]));
        const float d = prm.sampling_propagation ? smp : mu;
        state[row * OS + o] = __fadd_rn(state[row * OS + o], d);
        if (prm.mu_out != nullptr) {
          const int64_t oi = row_meta[2 * TM + row] * O + o;
          prm.mu_out[oi] = mu;
          prm.var_out[oi] = var;
          if (prm.sample_out != nullptr) prm.sample_out[oi] = smp;
        }
      }
    }
    __syncthreads();

    // ---- per-row scoring of (s_t, s_{t+1}) -----------------------------------------------------
    if (my_valid) {
      const float* srow = state + tid * OS;
      row_score_step(rs, prm.scorer, done_first, t, [&](int b) { return srow[b]; });
    }
    if (prm.traj_out != nullptr) {
      for (int idx = tid; idx < TM * O; idx += NT) {
        const int row = idx / O, o = idx - row * O;
        if (row < tile.count)
          prm.traj_out[(row_meta[2 * TM + row] * (H + 1) + (t + 1)) * O + o] = state[row * OS + o];
      }
    }
    // next step's input build reads `state`; the update phase of this step is already fenced by
    // the __syncthreads above, and buf0/buf1 reuse is fenced by the chunk-loop barriers.
  }
  cp_async_wait<0>();

  if (my_valid && prm.row_return != nullptr) {
    prm.row_return[my.out] = rs.cum;
    prm.row_costmask[my.out] = rs.cmask;
    prm.row_costsum[my.out] = rs.costsum;
  }
}

static size_t f32_smem_bytes(int O, int A, int act_rows) {
  const int IN = O + A;
  const int OS = O | 1;
  size_t floats = (size_t)WSTAGES * CHUNK + 2 * (size_t)act_rows * TM + (size_t)TM * OS + 2 * IN;
  floats += (2 * IN) & 1;
  return floats * sizeof(float) + 5 * TM * sizeof(int64_t) + 16;
}

static int round_up(int x, int m) { return (x + m - 1) / m * m; }

// The image the kernel streams, per member: layer -> column block (NB) -> k chunk (KC), the heads fused as N = 2 O
// (mu columns [0, O), raw variance [O, 2 O)), zero-padded to n_chunks whole chunks; the biases per layer, padded
// to whole column blocks (bias_stride floats). act_rows: rows of an activation buffer, the widest padded layer.
int rollout_f32_pack(const ModelWeights& mw, std::vector<float>& w, std::vector<float>& b, int& n_chunks,
                     int& bias_stride, int& act_rows) {
  const auto& c = mw.cfg;
  const int L = c.n_layers, E = c.ensemble_size, U = c.units, O = c.obs_dim, IN = c.obs_dim + c.act_dim;
  n_chunks = 0; bias_stride = 0; act_rows = round_up(IN, KC);
  for (int l = 0; l <= L; ++l) {
    const int K = l == 0 ? IN : U, N = l == L ? 2 * O : U;
    const int Kp = round_up(K, KC), Np = round_up(N, NB);
    n_chunks += (Np / NB) * (Kp / KC);
    bias_stride += Np;
    act_rows = std::max(act_rows, std::max(Kp, Np));
  }
  // the kernel keeps two activation tiles [act_rows x 32 rows] in shared memory: very wide layers (> ~780 units)
  // do not fit and are rejected here rather than at the first launch
  if (f32_smem_bytes(O, c.act_dim, act_rows) > 227 * 1024)
    return set_error(SIMBA_ERR_UNSUPPORTED, "units %d: the rollout kernels keep a row tile's activations in "
                     "shared memory, which holds at most ~780 hidden units", U);
  w.assign((size_t)E * n_chunks * CHUNK, 0.0f);
  b.assign((size_t)E * bias_stride, 0.0f);
  for (int e = 0; e < E; ++e) {
    size_t chunk = (size_t)e * n_chunks;
    int boff = 0;
    for (int l = 0; l <= L; ++l) {
      const int K = l == 0 ? IN : U, N = l == L ? 2 * O : U;
      const int Kp = round_up(K, KC), Np = round_up(N, NB);
      auto weight = [&](int k, int n) -> float {
        if (k >= K || n >= N) return 0.0f;
        if (l < L) return mw.kernel(e, l)[(size_t)k * U + n];
        if (n < O) return mw.kernel(e, L)[(size_t)k * O + n];            // mu head
        return mw.kernel(e, L + 1)[(size_t)k * O + (n - O)];             // var head
      };
      for (int nb = 0; nb < Np; nb += NB)
        for (int kc = 0; kc < Kp; kc += KC, ++chunk)
          for (int kk = 0; kk < KC; ++kk)
            for (int n = 0; n < NB; ++n)
              w[(chunk * KC + kk) * NB + n] = weight(kc + kk, nb + n);
      for (int n = 0; n < N; ++n)
        b[(size_t)e * bias_stride + boff + n] = l < L ? mw.bias(e, l)[n] : n < O ? mw.bias(e, L)[n] : mw.bias(e, L + 1)[n - O];
      boff += Np;
    }
  }
  return SIMBA_OK;
}

cudaError_t launch_rollout_f32(const RolloutParams& prm, cudaStream_t stream) {
  const size_t smem = f32_smem_bytes(prm.g.O, prm.g.A, prm.act_rows);
  // set on every launch: the attribute is per device and per function, and launches happen only at
  // graph capture or in the non-graph entry points, never on the replayed hot path
  {
    cudaError_t e = cudaFuncSetAttribute(rollout_f32_kernel,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  rollout_f32_kernel<<<prm.n_tiles, NT, smem, stream>>>(prm);
  return cudaGetLastError();
}

}  // namespace simba

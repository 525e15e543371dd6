// Shared device-side definitions of the CEM-MPC planner kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/simba_b200.h"

namespace simba {

// ---------------------------------------------------------------------------------------------
// Row geometry. A "row" is one (state s, particle p, candidate i) rollout. Rows of one ensemble
// member form a list of S * rows_per_state[e] entries (state-major); a tile is a slice of that
// list, so tiles never mix members and batched states fill tiles without per-state padding.
//   entry k of member e ->  s = k / M_e,  lr = lr_lo[e] + k % M_e   (lr = p * N_local + i_local)
// This reproduces tf.split of the particle-major batch (simba/models/mlp_ensemble.py:123,
// simba/policies/cem_mpc.py:49-51): with one rank lr is the reference's row index r.
// ---------------------------------------------------------------------------------------------
struct RowGeom {
  int32_t S, P, N, N_local, cand0;   // N = global population, cand0 = first local candidate
  int32_t H, O, A, E;
  int32_t lr_lo[SIMBA_MAX_MEMBERS];
  int32_t rows_per_state[SIMBA_MAX_MEMBERS];
};

struct Tile {        // host-built work list
  int32_t member;
  int32_t k0;        // first entry of the member's row list
  int32_t count;     // valid rows in this tile
  int32_t pad;
};

struct RowId {
  int32_t s, p, i_local, i_global;
  int64_t r_global;   // p * N + i_global : eps / Philox row (shard invariant)
  int64_t out;        // (s * P + p) * N_local + i_local
};

__device__ __forceinline__ RowId decode_row(const RowGeom& g, int member, int k) {
  RowId id;
  const int m = g.rows_per_state[member];
  id.s = k / m;
  const int lr = g.lr_lo[member] + (k - id.s * m);
  id.p = lr / g.N_local;
  id.i_local = lr - id.p * g.N_local;
  id.i_global = g.cand0 + id.i_local;
  id.r_global = (int64_t)id.p * g.N + id.i_global;
  id.out = ((int64_t)id.s * g.P + id.p) * g.N_local + id.i_local;
  return id;
}

// ---------------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al., SC'11). Counter map documented in oracle/philox.py.
// ---------------------------------------------------------------------------------------------
constexpr uint32_t kPhiloxM0 = 0xD2511F53u, kPhiloxM1 = 0xCD9E8D57u;
constexpr uint32_t kPhiloxW0 = 0x9E3779B9u, kPhiloxW1 = 0xBB67AE85u;
constexpr uint32_t kStreamAction = 1u, kStreamNoise = 2u, kStreamFinal = 3u;

__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(kPhiloxM0, c.x), lo0 = kPhiloxM0 * c.x;
    const uint32_t hi1 = __umulhi(kPhiloxM1, c.z), lo1 = kPhiloxM1 * c.z;
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
    k.x += kPhiloxW0;
    k.y += kPhiloxW1;
  }
  return c;
}

__device__ __forceinline__ float u01(uint32_t x) {   // ((x >> 8) + 0.5) * 2^-24, never 0
  return __fmul_rn(__fadd_rn((float)(x >> 8), 0.5f), 5.9604644775390625e-08f);
}

// Box-Muller on (x, y) and (z, w). kFast = approximate MUFU path (bf16 rollout), else the
// accurate libdevice path (fp32 parity contract: a few ulp from the f64-evaluated oracle).
template <bool kFast>
__device__ __forceinline__ float4 normals4(uint4 b) {
  const float ua = u01(b.x), ub = u01(b.y), uc = u01(b.z), ud = u01(b.w);
  float ra, rb, sa, ca, sb, cb;
  if (kFast) {
    ra = sqrtf(-1.3862943611198906f * __log2f(ua));   // -2 ln u = -2 ln2 * log2 u
    rb = sqrtf(-1.3862943611198906f * __log2f(uc));
    __sincosf(6.283185307179586f * ub, &sa, &ca);
    __sincosf(6.283185307179586f * ud, &sb, &cb);
  } else {
    ra = sqrtf(-2.0f * logf(ua));
    rb = sqrtf(-2.0f * logf(uc));
    sincospif(2.0f * ub, &sa, &ca);
    sincospif(2.0f * ud, &sb, &cb);
  }
  return make_float4(ra * ca, ra * sa, rb * cb, rb * sb);
}

// NOISE stream: 8 normals per Philox block from 16-bit uniforms (see oracle/philox.py). Every
// 32-bit word gives one Box-Muller pair: u_a from the low half, u_b from the high half.
__device__ __forceinline__ float u01_16(uint32_t h) {   // (h + 0.5) * 2^-16, exact in fp32
  return fmaf((float)h, 1.52587890625e-05f, 7.62939453125e-06f);
}
template <bool kFast>
__device__ __forceinline__ void normals8(uint4 b, float (&z)[8]) {
  const uint32_t w[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float ua = u01_16(w[i] & 0xffffu), ub = u01_16(w[i] >> 16);
    float r, sn, cs;
    if (kFast) {
      asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(-1.3862943611198906f * __log2f(ua)));
      __sincosf(6.283185307179586f * ub, &sn, &cs);
    } else {
      r = sqrtf(-2.0f * logf(ua));
      sincospif(2.0f * ub, &sn, &cs);
    }
    z[2 * i] = r * cs;
    z[2 * i + 1] = r * sn;
  }
}

template <bool kFast>
__device__ __forceinline__ void philox_noise8(uint64_t seed, uint32_t s, uint32_t iteration,
                                              uint32_t t, uint32_t row, uint32_t block8, float (&z)[8]) {
  const uint4 ctr = make_uint4(block8, row, t | (iteration << 16), s | (kStreamNoise << 28));
  normals8<kFast>(philox4x32_10(ctr, make_uint2((uint32_t)seed, (uint32_t)(seed >> 32))), z);
}

__device__ __forceinline__ uint2 philox_key(uint64_t seed) {
  return make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
}

template <bool kFast>
__device__ __forceinline__ float4 philox_normals(uint64_t seed, uint32_t stream, uint32_t s,
                                                 uint32_t iteration, uint32_t t, uint32_t row,
                                                 uint32_t block) {
  const uint4 ctr = make_uint4(block, row, t | (iteration << 16), s | (stream << 28));
  return normals4<kFast>(philox4x32_10(ctr, philox_key(seed)));
}

// ---------------------------------------------------------------------------------------------
// tf.math.softplus restated (TF core/kernels/softplus_op.h) — GaussianHead, mlp_ensemble.py:30
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float softplus_tf(float x) {
  const float threshold = -13.942385f;   // log(FLT_EPSILON) + 2
  if (x > -threshold) return x;
  const float e = expf(x);
  if (x < threshold) return e;
  return log1pf(e);
}

// Hidden-layer activation (simba_model_set_activation), a compile-time parameter of the kernel bodies.
constexpr int kActRelu = SIMBA_ACT_RELU, kActSwish = SIMBA_ACT_SWISH;

// fp32 swish (tf.nn.swish) and its derivative, accurate libm expf and explicit round-to-nearest operations in the
// order of the oracle's float32 numpy: sigmoid(z) = 1 / (1 + exp(-z)), swish(z) = z * sigmoid(z),
// swish'(z) = sigmoid(z) * (1 + z * (1 - sigmoid(z)))
__device__ __forceinline__ float sigmoid_f32(float z) { return __fdiv_rn(1.0f, __fadd_rn(1.0f, expf(-z))); }
__device__ __forceinline__ float swish_f32(float z) { return __fmul_rn(z, sigmoid_f32(z)); }
__device__ __forceinline__ float swish_grad_f32(float z) {
  const float s = sigmoid_f32(z);
  return __fmul_rn(s, __fadd_rn(1.0f, __fmul_rn(z, __fsub_rn(1.0f, s))));
}

// ---------------------------------------------------------------------------------------------
// SafetyGymStateScorer pieces (simba/environment_utils/safety_gym.py:110-192). Arithmetic is
// written with explicit round-to-nearest ops so nvcc cannot contract it into FMAs: the scoring
// thresholds (dist <= 0.24, hazard <= 0.2) are hard decisions and must see the oracle's values.
// ---------------------------------------------------------------------------------------------
struct ScorerDev {
  simba_scorer_t c;
};

// closest_distance, safety_gym.py:188-192: min_bins clip(D - D*(1 - l), 0, D)
template <class Load>
__device__ __forceinline__ float closest_distance(Load ld, int begin, int end, float D) {
  float best = INFINITY;
  for (int b = begin; b < end; ++b) {
    float v = __fsub_rn(D, __fmul_rn(D, __fsub_rn(1.0f, ld(b))));
    v = fminf(fmaxf(v, 0.0f), D);
    best = fminf(best, v);
  }
  return best;
}

// goal_distance_metric, safety_gym.py:168-176
template <class Load>
__device__ __forceinline__ float goal_distance(const simba_scorer_t& c, Load ld) {
  if (c.goal_dist_index >= 0) return fmaxf(ld(c.goal_dist_index), 0.0f);
  return closest_distance(ld, c.goal_begin, c.goal_end, c.lidar_max_dist);
}

// cost(), safety_gym.py:145-166
template <class Load>
__device__ __forceinline__ float state_cost(const simba_scorer_t& c, Load ld) {
  float cost = 0.0f;
  for (int j = 0; j < c.n_constraints; ++j) {
    const float d = closest_distance(ld, c.con_begin[j], c.con_end[j], c.lidar_max_dist);
    cost += (d <= c.con_size[j]) ? 1.0f : 0.0f;
  }
  if (c.constrain_indicator) return cost > 0.0f ? 1.0f : 0.0f;
  return cost;
}

// reward(), safety_gym.py:110-143 (goal branch), given the two goal distances
__device__ __forceinline__ float step_reward(const simba_scorer_t& c, float dist, float next_dist,
                                             bool goal_achieved) {
  float r = __fadd_rn(__fmul_rn(__fsub_rn(dist, next_dist), c.reward_distance),
                      __fmul_rn(goal_achieved ? 1.0f : 0.0f, c.reward_goal));
  r = __fadd_rn(0.0f, r);
  if (c.reward_clip != 0.0f) r = fminf(fmaxf(r, -c.reward_clip), c.reward_clip);
  return r;
}

// Per-row objective accumulator: the per-row part of MpcPolicy.compute_objective
// (simba/policies/mpc_policy.py:30-37) and SafeCemMpc.compute_objective
// (simba/policies/safe_cem_mpc.py:82-93). The two differ in WHEN done is updated (SURVEY q1).
struct RowScore {
  float cum;        // cumulative masked reward
  float costsum;    // sum_t cost(s_t), no done mask (safe_cem_mpc.py:98-108)
  uint64_t cmask;   // the current word of the cost history: bit t & 63 = cost(s_t) * (1 - done) > 0
  float dist;       // goal distance of the current state s_t
  float cost;       // cost(s_t)
  bool done;
};

// A row's cost history is W = ceil(H / 64) 64-bit words, stored as planes [W, S, P, N_local] (plane stride
// S * P * N_local rows): plane w holds steps [64 w, 64 w + 64), so with H <= 64 plane 0 is the whole history.
__host__ __device__ __forceinline__ int cmask_planes(int H) { return (H + 63) >> 6; }
// True after step t when the current word is complete and more steps follow: the caller stores it to plane
// t >> 6 and starts a new word. The last word (plane W - 1) is stored after the last step, as with H <= 64,
// where this is never true.
__host__ __device__ __forceinline__ bool cmask_word_ends(int t, int H) { return (t & 63) == 63 && t + 1 < H; }
__host__ __device__ __forceinline__ int64_t cmask_plane_stride(const RowGeom& g) {
  return (int64_t)g.S * g.P * g.N_local;
}

template <class Load>
__device__ __forceinline__ void row_score_init(RowScore& rs, const simba_scorer_t& c, Load ld) {
  rs.cum = 0.0f; rs.costsum = 0.0f; rs.cmask = 0ull; rs.done = false;
  rs.dist = goal_distance(c, ld);
  rs.cost = state_cost(c, ld);
}

// advance with s_{t+1} readable through ld
template <class Load>
__device__ __forceinline__ void row_score_step(RowScore& rs, const simba_scorer_t& c,
                                               bool done_first, int t, Load ld_next) {
  const float next_dist = goal_distance(c, ld_next);
  const float next_cost = state_cost(c, ld_next);
  const bool goal = rs.dist <= c.goal_threshold;
  const float r = step_reward(c, rs.dist, next_dist, goal);
  if (done_first) {                                  // safe_cem_mpc.py:87-93
    rs.done = rs.done || goal;
    if (!rs.done && rs.cost > 0.0f) rs.cmask |= (1ull << (t & 63));
    rs.cum = __fadd_rn(rs.cum, __fmul_rn(r, rs.done ? 0.0f : 1.0f));
  } else {                                           // mpc_policy.py:35-37
    rs.cum = __fadd_rn(rs.cum, __fmul_rn(r, rs.done ? 0.0f : 1.0f));
    if (!rs.done && rs.cost > 0.0f) rs.cmask |= (1ull << (t & 63));
    rs.done = rs.done || goal;
  }
  rs.costsum = __fadd_rn(rs.costsum, rs.cost);
  rs.dist = next_dist;
  rs.cost = next_cost;
}

__host__ __device__ __forceinline__ bool objective_done_first(int objective) {
  return objective == SIMBA_OBJ_SAFE_PENALTY || objective == SIMBA_OBJ_FEASIBLE_FIRST;
}

}  // namespace simba

// The Gaussian-head / state / scoring pass shared by the two tcgen05 rollout kernels (rollout_tc.cu:
// A operand in tensor memory; rollout_tc_wide.cu: A operand in a swizzled shared-memory tile), plus
// the NOISE-stream generator they both use. One implementation, so a parity fix lands once. Where the
// pass's values go besides tensor memory is its sink: nowhere (planning), the trajectory (simba_unfold_tc)
// or the Gaussian head's mu, var and sample (simba_ensemble_forward_tc).
//
// What the pass replaces, per rollout row and step (SURVEY.md section 8 a6-a13):
//   mlp_ensemble.py:28-34,189-193   mu, var = softplus(raw) + 1e-4, delta = mu + sqrt(var) * eps
//   transition_model.py:72-75,79-87 s_{t+1} = s_t + delta; x_{t+1} = scale([s_{t+1}, a_{t+1}])
//   safety_gym.py:188-192           closest_distance: min over a lidar slice (partial minima here)
//
// A thread owns OW consecutive outputs (= state dims = layer-0 K elements) of one row and walks them
// in 8-wide chunks: TMEM loads of chunk c + 1 are in flight while chunk c is computed.
#pragma once
#include "common.cuh"
#include "tc_ptx.cuh"

namespace simba {
namespace {

constexpr int kHeadParts = 1 + SIMBA_MAX_CONSTRAINTS;   // goal + constrained lidar partial minima

// ---- NOISE stream (oracle/philox.py): 8 normals per Philox4x32-10 block from 16-bit uniforms ------
// Returned as four bf16x2 words (element 2i in the low half of word i): the bf16 rollout consumes
// its Gaussian draws rounded to bf16 (DESIGN.md section 5).
__device__ __forceinline__ uint32_t box_muller_pair_bf16(uint32_t w) {
  // 2^23 + h is exact in fp32, so (h + 0.5) * 2^-16 comes out of one FMA without an I2F
  const float fa = __uint_as_float(__byte_perm(w, 0x4b000000u, 0x7610));   // 2^23 + (w & 0xffff)
  const float fb = __uint_as_float(__byte_perm(w, 0x4b000000u, 0x7632));   // 2^23 + (w >> 16)
  const float ua = fmaf(fa, 1.52587890625e-05f, -128.0f + 7.62939453125e-06f);
  const float ub = fmaf(fb, 1.52587890625e-05f, -128.0f + 7.62939453125e-06f);
  // u_a >= 2^-17 is never denormal: the .ftz forms are exact here and skip the denormal fix-ups
  float lg, r, sn, cs;
  const float th = 6.283185307179586f * ub;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(lg) : "f"(ua));
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(-1.3862943611198906f * lg));   // -2 ln u = -2 ln 2 lg2 u
  asm("sin.approx.ftz.f32 %0, %1;" : "=f"(sn) : "f"(th));
  asm("cos.approx.ftz.f32 %0, %1;" : "=f"(cs) : "f"(th));
  return pack_bf16(r * cs, r * sn);
}

struct PhiloxState {
  uint32_t c0, c1, c2, c3, k0, k1;
};
template <int kRounds>
__device__ __forceinline__ void philox_rounds(PhiloxState& p) {
#pragma unroll
  for (int r = 0; r < kRounds; ++r) {
    uint32_t lo0, hi0, lo1, hi1;                          // one IMAD.WIDE per product
    asm("{\n\t.reg .b64 p;\n\tmul.wide.u32 p, %2, %3;\n\tmov.b64 {%0, %1}, p;\n\t}" : "=r"(lo0), "=r"(hi0) : "r"(p.c0), "r"(kPhiloxM0));
    asm("{\n\t.reg .b64 p;\n\tmul.wide.u32 p, %2, %3;\n\tmov.b64 {%0, %1}, p;\n\t}" : "=r"(lo1), "=r"(hi1) : "r"(p.c2), "r"(kPhiloxM1));
    const uint32_t n0 = hi1 ^ p.c1 ^ p.k0, n2 = hi0 ^ p.c3 ^ p.k1;
    p.c1 = lo1; p.c3 = lo0; p.c0 = n0; p.c2 = n2;
    p.k0 += kPhiloxW0; p.k1 += kPhiloxW1;
  }
}
__device__ __forceinline__ uint4 philox_finish_noise8_bf16(const PhiloxState& p) {
  return make_uint4(box_muller_pair_bf16(p.c0), box_muller_pair_bf16(p.c1), box_muller_pair_bf16(p.c2),
                    box_muller_pair_bf16(p.c3));
}
__device__ __forceinline__ uint4 philox_noise8_bf16(uint2 key, uint32_t c0, uint32_t c1, uint32_t c2,
                                                    uint32_t c3) {
  PhiloxState p{c0, c1, c2, c3, key.x, key.y};
  philox_rounds<10>(p);
  return philox_finish_noise8_bf16(p);
}

// zero the draws of padded outputs (o >= O) of the block that starts at output o0
__device__ __forceinline__ uint4 mask_noise8(uint4 z, int o0, int O) {
  uint32_t w[4] = {z.x, z.y, z.z, z.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    if (o0 + 2 * i >= O) w[i] = 0u;
    else if (o0 + 2 * i + 1 >= O) w[i] &= 0xffffu;
  }
  return make_uint4(w[0], w[1], w[2], w[3]);
}

// externally supplied draws (parity mode): 8 consecutive floats of one row, zero beyond O
__device__ __forceinline__ uint4 external_noise8_bf16(const float* ep, int o0, int O) {
  float z[8];
#pragma unroll
  for (int q = 0; q < 8; ++q) z[q] = (o0 + q < O) ? ep[o0 + q] : 0.0f;
  return make_uint4(pack_bf16(z[0], z[1]), pack_bf16(z[2], z[3]), pack_bf16(z[4], z[5]), pack_bf16(z[6], z[7]));
}

// ---- lookup tables of the pass (shared memory, filled once per CTA) -------------------------------
//   scale[0][k], scale[1][k]: x_scaled[k] = fma(x[k], a, b) (transition_model.py:79-87), zero beyond
//                             O + A; `ones_at >= 0` turns k = ones_at, ones_at + 1 into the constant
//                             1 that multiplies the bias rows riding in the K padding of layer 0
//   pen[p][o]: 0 where state dim o belongs to part p's lidar slice, +inf elsewhere, so that
//              min_o (s[o] + pen[p][o]) is the slice minimum (part 0: goal lidar or the goal_dist dim)
// Both tables are kTW entries wide per row: the kernel's state width (64, or 128 for rollout_tc_wide.cu's
// wide-observation variant); sa / sb hold at least kTW entries.
template <int kTW = 64>
__device__ __forceinline__ void head_tables_init(float* scale_smem, float* pen_smem, const float* sa,
                                                 const float* sb, const simba_scorer_t& sc, int ones_at,
                                                 int tid, int nthreads) {
  for (int i = tid; i < kTW; i += nthreads) {
    const bool one = ones_at >= 0 && (i == ones_at || i == ones_at + 1);
    scale_smem[i] = one ? 0.0f : sa[i];
    scale_smem[kTW + i] = one ? 1.0f : sb[i];
    const bool in_goal = sc.goal_dist_index >= 0 ? (i == sc.goal_dist_index) : (i >= sc.goal_begin && i < sc.goal_end);
    pen_smem[i] = in_goal ? 0.0f : INFINITY;
    for (int q = 0; q < SIMBA_MAX_CONSTRAINTS; ++q)
      pen_smem[(1 + q) * kTW + i] =
          (q < sc.n_constraints && i >= sc.con_begin[q] && i < sc.con_end[q]) ? 0.0f : INFINITY;
  }
}

// 5 bits per 8-wide chunk of this thread's outputs: bit 0 = chunk intersects part 0 (goal), bit 1 + q =
// chunk intersects constrained slice q. Warp-uniform, so chunks outside every slice do no scoring.
template <int OW>
__device__ __forceinline__ uint32_t head_slice_bits(const simba_scorer_t& sc, int o_base) {
  uint32_t bits = 0;
#pragma unroll
  for (int c = 0; c < OW / 8; ++c) {
    const int lo = o_base + c * 8, hi = lo + 8;
    if (sc.goal_dist_index >= 0 ? (sc.goal_dist_index >= lo && sc.goal_dist_index < hi)
                                : (sc.goal_begin < hi && sc.goal_end > lo)) bits |= 1u << (c * 5);
    for (int q = 0; q < sc.n_constraints; ++q)
      if (sc.con_begin[q] < hi && sc.con_end[q] > lo) bits |= 1u << (c * 5 + 1 + q);
  }
  return bits;
}

struct HeadCtx {
  uint32_t t_acc;        // TMEM address of this row's head accumulators: mu at + o, raw var at + kVar + o
                         // (kVar = the head stride of head_step_pass: 64, or 128 for wide observations)
  uint32_t t_state;      // TMEM address of this row's fp32 state columns
  int o_base;            // first output / state dim of this thread
  int O, A;
  uint32_t slice_bits;   // head_slice_bits
  int n_constraints;
  const float* scale_smem;   // head_tables_init tables, kTW entries per row
  const float* pen_smem;
  float* part;           // this thread's slot of the partial-minima exchange: part p at part[p * 128]
  // two-CTA variant of rollout_tc.cu, CTA 1: the slot lives in CTA 0 (shared::cluster address of part p = 0,
  // 0 = the slot is local) and every store completes 4 bytes on that CTA's mbarrier
  uint32_t part_remote = 0, part_mbar = 0;
};

// sqrt(softplus(x) + 1e-4) on the MUFU path (mlp_ensemble.py:30, :192): ln(1 + e^x) =
// ln 2 * lg2(1 + ex2(x log2 e)). The raw-variance head's weights and bias are packed pre-scaled by
// log2(e) (simba_model_commit), so the accumulator holds x log2 e. Flush-to-zero ex2 (e^x < 2^-126
// adds nothing to 1), the clamp keeps e^x finite so that large x gives softplus(x) = x. The rounding
// of 1 + e costs <= 6e-8 absolute, i.e. <= 6e-4 relative to the variance because of its 1e-4 floor —
// far inside the bf16 tolerance.
__device__ __forceinline__ float head_stddev(float x_log2e) {
  float e, l, sd;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(fminf(x_log2e, 120.0f)));
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(l) : "f"(1.0f + e));
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(sd) : "f"(fmaf(l, 0.6931471805599453f, 1e-4f)));
  return sd;
}

// min over 8 values of v + pen (pen = 0 inside the slice, +inf outside)
__device__ __forceinline__ float slice_min8(const float (&v)[8], const float* pen, float acc) {
  const float4 p0 = *reinterpret_cast<const float4*>(pen);
  const float4 p1 = *reinterpret_cast<const float4*>(pen + 4);
  const float a = fminf(fminf(v[0] + p0.x, v[1] + p0.y), fminf(v[2] + p0.z, v[3] + p0.w));
  const float b = fminf(fminf(v[4] + p1.x, v[5] + p1.y), fminf(v[6] + p1.z, v[7] + p1.w));
  return fminf(acc, fminf(a, b));
}

// scoring + next-step input of one chunk, given the new state values sv[8] of dims [oc, oc + 8). The
// action a_{t+1} sits in state columns [O, O + A) (head_store_actions), so x = scale([s, a]) needs no
// special case here.
template <int kTW, class AStore>
__device__ __forceinline__ void head_chunk_tail(const HeadCtx& c, const AStore& astore, int oc, uint32_t bits,
                                                const float (&sv)[8], bool write_next, float& gmin,
                                                float (&cmin)[SIMBA_MAX_CONSTRAINTS]) {
  if (bits) {                                              // warp-uniform
    if (bits & 1u) gmin = slice_min8(sv, c.pen_smem + oc, gmin);
    if (bits >> 1) {
#pragma unroll
      for (int q = 0; q < SIMBA_MAX_CONSTRAINTS; ++q)
        if ((bits >> (1 + q)) & 1u) cmin[q] = slice_min8(sv, c.pen_smem + (1 + q) * kTW + oc, cmin[q]);
    }
  }
  if (write_next) {
    const ulonglong2 a0 = *reinterpret_cast<const ulonglong2*>(c.scale_smem + oc);
    const ulonglong2 a1 = *reinterpret_cast<const ulonglong2*>(c.scale_smem + oc + 4);
    const ulonglong2 b0 = *reinterpret_cast<const ulonglong2*>(c.scale_smem + kTW + oc);
    const ulonglong2 b1 = *reinterpret_cast<const ulonglong2*>(c.scale_smem + kTW + oc + 4);
    float x[8];
    f2_unpack(f2_fma(f2_pack(sv[0], sv[1]), a0.x, b0.x), x[0], x[1]);
    f2_unpack(f2_fma(f2_pack(sv[2], sv[3]), a0.y, b0.y), x[2], x[3]);
    f2_unpack(f2_fma(f2_pack(sv[4], sv[5]), a1.x, b1.x), x[4], x[5]);
    f2_unpack(f2_fma(f2_pack(sv[6], sv[7]), a1.y, b1.y), x[6], x[7]);
    astore.store8(oc, pack_bf16(x[0], x[1]), pack_bf16(x[2], x[3]), pack_bf16(x[4], x[5]), pack_bf16(x[6], x[7]));
  }
}

// The thread whose column slice starts the action block writes a_{t+1} (prefetched from global
// memory) into state columns [O, O + 4) of its row: the head outputs there are exactly zero (zero
// weights, bias and noise), so the pass carries them through unchanged into x_{t+1}. Columns beyond
// O + A hold zeros (their scale is 0, or the constant-one trick of the layer-0 bias rows).
__device__ __forceinline__ void head_store_actions(const HeadCtx& c, const float (&act)[4]) {
  const uint32_t v[4] = {__float_as_uint(act[0]), __float_as_uint(act[1]), __float_as_uint(act[2]),
                         __float_as_uint(act[3])};
  tmem_st<4>(c.t_state + c.O, v);
}

__device__ __forceinline__ void head_publish(const HeadCtx& c, float gmin, const float (&cmin)[SIMBA_MAX_CONSTRAINTS]) {
  if (c.part_remote != 0u) {
    st_async_b32(c.part_remote, __float_as_uint(gmin), c.part_mbar);
#pragma unroll
    for (int q = 0; q < SIMBA_MAX_CONSTRAINTS; ++q)
      if (q < c.n_constraints) st_async_b32(c.part_remote + (uint32_t)((1 + q) * 128 * 4), __float_as_uint(cmin[q]), c.part_mbar);
    return;
  }
  c.part[0] = gmin;
#pragma unroll
  for (int q = 0; q < SIMBA_MAX_CONSTRAINTS; ++q)
    if (q < c.n_constraints) c.part[(1 + q) * 128] = cmin[q];
}

// Where the values of a head pass go besides TMEM. The planning kernels keep nothing (NoTraj: the pass
// scores the states). The trajectory form of the kernels (simba_unfold_tc) writes the states to its row of
// traj_out [B, H + 1, O] (TrajSink) and skips the scoring: no slice minima, nothing published. The forward
// form (simba_ensemble_forward_tc) keeps the Gaussian head's per-element mu, var and sample instead of the
// state (ForwardSink, kState = false: the sampling head pass hands each chunk to head8 and neither reads nor
// writes the state columns).
struct NoTraj {
  static constexpr bool kScore = true, kState = true;
  __device__ __forceinline__ void put8(int, const float (&)[8]) const {}
};
struct TrajSink {
  static constexpr bool kScore = false, kState = true;
  float* row;   // this row's state of the current step in traj_out, null for a padding row
  int O;
  // outputs [oc, oc + 8) below O: 16-byte stores where the address allows (row offsets are not 16-byte
  // aligned for odd O), streaming (the trajectories are written once and read by the caller)
  __device__ __forceinline__ void put8(int oc, const float (&v)[8]) const {
    if (row == nullptr || oc >= O) return;
    float* p = row + oc;
    if (oc + 8 <= O && (reinterpret_cast<uintptr_t>(p) & 15u) == 0) {
      __stcs(reinterpret_cast<float4*>(p), make_float4(v[0], v[1], v[2], v[3]));
      __stcs(reinterpret_cast<float4*>(p + 4), make_float4(v[4], v[5], v[6], v[7]));
    } else if (oc + 8 <= O && (reinterpret_cast<uintptr_t>(p) & 7u) == 0) {
#pragma unroll
      for (int i = 0; i < 8; i += 2) __stcs(reinterpret_cast<float2*>(p + i), make_float2(v[i], v[i + 1]));
    } else {
#pragma unroll
      for (int i = 0; i < 8; ++i)
        if (oc + i < O) __stcs(p + i, v[i]);
    }
  }
};
struct ForwardSink {
  static constexpr bool kScore = false, kState = false;
  float* mu;       // mu_out / var_out / sample_out [B, O] (sample null when no sample is asked for)
  float* var;
  float* sample;
  int row;         // this thread's row of them, -1 for a padding row
  int O;
  // mu: the fp32 accumulator; v: softplus(raw) + 1e-4 before its square root; smp: mu + sqrt(var) * eps.
  // Stored as TrajSink stores a state chunk.
  __device__ __forceinline__ void head8(int oc, const uint32_t (&mu_bits)[8], const float (&v)[8],
                                        const float (&smp)[8]) const {
    if (row < 0) return;
    const int64_t off = (int64_t)row * O;
    float m[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) m[i] = __uint_as_float(mu_bits[i]);
    TrajSink{mu + off, O}.put8(oc, m);
    TrajSink{var + off, O}.put8(oc, v);
    if (sample != nullptr) TrajSink{sample + off, O}.put8(oc, smp);
  }
  __device__ __forceinline__ void put8(int, const float (&)[8]) const {}
};

// Trajectory form: every thread whose slice [o_base, o_base + OW) meets the action columns [O, O + A) stores
// its own columns of a_{t+1}, so that no column is written by two warps and an action block that crosses
// into the next slice (O = 47, A = 2) is carried whole (head_store_actions writes all four from the owner).
template <int OW>
__device__ __forceinline__ void head_store_own_actions(const HeadCtx& c, const float (&act)[4]) {
#pragma unroll
  for (int a = 0; a < 4; ++a) {
    if (a < c.A && c.O + a >= c.o_base && c.O + a < c.o_base + OW) {   // warp-uniform
      const uint32_t v[1] = {__float_as_uint(act[a])};
      tmem_st<1>(c.t_state + (uint32_t)(c.O + a), v);
    }
  }
}

// s_0 from global memory: state -> TMEM, x_0 -> A operand, partial minima (once per launch)
template <int OW, int kTW = 64, class AStore, class Sink = NoTraj>
__device__ __forceinline__ void head_first_pass(const HeadCtx& c, const AStore& astore, const float* s0_ptr,
                                                bool row_ok, const float (&act0)[4], const Sink& sink = Sink()) {
  float gmin = INFINITY, cmin[SIMBA_MAX_CONSTRAINTS];
#pragma unroll
  for (int q = 0; q < SIMBA_MAX_CONSTRAINTS; ++q) cmin[q] = INFINITY;
#pragma unroll 1
  for (int ch = 0; ch < OW / 8; ++ch) {
    const int oc = c.o_base + ch * 8;
    float sv[8];
    uint32_t st[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      sv[i] = (row_ok && oc + i < c.O) ? s0_ptr[oc + i] : 0.0f;
#pragma unroll
      for (int a = 0; a < 4; ++a)
        if (oc + i == c.O + a) sv[i] = act0[a];             // a_0 (zero beyond A)
      st[i] = __float_as_uint(sv[i]);
    }
    tmem_st<8>(c.t_state + oc, st);
    sink.put8(oc, sv);                                      // s_0 as read: the action columns lie beyond O
    head_chunk_tail<kTW>(c, astore, oc, Sink::kScore ? (c.slice_bits >> (ch * 5)) & 31u : 0u, sv, true, gmin, cmin);
  }
  if constexpr (Sink::kScore) head_publish(c, gmin, cmin);
}

// The same for a thread that owns one 8-wide chunk and already holds its eight s_0 values (zero beyond O or
// for a padding row) in registers: rollout_tc.cu's CTA-pair variant loads them before the dependency wait.
template <class AStore>
__device__ __forceinline__ void head_first_pass_vals(const HeadCtx& c, const AStore& astore, const float (&s0v)[8],
                                                     const float (&act0)[4]) {
  float gmin = INFINITY, cmin[SIMBA_MAX_CONSTRAINTS];
#pragma unroll
  for (int q = 0; q < SIMBA_MAX_CONSTRAINTS; ++q) cmin[q] = INFINITY;
  const int oc = c.o_base;
  float sv[8];
  uint32_t st[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    sv[i] = s0v[i];
#pragma unroll
    for (int a = 0; a < 4; ++a)
      if (oc + i == c.O + a) sv[i] = act0[a];             // a_0 (zero beyond A)
    st[i] = __float_as_uint(sv[i]);
  }
  tmem_st<8>(c.t_state + oc, st);
  head_chunk_tail<64>(c, astore, oc, c.slice_bits & 31u, sv, true, gmin, cmin);
  head_publish(c, gmin, cmin);
}

// Step t: s_{t+1} = s_t + mu (+ sqrt(softplus(raw var) + 1e-4) * eps), state back to TMEM, scaled bf16
// x_{t+1} into the A operand, partial lidar minima of s_{t+1} published. Padded outputs (o >= O) have
// zero weights, zero bias and zero noise, so their delta is exactly 0 and needs no mask. kVar: TMEM column
// offset of the raw-variance head from the mu head; kTW: width of the tables (both = the state width).
template <int OW, bool kSample, int kVar = 64, int kTW = 64, class Noise, class AStore, class Sink = NoTraj>
__device__ __forceinline__ void head_step_pass(const HeadCtx& c, const Noise& noise, const AStore& astore,
                                               bool write_next, const Sink& sink = Sink()) {
  constexpr int NCH = OW / 8;
  float gmin = INFINITY, cmin[SIMBA_MAX_CONSTRAINTS];
#pragma unroll
  for (int q = 0; q < SIMBA_MAX_CONSTRAINTS; ++q) cmin[q] = INFINITY;
  static_assert(Sink::kState || kSample, "the forward form forms the variance");
  uint32_t vm[2][8], vv[2][8], st[2][8];
  tmem_ld<8>(c.t_acc + c.o_base, vm[0]);
  if (kSample) tmem_ld<8>(c.t_acc + kVar + c.o_base, vv[0]);
  if constexpr (Sink::kState) tmem_ld<8>(c.t_state + c.o_base, st[0]);
#pragma unroll
  for (int ch = 0; ch < NCH; ++ch) {
    const int oc = c.o_base + ch * 8;
    const int cur = ch & 1, nxt = cur ^ 1;
    tmem_ld_wait();
    if (ch + 1 < NCH) {                                    // next chunk's loads fly during this chunk's math
      tmem_ld<8>(c.t_acc + oc + 8, vm[nxt]);
      if (kSample) tmem_ld<8>(c.t_acc + kVar + oc + 8, vv[nxt]);
      if constexpr (Sink::kState) tmem_ld<8>(c.t_state + oc + 8, st[nxt]);
    }
    float sv[8];
    if (kSample) {
      const uint4 nz = noise.get4(ch);
      const uint32_t nw[4] = {nz.x, nz.y, nz.z, nz.w};
      // two outputs per instruction wherever the op exists as fp32x2 (the MUFU ops and the clamp do not)
      const f32x2 kOne = f2_pack(1.0f, 1.0f);
      const f32x2 kLn2 = f2_pack(0.6931471805599453f, 0.6931471805599453f), kFloor = f2_pack(1e-4f, 1e-4f);
      float hv[8], hd[8];                                  // !kState: var and mu + stddev * eps, for sink.head8
#pragma unroll
      for (int q = 0; q < 8; q += 2) {
        float e0, e1, l0, l1, s0, s1;
        // sqrt(softplus(x) + 1e-4), see head_stddev; the accumulator already holds x log2(e)
        asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e0) : "f"(fminf(__uint_as_float(vv[cur][q]), 120.0f)));
        asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e1) : "f"(fminf(__uint_as_float(vv[cur][q + 1]), 120.0f)));
        f2_unpack(f2_add(f2_pack(e0, e1), kOne), l0, l1);
        asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(l0) : "f"(l0));
        asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(l1) : "f"(l1));
        f2_unpack(f2_fma(f2_pack(l0, l1), kLn2, kFloor), s0, s1);
        if constexpr (!Sink::kState) { hv[q] = s0; hv[q + 1] = s1; }
        asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(s0) : "f"(s0));
        asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(s1) : "f"(s1));
        const f32x2 eps = f2_pack(__uint_as_float(nw[q >> 1] << 16), __uint_as_float(nw[q >> 1] & 0xffff0000u));
        const f32x2 mu = f2_pack(__uint_as_float(vm[cur][q]), __uint_as_float(vm[cur][q + 1]));
        if constexpr (Sink::kState) {
          const f32x2 old = f2_pack(__uint_as_float(st[cur][q]), __uint_as_float(st[cur][q + 1]));
          f2_unpack(f2_add(old, f2_fma(f2_pack(s0, s1), eps, mu)), sv[q], sv[q + 1]);
        } else {
          f2_unpack(f2_fma(f2_pack(s0, s1), eps, mu), hd[q], hd[q + 1]);
        }
      }
      if constexpr (!Sink::kState) sink.head8(oc, vm[cur], hv, hd);
    } else {
#pragma unroll
      for (int q = 0; q < 8; ++q) sv[q] = __uint_as_float(st[cur][q]) + __uint_as_float(vm[cur][q]);
    }
    if constexpr (Sink::kState) {
      {
        uint32_t so[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) so[i] = __float_as_uint(sv[i]);
        tmem_st<8>(c.t_state + oc, so);
      }
      sink.put8(oc, sv);                                   // s_{t+1} as stored to TMEM
      head_chunk_tail<kTW>(c, astore, oc, Sink::kScore ? (c.slice_bits >> (ch * 5)) & 31u : 0u, sv, write_next,
                           gmin, cmin);
    }
  }
  if constexpr (Sink::kScore) head_publish(c, gmin, cmin);
}

// closest_distance (safety_gym.py:188-192) of a slice from its raw minimum m = min_b s[b]:
// v -> clip(D - D (1 - v), 0, D) is monotone non-decreasing in every rounding step, so
// min_b f(s[b]) == f(min_b s[b]) bit for bit.
__device__ __forceinline__ float closest_from_min(float m, float D) {
  const float w = __fsub_rn(D, __fmul_rn(D, __fsub_rn(1.0f, m)));
  return fminf(fmaxf(w, 0.0f), D);
}

// combine the Q partials of a row: goal distance (safety_gym.py:168-176) and cost (:145-166)
template <int Q>
__device__ __forceinline__ void head_combine(const simba_scorer_t& sc, const float* part_row, int nparts,
                                             float& dist, float& cost) {
  float g = INFINITY;
#pragma unroll
  for (int c = 0; c < Q; ++c) g = fminf(g, part_row[(c * nparts) * 128]);
  dist = sc.goal_dist_index >= 0 ? fmaxf(g, 0.0f) : closest_from_min(g, sc.lidar_max_dist);
  float cst = 0.0f;
  for (int q = 0; q < sc.n_constraints; ++q) {
    float m = INFINITY;
#pragma unroll
    for (int c = 0; c < Q; ++c) m = fminf(m, part_row[(c * nparts + 1 + q) * 128]);
    cst += (closest_from_min(m, sc.lidar_max_dist) <= sc.con_size[q]) ? 1.0f : 0.0f;
  }
  cost = sc.constrain_indicator ? (cst > 0.0f ? 1.0f : 0.0f) : cst;
}

// one step of the per-row objective (mpc_policy.py:30-37 / safe_cem_mpc.py:82-93), given the goal
// distance / cost of s_{t+1}
__device__ __forceinline__ void head_score_step(RowScore& rs, const simba_scorer_t& sc, bool done_first, int t,
                                                float next_dist, float next_cost) {
  const bool goal = rs.dist <= sc.goal_threshold;
  const float rew = step_reward(sc, rs.dist, next_dist, goal);
  if (done_first) {                                  // safe_cem_mpc.py:87-93
    rs.done = rs.done || goal;
    if (!rs.done && rs.cost > 0.0f) rs.cmask |= (1ull << t);
    rs.cum += rs.done ? 0.0f : rew;
  } else {                                           // mpc_policy.py:35-37
    rs.cum += rs.done ? 0.0f : rew;
    if (!rs.done && rs.cost > 0.0f) rs.cmask |= (1ull << t);
    rs.done = rs.done || goal;
  }
  rs.costsum += rs.cost;
  rs.dist = next_dist;
  rs.cost = next_cost;
}

}  // namespace
}  // namespace simba

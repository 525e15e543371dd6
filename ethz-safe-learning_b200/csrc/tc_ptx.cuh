// PTX wrappers shared by the tcgen05 rollout kernels (rollout_tc.cu, rollout_tc_wide.cu): mbarrier,
// TMA bulk copy, tcgen05 alloc / mma / commit / ld / st, UMMA descriptors, packed conversions.
#pragma once
#include <cuda_bf16.h>

#include <cstdint>

#include "common.cuh"

namespace simba {
namespace {

// ---- PTX wrappers ------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes)
               : "memory");
}
// suspend-time hint: the waiting warp sleeps in hardware until the phase completes (or this many
// ns pass), instead of burning issue slots in a polling loop next to the working warps
constexpr uint32_t kSuspendHintNs = 100000;
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
#ifdef SIMBA_TC_SPIN
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
#else
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
#endif
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity), "r"(kSuspendHintNs)
      : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug must fault the kernel, never hang the GPU. try_wait suspends the
// warp in hardware for a bounded time, so the spin count is the only bookkeeping on the slow path.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > (1u << 20)) __trap();
  }
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
      "l"(src), "r"(bytes), "r"(bar)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem),
               "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
               : "memory");
}
// D[tmem] (+)= A[smem] * B[smem], bf16 x bf16 -> fp32, single CTA
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc,
                                          uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]: the A operand (activations) is read from tensor memory, so one
// MMA streams only the weight tile from shared memory (half the SMEM traffic of the SS form)
__device__ __forceinline__ void umma_bf16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc,
                                             uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem),
      "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar)
               : "memory");
}
// width-generic TMEM row accessors: N consecutive 32-bit columns of this thread's lane
template <int N>
__device__ __forceinline__ void tmem_ld(uint32_t taddr, uint32_t (&v)[N]) {
  static_assert(N == 4 || N == 8 || N == 16 || N == 32, "unsupported TMEM load width");
  if constexpr (N == 4)
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]) : "r"(taddr) : "memory");
  if constexpr (N == 8)
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]) : "r"(taddr) : "memory");
  if constexpr (N == 16)
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]) : "r"(taddr) : "memory");
  if constexpr (N == 32)
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31]) : "r"(taddr) : "memory");
}
template <int N>
__device__ __forceinline__ void tmem_st(uint32_t taddr, const uint32_t (&v)[N]) {
  static_assert(N == 1 || N == 4 || N == 8 || N == 16, "unsupported TMEM store width");
  if constexpr (N == 1)
    asm volatile("tcgen05.st.sync.aligned.32x32b.x1.b32 [%0], {%1};" :: "r"(taddr), "r"(v[0]) : "memory");
  if constexpr (N == 4)
    asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};"
                 :: "r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]) : "memory");
  if constexpr (N == 8)
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
                 :: "r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]) : "memory");
  if constexpr (N == 16)
    asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
                 :: "r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_st_wait() {
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}
// relu(a), relu(b) -> packed bf16x2 (a in the low half)
__device__ __forceinline__ uint32_t pack_relu_bf16(float a, float b) {
  uint32_t r;
  asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
  return r;
}
__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
  return r;
}
// swish(z) = z sigmoid(z) = h + h tanh(h) with h = z / 2: one MUFU op (tanh.approx.f32) per element
__device__ __forceinline__ float swish_approx(float z) {
  const float h = 0.5f * z;
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(h));
  return fmaf(h, t, h);
}
// act(a), act(b) -> packed bf16x2 (a in the low half), for the activation ACT (kActRelu, kActSwish)
template <int ACT>
__device__ __forceinline__ uint32_t pack_act_bf16(float a, float b) {
  if constexpr (ACT == kActSwish) return pack_bf16(swish_approx(a), swish_approx(b));
  else return pack_relu_bf16(a, b);
}
// packed fp32x2 add (FADD2): one issue slot for two bias adds
__device__ __forceinline__ float2 add2(uint32_t lo, uint32_t hi, float2 b) {
  unsigned long long a = ((unsigned long long)hi << 32) | lo, bb, r;
  bb = ((unsigned long long)__float_as_uint(b.y) << 32) | __float_as_uint(b.x);
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(bb));
  return make_float2(__uint_as_float((uint32_t)r), __uint_as_float((uint32_t)(r >> 32)));
}
// ---- packed fp32x2 arithmetic (sm_100: one issue slot for two fp32 results) --------------------------
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 f2_pack(float lo, float hi) {
  f32x2 r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void f2_unpack(f32x2 v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ f32x2 f2_fma(f32x2 a, f32x2 b, f32x2 c) {
  f32x2 r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}
__device__ __forceinline__ f32x2 f2_mul(f32x2 a, f32x2 b) {
  f32x2 r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ f32x2 f2_add(f32x2 a, f32x2 b) {
  f32x2 r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}

__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c,
                                             uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d)
               : "memory");
}
// Programmatic dependent launch (PDL): let the next kernel in the stream start its prologue while
// this one runs, and wait for the previous kernel's results only where they are first needed.
__device__ __forceinline__ void pdl_launch_dependents() {
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}
__device__ __forceinline__ void pdl_wait_prior_grid() {
  asm volatile("griddepcontrol.wait;" ::: "memory");
}
__device__ __forceinline__ float sqrt_approx(float x) {
  float r;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
template <int kThreads>
__device__ __forceinline__ void named_bar_sync(int id) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "n"(kThreads) : "memory");
}

// true in exactly one (the lowest) lane of the converged warp
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

// producer side of a named barrier: counts this warp in without waiting (pairs with bar.sync)
template <int kThreads>
__device__ __forceinline__ void named_bar_arrive(int id) {
  asm volatile("bar.arrive %0, %1;" ::"r"(id), "n"(kThreads) : "memory");
}

// the same with the thread count in a register
__device__ __forceinline__ void named_bar_sync_n(int id, int threads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory");
}
__device__ __forceinline__ void named_bar_arrive_n(int id, int threads) {
  asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(threads) : "memory");
}

// ---- thread-block clusters: the peer CTA's shared memory (DSMEM) -----------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
// shared::cluster address of `smem_addr` (a shared::cta address of this CTA) in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t cluster_map_u32(uint32_t smem_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_addr), "r"(rank));
  return r;
}
// generic pointer to the same variable in CTA `rank`
template <class T>
__device__ __forceinline__ T* cluster_map_ptr(T* p, uint32_t rank) {
  uint64_t r;
  asm volatile("mapa.u64 %0, %1, %2;" : "=l"(r) : "l"(reinterpret_cast<uint64_t>(p)), "r"(rank));
  return reinterpret_cast<T*>(r);
}
// Asynchronous store into another CTA's shared memory that completes `bytes` transactions on an mbarrier
// of THAT CTA: the data is visible to whoever observes the barrier's phase completion, with no fence
// and no arrive on the producer side. (A release.cluster arrive compiles to MEMBAR.ALL.GPU + error
// barriers and the matching acquire to CCTL.IVALL: ~1.4 k cycles per hand-off, measured.)
__device__ __forceinline__ void st_async_v4(uint32_t cluster_addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d,
                                            uint32_t cluster_mbar) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.b32 [%0], {%1, %2, %3, %4}, [%5];"
               ::"r"(cluster_addr), "r"(a), "r"(b), "r"(c), "r"(d), "r"(cluster_mbar) : "memory");
}
__device__ __forceinline__ void st_async_b32(uint32_t cluster_addr, uint32_t v, uint32_t cluster_mbar) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.b32 [%0], %1, [%2];"
               ::"r"(cluster_addr), "r"(v), "r"(cluster_mbar) : "memory");
}
// all threads of all CTAs of the cluster (no CTA may exit while a peer can still touch its shared memory)
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// UMMA shared-memory descriptor: K-major, SWIZZLE_128B, 8-row groups 1024 B apart (dense 128 B rows)
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);        // start address
  d |= (uint64_t)1 << 16;                              // leading byte offset (unused for SW128 K-major)
  d |= (uint64_t)(1024 >> 4) << 32;                    // stride byte offset
  d |= (uint64_t)1 << 46;                              // descriptor version (sm_100)
  d |= (uint64_t)2 << 61;                              // SWIZZLE_128B
  return d;
}
// K-major, SWIZZLE_NONE tile of [128 rows][16 k] bf16: 8-row x 16-byte core matrices, K halves 128 B apart
// (leading byte offset), 8-row groups 256 B apart (stride byte offset). Used for the bias K-block.
__device__ __forceinline__ uint64_t umma_desc_k16_noswizzle(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)(128 >> 4) << 16;
  d |= (uint64_t)(256 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  return d;                                            // layout type 0 = SWIZZLE_NONE
}
// instruction descriptor: D=f32, A=B=bf16, both K-major, N=128, M=128
constexpr uint32_t kIdesc = (1u << 4) | (1u << 7) | (1u << 10) | ((128u >> 3) << 17) | ((128u >> 4) << 24);

// softplus on the MUFU path: ln(1 + e^x) = lg2(1 + ex2(x * log2 e)) * ln 2. The rounding of 1 + e
// costs at most 6e-8 absolute, i.e. <= 6e-4 relative to the variance because of its 1e-4 floor
// (mlp_ensemble.py:30) — far inside the bf16 path's tolerance.
__device__ __forceinline__ float softplus_fast(float x) {
  const float e = exp2f(fminf(x, 80.0f) * 1.4426950408889634f);
  return __log2f(1.0f + e) * 0.6931471805599453f;
}

// instruction descriptor for an arbitrary N (multiple of 16, <= 256): D=f32, A=B=bf16, K-major, M=128
__device__ __forceinline__ constexpr uint32_t umma_idesc_n(uint32_t n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((n >> 3) << 17) | ((128u >> 4) << 24);
}

}  // namespace
}  // namespace simba

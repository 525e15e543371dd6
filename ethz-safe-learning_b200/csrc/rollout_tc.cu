// bf16 tcgen05 fused rollout + scoring kernel (sm_100a) — the throughput path of the planner.
//
// Same contract as rollout_f32.cu (one launch per CEM iteration replaces cem_mpc.py:49-55,
// transition_model.py:64-87, mlp_ensemble.py:122-132,189-193, safety_gym.py:110-166 and the per-row
// part of mpc_policy.py:30-37 / safe_cem_mpc.py:82-93), with the per-layer GEMMs on the 5th-gen
// tensor cores:
//
//   * PERSISTENT CTAs, one per SM: a CTA walks work items (one ensemble member x NTILES row tiles of 128
//     rollouts) c, c + grid, ...; the member's whole bf16 weight set (144 KB for 4x128) is staged in
//     shared memory by the TMA engine (cp.async.bulk of pre-swizzled UMMA images), reused for all H steps
//     x (L+1) layers of every item of that member and re-staged only when the member changes. Everything
//     that does not depend on the previous kernel sits before griddepcontrol.wait (PDL);
//   * single plans (at most SMs / 2 tiles) run a CLUSTER OF TWO CTAs per tile that splits the head pass
//     by output columns and exchanges the slices through DSMEM (template parameter PAIR, below);
//   * activations are the A operand and live in TENSOR MEMORY (TS-mode tcgen05.mma: A from TMEM,
//     B = weights from shared memory), so an MMA streams only the weight tile from SMEM. The bias
//     of a layer is one more K = 16 MMA (constant ones tile x [bf16(b), bf16(b - hi)] block); layer 0
//     carries it in its K padding (k = O + A, O + A + 1 of the input are the constant 1);
//   * warp roles: Q epilogue threads per rollout row (Q = 4, one tile: latency configuration for
//     small populations; Q = 2, two tiles: throughput configuration) + ONE DEDICATED MMA-ISSUER WARP
//     PER TILE. tcgen05.mma issue blocks the issuing thread at the tensor pipe's own rate (a layer's
//     nine MMAs hold it for ~600 cycles), so an elected epilogue thread would stall its warp's 32 rows
//     and, through the tile's hand-off, the whole tile. Hand-offs are hardware named barriers in
//     producer / consumer form, which cost no issue slots while waiting (sixteen warps polling an
//     mbarrier spent 19 % of the kernel's issued instructions in try_wait loops): every epilogue warp
//     bar.arrive's on the tile's "A ready" barrier once its slice of the next A operand is in TMEM
//     (after tcgen05.wait::st + fence) and moves on; the issuer warp bar.sync's on it, issues the
//     layer, tcgen05.commit's onto the tile's mbarrier, waits for that (the only mbarrier poller of
//     the tile) and bar.arrive's on the tile's "accumulator ready" barrier, on which the epilogue
//     warps bar.sync. The one-tile variants split every layer into two 64-column halves on
//     double-buffered accumulators and A operands, each half with its own pair of barriers, so one
//     half drains while the other is still multiplied (see the issuer warp);
//   * per hidden layer an epilogue thread reads its column slice of the fp32 accumulator row
//     (tcgen05.ld 32x32b), applies ReLU, packs bf16 and writes the next layer's A operand
//     (tcgen05.st); in the shadow of the following MMAs it produces one Philox block of the step's
//     Gaussian draws (tc_head.cuh), parked as bf16 pairs in shared memory (two-tile variant) or
//     registers (one-tile variant);
//   * the rollout state s_t (fp32) lives in spare TMEM columns next to the accumulators. The
//     Gaussian-head / state pass is tc_head.cuh's head_step_pass (shared with rollout_tc_wide.cu); it
//     publishes each thread's partial lidar minima in a small shared-memory exchange;
//   * ONE SCORER WARP PER TILE combines those partials into goal distance / cost per row and keeps
//     the per-row objective (reward, done masks, cost bits), so that no epilogue warp and no tile-wide
//     barrier sits between a head pass and the next step's layer 0.
#include <cuda_bf16.h>

#include <cstdlib>
#include <type_traits>

#include "common.cuh"
#include "internal.h"
#include "rollout_params.cuh"
#include "tc_head.cuh"
#include "tc_ptx.cuh"

namespace simba {

// Debug timeline (compile with -DSIMBA_TC_TIMELINE): two threads of CTA 0 stamp clock64() at phase
// boundaries into prm.timeline (a scratch buffer handed in by tools/tc_timeline.py).
#ifdef SIMBA_TC_TIMELINE
#define TL(ev)                                                                                   \
  do {                                                                                           \
    if (tl_who >= 0 && blockIdx.x == 0)                                                          \
      prm.timeline[(tl_who * 64 + tl_t) * 64 + (ev)] = clock64();  \
  } while (0)
#else
#define TL(ev) do { } while (0)
#endif

namespace {

constexpr int kU = 128;                 // hidden width this kernel covers
constexpr int kMaxO = 60;               // observation dims (two Gaussian heads padded to 2 x 64 columns)
constexpr int kAtomBytes = 128 * 128;   // one 64-wide K atom of a 128-row tile (bf16, SW128)
constexpr int kBiasBlockBytes = 4096;   // one layer's bias as a K = 16 B operand (rollout_tc_pack)
constexpr int kBoundThreads = 640;      // launch bound: the hardware allocates warps in fours, so 17 - 19
                                        // warps occupy 20 warp slots -> 96 registers per thread

// A member's image (rollout_tc_pack) is staged into shared memory as it is: the layers' weight atoms, layer 0
// one and every later layer two (K = 128), then the L + 1 bias K-blocks.
__host__ __device__ constexpr uint32_t tc_weight_bytes(int L) { return kAtomBytes + (uint32_t)L * 2 * kAtomBytes; }
__host__ __device__ constexpr uint32_t tc_member_bytes(int L) {
  return tc_weight_bytes(L) + (uint32_t)(L + 1) * kBiasBlockBytes;
}
// Layer 0 carries its bias in the K padding when the input of IN = O + A elements leaves room for the constant
// ones at k = IN, IN + 1; otherwise it takes the bias K-step as every other layer does.
__host__ __device__ constexpr bool tc_l0_pad_bias(int in_dim) { return in_dim + 2 <= 64; }

struct TileInfo {
  int32_t member, k0, count, valid;
};

// Gaussian draws of the current step: one uint4 (8 outputs as bf16 pairs) per Philox block
template <int NB, int kThreads>
struct NoiseSmem {                       // [block][thread] uint4: conflict-free 16-byte accesses
  uint4* base;
  __device__ __forceinline__ uint4 get4(int b) const { return base[b * kThreads]; }
  __device__ __forceinline__ void put4(int b, uint4 v) { base[b * kThreads] = v; }
  __device__ __forceinline__ void put4_dyn(int b, uint4 v) { base[b * kThreads] = v; }
};
template <int NB>
struct NoiseRegs {
  uint4 v[NB];
  __device__ __forceinline__ uint4 get4(int b) const { return v[b]; }
  __device__ __forceinline__ void put4(int b, uint4 x) { v[b] = x; }
  __device__ __forceinline__ void put4_dyn(int b, uint4 x) {          // run-time index without local memory
#pragma unroll
    for (int i = 0; i < NB; ++i)
      if (i == b) v[i] = x;
  }
};

// A operand in tensor memory: K elements [k0, k0 + 8) of this thread's row = 4 columns of bf16 pairs
struct AStoreTmem {
  uint32_t t_a;
  __device__ __forceinline__ void store8(int k0, uint32_t p0, uint32_t p1, uint32_t p2, uint32_t p3) const {
    const uint32_t pk[4] = {p0, p1, p2, p3};
    tmem_st<4>(t_a + (uint32_t)(k0 >> 1), pk);
  }
};

// PAIR variant: the slice also goes into the peer CTA's exchange buffer (one 16-byte slot per thread
// and step parity; the peer's thread of the same row and column group moves it into its own A operand)
struct AStorePair {
  uint32_t t_a;
  uint32_t peer_slot;     // shared::cluster address of this thread's slot in the peer's buffer 0
  uint32_t buf_off;       // byte offset of the current step's buffer
  uint32_t peer_bar;      // shared::cluster address of the peer's mbarrier of the current step
  __device__ __forceinline__ void store8(int k0, uint32_t p0, uint32_t p1, uint32_t p2, uint32_t p3) const {
    const uint32_t pk[4] = {p0, p1, p2, p3};
    tmem_st<4>(t_a + (uint32_t)(k0 >> 1), pk);
    st_async_v4(peer_slot + buf_off, p0, p1, p2, p3, peer_bar);
  }
};

}  // namespace

// NTILES row tiles per CTA, Q epilogue threads per rollout row.
//
// PAIR (latency variant for plans with at most half as many tiles as SMs): a CLUSTER OF TWO CTAs works
// on one row tile. The hidden layers are computed redundantly by both (no exchange, no extra latency:
// the SMs would be idle otherwise); the Gaussian-head / state pass — the longest single stage of a step,
// bound by the SM's MUFU rate — is split by output columns: CTA c owns state dims [32 c, 32 c + 32),
// its threads push their 8 scaled bf16 inputs of the next step into the peer's shared memory (DSMEM)
// as well as into their own A operand, and their partial lidar minima into CTA 0's exchange buffer, with
// st.async: each store completes its bytes on an mbarrier of the destination CTA, which that CTA's scorer
// warp arms with the step's byte count (expect_tx), so there is no fence and no arrive on the producer
// side. The receiving thread waits for the phase, moves its row's 16 bytes into the A operand and
// publishes it. Exchange buffers and their mbarriers alternate by step parity; buffer p of step t + 2 is
// written only after the peer has sent all of step t + 1, which it does after consuming step t, so two
// suffice (and a barrier is re-armed for step t + 2 long before that step's bytes can arrive; were they
// early, a negative transaction count is legal and the pending arm keeps the phase open).
//
// TRAJ (simba_unfold_tc): the trajectory form. The epilogue threads write s_0 and every s_{t+1} of their
// valid rows to prm.traj_out [B, H + 1, O] (tc_head.cuh TrajSink) and score nothing: the scorer warps
// idle, no partial minima are published, the scorer struct is not read. Each thread whose column slice
// meets the action block stores its own action columns (head_store_own_actions). H is bounded only by
// the 16 bits of the Philox step counter.
//
// FWD (simba_ensemble_forward_tc): the forward form, a TRAJ form at H = 1 whose epilogue threads write, instead of
// the state, the Gaussian head's mu, var and (with external draws) sample of their valid rows to prm.mu_out,
// var_out and sample_out [B, O] (tc_head.cuh ForwardSink). Its head pass always forms the variance; without draws
// the noise stays zero.
template <int NTILES, int Q, bool PAIR, bool TRAJ, bool FWD = false>
__device__ __forceinline__ void rollout_tc_body(const RolloutParams& prm) {
  static_assert(!PAIR || (NTILES == 1 && Q == 4), "the pair variant is the one-tile latency configuration");
  static_assert(!(PAIR && TRAJ), "the trajectory form has no pair variant");
  static_assert(!FWD || TRAJ, "the forward form is a trajectory form");
  constexpr int kTileThreads = Q * 128;
  constexpr int kTileWarps = Q * 4;
  constexpr int kEpiThreads = NTILES * kTileThreads;
  constexpr int kEpiWarps = kEpiThreads / 32;
  constexpr int OW = (PAIR ? 32 : 64) / Q;   // head outputs (= state dims = layer-0 K elements) per thread
  constexpr int NSL = PAIR ? 2 * Q : Q;      // column slices of a row's head outputs (one partial minimum each)
  constexpr int NB = OW / 8;          // Philox blocks / 8-wide chunks per thread and step
  constexpr int HCOLS = 128 / Q;      // accumulator columns per thread and hidden layer
  // TMEM columns per tile: 128 fp32 accumulator columns, 64 fp32 state columns and 64 columns that
  // hold the bf16 A operand (128 K-elements, two per 32-bit column).
  //   two tiles: [2 x 128 acc][2 x 64 state][2 x 64 A] = 512 columns
  //   one tile (kDbl): [2 x 128 acc][64 state][2 x 64 A] = 448 of 512 allocated columns. The accumulator and
  //   the A operand are double-buffered: consecutive GEMMs of a step alternate between buffers 0 and 1, so a
  //   layer's two 64-column halves can drain while the other half is still being multiplied (see the issuer).
  // Taking all 512 columns of the SM is safe only because no second CTA of these kernels can be resident on
  // the SM and block in tcgen05.alloc: a CTA holds more than half of the SM's registers (576 or 640 threads
  // under the 96-register bound) and, at C1 depth, of its shared memory.
  constexpr bool kDbl = NTILES == 1;
  static_assert(!kDbl || Q == 4, "the one-tile variants split the columns into halves of two column groups");
  constexpr int kTmemCols = 512;
  constexpr uint32_t kStateCol = kDbl ? 256 : NTILES * 128;
  constexpr uint32_t kACol = kDbl ? 320 : NTILES * 192;
  // Throughput variant: the step's noise and the per-row running objective are parked in shared
  // memory to free registers. Latency variant (one tile): they stay in registers.
  constexpr bool kPark = NTILES > 1;
  constexpr int kBarAcc = 2, kBarA = 2 + NTILES, kBarPart = 2 + 2 * NTILES, kBarFree = 2 + 3 * NTILES;   // ids (+ tile)
  // one tile: kBarAcc / kBarA are "accumulator ready" / "A ready" of the low column half (columns 0-63, the
  // warps of column groups 0-1); these two are the high half's (column groups 2-3)
  constexpr int kBarAccHi = 6, kBarAHi = 7;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const RowGeom& g = prm.g;
  const int L = prm.L;
  const int H = g.H;
  const int O = g.O, A = g.A;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t crank = PAIR ? cluster_ctarank() : 0u;            // CTA within the pair
  // Persistent CTAs: work item = NTILES consecutive tiles of one member; CTA c takes items c, c + n_ctas, ...
  // (the grid is one CTA per SM when there are more items than SMs). A CTA's items mostly belong to the
  // same member, so the 144 KB weight set is staged once per member change instead of once per item, and
  // TMEM allocation, barrier setup, table fills and the CTA launch itself are paid once per SM.
  const int n_items = (prm.n_tiles + NTILES - 1) / NTILES;
  const int cta_item0 = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  const int n_ctas = PAIR ? (int)(gridDim.x >> 1) : (int)gridDim.x;       // PAIR: one item per cluster (launch_variant)
  const bool l0_pad_bias = tc_l0_pad_bias(O + A);
  constexpr int n_quarters = 4;                   // TMEM lane quarters (= warps per column group) of a tile
  constexpr int tile_bar_threads = Q * 128 + 32;  // a tile's epilogue warps + one partner warp (issuer / scorer)
  constexpr int half_bar_threads = Q * 64 + 32;   // one tile: the epilogue warps of a column half + the issuer or relay warp

  // ---- shared memory carve-up (base is 1024-aligned: required by SWIZZLE_128B) -------------------
  const uint32_t w_bytes = tc_weight_bytes(L);
  uint8_t* w_smem = smem_raw;
  uint8_t* biask_smem = w_smem + w_bytes;                                  // [(L+1)][4096]: bias K-blocks (B operand)
  uint8_t* ones_smem = biask_smem + (L + 1) * 4096;                        // [4096]: A operand of the bias K-step
  float* scale_smem = reinterpret_cast<float*>(ones_smem + 4096);          // [2][64]: a, b of x*a+b
  float* pen_smem = scale_smem + 128;                                      // [kHeadParts][64]
  const int nparts = TRAJ ? 1 : 1 + prm.scorer.n_constraints;              // goal + constrained lidars
  float* part_smem = pen_smem + kHeadParts * 64;                           // [1 or 2 (PAIR)][NTILES][NSL][nparts][128]
  const int part_buf_floats = NTILES * NSL * nparts * 128;
  uint4* xch_smem = reinterpret_cast<uint4*>(part_smem + (PAIR ? 2 : 1) * part_buf_floats);   // PAIR: [2][Q][128] x 16 B
  uint4* noise_smem = xch_smem + (PAIR ? 2 * Q * 128 : 0);                                    // [NB][threads]
  // running objective of every rollout row (RowScore fields, field-major), kept by the tile's scorer warp
  uint32_t* rs_smem = reinterpret_cast<uint32_t*>(noise_smem + (kPark ? NB * kEpiThreads : 0));   // [NTILES][8][128]
  uint64_t* bars = reinterpret_cast<uint64_t*>(rs_smem + NTILES * 8 * 128);
  // bars[0] = weights landed; bars[1 + j] = MMAs of tile j committed. Named barriers: 0 = CTA, 1 = all
  // epilogue threads, 2 + j = "accumulator ready" of tile j, 2 + NTILES + j = "A ready"
  // PAIR: bars[1 + NTILES + p] = the peer's warps have sent their step-parity-p slices
  // one tile: bars[1] = the low column half's MMAs committed, bars[3 + NTILES] = the high half's
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 1 + NTILES + 2 + (kDbl ? 1 : 0));
  TileInfo* tinfo = reinterpret_cast<TileInfo*>(tmem_slot + 2);
  uint64_t* seed_sh = reinterpret_cast<uint64_t*>(tinfo + NTILES);
  int32_t* w_state_sh = reinterpret_cast<int32_t*>(seed_sh + 1);     // [0] member whose weights are staged, [1] loads issued

  const uint32_t bar_w = smem_u32(&bars[0]);

#ifdef SIMBA_TC_TIMELINE
  // launch anatomy (thread 0 of CTA 0): row 3 of the timeline = entry, setup done, PDL wait passed, first
  // A published, items done, exit
#define TLK(k) do { if (blockIdx.x == 0 && threadIdx.x == 0) { prm.timeline[(3 * 64) * 64 + (k)] = clock64(); \
    unsigned long long gt_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt_)); \
    prm.timeline[(3 * 64 + 10 + prm.iteration) * 64 + (k)] = (long long)gt_; } } while (0)
#else
#define TLK(k) do { } while (0)
#endif
  TLK(0);
  pdl_launch_dependents();
  // member whose weights this CTA stages (-1: no rows at all); fixed geometry, readable before the PDL wait
  auto item_member = [&](int item) {
    int wm = -1;
    for (int q = 0; q < NTILES; ++q)
      if (item * NTILES + q < prm.n_tiles && prm.tiles[item * NTILES + q].count > 0) wm = prm.tiles[item * NTILES + q].member;
    return wm;
  };
  // one TMA bulk copy per layer and one of the bias K-blocks, which end the member's image, all onto bars[0] (thread 0
  // only; every MMA that read the previous set has completed)
  auto stage_weights = [&](int wm) {
    const uint8_t* wsrc = reinterpret_cast<const uint8_t*>(prm.w_tc) + (size_t)wm * prm.w_tc_member_bytes;
    const uint32_t bk_bytes = (uint32_t)(L + 1) * 4096u;
    mbar_expect_tx(bar_w, w_bytes + bk_bytes);
    uint32_t off = 0;
    for (int l = 0; l <= L; ++l) {
      const uint32_t nb = (l == 0) ? kAtomBytes : 2 * kAtomBytes;
      bulk_g2s(smem_u32(w_smem + off), wsrc + off, nb, bar_w);
      off += nb;
    }
    bulk_g2s(smem_u32(biask_smem), wsrc + (prm.w_tc_member_bytes - bk_bytes), bk_bytes, bar_w);
    w_state_sh[0] = wm;
    w_state_sh[1] += 1;
  };
  if (threadIdx.x == 0) {
    mbar_init(bar_w, 1);
#pragma unroll
    for (int j = 0; j < NTILES; ++j) {
      mbar_init(smem_u32(&bars[1 + j]), 1);                      // tcgen05.commit
    }
    if (kDbl) mbar_init(smem_u32(&bars[3 + NTILES]), 1);         // tcgen05.commit of the high half
    if (PAIR) {                                                  // armed below, once the tile is known to be live
      mbar_init(smem_u32(&bars[1 + NTILES]), 1);
      mbar_init(smem_u32(&bars[2 + NTILES]), 1);
    }
    fence_barrier_init();
    // The member's weights do not depend on the previous kernel (the tile list is fixed geometry), so
    // the copies for the first item start before the programmatic-dependency wait and overlap the CEM
    // update's tail. A CTA whose tiles turn out inactive still drains them before it exits.
    w_state_sh[0] = -1;
    w_state_sh[1] = 0;
    const int wm = cta_item0 < n_items ? item_member(cta_item0) : -1;
    if (wm >= 0) stage_weights(wm);
  }
  auto load_tile = [&](int ti) {                                // fixed geometry: valid = has rows
    TileInfo info{0, 0, 0, 0};
    if (ti < prm.n_tiles) {
      const Tile t = prm.tiles[ti];
      info.member = t.member; info.k0 = t.k0; info.count = t.count;
      info.valid = t.count > 0 ? 1 : 0;
    }
    return info;
  };
  if (threadIdx.x < NTILES) tinfo[threadIdx.x] = load_tile(cta_item0 * NTILES + threadIdx.x);
  if (warp == 0) tmem_alloc(smem_u32(tmem_slot), kTmemCols);
  if (warp < kEpiWarps) {
    // constant tables of this CTA (all epilogue threads cooperate)
    // A operand of the bias K-step: ones[m][0] = ones[m][1] = 1, rest 0 (same core-matrix layout)
    for (int i = threadIdx.x; i < 1024; i += kEpiThreads) {
      const int byte = i * 4;                           // [16 groups][2 K halves][8 rows][16 B]
      const bool first = ((byte & 255) < 128) && ((byte & 15) == 0);   // K half 0, elements 0 and 1
      reinterpret_cast<uint32_t*>(ones_smem)[i] = first ? 0x3F803F80u : 0u;
    }
    fence_proxy_async();                                // generic-proxy writes -> visible to the MMA
    if constexpr (TRAJ) {                               // the penalty table is never read
      head_tables_init(scale_smem, pen_smem, prm.tc_scale_a, prm.tc_scale_b, simba_scorer_t{},
                       l0_pad_bias ? O + A : -1, threadIdx.x, kEpiThreads);
    } else {
      head_tables_init(scale_smem, pen_smem, prm.tc_scale_a, prm.tc_scale_b, prm.scorer,
                       l0_pad_bias ? O + A : -1, threadIdx.x, kEpiThreads);
    }
  }
  if (PAIR && threadIdx.x == 0) {
    // arm the exchange barriers for s_0 (step -1, barrier 1) and step 0 (barrier 0); see the scorer warps
    const uint32_t per_step = crank == 0 ? (uint32_t)(kEpiThreads * 4 * nparts) : 0u;
    mbar_expect_tx(smem_u32(&bars[2 + NTILES]), per_step + (uint32_t)(kEpiThreads * 16));
    const uint32_t b0 = per_step + (1 < H ? (uint32_t)(kEpiThreads * 16) : 0u);
    if (b0 != 0u) mbar_expect_tx(smem_u32(&bars[1 + NTILES]), b0);
  }
  tc_fence_before();
  __syncthreads();
  if (PAIR) cluster_sync_all();                                 // the peer's mbarriers are armed before any store can reach them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  TLK(1);
  // everything above (barriers, the first weight copy, TMEM, constant tables, the cluster handshake) is
  // independent of the previous kernel — the CEM update that wrote the actions, the active flags and the
  // seed — and overlaps its tail under programmatic dependent launch; from here on its results are needed
  // PAIR (one item per CTA, the latency path): the wait moves further down, into each warp role behind its
  // own per-item setup (row decoding, pointers, the s_0 loads), which depends only on fixed geometry and on
  // the states; each role then checks the active flags itself (late_gate).
  constexpr bool kLateWait = PAIR;
  if (!kLateWait) pdl_wait_prior_grid();
  TLK(2);
  // (the plan's seed is uploaded before the plan's first kernel, a full dependency of every kernel of the plan)
  if (threadIdx.x == 0) *seed_sh = prm.seed_ptr ? *prm.seed_ptr : prm.seed;   // published by the item loop's first barrier
  // whether any state a tile touches is still planning (cem_mpc.py:66-67 early exit)
  auto tile_active = [&](const TileInfo& t) {
    if (prm.active == nullptr) return true;
    const int m = g.rows_per_state[t.member];
    bool any = false;
    for (int s = t.k0 / m; s <= (t.k0 + t.count - 1) / m; ++s) any = any || prm.active[s] != 0;
    return any;
  };
  auto late_gate = [&](const TileInfo& t) {
    if (!kLateWait) return true;                       // the item loop already waited and filtered
    pdl_wait_prior_grid();
    return tile_active(t);
  };
  uint32_t ph = 0;                                    // phase of the tile's commit mbarrier (issuer warps), runs across items

#pragma unroll 1
  for (int item = cta_item0; item < n_items; item += n_ctas) {
  if (threadIdx.x < NTILES) {
    TileInfo info = tinfo[threadIdx.x];                       // first item: fetched before the PDL wait
    if (item != cta_item0) info = load_tile(item * NTILES + threadIdx.x);
    if (!kLateWait && info.valid) info.valid = tile_active(info) ? 1 : 0;
    tinfo[threadIdx.x] = info;
  }
  __syncthreads();
  bool any_valid = false;
  int member = -1;
#pragma unroll
  for (int j = 0; j < NTILES; ++j)
    if (tinfo[j].valid) { any_valid = true; member = tinfo[j].member; }
  // another member than the one staged: every MMA of the previous item has completed (its last accumulator
  // was consumed before the CTA barrier that ended the item), so the set can be overwritten
  if (threadIdx.x == 0 && any_valid && member != w_state_sh[0]) {
    if (w_state_sh[1] > 0) mbar_wait(bar_w, (uint32_t)(w_state_sh[1] - 1) & 1u);   // a copy nobody waited for (inactive item)
    stage_weights(member);
  }
  __syncthreads();

  if (any_valid) {
    if (kDbl && warp == kEpiWarps + 2 * NTILES) {
      // ====================== relay warp (one tile): commit 0 -> "accumulator low ready", commit 1 -> "high ready" ===
      // The low half drains while the high half's last MMAs run. tcgen05.mma blocks the issuing thread at the
      // pipe's rate, so the issuer itself would see commit 0 only after it has issued the high half's MMAs; this
      // warp sleeps on the commit mbarriers instead (the tile's only mbarrier poller). The head pass reads both
      // halves, so there the low half waits for commit 1 as well, which completes after every earlier MMA (commit
      // 0's phase passes unobserved and is not waited for again). Neither barrier can run two phases ahead: the
      // next commit onto it follows an "A ready" of the warps this relay releases.
      if (tinfo[0].valid && late_gate(tinfo[0])) {
        const uint32_t bar_lo = smem_u32(&bars[1]), bar_hi = smem_u32(&bars[3 + NTILES]);
        for (int t = 0; t < H; ++t) {
          for (int layer = 0; layer <= L; ++layer) {
            mbar_wait(layer < L ? bar_lo : bar_hi, ph);
            tc_fence_before();
            named_bar_arrive_n(kBarAcc, half_bar_threads);
            mbar_wait(bar_hi, ph);
            ph ^= 1;
            tc_fence_before();
            named_bar_arrive_n(kBarAccHi, half_bar_threads);
          }
        }
      }
    } else if (warp >= kEpiWarps + NTILES) {
      // ====================== scorer warp of tile j: the per-row objective, off everybody's critical path ======
      // (mpc_policy.py:30-37 / safe_cem_mpc.py:82-93 on safety_gym.py:110-166). Lane i owns rows i, i + 32,
      // i + 64, i + 96 of the tile. After every head pass the epilogue warps bar.arrive on "partials
      // published"; this warp bar.sync's on it, combines the Q partial lidar minima of each row into the
      // goal distance / cost of s_{t+1}, advances the row's objective, and bar.arrive's on "partials free",
      // which the epilogue warps pass (normally without waiting: it is L layers old by then) before their
      // next head pass overwrites the exchange buffer.
      const int j = warp - kEpiWarps - NTILES;
      const TileInfo tis = tinfo[j];
      // PAIR: bytes the peer sends into this CTA for step t — CTA 1's partial minima go to CTA 0 every step,
      // the 16-byte next-input slices go both ways whenever a next step follows
      auto xbytes = [&](int t) -> uint32_t {
        return (crank == 0 ? (uint32_t)(kEpiThreads * 4 * nparts) : 0u) + (t + 1 < H ? (uint32_t)(kEpiThreads * 16) : 0u);
      };
      const uint32_t xbar = smem_u32(&bars[1 + NTILES]);
      if (PAIR && tis.valid && crank != 0 && late_gate(tis)) {
        // CTA 1 keeps no objective: its scorer warp only re-arms the two exchange barriers, each for the
        // step after next once the current one has completed
        for (int ts = -1; ts + 1 < H; ++ts) {
          mbar_wait(xbar + 8u * ((uint32_t)ts & 1u), (uint32_t)((ts + 1) >> 1) & 1u);
          if (lane == 0 && xbytes(ts + 2) != 0u) mbar_expect_tx(xbar + 8u * ((uint32_t)ts & 1u), xbytes(ts + 2));
        }
      }
      if (!TRAJ && tis.valid && crank == 0) {                              // PAIR: CTA 0 keeps the objective
        const simba_scorer_t& sc = prm.scorer;
        const bool done_first = objective_done_first(prm.objective);
        // the objective of the lane's four rows is parked in shared memory (field-major), so the row
        // loop stays rolled: this warp is never on the critical path and the kernel already exceeds the
        // instruction cache
        uint32_t* my_rs = rs_smem + j * 8 * 128 + lane;                    // [8 fields][128 rows]
        const float* part_tile0 = part_smem + (j * NSL * nparts) * 128;    // [NSL][nparts][128 rows]
#pragma unroll 1
        for (int i = 0; i < n_quarters; ++i) {
          const int row = lane + 32 * i;
#pragma unroll
          for (int f = 0; f < 7; ++f) my_rs[f * 128 + 32 * i] = 0u;
          my_rs[7 * 128 + 32 * i] = row < tis.count ? (uint32_t)decode_row(g, tis.member, tis.k0 + row).out : 0xffffffffu;
        }
        const bool live = late_gate(tis);
        for (int ts = -1; live && ts < H; ++ts) {                          // ts = -1: distance / cost of s_0
          named_bar_sync_n(kBarPart + j, tile_bar_threads);
          const float* part_tile = part_tile0;
          if (PAIR) {                                                      // + the peer CTA's slices of this step
            mbar_wait(xbar + 8u * ((uint32_t)ts & 1u), (uint32_t)((ts + 1) >> 1) & 1u);
            if (lane == 0 && ts + 2 < H) mbar_expect_tx(xbar + 8u * ((uint32_t)ts & 1u), xbytes(ts + 2));
            part_tile += (ts & 1) * part_buf_floats;
          }
#pragma unroll 1
          for (int i = 0; i < n_quarters; ++i) {
            uint32_t* q = my_rs + 32 * i;
            float nd, nc;
            head_combine<NSL>(sc, part_tile + lane + 32 * i, nparts, nd, nc);
            if (ts < 0) {
              q[4 * 128] = __float_as_uint(nd);
              q[5 * 128] = __float_as_uint(nc);
            } else {
              RowScore rs;
              rs.cum = __uint_as_float(q[0]);
              rs.costsum = __uint_as_float(q[128]);
              rs.cmask = (uint64_t)q[2 * 128] | ((uint64_t)q[3 * 128] << 32);
              rs.dist = __uint_as_float(q[4 * 128]);
              rs.cost = __uint_as_float(q[5 * 128]);
              rs.done = q[6 * 128] != 0u;
              head_score_step(rs, sc, done_first, ts, nd, nc);
              q[0] = __float_as_uint(rs.cum);
              q[128] = __float_as_uint(rs.costsum);
              q[2 * 128] = (uint32_t)rs.cmask;
              q[3 * 128] = (uint32_t)(rs.cmask >> 32);
              q[4 * 128] = __float_as_uint(rs.dist);
              q[5 * 128] = __float_as_uint(rs.cost);
              q[6 * 128] = rs.done ? 1u : 0u;
            }
          }
          if (ts + 1 < H) named_bar_arrive_n(kBarFree + j, tile_bar_threads);
        }
        if (live && prm.row_return != nullptr) {
#pragma unroll 1
          for (int i = 0; i < n_quarters; ++i) {
            const uint32_t* q = my_rs + 32 * i;
            const uint32_t slot = q[7 * 128];
            if (slot != 0xffffffffu) {
              prm.row_return[slot] = __uint_as_float(q[0]);
              prm.row_costmask[slot] = (uint64_t)q[2 * 128] | ((uint64_t)q[3 * 128] << 32);
              prm.row_costsum[slot] = __uint_as_float(q[128]);
            }
          }
        }
      }
    } else if (warp >= kEpiWarps) {
      // ====================== MMA issuer warp of tile j (lane 0 issues; the warp stays converged) ==============
      const int j = warp - kEpiWarps;
      if (tinfo[j].valid) {
        const uint32_t bar_acc = smem_u32(&bars[1 + j]);
        const uint32_t d_tmem = tmem_base + (uint32_t)j * 128;
        const uint32_t a_tmem = tmem_base + (uint32_t)(kACol + j * 64);              // lane 0, A columns
        const uint64_t ones_desc = umma_desc_k16_noswizzle(smem_u32(ones_smem));
        mbar_wait(bar_w, (uint32_t)(w_state_sh[1] - 1) & 1u);   // this member's weights have landed before the first MMA
#ifdef SIMBA_TC_TIMELINE
        const int tl_who = (j == 0 && lane == 0) ? 2 : -1;
#endif
        const bool live = late_gate(tinfo[j]);
        if constexpr (kDbl) {
          // One tile: every GEMM is issued as two N = 64 column halves, so that one half drains while the other
          // is multiplied. Order: N0 x K[0,64) and N1 x K[0,64) (these read only A's low half), then, once the
          // high half of A is in TMEM, N0 x K[64,128) + bias -> commit 0, N1 x K[64,128) + bias -> commit 1.
          // Every output element still accumulates K-steps 0..7, then the bias, as the N = 128 MMAs of the
          // two-tile kernel do (its rows are bit-identical). Layer 0 (K = 64): N0 (+ bias), commit 0, N1 (+ bias),
          // commit 1. The pair's head GEMM multiplies only this CTA's columns: mu [32 c, 32 c + 32) and raw
          // variance [64 + 32 c, ...), two N = 32 MMAs per K-step in place of the halves.
          // Why no MMA reads or writes TMEM that an epilogue warp is still using: GEMM n reads A[n & 1] and
          // accumulates into acc[n & 1];
          //  * A[n & 1] is rewritten by the drain of GEMM n + 1 (or the head pass), which starts after a commit of
          //    GEMM n + 1, and a commit completes only when every earlier MMA of this thread has, GEMM n included;
          // The issuer waits for no commit: the relay warp below hands them to the epilogue warps.
          //  * acc[n & 1] is next written by GEMM n + 2. Its low-half MMAs are issued after "A low ready" of
          //    GEMM n + 2, its high-half MMAs after GEMM n + 1 was fully issued, i.e. after "A high ready" of
          //    GEMM n + 1: each half's warps publish that only after their tcgen05.ld of acc[n & 1] was waited;
          //  * the head pass -> layer 0 boundary stays a full synchronisation: the head pass reads both halves of
          //    its accumulator (both commits), and layer 0 waits for the x slices of all warps (both "A ready").
          const uint32_t bar_acc_hi = smem_u32(&bars[3 + NTILES]);
          constexpr uint32_t kIdesc64 = umma_idesc_n(64u), kIdesc32 = umma_idesc_n(32u);
          uint32_t par = 0;                                 // buffers of the next GEMM
          // K-steps [kb, kb + 4) of one half: D columns d, B descriptor b (its rows = those columns)
          auto mma4 = [&](uint32_t d, uint32_t a, uint64_t b, uint32_t idesc, int kb) {
#pragma unroll
            for (int k = 0; k < 4; ++k)
              umma_bf16_ts(d, a + (uint32_t)(kb + k) * 8, b + (uint64_t)(((kb ? kAtomBytes : 0) + k * 32) >> 4), idesc,
                           (kb + k) > 0 ? 1u : 0u);
          };
          // bias block rows from `col` (8-row groups of 256 bytes)
          auto mma_bias = [&](uint32_t d, uint32_t bias_sm, uint32_t col, uint32_t idesc) {
            umma_bf16(d, ones_desc, umma_desc_k16_noswizzle(bias_sm + col * 32), idesc, 1u);
          };
          for (int t = 0; live && t < H; ++t) {
#ifdef SIMBA_TC_TIMELINE
            const int tl_t = t;
#endif
            {                                               // layer 0 (K = 64): needs the x slices of all warps
              const uint32_t d = d_tmem + par * 128, a = a_tmem + par * 64;
              const uint64_t b = umma_desc_sw128(smem_u32(w_smem));
              const uint32_t bias_sm = smem_u32(biask_smem);
              named_bar_sync_n(kBarA, half_bar_threads);
              named_bar_sync_n(kBarAHi, half_bar_threads);
              tc_fence_after();
              TL(0);
              if (elect_one()) {
                mma4(d, a, b, kIdesc64, 0);
                if (!l0_pad_bias) mma_bias(d, bias_sm, 0u, kIdesc64);
                umma_commit(bar_acc);
                mma4(d + 64, a, b + (uint64_t)((64 * 128) >> 4), kIdesc64, 0);
                if (!l0_pad_bias) mma_bias(d + 64, bias_sm, 64u, kIdesc64);
                umma_commit(bar_acc_hi);
              }
              TL(1);
              __syncwarp();
              par ^= 1;                                     // the relay warp releases the epilogue warps
            }
            for (int layer = 1; layer <= L; ++layer) {
              const uint32_t d = d_tmem + par * 128, a = a_tmem + par * 64;
              const bool own_head = PAIR && layer == L;
              const uint32_t c0 = own_head ? crank * 32 : 0u, c1 = own_head ? 64u + crank * 32 : 64u;   // columns = B rows
              const uint32_t idesc = own_head ? kIdesc32 : kIdesc64;
              // B rows c0 / c1 start whole 1024-byte swizzle groups (SW128)
              const uint64_t bw = umma_desc_sw128(smem_u32(w_smem + kAtomBytes + (layer - 1) * 2 * kAtomBytes));
              const uint64_t b0 = bw + (uint64_t)((c0 * 128) >> 4), b1 = bw + (uint64_t)((c1 * 128) >> 4);
              const uint32_t bias_sm = smem_u32(biask_smem + layer * 4096);
              named_bar_sync_n(kBarA, half_bar_threads);      // the low half of this GEMM's A is in TMEM
              tc_fence_after();
              TL(2 * layer);
              if (elect_one()) {                              // K[0, 64) of both halves
                mma4(d + c0, a, b0, idesc, 0);
                mma4(d + c1, a, b1, idesc, 0);
              }
              TL(2 * layer + 1);
              __syncwarp();
              named_bar_sync_n(kBarAHi, half_bar_threads);    // the high half of A
              tc_fence_after();
              TL(20 + 2 * layer);
              if (elect_one()) {                              // K[64, 128) + bias, one half after the other
                mma4(d + c0, a, b0, idesc, 4);
                mma_bias(d + c0, bias_sm, c0, idesc);
                umma_commit(bar_acc);
                mma4(d + c1, a, b1, idesc, 4);
                mma_bias(d + c1, bias_sm, c1, idesc);
                umma_commit(bar_acc_hi);
              }
              TL(21 + 2 * layer);
              __syncwarp();
              par ^= 1;
            }
          }
        } else
        for (int t = 0; live && t < H; ++t) {
#ifdef SIMBA_TC_TIMELINE
          const int tl_t = t;
#endif
          for (int layer = 0; layer <= L; ++layer) {
            named_bar_sync_n(kBarA + j, tile_bar_threads);     // every epilogue warp's slice of this layer's A is in TMEM
            tc_fence_after();
            TL(2 * layer);
            if (elect_one()) {                                // ptxas must KNOW one lane is active: with a plain
                                                              // lane test every UTCHMMA gets an operand waterfall loop
              // descriptor arithmetic hoisted out of the K loop: one add per MMA on the 14-bit address field
              const uint32_t woff = (layer == 0) ? 0u : (uint32_t)(kAtomBytes + (layer - 1) * 2 * kAtomBytes);
              const uint64_t b0 = umma_desc_sw128(smem_u32(w_smem + woff));
#pragma unroll
              for (int k = 0; k < 4; ++k)                     // K = 64 (layer 0) ...
                umma_bf16_ts(d_tmem, a_tmem + (uint32_t)k * 8, b0 + (uint64_t)((k * 32) >> 4), kIdesc, k > 0 ? 1u : 0u);
              if (layer > 0) {
#pragma unroll
                for (int k = 4; k < 8; ++k)                   // ... or 128; UMMA_K = 16 = 8 TMEM columns of bf16 pairs
                  umma_bf16_ts(d_tmem, a_tmem + (uint32_t)k * 8, b0 + (uint64_t)((kAtomBytes + (k - 4) * 32) >> 4),
                               kIdesc, 1u);
              }
              // + bias: ones[128 x 16] * biasK[16 x 128] (bf16 hi + lo rows), both operands from SMEM
              if (layer > 0 || !l0_pad_bias)
                umma_bf16(d_tmem, ones_desc, umma_desc_k16_noswizzle(smem_u32(biask_smem + layer * 4096)), kIdesc, 1u);
              umma_commit(bar_acc);
            }
            TL(2 * layer + 1);
            __syncwarp();
            mbar_wait(bar_acc, ph);                           // the layer's MMAs have completed
            ph ^= 1;
            tc_fence_before();
            named_bar_arrive_n(kBarAcc + j, tile_bar_threads); // wake the tile's epilogue warps
          }
        }
      }
    } else {
      // ============ epilogue warps: Q threads per rollout row, each owns a column slice ============
      const int j = warp / kTileWarps;                    // tile of this warp
      const int wl = warp - j * kTileWarps;               // warp within the tile
      const int cgp = wl >> 2;                            // column group in [0, Q)
      const int r = (wl & 3) * 32 + lane;                 // row in tile == TMEM lane
      const TileInfo ti = tinfo[j];
      if (ti.valid) {
        const bool row_ok = r < ti.count;
        const RowId id = decode_row(g, ti.member, ti.k0 + (row_ok ? r : 0));
        const uint32_t lane_base = tmem_base + ((uint32_t)((wl & 3) * 32) << 16);
        const uint32_t t_acc = lane_base + (uint32_t)j * 128;
        const uint32_t t_a = lane_base + (uint32_t)(kACol + j * 64);          // this row's A-operand columns (one tile: buffer 0)
        const float* act_ptr = prm.actions + ((int64_t)id.s * g.N + id.i_global) * prm.action_stride;
        const simba_scorer_t& sc = prm.scorer;

        HeadCtx hc;
        hc.t_acc = t_acc;
        hc.t_state = lane_base + (uint32_t)(kStateCol + j * 64);
        hc.o_base = (PAIR ? (int)crank * 32 : 0) + cgp * OW;
        hc.O = O; hc.A = A;
        hc.slice_bits = TRAJ ? 0u : head_slice_bits<OW>(sc, hc.o_base);
        hc.n_constraints = TRAJ ? 0 : sc.n_constraints;
        hc.scale_smem = scale_smem;
        hc.pen_smem = pen_smem;
        // partial minima: slice crank * Q + cgp of the buffer the scorer warp (PAIR: of CTA 0) reads
        float* part_slot0 = part_smem + ((j * NSL + (int)crank * Q + cgp) * nparts) * 128 + r;   // [nparts] stride 128
        hc.part = part_slot0 + (PAIR ? part_buf_floats : 0);                  // s_0 counts as step -1: buffer 1
        typename std::conditional<PAIR, AStorePair, AStoreTmem>::type astore;
        astore.t_a = t_a;
        const uint32_t my_xbar = smem_u32(&bars[1 + NTILES]);                 // PAIR: [2] mbarriers, 8 bytes apart
        const uint32_t peer_xbar = PAIR ? cluster_map_u32(my_xbar, crank ^ 1u) : 0u;
        const bool keeps_score = !TRAJ && (!PAIR || crank == 0);              // this CTA's scorer warp is the live one
        const uint32_t part_remote0 = (PAIR && crank != 0) ? cluster_map_u32(smem_u32(part_slot0), 0u) : 0u;
        if constexpr (PAIR) {
          astore.peer_slot = cluster_map_u32(smem_u32(xch_smem + cgp * 128 + r), crank ^ 1u);
          astore.buf_off = (uint32_t)(Q * 128 * sizeof(uint4));               // buffer 1
          astore.peer_bar = peer_xbar + 8u;
          if (crank != 0) {                                                   // CTA 1: partial minima go to CTA 0 (peer)
            hc.part_remote = part_remote0 + (uint32_t)(part_buf_floats * sizeof(float));
            hc.part_mbar = peer_xbar + 8u;
          }
        }
        // PAIR: hand this warp's slices of step t to the peer (t = -1: s_0) and, when a next step follows,
        // fetch the peer's half of x_{t+1} into the A operand
        auto exchange = [&](int t, bool next_step) {
          if constexpr (PAIR) {
            const uint32_t b = (uint32_t)t & 1u;
            if (next_step) {
              mbar_wait(my_xbar + 8u * b, (uint32_t)((t + 1) >> 1) & 1u);     // all of the peer's step-t stores have landed
              const uint4 v = xch_smem[(b * Q + cgp) * 128 + r];
              const uint32_t pk[4] = {v.x, v.y, v.z, v.w};
              tmem_st<4>(astore.t_a + (uint32_t)((((int)crank ^ 1) * 32 + cgp * 8) >> 1), pk);
            }
          }
        };
        const float* s0_ptr = prm.states + (prm.state_per_row ? id.r_global : (int64_t)id.s) * prm.state_stride;
        // TRAJ: this row's s_t in traj_out, advanced by one step before every head pass; FWD: its outputs
        typename std::conditional<FWD, ForwardSink, typename std::conditional<TRAJ, TrajSink, NoTraj>::type>::type sink{};
        if constexpr (FWD) {
          sink = ForwardSink{prm.mu_out, prm.var_out, prm.sample_out, row_ok ? (int)id.out : -1, O};
        } else if constexpr (TRAJ) {
          sink.row = row_ok ? prm.traj_out + id.out * (int64_t)(H + 1) * O : nullptr;
          sink.O = O;
        }

#ifdef SIMBA_TC_TIMELINE
        const int tl_who = (j == 0 && lane == 0) ? (wl == 0 ? 0 : (wl == kTileWarps - 1 ? 1 : -1)) : -1;
        int tl_t = 0;
#endif
        // this warp's slice of the tile's next A operand is complete: stores landed and ordered before
        // the issuer's MMAs; count the warp in on "A ready" without waiting
        // one tile: the warps of column groups 0-1 hand off through the low half's barriers, 2-3 the high half's
        static_assert(!kDbl || kBarAccHi - kBarAcc == kBarAHi - kBarA, "one offset selects both barriers of a half");
        const int bar_off = kDbl ? (cgp >= Q / 2 ? kBarAHi - kBarA : 0) : j;
        const int bar_acc_mine = kBarAcc + bar_off, bar_a_mine = kBarA + bar_off;
        const int hand_off_threads = kDbl ? half_bar_threads : tile_bar_threads;
        auto publish_a = [&]() {
          tmem_st_wait();
          tc_fence_before();
          named_bar_arrive_n(bar_a_mine, hand_off_threads);
        };
        auto wait_accumulator = [&]() {
          // released by the issuer warp's arrive. (Letting the sixteen epilogue warps sleep on the commit
          // mbarrier themselves is slower even in the one-tile variant: commit -> accumulator seen 496
          // cycles instead of 408 through the relay, measured.)
          named_bar_sync_n(bar_acc_mine, hand_off_threads);
          tc_fence_after();
        };
        // one tile: buffers of GEMM l of step t (GEMM n of the item uses accumulator and A buffer n & 1)
        auto gemm_par = [&](int t, int l) { return (uint32_t)(t * (L + 1) + l) & 1u; };

        // the thread whose column slice holds state column O prefetches a_{t+1} one step ahead (the L2
        // latency is off the critical path) and parks it in state columns [O, O + A) of its row
        // (tc_head.cuh head_store_actions; A <= 4 on this path). TRAJ: every thread whose slice meets
        // [O, O + A) fetches the actions and stores its own columns of them (head_store_own_actions).
        const bool owns_actions = TRAJ ? (O < hc.o_base + OW) && (O + A > hc.o_base)
                                       : (O >= hc.o_base) && (O < hc.o_base + OW);
        float act_pf[4] = {0.f, 0.f, 0.f, 0.f};
        auto prefetch_actions = [&](int tn) {
          if (owns_actions && row_ok && tn < H) {
#pragma unroll
            for (int a = 0; a < 4; ++a)
              if (a < A) act_pf[a] = act_ptr[tn * A + a];
          }
        };

        // N(0,1) draws of this thread's OW outputs for the current step. They depend only on
        // (seed, iteration, t, row, o), not on the network, so they are produced one Philox block
        // (8 normals) at a time right after this warp has handed a hidden layer's A slice to the
        // issuer, i.e. in the shadow of the tensor-core work instead of inside the head epilogue.
        typename std::conditional<kPark, NoiseSmem<NB, kEpiThreads>, NoiseRegs<NB>>::type noise;
        if constexpr (kPark) noise.base = noise_smem + threadIdx.x;
#pragma unroll
        for (int b = 0; b < NB; ++b) noise.put4(b, make_uint4(0u, 0u, 0u, 0u));
        const uint32_t c3_noise = (uint32_t)id.s | (kStreamNoise << 28);
        const uint32_t row32 = (uint32_t)id.r_global;
        const float* eps_row = prm.eps == nullptr ? nullptr
            : prm.eps + ((int64_t)id.s * H * ((int64_t)g.P * g.N) + id.r_global) * O;
        const int64_t eps_step = (int64_t)g.P * g.N * O;
        // One Philox block (8 draws) of step t; b may be a run-time value (one call site per layer keeps the
        // layer loop small: the kernel is far larger than the instruction cache).
        const uint64_t seed64 = *seed_sh;
        const uint2 key = make_uint2((uint32_t)seed64, (uint32_t)(seed64 >> 32));
        const uint32_t c2_base = (uint32_t)prm.iteration << 16;
        auto make_noise = [&](int b, int t) {
          const int o0 = hc.o_base + b * 8;
          if (o0 >= O) return;                              // warp-uniform: nothing to draw
          uint4 z;
          if (FWD || eps_row != nullptr) {                 // FWD: external draws only (sampling_propagation)
            z = external_noise8_bf16(eps_row + t * eps_step, o0, O);
          } else {
#ifdef SIMBA_TC_TIMELINE
            {
              PhiloxState p{(uint32_t)(o0 >> 3), row32, (uint32_t)t | c2_base, c3_noise, key.x, key.y};
              TL(50);
              philox_rounds<10>(p);
              if (p.c0 == 0x12345u) TL(53);
              TL(51);
              z = philox_finish_noise8_bf16(p);
              if (z.x == 0x12345u) TL(53);
              TL(52);
            }
#else
            z = philox_noise8_bf16(key, (uint32_t)(o0 >> 3), row32, (uint32_t)t | c2_base, c3_noise);
#endif
            if (o0 + 8 > O) z = mask_noise8(z, o0, O);      // padded outputs draw nothing (their delta is 0)
          }
          noise.put4_dyn(b, z);
        };
        // PAIR: s_0 does not depend on the previous kernel — its loads are in flight across the dependency wait
        float s0v[8];
        if constexpr (PAIR) {
#pragma unroll
          for (int i = 0; i < 8; ++i) s0v[i] = (row_ok && hc.o_base + i < O) ? s0_ptr[hc.o_base + i] : 0.0f;
        }
        const bool live = late_gate(ti);
        if (live) {
        prefetch_actions(0);
        if constexpr (PAIR) head_first_pass_vals(hc, astore, s0v, act_pf);
        else head_first_pass<OW>(hc, astore, s0_ptr, row_ok, act_pf, sink);
        prefetch_actions(1);
        exchange(-1, true);
        publish_a();                                        // layer-0 input of step 0
        TLK(3);
        if (keeps_score) named_bar_arrive_n(kBarPart + j, tile_bar_threads);  // partial minima of s_0 published (scorer warp)

        PhiloxState ps{0u, 0u, 0u, 0u, 0u, 0u};             // a noise block in flight across two layers (latency variant)
        for (int t = 0; t < H; ++t) {
#ifdef SIMBA_TC_TIMELINE
          tl_t = t;
#endif
          TL(0);
          if (owns_actions) {                                 // a_{t+1}, fetched during step t - 1
            if constexpr (TRAJ) head_store_own_actions<OW>(hc, act_pf);
            else head_store_actions(hc, act_pf);
          }
          prefetch_actions(t + 2);
          // ---- hidden layers: TMEM accumulator (bias included) -> ReLU -> bf16 -> next A operand ------
          for (int l = 0; l < L; ++l) {
            wait_accumulator();
            TL(1 + l * 4);
            {
              constexpr int NLD = HCOLS / 32;                // 32-column loads per thread (2 at Q = 2)
              uint32_t v[NLD][32];
#pragma unroll
              for (int i = 0; i < NLD; ++i) tmem_ld<32>(t_acc + (kDbl ? gemm_par(t, l) * 128 : 0u) + (uint32_t)(cgp * HCOLS + i * 32), v[i]);
              tmem_ld_wait();
#pragma unroll
              for (int i = 0; i < NLD; ++i) {
                uint32_t pk[16];
#pragma unroll
                for (int q = 0; q < 16; ++q)
                  pk[q] = pack_relu_bf16(__uint_as_float(v[i][2 * q]), __uint_as_float(v[i][2 * q + 1]));
                tmem_st<16>(t_a + (kDbl ? (gemm_par(t, l) ^ 1u) * 64 : 0u) + (uint32_t)((cgp * HCOLS + i * 32) / 2), pk);
              }
            }
            TL(2 + l * 4);
            publish_a();
            TL(3 + l * 4);
            if (prm.sampling_propagation) {
              if (!FWD && NTILES == 1 && L >= 2 * NB && eps_row == nullptr) {
                // latency variant: a whole block (~1.3 k cycles for a lone warp: two serial dependency
                // chains) is longer than one layer's MMA shadow, so it is split over two layers — the ten
                // Philox rounds after an even layer, Box-Muller after the following odd one
                const int b = l >> 1, o0 = hc.o_base + b * 8;
                if (b < NB && o0 < O) {
                  if ((l & 1) == 0) {
                    ps = PhiloxState{(uint32_t)(o0 >> 3), row32, (uint32_t)t | c2_base, c3_noise, key.x, key.y};
                    philox_rounds<10>(ps);
                  } else {
                    uint4 z = philox_finish_noise8_bf16(ps);
                    if (o0 + 8 > O) z = mask_noise8(z, o0, O);
                    noise.put4_dyn(b, z);
                  }
                }
              } else {
                // the NB Philox blocks of the step, one per hidden layer (the last layer takes the rest)
                if (l < NB) make_noise(l, t);
                if (l == L - 1)
                  for (int b = L; b < NB; ++b) make_noise(b, t);
              }
            }
            TL(4 + l * 4);
          }

          // ---- Gaussian heads + state update + next input + partial minima (one fused pass) --------
          wait_accumulator();
          if (keeps_score) named_bar_sync_n(kBarFree + j, tile_bar_threads);  // the scorer warp is done with the previous partials
          TL(40);
          if constexpr (PAIR) {
            hc.part = part_slot0 + (t & 1) * part_buf_floats;
            astore.buf_off = (uint32_t)((t & 1) * Q * 128 * sizeof(uint4));
            astore.peer_bar = peer_xbar + 8u * ((uint32_t)t & 1u);
            if (crank != 0) {
              hc.part_remote = part_remote0 + (uint32_t)((t & 1) * part_buf_floats * sizeof(float));
              hc.part_mbar = astore.peer_bar;
            }
          }
          if constexpr (TRAJ && !FWD) {
            if (sink.row != nullptr) sink.row += O;
          }
          if constexpr (kDbl) {                             // the head GEMM's accumulator, x_{t+1} into the other A buffer
            hc.t_acc = t_acc + gemm_par(t, L) * 128;
            astore.t_a = t_a + (gemm_par(t, L) ^ 1u) * 64;
          }
          if constexpr (FWD) head_step_pass<OW, true>(hc, noise, astore, false, sink);
          else if (prm.sampling_propagation) head_step_pass<OW, true>(hc, noise, astore, t + 1 < H, sink);
          else head_step_pass<OW, false>(hc, noise, astore, t + 1 < H, sink);
          TL(41);
          exchange(t, t + 1 < H);
          if (t + 1 < H) publish_a();                       // next step's layer 0 goes out
          if (keeps_score) named_bar_arrive_n(kBarPart + j, tile_bar_threads);  // partial minima of s_{t+1} published (scorer warp)
          TL(42);
        }
        TLK(6);
        }  // live
      }
    }
  }

  tc_fence_before();
  __syncthreads();                                  // end of the item: tile info, exchange buffers and TMEM columns are free again
  tc_fence_after();
  }  // items

  if (threadIdx.x == 0 && w_state_sh[1] > 0) mbar_wait(bar_w, (uint32_t)(w_state_sh[1] - 1) & 1u);   // never exit with a bulk copy into this CTA's memory pending
  tc_fence_before();
  __syncthreads();
  // PAIR: no cluster barrier is needed here. The last stores into the peer's memory are the step H - 2 input
  // slices, which the peer consumed before its last step, and CTA 1's last partial minima, which CTA 0's
  // scorer warp waited for before the barrier above; st.async data travels from registers, so the sender
  // may exit first.
  TLK(4);
  if (warp == 0) tmem_dealloc(tmem_base, kTmemCols);
  TLK(5);
}

template <int NTILES, int Q, bool PAIR>
__global__ void __launch_bounds__(kBoundThreads, 1) rollout_tc_kernel(const RolloutParams prm) {
  rollout_tc_body<NTILES, Q, PAIR, false>(prm);
}

// the trajectory form (simba_unfold_tc): <1, 4> and the persistent two-tile <2, 2>
template <int NTILES, int Q>
__global__ void __launch_bounds__(kBoundThreads, 1) unfold_tc_kernel(const RolloutParams prm) {
  rollout_tc_body<NTILES, Q, false, true>(prm);
}

// the forward form (simba_ensemble_forward_tc): the same two variants at H = 1
template <int NTILES, int Q>
__global__ void __launch_bounds__(kBoundThreads, 1) forward_tc_kernel(const RolloutParams prm) {
  rollout_tc_body<NTILES, Q, false, true, true>(prm);
}

// ---- host side ------------------------------------------------------------------------------------
static size_t tc_smem_bytes(int L, int ntiles, int q, int nparts, bool pair = false) {
  size_t b = tc_member_bytes(L) + 4096;                            // weights, bias K-blocks + ones tile
  b += 128 * sizeof(float);                                        // scaler
  b += kHeadParts * 64 * sizeof(float);                            // slice penalty table
  b += (size_t)ntiles * q * nparts * 128 * sizeof(float) * (pair ? 4 : 1);   // partial minima exchange (pair: 2 x 2 q slices)
  if (pair) b += (size_t)2 * q * 128 * sizeof(uint4);              // next-input slices from the peer CTA
  if (ntiles > 1)                                                  // parking area of the two-tile variant:
    b += (size_t)(64 / q / 8) * (ntiles * q * 128) * sizeof(uint4);      // bf16x2 noise of the current step
  b += (size_t)8 * ntiles * 128 * sizeof(uint32_t);                      // per-row running objective
  b += (3 + ntiles + (ntiles == 1 ? 1 : 0)) * sizeof(uint64_t) + 2 * sizeof(uint32_t) + ntiles * sizeof(TileInfo) + sizeof(uint64_t) + 2 * sizeof(int32_t);
  return b + 1024;                                                 // alignment slack
}

constexpr size_t kMaxSmem = 227 * 1024;

bool rollout_tc_supported(int O, int A, int L, int U) {
  // narrower hidden layers run zero-padded to 128 units (rollout_tc_pack pads the image); the
  // member's whole weight set must fit in shared memory next to the one-tile variant's buffers
  return U >= 1 && U <= kU && O >= 1 && O <= kMaxO && O + A <= 64 && A <= 4 && L >= 1 &&
         tc_smem_bytes(L, 1, 4, kHeadParts) + 1024 <= kMaxSmem;
}

// The image, per member, in the order stage_weights copies it into shared memory:
//   * per layer the UMMA B operand B[n][k] = W[k][n], K-major SWIZZLE_128B: one [128 rows][128 bytes] slab per
//     64-wide K atom, layer 0 one atom (K = O + A, zero-padded), every later layer two (K = units, zero-padded to
//     128). Heads: mu -> rows [0, O), var -> rows [64, 64 + O), the raw-variance head pre-scaled by log2(e). When
//     tc_l0_pad_bias, layer 0 carries its bias as bf16 hi / lo in k = IN, IN + 1, where the kernel feeds ones;
//   * then per layer its bias as one more K = 16 block of its GEMM, B[n][0] = hi, B[n][1] = lo, K-major
//     SWIZZLE_NONE: 8-row x 16-byte core matrices, the two K halves 128 B apart (leading byte offset), 8-row groups
//     256 B apart (stride byte offset) -> kBiasBlockBytes per layer.
int64_t rollout_tc_pack(const ModelWeights& mw, std::vector<uint16_t>& img) {
  const auto& c = mw.cfg;
  const int L = c.n_layers, E = c.ensemble_size, U = c.units, O = c.obs_dim, IN = c.obs_dim + c.act_dim;
  const int64_t member_bytes = tc_member_bytes(L);
  img.assign((size_t)E * member_bytes / 2, 0);
  for (int e = 0; e < E; ++e) {
    uint16_t* w = &img[(size_t)e * member_bytes / 2];
    uint16_t* bias_k16 = w + tc_weight_bytes(L) / 2;
    for (int l = 0; l <= L; ++l) {
      const int K = l == 0 ? IN : U;
      auto weight = [&](int k, int n) -> uint16_t {     // n = tile row (output feature)
        if (l == 0 && tc_l0_pad_bias(IN) && (k == IN || k == IN + 1) && n < U) {
          uint16_t hi, lo;
          bf16_split(mw.bias(e, 0)[n], hi, lo);
          return k == IN ? hi : lo;
        }
        if (k >= K) return 0;
        if (l < L) return n < U ? bf16_bits(mw.kernel(e, l)[(size_t)k * U + n]) : 0;
        if (n < O) return bf16_bits(mw.kernel(e, L)[(size_t)k * O + n]);
        if (n >= 64 && n < 64 + O) return bf16_bits(kLog2e * mw.kernel(e, L + 1)[(size_t)k * O + (n - 64)]);
        return 0;
      };
      const int atoms = l == 0 ? 1 : 2;
      for (int at = 0; at < atoms; ++at)
        for (int n = 0; n < 128; ++n)
          for (int kk = 0; kk < 64; ++kk) w[(at * kAtomBytes + sw128_offset(n, kk)) / 2] = weight(at * 64 + kk, n);
      w += atoms * kAtomBytes / 2;
      for (int n = 0; n < 128; ++n) {
        float bv = 0.0f;
        if (l < L) bv = n < U ? mw.bias(e, l)[n] : 0.0f;
        else if (n < O) bv = mw.bias(e, L)[n];
        else if (n >= 64 && n < 64 + O) bv = kLog2e * mw.bias(e, L + 1)[n - 64];
        uint16_t* bk = bias_k16 + l * kBiasBlockBytes / 2 + (n / 8) * 128 + (n % 8) * 8;
        bf16_split(bv, bk[0], bk[1]);
      }
    }
  }
  return member_bytes;
}

// whether the two-tile throughput variant (and its shared-memory parking areas) fits for this depth
bool rollout_tc_two_tiles_fit(int L, int n_constraints) {
  return tc_smem_bytes(L, 2, 2, 1 + n_constraints) + 1024 <= kMaxSmem;
}

// whether the two-CTA latency variant (doubled partial-minima buffers + the peer exchange) fits
bool rollout_tc_pair_fits(int L, int n_constraints) {
  return tc_smem_bytes(L, 1, 4, 1 + n_constraints, true) + 1024 <= kMaxSmem;
}

template <int NTILES, int Q, bool PAIR, bool TRAJ, bool FWD = false>
static cudaError_t launch_variant(const RolloutParams& prm, cudaStream_t stream) {
  void (*kern)(const RolloutParams) = rollout_tc_kernel<NTILES, Q, PAIR>;
  if constexpr (FWD) kern = forward_tc_kernel<NTILES, Q>;
  else if constexpr (TRAJ) kern = unfold_tc_kernel<NTILES, Q>;
  const size_t smem = tc_smem_bytes(prm.L, NTILES, Q, TRAJ ? 1 : 1 + prm.scorer.n_constraints, PAIR);
  const int n_items = (prm.n_tiles + NTILES - 1) / NTILES;
  const int sms = prm.n_sms;
  if (sms <= 0) return cudaErrorInvalidValue;
  // persistent CTAs (one per SM, 1 CTA / SM by shared memory and TMEM); the pair variant runs one item per cluster
  const int grid = PAIR ? 2 * n_items : (n_items < sms ? n_items : sms);
  // epilogue warps + an issuer and a scorer warp per tile (+ the one-tile variants' relay warp)
  return launch_kernel(kern, grid, NTILES * Q * 128 + 64 * NTILES + (NTILES == 1 ? 32 : 0), smem, stream, PAIR ? 2 : 1, prm.pdl, prm);
}

cudaError_t launch_rollout_tc(const RolloutParams& prm, cudaStream_t stream) {
  if (prm.mu_out != nullptr) {
    switch (prm.kernel) {   // the forward form: the trajectory form's variants
      case RolloutKernel::kTcOneCta: return launch_variant<1, 4, false, true, true>(prm, stream);
      case RolloutKernel::kTcTwoTile: return launch_variant<2, 2, false, true, true>(prm, stream);
      default: return cudaErrorInvalidValue;
    }
  }
  if (prm.traj_out == nullptr) {
    switch (prm.kernel) {
      case RolloutKernel::kTcOneCta: return launch_variant<1, 4, false, false>(prm, stream);
      case RolloutKernel::kTcPair: return launch_variant<1, 4, true, false>(prm, stream);
      case RolloutKernel::kTcTwoTile: return launch_variant<2, 2, false, false>(prm, stream);
      default: return cudaErrorInvalidValue;
    }
  }
  switch (prm.kernel) {   // the trajectory form has no pair variant
    case RolloutKernel::kTcOneCta: return launch_variant<1, 4, false, true>(prm, stream);
    case RolloutKernel::kTcTwoTile: return launch_variant<2, 2, false, true>(prm, stream);
    default: return cudaErrorInvalidValue;
  }
}

}  // namespace simba

// bf16 tcgen05 rollout + scoring kernel for WIDE ensembles (128 < units <= 416, e.g. the 4x400
// model of BASELINE configs[4]) — same contract as rollout_tc.cu / rollout_f32.cu.
//
// A member's weights (1.2 MB for 4x400) no longer fit in shared memory, and a 400-column fp32
// accumulator fills tensor memory, so the kernel is a warp-specialised streaming pipeline:
//
//   * producer warp: streams the member's pre-swizzled UMMA weight tiles ([units n x 64 k] bf16,
//     51 KB) from L2 through a two-stage TMA ring (cp.async.bulk + full / empty mbarriers). The
//     tile sequence of a rollout step (layer 0, (L-1) x KA hidden K-blocks, KA head K-blocks) is
//     the same for every step, so the producer just cycles through it, decoupled from the math;
//   * MMA warp (one thread chosen with elect.sync, so that ptxas keeps the tcgen05.mma operands in
//     uniform registers instead of wrapping every MMA in an operand waterfall loop): per layer
//     bar.sync's on "A ready", then per K-block waits for the stage, issues 4 x tcgen05.mma (K = 16)
//     per N half (N = 208 + 192 for 400 units; N = 128 for the heads) with both operands in shared
//     memory, and tcgen05.commit's the stage back to the producer; after the last K-block it commits
//     onto an mbarrier, waits for it and bar.arrive's on "accumulator ready";
//   * 4 x 128 epilogue threads (Q = 4 per rollout row, as in rollout_tc.cu): bar.sync on
//     "accumulator ready" (hardware named barrier: no polling), drain the fp32 accumulator row from
//     TMEM, ReLU, pack bf16 and store 16-byte chunks into the 128B-swizzled K-major A tile in
//     shared memory (7 atoms of [128 x 64] for 400 units), fence to the async proxy and bar.arrive
//     on "A ready". The Gaussian-head / state / scoring pass is tc_head.cuh's (shared with
//     rollout_tc.cu: state in spare TMEM columns, Philox noise in the shadow of the hidden layers),
//     writing the next step's scaled input into atom 0 of the A tile.
//   * biases ride in the K padding: the A tile holds constant ones at k = K_real, K_real + 1 and
//     the weight tiles hold bf16(b) and bf16(b - hi) in those two k rows, so no epilogue touches
//     a bias (K_real = 62 -> 64 for layer 0, 400 -> 448 for the others).
//
// The state width kSW is a template parameter. kSW = 64 is the wide-model kernel described above (TMEM
// state columns [448, 512), heads N = 128: mu in rows [0, O), raw var in rows [64, 64 + O)). kSW = 128
// runs observations up to obs_dim + act_dim + 2 = 128 for any hidden width up to 384: layer 0 spans two
// K atoms, the state sits in TMEM columns [384, 512), the heads are one N = 256 MMA per K-step (mu in rows
// [0, O), raw var in rows [128, 128 + O)) and each epilogue thread owns 32 outputs (4 Philox blocks per
// step; obs_dim <= 124, so that the four action columns at O stay inside the state). Its hidden widths are padded
// to at least 128, so the hidden layers' constant ones (k = U, U + 1)
// lie beyond the layer-0 input that the head pass rewrites every step (k < 128).
#include <algorithm>
#include <cstdlib>
#include <type_traits>

#include "common.cuh"
#include "internal.h"
#include "rollout_params.cuh"
#include "tc_head.cuh"
#include "tc_ptx.cuh"

namespace simba {

// Debug timeline (compile with -DSIMBA_TC_TIMELINE): epilogue thread 0 and the last epilogue warp's
// lane 0 of CTA 0 stamp clock64() at phase boundaries into prm.timeline (tools/tc_timeline.py c5).
#ifdef SIMBA_TC_TIMELINE
#define TLW(ev)                                                                                  \
  do {                                                                                           \
    if (tl_who >= 0 && blockIdx.x == 0)                                                          \
      prm.timeline[(tl_who * 64 + tl_t) * 64 + (ev)] = clock64();  \
  } while (0)
#else
#define TLW(ev) do { } while (0)
#endif

namespace {

constexpr int kQ = 4;                         // epilogue threads per rollout row
constexpr int kEpiThreads = kQ * 128;
constexpr int kWideThreads = kEpiThreads + 64;   // + producer warp + MMA warp
constexpr int kAtomBytes = 128 * 128;         // one 64-wide K atom of a 128-row tile (bf16, SW128)
constexpr int kStages = 2;
constexpr int kBarEpi = 1, kBarAcc = 2, kBarA = 3, kBarScore = 4;   // named barrier ids
constexpr int kTmemCols = 512;

// Layout constants of the variant with state width kSW (64 or 128)
template <int kSW>
struct WideCfg {
  static constexpr int kStateCol = kTmemCols - kSW;   // TMEM: accumulator columns [0, units), state [kStateCol, 512)
  static constexpr int OW = kSW / kQ;                 // head outputs / state dims / layer-0 K elements per thread
  static constexpr int NB = OW / 8;                   // Philox blocks / 8-wide chunks per thread and step
  static constexpr int kL0Atoms = kSW / 64;           // K-blocks of layer 0
  static constexpr int kHeadN = 2 * kSW;              // head rows: mu at [0, O), raw var at [kSW, kSW + O)
  // head K-blocks ([kHeadN x 64] bf16: 16 or 32 KB) fetched per TMA tile. At kSW = 128 a block alone is as
  // large as three of the narrow variant's, and two per stage would not leave room for a 320-unit A tile.
  static constexpr int kHeadGroup = kSW == 64 ? 3 : 1;
  static constexpr int kMinUnits = kSW == 64 ? 0 : 128;   // see the file comment
  static constexpr int kMaxUnits = kSW == 64 ? 448 - 2 : kStateCol;
};

struct WideShape {
  int U, KA, L;
  uint32_t hid_tile_bytes;      // [U x 64] bf16
  uint32_t head_tile_bytes;     // [kHeadN x 64] bf16 (one K-block; kHeadGroup of them travel together)
  int head_tiles;               // ceil(KA / kHeadGroup)
  int tiles_per_step;
};

template <int kSW>
__host__ __device__ inline WideShape wide_shape(int U, int L) {
  using C = WideCfg<kSW>;
  WideShape s;
  s.U = U; s.L = L;
  s.KA = (U + 2 + 63) / 64;
  s.hid_tile_bytes = (uint32_t)U * 128u;
  s.head_tile_bytes = (uint32_t)C::kHeadN * 128u;
  s.head_tiles = (s.KA + C::kHeadGroup - 1) / C::kHeadGroup;
  s.tiles_per_step = C::kL0Atoms + (L - 1) * s.KA + s.head_tiles;
  return s;
}

template <int kSW>
__host__ __device__ inline uint32_t wide_stage_bytes(const WideShape& s) {
  const uint32_t head = (uint32_t)WideCfg<kSW>::kHeadGroup * s.head_tile_bytes;
  const uint32_t big = s.hid_tile_bytes > head ? s.hid_tile_bytes : head;
  return (big + 1023u) & ~1023u;
}

// source offset / size of tile `i` of the per-step stream
template <int kSW>
__device__ __forceinline__ void wide_tile(const WideShape& s, int i, uint32_t& off, uint32_t& bytes) {
  constexpr int kHeadGroup = WideCfg<kSW>::kHeadGroup;
  const int n_hid = WideCfg<kSW>::kL0Atoms + (s.L - 1) * s.KA;
  if (i < n_hid) { off = (uint32_t)i * s.hid_tile_bytes; bytes = s.hid_tile_bytes; return; }
  // the heads' K-blocks are small (16 KB), so kHeadGroup consecutive ones travel as one tile: with
  // one block per tile the two-stage ring was latency-bound there (4.9 k cycles for 2.6 k of MMAs)
  const int ht = i - n_hid;
  const int blocks = min(kHeadGroup, s.KA - ht * kHeadGroup);
  off = (uint32_t)n_hid * s.hid_tile_bytes + (uint32_t)(ht * kHeadGroup) * s.head_tile_bytes;
  bytes = (uint32_t)blocks * s.head_tile_bytes;
}

struct TileInfoW {
  int32_t member, k0, count, valid;
};

}  // namespace

// TRAJ (simba_unfold_tc): the trajectory form. The epilogue threads write s_0 and every s_{t+1} of their valid
// rows to prm.traj_out [B, H + 1, O] (tc_head.cuh TrajSink) and score nothing (no partial minima, no objective,
// no scorer struct read). Each thread whose column slice meets the action block stores its own action columns
// (head_store_own_actions). H is bounded only by the 16 bits of the Philox step counter.
//
// FWD (simba_ensemble_forward_tc): the forward form, a TRAJ form at H = 1 that writes the Gaussian head's mu, var
// and (with external draws) sample of its valid rows to prm.mu_out, var_out and sample_out [B, O] instead of the
// state (tc_head.cuh ForwardSink). Its head pass always forms the variance; without draws the noise stays zero.
// ACT: the hidden layers' activation, applied where drain_chunks packs the accumulator to bf16 (rollout_tc.cu)
template <int kSW, bool TRAJ, bool FWD = false, int ACT = kActRelu>
__device__ __forceinline__ void rollout_tc_wide_body(const RolloutParams& prm) {
  static_assert(!FWD || TRAJ, "the forward form is a trajectory form");
  using C = WideCfg<kSW>;
  constexpr int kStateCol = C::kStateCol, OW = C::OW, NB = C::NB, kHeadGroup = C::kHeadGroup;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const RowGeom& g = prm.g;
  const int L = prm.L, U = prm.U;
  const int H = g.H;
  const int O = g.O, A = g.A;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const WideShape ws = wide_shape<kSW>(U, L);
  const int KA = ws.KA;

  // ---- shared memory carve-up (base is 1024-aligned: required by SWIZZLE_128B) -------------------
  uint8_t* a_smem = smem_raw;                                              // [KA][128 x 64] bf16 SW128
  uint8_t* b_smem = a_smem + (size_t)KA * kAtomBytes;                      // [kStages][U x 64] bf16 SW128
  const uint32_t stage_bytes = wide_stage_bytes<kSW>(ws);
  float* scale_smem = reinterpret_cast<float*>(b_smem + (size_t)kStages * stage_bytes);   // [2][kSW]
  float* pen_smem = scale_smem + 2 * kSW;                                  // [kParts][kSW]
  const int nparts = TRAJ ? 1 : 1 + prm.scorer.n_constraints;
  float* part_smem = pen_smem + kHeadParts * kSW;                              // [kQ][nparts][128]
  // running objective of every rollout row (RowScore fields, field-major), see rollout_tc.cu
  uint32_t* rs_smem = reinterpret_cast<uint32_t*>(part_smem + kQ * nparts * 128);   // [8][128]
  uint64_t* bars = reinterpret_cast<uint64_t*>(rs_smem + 8 * 128);
  // bars: [0,1] full, [2,3] empty, [5] MMAs of the layer committed ("A ready" / "accumulator ready" hand-offs
  // are named barriers)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 6);
  TileInfoW* tinfo = reinterpret_cast<TileInfoW*>(tmem_slot + 2);

  const uint32_t bar_full[kStages] = {smem_u32(&bars[0]), smem_u32(&bars[1])};
  const uint32_t bar_empty[kStages] = {smem_u32(&bars[2]), smem_u32(&bars[3])};
  const uint32_t bar_acc = smem_u32(&bars[5]);

  pdl_launch_dependents();
  if (threadIdx.x == 0) {
    for (int s = 0; s < kStages; ++s) { mbar_init(bar_full[s], 1); mbar_init(bar_empty[s], 1); }
    mbar_init(bar_acc, 1);
    fence_barrier_init();
  }
  if (warp == 0) tmem_alloc(smem_u32(tmem_slot), kTmemCols);
  pdl_wait_prior_grid();
  if (threadIdx.x == 0) {
    TileInfoW info{0, 0, 0, 0};
    if ((int)blockIdx.x < prm.n_tiles) {
      const Tile t = prm.tiles[blockIdx.x];
      info.member = t.member; info.k0 = t.k0; info.count = t.count;
      bool any = t.count > 0;
      if (any && prm.active != nullptr) {                     // cem_mpc.py:66-67 early exit
        const int m = g.rows_per_state[t.member];
        any = false;
        for (int s = t.k0 / m; s <= (t.k0 + t.count - 1) / m; ++s) any = any || prm.active[s] != 0;
      }
      info.valid = any ? 1 : 0;
    }
    tinfo[0] = info;
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const TileInfoW ti = tinfo[0];

  if (ti.valid) {
    if (warp == kEpiThreads / 32) {
      // ===================== producer warp: weight tiles through the TMA ring =====================
      if (elect_one()) {
        const uint8_t* wsrc = reinterpret_cast<const uint8_t*>(prm.w_tc) + (size_t)ti.member * prm.w_tc_member_bytes;
        const int total = H * ws.tiles_per_step;
        int in_step = 0;
        for (int i = 0; i < total; ++i) {
          const int s = i % kStages;
          if (i >= kStages) mbar_wait(bar_empty[s], ((i / kStages) - 1) & 1);
          uint32_t off, bytes;
          wide_tile<kSW>(ws, in_step, off, bytes);
          mbar_expect_tx(bar_full[s], bytes);
          bulk_g2s(smem_u32(b_smem + (size_t)s * stage_bytes), wsrc + off, bytes, bar_full[s]);
          if (++in_step == ws.tiles_per_step) in_step = 0;
        }
      }
    } else if (warp == kEpiThreads / 32 + 1) {
      // ===================== MMA warp: one elected thread issues every tcgen05.mma ================
      const int N1 = ((U / 2 + 15) / 16) * 16, N2 = U - N1;        // two N halves, multiples of 16
      const uint32_t idesc1 = umma_idesc_n((uint32_t)N1), idesc2 = umma_idesc_n((uint32_t)N2);
      const uint32_t idesc_head = umma_idesc_n((uint32_t)C::kHeadN);
      const uint32_t a_base = smem_u32(a_smem);
      int tile0 = 0;                                               // ring position at the start of the layer
      uint32_t acc_ph = 0;
      for (int t = 0; t < H; ++t) {
        for (int layer = 0; layer <= L; ++layer) {
          named_bar_sync<kEpiThreads + 32>(kBarA);                 // this layer's A tile is complete
          tc_fence_after();
          const int n_tiles_layer = layer < L ? (layer == 0 ? C::kL0Atoms : KA) : ws.head_tiles;
          if (elect_one()) {
            int tile = tile0;                                      // running index into the ring
            if (layer < L) {
              const int kblocks = layer == 0 ? C::kL0Atoms : KA;
              for (int kb = 0; kb < kblocks; ++kb, ++tile) {
                const int s = tile % kStages;
                mbar_wait(bar_full[s], (tile / kStages) & 1);
                tc_fence_after();
                const uint64_t a_desc = umma_desc_sw128(a_base + (uint32_t)kb * kAtomBytes);
                const uint64_t b_desc = umma_desc_sw128(smem_u32(b_smem + (size_t)s * stage_bytes));
                const uint64_t b2_off = (uint64_t)(((uint32_t)N1 * 128u) >> 4);
#pragma unroll
                for (int k = 0; k < 4; ++k) {                      // UMMA_K = 16 -> 32 bytes along K (2 descriptor units)
                  const uint32_t acc = (kb > 0 || k > 0) ? 1u : 0u;
                  umma_bf16(tmem_base, a_desc + (uint64_t)(2 * k), b_desc + (uint64_t)(2 * k), idesc1, acc);
                  umma_bf16(tmem_base + (uint32_t)N1, a_desc + (uint64_t)(2 * k), b_desc + b2_off + (uint64_t)(2 * k),
                            idesc2, acc);
                }
                umma_commit(bar_empty[s]);                         // stage free once these MMAs retire
              }
            } else {
              for (int ht = 0; ht < ws.head_tiles; ++ht, ++tile) {
                const int s = tile % kStages;
                mbar_wait(bar_full[s], (tile / kStages) & 1);
                tc_fence_after();
                const uint64_t b_desc = umma_desc_sw128(smem_u32(b_smem + (size_t)s * stage_bytes));
                const int blocks = min(kHeadGroup, KA - ht * kHeadGroup);
                for (int jb = 0; jb < blocks; ++jb) {
                  const int kb = ht * kHeadGroup + jb;
                  const uint64_t a_desc = umma_desc_sw128(a_base + (uint32_t)kb * kAtomBytes);
                  const uint64_t bj = b_desc + (uint64_t)(((uint32_t)jb * ws.head_tile_bytes) >> 4);
#pragma unroll
                  for (int k = 0; k < 4; ++k)
                    umma_bf16(tmem_base, a_desc + (uint64_t)(2 * k), bj + (uint64_t)(2 * k), idesc_head,
                              (kb > 0 || k > 0) ? 1u : 0u);
                }
                umma_commit(bar_empty[s]);
              }
            }
            umma_commit(bar_acc);                                  // this layer's MMAs, all of them
          }
          tile0 += n_tiles_layer;                                  // every lane tracks the ring position
          __syncwarp();
          mbar_wait(bar_acc, acc_ph);                              // accumulator of this layer complete
          acc_ph ^= 1;
          tc_fence_before();
          named_bar_arrive<kEpiThreads + 32>(kBarAcc);             // wake the epilogue warps
        }
      }
    } else {
      // ============ epilogue warps: kQ threads per rollout row, each owns a column slice ============
      const int wl = warp;                                  // warp within the tile
      const int cgp = wl >> 2;                              // column group in [0, kQ)
      const int r = (wl & 3) * 32 + lane;                   // row in tile == TMEM lane
      // scaler / penalty tables, zeroed A tile with the constant ones of the bias rows
      {
        if constexpr (TRAJ)                                  // the penalty table is never read
          head_tables_init<kSW>(scale_smem, pen_smem, prm.tc_scale_a, prm.tc_scale_b, simba_scorer_t{}, O + A,
                                threadIdx.x, kEpiThreads);
        else
          head_tables_init<kSW>(scale_smem, pen_smem, prm.tc_scale_a, prm.tc_scale_b, prm.scorer, O + A, threadIdx.x,
                                kEpiThreads);
        uint32_t* a32 = reinterpret_cast<uint32_t*>(a_smem);
        for (int i = threadIdx.x; i < KA * kAtomBytes / 4; i += kEpiThreads) a32[i] = 0u;
        named_bar_sync<kEpiThreads>(kBarEpi);
        // ones at k = U, U + 1 of every row (same 16-byte chunk; U is a multiple of 8)
        if (threadIdx.x < 128) {
          const int row = threadIdx.x, c8 = U >> 3, atom = c8 >> 3, cin = c8 & 7;
          uint32_t* p = reinterpret_cast<uint32_t*>(a_smem + (size_t)atom * kAtomBytes + (row >> 3) * 1024 +
                                                    (row & 7) * 128 + ((cin ^ (row & 7)) * 16));
          p[0] = 0x3F803F80u;                                 // bf16 1.0, 1.0
        }
        fence_proxy_async();
        named_bar_sync<kEpiThreads>(kBarEpi);
      }
      const bool row_ok = r < ti.count;
      const RowId id = decode_row(g, ti.member, ti.k0 + (row_ok ? r : 0));
      const uint64_t seed = prm.seed_ptr ? *prm.seed_ptr : prm.seed;
      const uint32_t t_lane = tmem_base + ((uint32_t)((wl & 3) * 32) << 16);
      const float* act_ptr = prm.actions + ((int64_t)id.s * g.N + id.i_global) * prm.action_stride;
      const bool done_first = objective_done_first(prm.objective);
      const simba_scorer_t& sc = prm.scorer;
      const float* s0_ptr = prm.states + (prm.state_per_row ? id.r_global : (int64_t)id.s) * prm.state_stride;
      // TRAJ: this row's s_t in traj_out, advanced by one step before every head pass; FWD: its outputs
      typename std::conditional<FWD, ForwardSink, typename std::conditional<TRAJ, TrajSink, NoTraj>::type>::type sink{};
      if constexpr (FWD) {
        sink = ForwardSink{prm.mu_out, prm.var_out, prm.sample_out, row_ok ? (int)id.out : -1, O};
      } else if constexpr (TRAJ) {
        sink.row = row_ok ? prm.traj_out + id.out * (int64_t)(H + 1) * O : nullptr;
        sink.O = O;
      }
      const uint32_t a_row = smem_u32(a_smem) + (uint32_t)(r >> 3) * 1024u + (uint32_t)(r & 7) * 128u;
      const uint32_t rsw = (uint32_t)(r & 7);

      HeadCtx hc;
      hc.t_acc = t_lane;
      hc.t_state = t_lane + (uint32_t)kStateCol;
      hc.o_base = cgp * OW;
      hc.O = O; hc.A = A;
      hc.slice_bits = TRAJ ? 0u : head_slice_bits<OW>(sc, hc.o_base);
      hc.n_constraints = TRAJ ? 0 : sc.n_constraints;
      hc.scale_smem = scale_smem;
      hc.pen_smem = pen_smem;
      hc.part = part_smem + (cgp * nparts) * 128 + r;
      const float* part_row = part_smem + r;

      // 16-byte chunk `c8` (k = 8 c8 .. 8 c8 + 7) of this row in the swizzled A tile
      auto a_chunk = [&](int c8) -> uint32_t {
        return a_row + (uint32_t)(c8 >> 3) * kAtomBytes + ((((uint32_t)c8 & 7u) ^ rsw) << 4);
      };
      // A operand in shared memory: K elements [k0, k0 + 8) of this thread's row = one 16-byte chunk of the
      // layer-0 input (atom 0, and atom 1 for k0 >= 64 at kSW = 128)
      struct AStoreSmem {
        uint32_t a_row, rsw;
        __device__ __forceinline__ void store8(int k0, uint32_t p0, uint32_t p1, uint32_t p2, uint32_t p3) const {
          uint32_t a = a_row + ((((uint32_t)(k0 >> 3) & 7u) ^ rsw) << 4);
          if (C::kL0Atoms > 1) a += (uint32_t)(k0 >> 6) * kAtomBytes;
          st_shared_v4(a, p0, p1, p2, p3);
        }
      };
      const AStoreSmem astore{a_row, rsw};
      // this warp's part of the layer's A tile is complete: fence to the async proxy, count the warp in
      auto publish_a = [&]() {
        fence_proxy_async();
        tc_fence_before();
        named_bar_arrive<kEpiThreads + 32>(kBarA);
      };
      auto wait_accumulator = [&]() {
        named_bar_sync<kEpiThreads + 32>(kBarAcc);            // released by the MMA warp's arrive
        tc_fence_after();
      };

      // TRAJ: every thread whose slice meets [O, O + A) fetches and stores its own action columns, every step
      const bool meets_actions = (O < hc.o_base + OW) && (O + A > hc.o_base);
      const bool owns_actions = TRAJ ? meets_actions : (O >= hc.o_base) && (O < hc.o_base + OW);
      // a_0 goes into the state columns [O, O + A) of whichever slices hold them (head_first_pass); at kSW = 128
      // they may straddle two slices (O = 63, A = 2), so every thread whose slice meets them fetches a_0. Later
      // actions come from the owner alone (head_store_actions writes all four columns).
      const bool needs_a0 = (kSW == 64 && !TRAJ) ? owns_actions : meets_actions;
      float act_pf[4] = {0.f, 0.f, 0.f, 0.f};
      auto prefetch_actions = [&](int tn, bool mine) {
        if (mine && row_ok && tn < H) {
#pragma unroll
          for (int a = 0; a < 4; ++a)
            if (a < A) act_pf[a] = act_ptr[tn * A + a];
        }
      };
      // N(0,1) draws of this thread's outputs for the current step (tc_head.cuh), in registers
      struct NoiseRegs {
        uint4 v[NB];
        __device__ __forceinline__ uint4 get4(int b) const { return v[b]; }
      } noise;
#pragma unroll
      for (int b = 0; b < NB; ++b) noise.v[b] = make_uint4(0u, 0u, 0u, 0u);
      const uint32_t c3_noise = (uint32_t)id.s | (kStreamNoise << 28);
      auto make_noise = [&](auto btag, int t) {
        constexpr int b = decltype(btag)::value;
        const int o0 = hc.o_base + b * 8;
        if (o0 >= O) return;
        uint4 z;
        if (FWD || prm.eps != nullptr) {                   // FWD: external draws only (sampling_propagation)
          const float* ep = prm.eps + (((int64_t)id.s * H + t) * ((int64_t)g.P * g.N) + id.r_global) * O;
          z = external_noise8_bf16(ep, o0, O);
        } else {
          z = philox_noise8_bf16(make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)), (uint32_t)(o0 >> 3),
                                 (uint32_t)id.r_global, (uint32_t)t | ((uint32_t)prm.iteration << 16), c3_noise);
          if (o0 + 8 > O) {                                   // padded outputs draw nothing (their delta is 0)
            uint32_t w[4] = {z.x, z.y, z.z, z.w};
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              if (o0 + 2 * i >= O) w[i] = 0u;
              else if (o0 + 2 * i + 1 >= O) w[i] &= 0xffffu;
            }
            z = make_uint4(w[0], w[1], w[2], w[3]);
          }
        }
        noise.v[b] = z;
      };

      uint32_t* my_rs = rs_smem + r;                      // cum, costsum, cmask lo / hi, dist, cost, done
      prefetch_actions(0, needs_a0);
      head_first_pass<OW, kSW>(hc, astore, s0_ptr, row_ok, act_pf, sink);
      prefetch_actions(1, owns_actions);
      tmem_st_wait();
      publish_a();                                       // layer-0 input of step 0
      if constexpr (!TRAJ) named_bar_sync<kEpiThreads>(kBarScore);   // partial minima of s_0 visible to the scorers
      if (!TRAJ && cgp == 0) {
        float d0, c0;
        head_combine<kQ>(sc, part_row, nparts, d0, c0);
        my_rs[0] = 0u; my_rs[128] = 0u; my_rs[256] = 0u; my_rs[384] = 0u;
        my_rs[512] = __float_as_uint(d0);
        my_rs[640] = __float_as_uint(c0);
        my_rs[768] = 0u;
      }

#ifdef SIMBA_TC_TIMELINE
      const int tl_who = (lane == 0) ? (wl == 0 ? 0 : (wl == 4 * kQ - 1 ? 1 : -1)) : -1;
      int tl_t = 0;
#endif
      const int n_chunks = U >> 3;                       // 16-byte chunks per hidden activation row
      const int my_c0 = cgp * (n_chunks / kQ) + min(cgp, n_chunks % kQ);
      const int my_c1 = my_c0 + n_chunks / kQ + (cgp < n_chunks % kQ ? 1 : 0);
      for (int t = 0; t < H; ++t) {
#ifdef SIMBA_TC_TIMELINE
        tl_t = t;
#endif
        TLW(0);
        if (owns_actions) {                                 // a_{t+1}, fetched during step t - 1
          if constexpr (TRAJ) head_store_own_actions<OW>(hc, act_pf);
          else head_store_actions(hc, act_pf);
        }
        prefetch_actions(t + 2, owns_actions);
        // ---- hidden layers: TMEM -> activation -> bf16 -> swizzled A tile (bias is in the accumulator) ----
        for (int l = 0; l < L; ++l) {
          wait_accumulator();
          TLW(1 + l * 4);
          // this column group's contiguous run of 16-byte chunks (8 accumulator columns each): four at a
          // time through one 32-column TMEM load, then a 16- and an 8-column tail
          {
            auto drain_chunks = [&](auto ntag, int c) {
              constexpr int NC = decltype(ntag)::value;       // chunks in this load
              uint32_t v[NC * 8];
              tmem_ld<NC * 8>(t_lane + (uint32_t)c * 8, v);
              tmem_ld_wait();
#pragma unroll
              for (int u = 0; u < NC; ++u)
                st_shared_v4(a_chunk(c + u),
                             pack_act_bf16<ACT>(__uint_as_float(v[u * 8 + 0]), __uint_as_float(v[u * 8 + 1])),
                             pack_act_bf16<ACT>(__uint_as_float(v[u * 8 + 2]), __uint_as_float(v[u * 8 + 3])),
                             pack_act_bf16<ACT>(__uint_as_float(v[u * 8 + 4]), __uint_as_float(v[u * 8 + 5])),
                             pack_act_bf16<ACT>(__uint_as_float(v[u * 8 + 6]), __uint_as_float(v[u * 8 + 7])));
            };
            int c = my_c0;
            for (; c + 4 <= my_c1; c += 4) drain_chunks(std::integral_constant<int, 4>{}, c);
            if (c + 2 <= my_c1) { drain_chunks(std::integral_constant<int, 2>{}, c); c += 2; }
            if (c < my_c1) drain_chunks(std::integral_constant<int, 1>{}, c);
          }
          TLW(2 + l * 4);
          tmem_st_wait();                                  // (the action columns stored at the top of the step)
          publish_a();
          TLW(3 + l * 4);
          if (prm.sampling_propagation) {
            // the NB (2 or 4) Philox blocks of the step ride in the shadow of the hidden layers' MMAs: block b
            // after layer b, the blocks beyond the last layer after that one
            if (l == 0) make_noise(std::integral_constant<int, 0>{}, t);
            if (l == (L > 1 ? 1 : 0)) make_noise(std::integral_constant<int, 1>{}, t);
            if constexpr (NB > 2) {
              if (l == (L > 2 ? 2 : L - 1)) make_noise(std::integral_constant<int, 2>{}, t);
              if (l == (L > 3 ? 3 : L - 1)) make_noise(std::integral_constant<int, 3>{}, t);
            }
          }
        }
        // ---- Gaussian heads + state update + next input + partial minima (tc_head.cuh) -----------------
        wait_accumulator();
        TLW(40);
        if constexpr (kSW == 128 && !TRAJ) {
          // 96 registers: re-derive the slice predicates every step instead of holding them (no spills)
          asm volatile("mov.b32 %0, %0;" : "+r"(hc.slice_bits));
        }
        if constexpr (TRAJ && !FWD) {
          if (sink.row != nullptr) sink.row += O;
        }
        if constexpr (FWD) head_step_pass<OW, true, kSW, kSW>(hc, noise, astore, false, sink);
        else if (prm.sampling_propagation) head_step_pass<OW, true, kSW, kSW>(hc, noise, astore, t + 1 < H, sink);
        else head_step_pass<OW, false, kSW, kSW>(hc, noise, astore, t + 1 < H, sink);
        TLW(41);
        tmem_st_wait();
        if (t + 1 < H) publish_a();
        TLW(42);
        if constexpr (!TRAJ) named_bar_sync<kEpiThreads>(kBarScore);   // partial minima of s_{t+1} visible to the scorers
        if (!TRAJ && cgp == 0) {
          float next_dist, next_cost;
          head_combine<kQ>(sc, part_row, nparts, next_dist, next_cost);
          RowScore rs;
          rs.cum = __uint_as_float(my_rs[0]);
          rs.costsum = __uint_as_float(my_rs[128]);
          rs.cmask = (uint64_t)my_rs[256] | ((uint64_t)my_rs[384] << 32);
          rs.dist = __uint_as_float(my_rs[512]);
          rs.cost = __uint_as_float(my_rs[640]);
          rs.done = my_rs[768] != 0u;
          head_score_step(rs, sc, done_first, t, next_dist, next_cost);
          my_rs[0] = __float_as_uint(rs.cum);
          my_rs[128] = __float_as_uint(rs.costsum);
          my_rs[256] = (uint32_t)rs.cmask;
          my_rs[384] = (uint32_t)(rs.cmask >> 32);
          my_rs[512] = __float_as_uint(rs.dist);
          my_rs[640] = __float_as_uint(rs.cost);
          my_rs[768] = rs.done ? 1u : 0u;
        }
        if (!TRAJ && cgp == 0 && cmask_word_ends(t, H)) {       // H > 64: word t >> 6 is complete
          if (row_ok && prm.row_return != nullptr)
            prm.row_costmask[(t >> 6) * cmask_plane_stride(g) + id.out] = (uint64_t)my_rs[256] | ((uint64_t)my_rs[384] << 32);
          my_rs[256] = 0u;
          my_rs[384] = 0u;
        }
        TLW(43);
      }
      if (!TRAJ && cgp == 0 && row_ok && prm.row_return != nullptr) {
        prm.row_return[id.out] = __uint_as_float(my_rs[0]);
        prm.row_costmask[((H - 1) >> 6) * cmask_plane_stride(g) + id.out] = (uint64_t)my_rs[256] | ((uint64_t)my_rs[384] << 32);
        prm.row_costsum[id.out] = __uint_as_float(my_rs[128]);
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, kTmemCols);
}

template <int kSW>
__global__ void __launch_bounds__(kWideThreads, 1) rollout_tc_wide_kernel(const RolloutParams prm) {
  rollout_tc_wide_body<kSW, false>(prm);
}

// the trajectory form (simba_unfold_tc)
template <int kSW>
__global__ void __launch_bounds__(kWideThreads, 1) unfold_tc_wide_kernel(const RolloutParams prm) {
  rollout_tc_wide_body<kSW, true>(prm);
}

// the forward form (simba_ensemble_forward_tc)
template <int kSW>
__global__ void __launch_bounds__(kWideThreads, 1) forward_tc_wide_kernel(const RolloutParams prm) {
  rollout_tc_wide_body<kSW, true, true>(prm);
}

// the swish forms of the three above (kActSwish)
template <int kSW>
__global__ void __launch_bounds__(kWideThreads, 1) rollout_swish_tc_wide_kernel(const RolloutParams prm) {
  rollout_tc_wide_body<kSW, false, false, kActSwish>(prm);
}
template <int kSW>
__global__ void __launch_bounds__(kWideThreads, 1) unfold_swish_tc_wide_kernel(const RolloutParams prm) {
  rollout_tc_wide_body<kSW, true, false, kActSwish>(prm);
}
template <int kSW>
__global__ void __launch_bounds__(kWideThreads, 1) forward_swish_tc_wide_kernel(const RolloutParams prm) {
  rollout_tc_wide_body<kSW, true, true, kActSwish>(prm);
}

// ---- host side ------------------------------------------------------------------------------------
template <int kSW>
static size_t wide_smem_bytes(int L, int U, int nparts) {
  const WideShape ws = wide_shape<kSW>(U, L);
  size_t b = (size_t)ws.KA * kAtomBytes;
  b += (size_t)kStages * wide_stage_bytes<kSW>(ws);
  b += 2 * kSW * sizeof(float) + kHeadParts * kSW * sizeof(float);
  b += (size_t)kQ * nparts * 128 * sizeof(float);
  b += (size_t)8 * 128 * sizeof(uint32_t);                          // per-row running objective
  b += 6 * sizeof(uint64_t) + 2 * sizeof(uint32_t) + sizeof(TileInfoW);
  return b + 1024;                                                 // alignment slack
}

static size_t wide_smem_bytes(int sw, int L, int UP, int nparts) {
  return sw == 64 ? wide_smem_bytes<64>(L, UP, nparts) : wide_smem_bytes<128>(L, UP, nparts);
}

// widths that are not a multiple of 16 run zero-padded to the next one; the 128-column variant pads to at
// least 128 (file comment)
static int rollout_tc_wide_units(int sw, int U) {
  const int UP = (U + 15) / 16 * 16;
  return sw == 64 ? UP : std::max(UP, WideCfg<128>::kMinUnits);
}

// shape check used when the weight images are packed (no scorer yet: one constraint slot assumed). The layer-0
// input needs O + A + 2 K elements; head_store_actions writes four state columns from O, so O + 4 <= kSW as well
// (the <64> variant's O <= 60 implies it).
bool rollout_tc_wide_supported(int sw, int O, int A, int L, int U) {
  const int UP = rollout_tc_wide_units(sw, U);
  const bool shape = sw == 64 ? U > 128 && UP <= WideCfg<64>::kMaxUnits && O <= 60 && O + A + 2 <= 64
                              : UP <= WideCfg<128>::kMaxUnits && O + A + 2 <= 128 && O + 4 <= 128;
  return shape && O >= 1 && A <= 4 && L >= 1 && L <= 6 &&
         wide_smem_bytes(sw, L, UP, 1) <= 227 * 1024;
}

// the A tile, the two-stage weight ring and the per-constraint exchange buffers must share 227 KB
bool rollout_tc_wide_fits(int sw, int L, int U, int n_constraints) {
  return wide_smem_bytes(sw, L, rollout_tc_wide_units(sw, U), 1 + n_constraints) <= 227 * 1024;
}

// The weight stream of the variant with state width sw, per member the tiles of one rollout step in consumption
// order: layer 0: sw / 64 tiles [UP x 64]; layers 1..L-1: KA tiles [UP x 64]; heads: KA tiles [2 sw x 64] (mu rows
// [0, O), var rows [sw, sw + O), the raw-variance head pre-scaled by log2(e)); each tile K-major SWIZZLE_128B. UP
// is the width rollout_tc_wide_units pads to, its extra units have zero weights and bias. The bias of a layer
// sits in k rows KB (hi) and KB + 1 (lo), which the kernel multiplies by constant ones in the A tile.
int64_t rollout_tc_wide_pack(int sw, const ModelWeights& mw, std::vector<uint16_t>& img) {
  const auto& c = mw.cfg;
  const int L = c.n_layers, E = c.ensemble_size, U = c.units, O = c.obs_dim, IN = c.obs_dim + c.act_dim;
  const int UP = rollout_tc_wide_units(sw, U);
  const WideShape ws = sw == 64 ? wide_shape<64>(UP, L) : wide_shape<128>(UP, L);
  const int KA = ws.KA;
  const int64_t member_bytes =
      (int64_t)(ws.tiles_per_step - ws.head_tiles) * ws.hid_tile_bytes + (int64_t)KA * ws.head_tile_bytes;
  img.assign((size_t)E * member_bytes / 2, 0);
  for (int e = 0; e < E; ++e) {
    int64_t off = (int64_t)e * member_bytes;
    for (int l = 0; l <= L; ++l) {
      const int K = l == 0 ? IN : U;                     // real input width
      const int KB = l == 0 ? IN : UP;                   // the A tile holds the constant ones at k = KB, KB + 1
      const int rows = l < L ? UP : 2 * sw;              // tile rows = output features
      const int tiles = l == 0 ? sw / 64 : KA;
      auto weight = [&](int k, int n) -> uint16_t {
        int layer = l, col = n;                          // Keras layer index and output column
        if (l == L) {
          if (n < O) { layer = L; col = n; }
          else if (n >= sw && n < sw + O) { layer = L + 1; col = n - sw; }
          else return 0;
        } else if (n >= U) {
          return 0;                                      // padded hidden unit: weights and bias 0
        }
        const int width = l < L ? U : O;
        const float pre = layer == L + 1 ? kLog2e : 1.0f;
        if (k < K) return bf16_bits(pre * mw.kernel(e, layer)[(size_t)k * width + col]);
        if (k == KB || k == KB + 1) {
          uint16_t hi, lo;
          bf16_split(pre * mw.bias(e, layer)[col], hi, lo);
          return k == KB ? hi : lo;
        }
        return 0;
      };
      for (int tI = 0; tI < tiles; ++tI) {
        for (int n = 0; n < rows; ++n)
          for (int kk = 0; kk < 64; ++kk) img[(off + sw128_offset(n, kk)) / 2] = weight(tI * 64 + kk, n);
        off += (int64_t)rows * 128;
      }
    }
  }
  return member_bytes;
}

template <int kSW, bool TRAJ, bool FWD = false>
static cudaError_t launch_wide(const RolloutParams& model_prm, cudaStream_t stream) {
  RolloutParams prm = model_prm;
  prm.U = rollout_tc_wide_units(kSW, prm.U);                       // the kernel runs the zero-padded width
  const bool swish = prm.act == kActSwish;
  void (*kern)(const RolloutParams) = swish ? rollout_swish_tc_wide_kernel<kSW> : rollout_tc_wide_kernel<kSW>;
  if constexpr (FWD) kern = swish ? forward_swish_tc_wide_kernel<kSW> : forward_tc_wide_kernel<kSW>;
  else if constexpr (TRAJ) kern = swish ? unfold_swish_tc_wide_kernel<kSW> : unfold_tc_wide_kernel<kSW>;
  const size_t smem = wide_smem_bytes<kSW>(prm.L, prm.U, TRAJ ? 1 : 1 + prm.scorer.n_constraints);
  return launch_kernel(kern, prm.n_tiles, kWideThreads, smem, stream, 1, prm.pdl, prm);
}

cudaError_t launch_rollout_tc_wide(const RolloutParams& prm, cudaStream_t stream) {
  if (prm.mu_out != nullptr) {
    switch (prm.kernel) {
      case RolloutKernel::kTcWide: return launch_wide<64, true, true>(prm, stream);
      case RolloutKernel::kTcWideObs: return launch_wide<128, true, true>(prm, stream);
      default: return cudaErrorInvalidValue;
    }
  }
  if (prm.traj_out == nullptr) {
    switch (prm.kernel) {
      case RolloutKernel::kTcWide: return launch_wide<64, false>(prm, stream);
      case RolloutKernel::kTcWideObs: return launch_wide<128, false>(prm, stream);
      default: return cudaErrorInvalidValue;
    }
  }
  switch (prm.kernel) {
    case RolloutKernel::kTcWide: return launch_wide<64, true>(prm, stream);
    case RolloutKernel::kTcWideObs: return launch_wide<128, true>(prm, stream);
    default: return cudaErrorInvalidValue;
  }
}

}  // namespace simba

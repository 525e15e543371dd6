// The small CEM kernels around the rollout: action sampling, cross-particle score reduction,
// elite selection (radix select), moment refit, final noise — plus the batch versions of the
// reference's public scorer / scale / compute_objective methods. All are HBM / latency bound:
// coalesced, vectorised where the layout allows, no tensor cores.
#include <cooperative_groups.h>

#include "cem_kernels.cuh"
#include "internal.h"

namespace cg = cooperative_groups;

namespace simba {

// =============================================================================================
// k1  action sampling — simba/policies/cem_mpc.py:44-48
//     a = clip_by_value(z * sigma + mu, lb, ub);  z external or Philox stream ACTION.
// One thread = 4 consecutive flattened (h, a) elements of one candidate (= one Philox block).
// =============================================================================================
// one Philox block = 4 consecutive flattened (h, a) elements of candidate i of state s
// n / d for 0 <= n < 2^22, 1 <= d < 2^22 with inv = 1.0f / d: a multiply and a fix-up instead of the
// ~30-instruction integer division. The latency kernels below run 32 warps on one SM, where every
// instruction all threads execute costs 8 issue cycles per scheduler.
__device__ __forceinline__ int div_small(int n, int d, float inv) {
  int q = (int)((float)n * inv);
  const int r = n - q * d;
  if (r < 0) --q;
  else if (r >= d) ++q;
  return q;
}

// the four N(0,1) draws of block j of candidate i: external (parity mode) or the ACTION stream
__device__ __forceinline__ void sample_draws4(const SampleParams& p, uint64_t seed, int s, int i, int j, float (&z)[4]) {
  const int HA = p.H * p.A;
  if (p.z != nullptr) {
    const long base = ((long)s * p.N + i) * HA + 4 * j;
#pragma unroll
    for (int q = 0; q < 4; ++q) z[q] = (4 * j + q < HA) ? p.z[base + q] : 0.0f;
  } else {
    const float4 n = philox_normals<false>(seed, kStreamAction, (uint32_t)s, (uint32_t)p.iteration, 0u, (uint32_t)i,
                                           (uint32_t)j);
    z[0] = n.x; z[1] = n.y; z[2] = n.z; z[3] = n.w;
  }
}
// clip(z * sigma + mu) — cem_mpc.py:44-48. mu_s / sigma_s: this state's H * A values (global memory, or
// the fused update kernel's shared copies)
__device__ __forceinline__ void sample_apply4(const SampleParams& p, const float* mu_s, const float* sigma_s,
                                              const float (&z)[4], int j, float (&out)[4]) {
  const int HA = p.H * p.A;
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const int e = 4 * j + q;
    out[q] = 0.0f;
    if (e < HA) {
      const int a = e % p.A;
      const float v = __fadd_rn(__fmul_rn(z[q], sigma_s[e]), mu_s[e]);
      out[q] = fminf(fmaxf(v, p.lb[a]), p.ub[a]);
    }
  }
}
__device__ __forceinline__ void sample_values4_from(const SampleParams& p, const float* mu_s, const float* sigma_s,
                                                    uint64_t seed, int s, int i, int j, float (&out)[4]) {
  float z[4];
  sample_draws4(p, seed, s, i, j, z);
  sample_apply4(p, mu_s, sigma_s, z, j, out);
}

__device__ __forceinline__ void sample_values4(const SampleParams& p, int s, int i, int j, float (&out)[4]) {
  const int HA = p.H * p.A;
  sample_values4_from(p, p.mu + s * HA, p.sigma + s * HA, p.seed_ptr ? *p.seed_ptr : p.seed, s, i, j, out);
}

__device__ __forceinline__ void store_block4(const SampleParams& p, int s, int i, int j, const float (&out)[4],
                                             float* dst_all) {
  const int HA = p.H * p.A;
  const long base = ((long)s * p.N + i) * HA + 4 * j;
  if ((HA & 3) == 0) {
    *reinterpret_cast<float4*>(dst_all + base) = make_float4(out[0], out[1], out[2], out[3]);
  } else {
#pragma unroll
    for (int q = 0; q < 4; ++q)
      if (4 * j + q < HA) dst_all[base + q] = out[q];
  }
}

__device__ __forceinline__ void sample_block_to(const SampleParams& p, int s, int i, int j, float* dst_all) {
  float out[4];
  sample_values4(p, s, i, j, out);
  store_block4(p, s, i, j, out, dst_all);
}

__device__ __forceinline__ void sample_block(const SampleParams& p, int s, int i, int j) {
  sample_block_to(p, s, i, j, p.out);
}

// true when candidate i was sampled by this rank (its row is in the action buffer)
__device__ __forceinline__ bool sampled_here(const SampleParams& p, int i) {
  return p.n_cand == 0 || (i >= p.cand0 && i < p.cand0 + p.n_cand);
}

__global__ void __launch_bounds__(256) sample_actions_kernel(SampleParams p) {
  // a rollout launched behind this kernel as a programmatic dependent may start its prologue now (it waits
  // for this grid's completion before it reads the actions); a no-op for plain launches
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  const int JB = (p.H * p.A + 3) >> 2;
  const int NC = p.n_cand ? p.n_cand : p.N;     // candidates this rank samples
  const long total = (long)p.S * NC * JB;
  for (long idx = blockIdx.x * (long)blockDim.x + threadIdx.x; idx < total;
       idx += (long)gridDim.x * blockDim.x) {
    const int j = (int)(idx % JB);
    const long si = idx / JB;                 // s * NC + local candidate
    const int s = (int)(si / NC);
    const int i = p.cand0 + (int)(si - (long)s * NC);
    if (p.active != nullptr && p.active[s] == 0) continue;
    sample_block(p, s, i, j);
  }
}

cudaError_t launch_sample_actions(const SampleParams& p, cudaStream_t st) {
  const int HA = p.H * p.A;
  const long total = (long)p.S * (p.n_cand ? p.n_cand : p.N) * ((HA + 3) / 4);
  int blocks = (int)((total + 255) / 256);
  if (blocks > 148 * 8) blocks = 148 * 8;
  if (blocks < 1) blocks = 1;
  sample_actions_kernel<<<blocks, 256, 0, st>>>(p);
  return cudaGetLastError();
}

// =============================================================================================
// k8  cross-particle reduction — simba/policies/mpc_policy.py:38-39,
//     simba/policies/safe_cem_mpc.py:94-96 (mean return), :110-120 (per-step particle counts of
//     the done-masked cost -> Beta posterior test), :98-108 (mean cost sum).
// One thread per (state, local candidate); loads are coalesced across candidates for each
// particle. Per-step counts use bit-sliced (carry-save) counters over the 64-bit cost masks, so
// the H x P popcount costs ~3 logic ops per particle and plane. Summation order over particles
// is fixed (p ascending) => bit-identical on every rank. Horizons beyond 64 steps run the
// counters once more per further 64-step plane of the masks (cmask_planes).
// =============================================================================================
// counter bits b = 0..7 of 64 steps: add one particle's mask word
__device__ __forceinline__ void bitsliced_add(uint64_t (&plane)[8], uint64_t carry) {
#pragma unroll
  for (int b = 0; b < 8; ++b) {
    const uint64_t t = plane[b] & carry;
    plane[b] ^= carry;
    carry = t;
  }
}
// the largest count among the first `steps` (>= 1) steps of the counters
__device__ __forceinline__ int bitsliced_max(const uint64_t (&plane)[8], int steps) {
  uint64_t cand = (steps >= 64) ? ~0ull : ((1ull << steps) - 1ull);
  int maxc = 0;
#pragma unroll
  for (int b = 7; b >= 0; --b) {
    const uint64_t m = cand & plane[b];
    if (m) { cand = m; maxc |= (1 << b); }
  }
  return maxc;
}

// H > 64: the largest per-step count of planes 1 .. W - 1 (steps [64, H)). Not inlined: the callers' H <= 64 code
// stays as it was, and the fused update kernel, bound by the latency of its serial path, does not grow.
__device__ __noinline__ int later_planes_max(const uint64_t* row_costmask, long base, int stride, int P, int H,
                                             long plane_stride) {
  int maxc = 0;
  for (int w = 1; w < cmask_planes(H); ++w) {          // steps [64 w, 64 w + 64)
    uint64_t plane[8];
#pragma unroll
    for (int b = 0; b < 8; ++b) plane[b] = 0ull;
    const uint64_t* mw = row_costmask + w * plane_stride;
#pragma unroll 4
    for (int q = 0; q < P; ++q) bitsliced_add(plane, mw[base + (long)q * stride]);
    maxc = max(maxc, bitsliced_max(plane, H - 64 * w));
  }
  return maxc;
}

// rows of candidate i: element base + q * stride of each array, q = 0 .. P - 1; mask plane w at
// row_costmask + w * plane_stride
__device__ __forceinline__ float2 reduce_rows(const float* row_return, const uint64_t* row_costmask,
                                              const float* row_costsum, long base, int stride, int P, int H,
                                              long plane_stride, int objective) {
  float ret = 0.0f, csum = 0.0f;
  uint64_t plane[8];
#pragma unroll
  for (int b = 0; b < 8; ++b) plane[b] = 0ull;
#pragma unroll 4
  for (int q = 0; q < P; ++q) {
    const long r = base + (long)q * stride;
    ret = __fadd_rn(ret, row_return[r]);
    csum = __fadd_rn(csum, row_costsum[r]);
    bitsliced_add(plane, row_costmask[r]);
  }
  const float mean_ret = __fdiv_rn(ret, (float)P);
  float cost = 0.0f;
  if (objective == SIMBA_OBJ_LEAST_COST) {
    cost = __fdiv_rn(csum, (float)P);
  } else if (objective != SIMBA_OBJ_REWARD) {
    int maxc = bitsliced_max(plane, H);
    if (H > 64) maxc = max(maxc, later_planes_max(row_costmask, base, stride, P, H, plane_stride));
    cost = (float)maxc;
  }
  return make_float2(mean_ret, cost);
}

__device__ __forceinline__ float2 reduce_candidate(const ReduceParams& p, int s, int i) {
  return reduce_rows(p.row_return, p.row_costmask, p.row_costsum, (long)s * p.P * p.N_local + i, p.N_local, p.P, p.H,
                     (long)p.S * p.P * p.N_local, p.objective);
}

__global__ void __launch_bounds__(256) score_reduce_kernel(ReduceParams p) {
  const long total = (long)p.S * p.N_local;
  const long idx = blockIdx.x * (long)blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int s = (int)(idx / p.N_local);
  const int i = (int)(idx - (long)s * p.N_local);
  if (p.active != nullptr && p.active[s] == 0) return;
  reinterpret_cast<float2*>(p.out_pairs)[idx] = reduce_candidate(p, s, i);
}

cudaError_t launch_score_reduce(const ReduceParams& p, cudaStream_t st) {
  const long total = (long)p.S * p.N_local;
  score_reduce_kernel<<<(int)((total + 255) / 256), 256, 0, st>>>(p);
  return cudaGetLastError();
}

// =============================================================================================
// k9  elite selection — simba/policies/cem_mpc.py:56-60
//     top_k(scores, K, sorted=False) with ties -> lower index; argmax; strict '>' best-so-far.
// One CTA per state. Candidates get a 64-bit order key (larger = better); an MSD radix select
// (8-bit digits, shared-memory histogram) finds the K-th largest key; one ordered compaction
// (two block scans) emits the elite set in ascending index order, which makes the refit's
// summation order — and therefore mu/sigma — bit-identical on every rank.
// =============================================================================================
__device__ __forceinline__ uint32_t ordered_u32(float f) {
  if (f != f) return 0u;                          // NaN (a diverged rollout) ranks below every number: never elite
  f = f + 0.0f;                                   // -0 -> +0 so that -0 == +0 ties by index
  const uint32_t u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

__device__ __forceinline__ float pair_score(int objective, float ret, float cost, float c_max) {
  switch (objective) {
    case SIMBA_OBJ_REWARD: return ret;
    case SIMBA_OBJ_LEAST_COST: return -cost;
    default:   // SAFE_PENALTY (safe_cem_mpc.py:96) and the score FEASIBLE_FIRST reports
      return __fsub_rn(ret, __fmul_rn(cost > c_max ? 1.0f : 0.0f, 100.0f));
  }
}

__device__ __forceinline__ uint64_t pair_key(int objective, float ret, float cost, float c_max) {
  if (objective == SIMBA_OBJ_FEASIBLE_FIRST) {
    if (cost <= c_max) return (1ull << 63) | (uint64_t)ordered_u32(ret);
    const uint32_t viol = (uint32_t)fminf(cost, 255.0f);
    return ((uint64_t)(255u - viol) << 32) | (uint64_t)ordered_u32(ret);
  }
  return (uint64_t)ordered_u32(pair_score(objective, ret, cost, c_max));
}

template <int NT>
__device__ __forceinline__ int block_exclusive_scan(int v, int* warp_sums, int* total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int incl = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const int n = __shfl_up_sync(0xffffffffu, incl, d);
    if (lane >= d) incl += n;
  }
  if (lane == 31) warp_sums[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    int w = (lane < NT / 32) ? warp_sums[lane] : 0;
    int wi = w;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int n = __shfl_up_sync(0xffffffffu, wi, d);
      if (lane >= d) wi += n;
    }
    if (lane < NT / 32) warp_sums[lane] = wi - w;     // exclusive warp offsets
    if (lane == 31) *total = wi;
  }
  __syncthreads();
  const int res = warp_sums[warp] + incl - v;
  __syncthreads();
  return res;
}

constexpr int kSelectThreads = 1024;

// Radix-select step: thread tid < 256 brings the count of bin 255 - tid; picks the bin that holds the
// need-th largest key (bins above it hold fewer than `need`) with one suffix scan over the 256 bins —
// eight warp scans and a seven-term carry — instead of up to 255 dependent shared-memory reads per
// thread (3.9 us per pass of the population-65536 selection, 4 passes per call). Ends with a CTA barrier.
__device__ __forceinline__ void pick_digit(int count_rev, int need, int* warp_tot, int* sh_digit, int* sh_need) {
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  int incl = count_rev;
  if (tid < 256) {
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int n = __shfl_up_sync(0xffffffffu, incl, d);
      if (lane >= d) incl += n;
    }
    if (lane == 31) warp_tot[w] = incl;
  }
  __syncthreads();
  if (tid < 256) {
    int above = incl - count_rev;                          // bins above this one inside the warp ...
    for (int q = 0; q < w; ++q) above += warp_tot[q];      // ... and in the warps holding higher bins
    if (above < need && need <= above + count_rev) { *sh_digit = 255 - tid; *sh_need = need - above; }
  }
  __syncthreads();
}

__global__ void __launch_bounds__(kSelectThreads) select_elites_kernel(SelectParams p) {
  const int s = blockIdx.x;
  if (p.active != nullptr && p.active[s] == 0) return;
  __shared__ int hist[256];
  __shared__ int warp_sums[32];
  __shared__ int sh_total;
  __shared__ int sh_digit, sh_need;
  __shared__ unsigned long long sh_best_key;
  __shared__ int sh_best_idx;
  const int tid = threadIdx.x;
  const int N = p.N, K = p.K;
  // candidate i lives at pairs_all[(g * S + s) * N_local + (i % N_local)], g = i / N_local
  auto load_pair = [&](int i) {
    const int gsh = i / p.N_local, il = i - gsh * p.N_local;
    return reinterpret_cast<const float2*>(p.pairs_all)[((long)gsh * p.S + s) * p.N_local + il];
  };

  // ---- stage the 64-bit order keys once (L2-resident scratch) and find their range --------------
  __shared__ unsigned long long sh_kmin, sh_kmax;
  if (tid == 0) { sh_best_key = 0ull; sh_best_idx = 0x7fffffff; sh_kmin = ~0ull; sh_kmax = 0ull; }
  __syncthreads();
  unsigned long long* keys = p.key_scratch + (long)s * N;
  {
    unsigned long long kmin = ~0ull, kmax = 0ull;
    for (int base = 0; base < N; base += 4 * kSelectThreads) {
      float2 pr[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int i = base + u * kSelectThreads + tid;
        pr[u] = i < N ? load_pair(i) : make_float2(0.f, 0.f);
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int i = base + u * kSelectThreads + tid;
        if (i < N) {
          const unsigned long long k = pair_key(p.objective, pr[u].x, pr[u].y, p.c_max);
          keys[i] = k;
          kmin = k < kmin ? k : kmin;
          kmax = k > kmax ? k : kmax;
        }
      }
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
      const unsigned long long a = __shfl_xor_sync(0xffffffffu, kmin, d), c = __shfl_xor_sync(0xffffffffu, kmax, d);
      kmin = a < kmin ? a : kmin;
      kmax = c > kmax ? c : kmax;
    }
    if ((tid & 31) == 0) { atomicMin(&sh_kmin, kmin); atomicMax(&sh_kmax, kmax); }
  }
  __syncthreads();                                         // also publishes keys[] to the whole CTA
  const unsigned long long kmin = sh_kmin, span = sh_kmax - sh_kmin;

  // ---- MSD radix select of the K-th largest key on (key - kmin): the digits of the normalised keys
  //      are spread over the bins (scores of one population share their exponent bits), and passes
  //      above the span's top byte are skipped. Histogram updates are warp-aggregated
  //      (__match_any_sync) so that heavy ties cost one shared-memory atomic per warp, not 32.
  uint64_t prefix = 0ull, mask = 0ull;
  int need = K;
  int top_byte = 7;
  while (top_byte > 0 && ((span >> (8 * top_byte)) & 0xffull) == 0ull) --top_byte;
  const int lane = tid & 31;
  for (int byte = top_byte; byte >= 0; --byte) {
    if (tid < 256) hist[tid] = 0;
    __syncthreads();
    const int shift = 8 * byte;
    for (int base = 0; base < N; base += 8 * kSelectThreads) {
      uint64_t kk[8];                                       // 8 independent L2 loads in flight per thread
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int i = base + u * kSelectThreads + tid;
        kk[u] = i < N ? keys[i] : 0ull;
      }
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int i = base + u * kSelectThreads + tid;
        int bin = -1;
        if (i < N) {
          const uint64_t k = kk[u] - kmin;
          if ((k & mask) == prefix) bin = (int)((k >> shift) & 0xffull);
        }
        const unsigned peers = __match_any_sync(0xffffffffu, bin);
        if (bin >= 0 && lane == __ffs(peers) - 1) atomicAdd(&hist[bin], __popc(peers));
      }
    }
    __syncthreads();
    pick_digit(tid < 256 ? hist[255 - tid] : 0, need, warp_sums, &sh_digit, &sh_need);
    prefix |= (uint64_t)sh_digit << shift;
    mask |= 0xffull << shift;
    need = sh_need;
    __syncthreads();
  }
  const uint64_t T = prefix + kmin;   // K-th largest key; `need` of the keys == T are taken, lowest index first

  // ---- ordered compaction: each thread owns a contiguous index range -------------------------
  const int V = (N + kSelectThreads - 1) / kSelectThreads;
  const int lo = min(N, tid * V), hi = min(N, lo + V);
  int eq_local = 0, gt_local = 0;
  uint64_t best_k = 0ull;
  int best_i = 0x7fffffff;
  for (int i = lo; i < hi; ++i) {
    const uint64_t k = keys[i];
    eq_local += (k == T);
    gt_local += (k > T);
    if (k > best_k || best_i == 0x7fffffff) { best_k = k; best_i = i; }   // first max in range
  }
  const int eq_before = block_exclusive_scan<kSelectThreads>(eq_local, warp_sums, &sh_total);
  const int eq_take = max(0, min(eq_local, need - eq_before));           // ties taken from this range
  int pos = block_exclusive_scan<kSelectThreads>(gt_local + eq_take, warp_sums, &sh_total);
  int eq_run = eq_before;
  for (int i = lo; i < hi; ++i) {
    const uint64_t k = keys[i];
    bool sel = k > T;
    if (k == T) { sel = eq_run < need; ++eq_run; }
    if (sel) p.out_elite[(long)s * K + pos++] = i;
    if (p.out_scores != nullptr) {
      const float2 pr = load_pair(i);
      p.out_scores[(long)s * N + i] = pair_score(p.objective, pr.x, pr.y, p.c_max);
    }
  }

  // ---- best of elite = global best key, lowest index among ties (argmax first max) -----------
  if (best_i != 0x7fffffff) atomicMax(&sh_best_key, (unsigned long long)best_k);
  __syncthreads();
  if (best_i != 0x7fffffff && best_k == sh_best_key) atomicMin(&sh_best_idx, best_i);
  __syncthreads();
  const int top = sh_best_idx;
  const float2 pr = load_pair(top);
  const float top_score = pair_score(p.objective, pr.x, pr.y, p.c_max);
  if (top_score > p.best_score[s]) {                       // cem_mpc.py:58 strict '>'
    if (tid < p.A) {
      if (p.regen && !sampled_here(p.sample, top)) {      // another rank sampled it: same counters, same row
        float v[4];
        sample_values4(p.sample, s, top, tid >> 2, v);
        p.best_action[s * p.A + tid] = v[tid & 3];
      } else {
        p.best_action[s * p.A + tid] = p.actions[((long)s * N + top) * p.H * p.A + tid];
      }
    }
    __syncthreads();
    if (tid == 0) p.best_score[s] = top_score;
  }
}

// ---------------------------------------------------------------------------------------------
// Large populations (configs[2]: N = 65536, K = 6554): the same selection on a thread-block
// CLUSTER of 8 CTAs per state. Each CTA keeps its contiguous slice of the order keys in shared
// memory; per radix pass the 8 slice histograms are combined through distributed shared memory
// (every CTA reads the other 7 and derives the same digit), so a pass costs one hardware cluster
// barrier instead of a trip through L2, and the ordered compaction uses the per-CTA (>, ==)
// counts as its cross-CTA prefix. Output is identical to select_elites_kernel: elites in
// ascending index order, ties to the lower index, argmax = first max.
// ---------------------------------------------------------------------------------------------
constexpr int kSelClusterSize = 8;
constexpr int kSelClusterMinN = 8192;          // below this one CTA is as fast
constexpr int kSelClusterMaxSlice = 16384;     // keys per CTA (128 KB of shared memory)

__global__ void __launch_bounds__(kSelectThreads)
select_elites_cluster_kernel(SelectParams p, int slice) {
  cg::cluster_group cluster = cg::this_cluster();
  const int rank = (int)cluster.block_rank();
  const int s = blockIdx.x / kSelClusterSize;
  if (p.active != nullptr && p.active[s] == 0) return;      // uniform over the cluster
  extern __shared__ __align__(16) unsigned long long keys[];   // [slice]
  __shared__ int hist[2][256];
  __shared__ int warp_sums[32];
  __shared__ int sh_total;
  __shared__ int sh_digit, sh_need;
  __shared__ unsigned long long sh_minmax[2];
  __shared__ int sh_counts[2];                     // (> T, == T) in this slice
  __shared__ unsigned long long sh_best_key;
  __shared__ int sh_best_idx;
  const int tid = threadIdx.x, lane = tid & 31;
  const int N = p.N, K = p.K;
  const int lo = min(N, rank * slice), hi = min(N, lo + slice), n_loc = hi - lo;
  auto load_pair = [&](int i) {
    const int gsh = i / p.N_local, il = i - gsh * p.N_local;
    return reinterpret_cast<const float2*>(p.pairs_all)[((long)gsh * p.S + s) * p.N_local + il];
  };

  // ---- stage this slice's order keys in shared memory, find the global key range ---------------
  if (tid == 0) { sh_best_key = 0ull; sh_best_idx = 0x7fffffff; sh_minmax[0] = ~0ull; sh_minmax[1] = 0ull; }
  __syncthreads();
  {
    unsigned long long kmin = ~0ull, kmax = 0ull;
    for (int base = 0; base < n_loc; base += 4 * kSelectThreads) {
      float2 pr[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int j = base + u * kSelectThreads + tid;
        pr[u] = j < n_loc ? load_pair(lo + j) : make_float2(0.f, 0.f);
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int j = base + u * kSelectThreads + tid;
        if (j < n_loc) {
          const unsigned long long k = pair_key(p.objective, pr[u].x, pr[u].y, p.c_max);
          keys[j] = k;
          kmin = k < kmin ? k : kmin;
          kmax = k > kmax ? k : kmax;
          if (p.out_scores != nullptr)
            p.out_scores[(long)s * N + lo + j] = pair_score(p.objective, pr[u].x, pr[u].y, p.c_max);
        }
      }
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
      const unsigned long long a = __shfl_xor_sync(0xffffffffu, kmin, d), c = __shfl_xor_sync(0xffffffffu, kmax, d);
      kmin = a < kmin ? a : kmin;
      kmax = c > kmax ? c : kmax;
    }
    if (lane == 0) { atomicMin(&sh_minmax[0], kmin); atomicMax(&sh_minmax[1], kmax); }
  }
  cluster.sync();
  unsigned long long kmin = ~0ull, kmax = 0ull;
  for (int r = 0; r < kSelClusterSize; ++r) {
    const unsigned long long* mm = cluster.map_shared_rank(sh_minmax, r);
    kmin = mm[0] < kmin ? mm[0] : kmin;
    kmax = mm[1] > kmax ? mm[1] : kmax;
  }
  const unsigned long long span = kmax - kmin;

  // ---- MSD radix select of the K-th largest key on (key - kmin) ---------------------------------
  uint64_t prefix = 0ull, mask = 0ull;
  int need = K;
  int top_byte = 7;
  while (top_byte > 0 && ((span >> (8 * top_byte)) & 0xffull) == 0ull) --top_byte;
  int buf = 0;
  for (int byte = top_byte; byte >= 0; --byte, buf ^= 1) {
    if (tid < 256) hist[buf][tid] = 0;
    __syncthreads();
    const int shift = 8 * byte;
    for (int base = 0; base < n_loc; base += kSelectThreads) {
      const int j = base + tid;
      int bin = -1;
      if (j < n_loc) {
        const uint64_t k = keys[j] - kmin;
        if ((k & mask) == prefix) bin = (int)((k >> shift) & 0xffull);
      }
      const unsigned peers = __match_any_sync(0xffffffffu, bin);
      if (bin >= 0 && lane == __ffs(peers) - 1) atomicAdd(&hist[buf][bin], __popc(peers));
    }
    cluster.sync();                            // every slice's histogram of this pass is complete
    int t = 0;
    if (tid < 256) {
      int part[kSelClusterSize];                             // eight independent DSMEM reads in flight
#pragma unroll
      for (int r = 0; r < kSelClusterSize; ++r) part[r] = cluster.map_shared_rank(&hist[buf][0], r)[255 - tid];
#pragma unroll
      for (int r = 0; r < kSelClusterSize; ++r) t += part[r];
    }
    pick_digit(t, need, warp_sums, &sh_digit, &sh_need);
    prefix |= (uint64_t)sh_digit << shift;
    mask |= 0xffull << shift;
    need = sh_need;
    __syncthreads();
    // hist[buf] may still be read by the other CTAs; it is only zeroed again two passes later,
    // after the next pass's cluster barrier
  }
  const uint64_t T = prefix + kmin;   // K-th largest key; `need` of the keys == T are taken, lowest index first

  // ---- ordered compaction: thread = contiguous range of the slice, CTA = contiguous slice -----
  const int V = (n_loc + kSelectThreads - 1) / kSelectThreads;
  const int tlo = min(n_loc, tid * V), thi = min(n_loc, tlo + V);
  int eq_local = 0, gt_local = 0;
  uint64_t best_k = 0ull;
  int best_i = 0x7fffffff;
  for (int j = tlo; j < thi; ++j) {
    const uint64_t k = keys[j];
    eq_local += (k == T);
    gt_local += (k > T);
    if (k > best_k || best_i == 0x7fffffff) { best_k = k; best_i = lo + j; }   // first max in range
  }
  const int eq_before_cta = block_exclusive_scan<kSelectThreads>(eq_local, warp_sums, &sh_total);
  const int eq_cta = sh_total;
  __syncthreads();
  (void)block_exclusive_scan<kSelectThreads>(gt_local, warp_sums, &sh_total);
  if (tid == 0) { sh_counts[0] = sh_total; sh_counts[1] = eq_cta; }
  if (best_i != 0x7fffffff) atomicMax(&sh_best_key, (unsigned long long)best_k);
  __syncthreads();
  if (best_i != 0x7fffffff && best_k == sh_best_key) atomicMin(&sh_best_idx, best_i);
  cluster.sync();                              // counts and per-slice best of every CTA are visible
  int eq_before = 0, pos_base = 0;
  unsigned long long gbest_key = 0ull;
  int gbest_idx = 0x7fffffff;
  for (int r = 0; r < kSelClusterSize; ++r) {
    const int* cnt = cluster.map_shared_rank(sh_counts, r);
    const int gt_r = cnt[0], eq_r = cnt[1];
    if (r < rank) {
      pos_base += gt_r + max(0, min(eq_r, need - eq_before));
      eq_before += eq_r;
    }
    const unsigned long long bk = *cluster.map_shared_rank(&sh_best_key, r);
    const int bi = *cluster.map_shared_rank(&sh_best_idx, r);
    if (bi != 0x7fffffff && (gbest_idx == 0x7fffffff || bk > gbest_key)) { gbest_key = bk; gbest_idx = bi; }
  }
  const int eq_seen = eq_before + eq_before_cta;                         // == T keys at lower indices
  const int eq_take = max(0, min(eq_local, need - eq_seen));
  int pos = pos_base + block_exclusive_scan<kSelectThreads>(gt_local + eq_take, warp_sums, &sh_total);
  int eq_run = eq_seen;
  for (int j = tlo; j < thi; ++j) {
    const uint64_t k = keys[j];
    bool sel = k > T;
    if (k == T) { sel = eq_run < need; ++eq_run; }
    if (sel) p.out_elite[(long)s * K + pos++] = lo + j;
  }

  // ---- best of elite = global best key, lowest index among ties (slices are index-ordered, so
  //      the first slice holding the maximum wins) ------------------------------------------------
  if (rank == 0) {
    const float2 pr = load_pair(gbest_idx);
    const float top_score = pair_score(p.objective, pr.x, pr.y, p.c_max);
    if (top_score > p.best_score[s]) {                       // cem_mpc.py:58 strict '>'
      if (tid < p.A) {
        if (p.regen && !sampled_here(p.sample, gbest_idx)) {   // another rank sampled it: same counters, same row
          float v[4];
          sample_values4(p.sample, s, gbest_idx, tid >> 2, v);
          p.best_action[s * p.A + tid] = v[tid & 3];
        } else {
          p.best_action[s * p.A + tid] = p.actions[((long)s * N + gbest_idx) * p.H * p.A + tid];
        }
      }
      __syncthreads();
      if (tid == 0) p.best_score[s] = top_score;
    }
  }
  cluster.sync();                              // no CTA may exit while its shared memory is being read
}

static bool use_cluster_path(int N) {
  return N >= kSelClusterMinN && (N + kSelClusterSize - 1) / kSelClusterSize <= kSelClusterMaxSlice;
}

cudaError_t launch_select_elites(const SelectParams& p, cudaStream_t st) {
  if (use_cluster_path(p.N)) {
    const int slice = (p.N + kSelClusterSize - 1) / kSelClusterSize;
    return launch_kernel(select_elites_cluster_kernel, p.S * kSelClusterSize, kSelectThreads,
                         (size_t)slice * sizeof(unsigned long long), st, kSelClusterSize, false, p, slice);
  }
  select_elites_kernel<<<p.S, kSelectThreads, 0, st>>>(p);
  return cudaGetLastError();
}

// =============================================================================================
// k10  refit — simba/policies/cem_mpc.py:61-67
//      elites = gather(actions, elite); mean, var = moments(elites, axes=0) (population, two-pass);
//      mu, sigma smoothing; early exit when mean(sigma) <= stddev_threshold.
// One CTA per state; thread = (column c = (h, a), row group); partials are combined in a fixed
// order (deterministic => bit-identical replicas).
// =============================================================================================
constexpr int kRefitThreads = 1024;

#ifdef SIMBA_TC_TIMELINE
__shared__ long long* s_rtl_ptr;                    // set by thread 0 of the kernels that call refit_body (debug stamps)
#define RTL(k) do { if (blockIdx.x == 0 && threadIdx.x == 0 && s_rtl_ptr != nullptr) s_rtl_ptr[k] = clock64(); } while (0)
#else
#define RTL(k) do { } while (0)
#endif
// `elite` may live in global or shared memory; `sh` needs (groups + 2) * HA floats.
// Must be called by all kRefitThreads threads of the CTA.
__device__ __forceinline__ void refit_body(const RefitParams& p, int s, const int* elite, float* sh,
                                           int* stopped_sh = nullptr, const float* acts_copy = nullptr) {
  const int HA = p.H * p.A;
  const int groups = p.groups;                            // max(1, kRefitThreads / HA), from the launch function
  float* part = sh;
  float* mean = part + groups * HA;
  float* sig = mean + HA;
  const int tid = threadIdx.x;
  // acts_copy: this state's [N, H * A] actions staged in shared memory by the fused update kernel
  const float* acts = acts_copy != nullptr ? acts_copy : p.actions + (long)s * p.N * HA;
  const float kf = (float)p.K;
  if (p.regen) {
    // population sharding: elite rows that other ranks sampled are recomputed into the action buffer
    // (same Philox counters, same mu / sigma => the owner's values bit for bit), then gathered as usual
    const int JB = (HA + 3) >> 2;
    for (int idx = tid; idx < p.K * JB; idx += kRefitThreads) {
      const int e = elite[idx / JB];
      if (!sampled_here(p.sample, e)) sample_block_to(p.sample, s, e, idx % JB, p.actions);
    }
    __syncthreads();
  }

  // Loads that do not depend on the two passes are issued before them, so that their L2 round trips
  // overlap the gathers (HA <= kRefitThreads, checked at creation: column cc == tid has one owner).
  const bool owns_col = tid < HA;
  float mu_old = 0.0f, sg_old = 0.0f;
  int iters_old = 0;
  if (owns_col) { mu_old = p.mu[s * HA + tid]; sg_old = p.sigma[s * HA + tid]; }
  if (tid == 0 && p.iterations_run != nullptr) iters_old = p.iterations_run[s];

  const int grp = div_small(tid, HA, 1.0f / (float)HA), c = tid - grp * HA;   // HA <= 1024 (checked at creation)
  RTL(10);
  // A single plan's elite set (K <= groups: one elite per row group at most) keeps the thread's one gathered
  // value in a register for the second pass. Same values, same accumulation order as the general loop below —
  // and a fraction of its code.
  const bool single = p.K <= groups;
  const bool works = grp < p.K;                                // this thread's group holds an elite (single only)
  float held = 0.0f;
  if (single && works) held = acts_copy != nullptr ? acts_copy[elite[grp] * HA + c] : acts[(long)elite[grp] * HA + c];
  for (int pass = 0; pass < 2; ++pass) {
    if (grp < groups) {
      float acc = 0.0f;
      if (single) {
        if (works) {
          if (pass) { const float d = __fsub_rn(held, mean[c]); acc = __fadd_rn(acc, __fmul_rn(d, d)); }
          else acc = __fadd_rn(acc, held);
        }
      } else {
        const float m = pass ? mean[c] : 0.0f;
        // gathers are independent: issue 8 at a time, accumulate in index order (deterministic)
        int k = grp;
        for (; k + 7 * groups < p.K; k += 8 * groups) {
          float v[8];
#pragma unroll
          for (int u = 0; u < 8; ++u) v[u] = acts[(long)elite[k + u * groups] * HA + c];
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            if (pass) { const float d = __fsub_rn(v[u], m); acc = __fadd_rn(acc, __fmul_rn(d, d)); }
            else acc = __fadd_rn(acc, v[u]);
          }
        }
        for (; k < p.K; k += groups) {
          const float v = acts[(long)elite[k] * HA + c];
          if (pass) { const float d = __fsub_rn(v, m); acc = __fadd_rn(acc, __fmul_rn(d, d)); }
          else acc = __fadd_rn(acc, v);
        }
      }
      part[grp * HA + c] = acc;
    }
    RTL(11 + 4 * pass);
    __syncthreads();
    RTL(12 + 4 * pass);
    if (owns_col) {
      const int cc = tid;
      float tot = 0.0f;
#pragma unroll 8
      for (int gI = 0; gI < groups; ++gI) tot = __fadd_rn(tot, part[gI * HA + cc]);   // fixed order; loads pipelined
      const float r = __fdiv_rn(tot, kf);
      if (pass == 0) mean[cc] = r;
      else {
        const float sd = sqrtf(r);                                        // cem_mpc.py:63
        const float mu_new = __fadd_rn(__fmul_rn(p.smoothing, mu_old), __fmul_rn(p.one_minus_smoothing, mean[cc]));
        const float sg_new = __fadd_rn(__fmul_rn(p.smoothing, sg_old), __fmul_rn(p.one_minus_smoothing, sd));
        p.mu[s * HA + cc] = mu_new;                                       // cem_mpc.py:64-65
        p.sigma[s * HA + cc] = sg_new;
        sig[cc] = sg_new;
        mean[cc] = mu_new;            // the fused update kernel samples the next iteration from these copies
      }
    }
    RTL(13 + 4 * pass);
    __syncthreads();
    RTL(14 + 4 * pass);
  }
  if (tid == 0) {
    float tot = 0.0f;
#pragma unroll 8
    for (int cc = 0; cc < HA; ++cc) tot = __fadd_rn(tot, sig[cc]);
    if (p.iterations_run != nullptr) p.iterations_run[s] = iters_old + 1;
    const bool stop = p.active != nullptr && __fdiv_rn(tot, (float)HA) <= p.stddev_threshold;  // cem_mpc.py:66-67
    if (stop) p.active[s] = 0;
    if (stopped_sh != nullptr) *stopped_sh = stop ? 1 : 0;
  }
}

// refit_body for an elite set with at most one elite per row group (K <= groups: a single plan's K = 15 against 34
// groups), on the staged actions of the fused update kernel. In that case refit_body's partial of group g is
// 0 + x_g (pass 0) or 0 + (x_g - mean)^2 (pass 1) for g < K and 0 for the idle groups, summed over the groups in
// ascending order — which one thread per column can do directly: the same additions in the same order, without
// the [groups][H A] partials, their four CTA barriers and the (group, column) thread layout.
__device__ __forceinline__ void refit_single(const RefitParams& p, int s, const int* elite, const float* acts_s,
                                             float* xs, float* mean, float* sig, int* stopped_sh, float mu_old,
                                             float sg_old, int iters_old) {
  const int HA = p.H * p.A, groups = p.groups, K = p.K, tid = threadIdx.x;
  const float kf = (float)K;
  RTL(10);
  // the K elite rows, gathered by K * HA threads at once into xs[K][HA] (the idle partials area), so that the
  // column threads below read plain rows: no dependent index -> value round trip inside their addition chains
  for (int i = tid; i < K * HA; i += kRefitThreads) {
    const int gI = div_small(i, HA, 1.0f / (float)HA);
    xs[i] = acts_s[elite[gI] * HA + (i - gI * HA)];
  }
  __syncthreads();
  RTL(11);
  if (tid < HA) {
    const int c = tid;
    float tot = 0.0f, tot2 = 0.0f;
    for (int g0 = 0; g0 < K; g0 += 8) {                       // eight independent reads, then their additions
      float x[8];
#pragma unroll
      for (int q = 0; q < 8; ++q) x[q] = xs[min(g0 + q, K - 1) * HA + c];
#pragma unroll
      for (int q = 0; q < 8; ++q)
        if (g0 + q < K) tot = __fadd_rn(tot, __fadd_rn(0.0f, x[q]));
    }
    for (int gI = K; gI < groups; ++gI) tot = __fadd_rn(tot, 0.0f);      // the idle groups' partials
    const float m = __fdiv_rn(tot, kf);
    for (int g0 = 0; g0 < K; g0 += 8) {
      float x[8];
#pragma unroll
      for (int q = 0; q < 8; ++q) x[q] = xs[min(g0 + q, K - 1) * HA + c];
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        const float d = __fsub_rn(x[q], m);
        if (g0 + q < K) tot2 = __fadd_rn(tot2, __fadd_rn(0.0f, __fmul_rn(d, d)));
      }
    }
    for (int gI = K; gI < groups; ++gI) tot2 = __fadd_rn(tot2, 0.0f);
    RTL(12);
    const float sd = sqrtf(__fdiv_rn(tot2, kf));                          // cem_mpc.py:63
    const float mu_new = __fadd_rn(__fmul_rn(p.smoothing, mu_old), __fmul_rn(p.one_minus_smoothing, m));
    const float sg_new = __fadd_rn(__fmul_rn(p.smoothing, sg_old), __fmul_rn(p.one_minus_smoothing, sd));
    p.mu[s * HA + c] = mu_new;                                            // cem_mpc.py:64-65
    p.sigma[s * HA + c] = sg_new;
    sig[c] = sg_new;
    mean[c] = mu_new;               // the next iteration is sampled from these copies
  }
  RTL(13);
  __syncthreads();
  RTL(14);
  if (tid < 32) {
    // mean(sigma) in column order: one read per lane, lane 0 takes the values through shuffles, so only the
    // additions are a dependent chain
    float tot = 0.0f;
    for (int c0 = 0; c0 < HA; c0 += 32) {
      const float mine = c0 + tid < HA ? sig[c0 + tid] : 0.0f;
#pragma unroll
      for (int q = 0; q < 32; ++q) {
        const float v = __shfl_sync(0xffffffffu, mine, q);
        if (c0 + q < HA) tot = __fadd_rn(tot, v);
      }
    }
    if (tid == 0) {
      if (p.iterations_run != nullptr) p.iterations_run[s] = iters_old + 1;
      const bool stop = p.active != nullptr && __fdiv_rn(tot, (float)HA) <= p.stddev_threshold;  // cem_mpc.py:66-67
      if (stop) p.active[s] = 0;
      *stopped_sh = stop ? 1 : 0;
    }
  }
  RTL(15);
}

__global__ void __launch_bounds__(kRefitThreads) refit_kernel(RefitParams p) {
  const int s = blockIdx.x;
  if (p.active != nullptr && p.active[s] == 0) return;
  extern __shared__ float sh[];           // [groups][HA] partials, then [HA] mean, [HA] sigma
#ifdef SIMBA_TC_TIMELINE
  if (threadIdx.x == 0) s_rtl_ptr = nullptr;
#endif
  refit_body(p, s, p.elite + (long)s * p.K, sh);
}

// Large elite sets: the K gathers are spread over a cluster of 8 CTAs per state; the per-CTA
// column sums are combined in rank order through distributed shared memory (every CTA derives the
// same mean / variance), two cluster barriers per refit.
__global__ void __launch_bounds__(kRefitThreads) refit_cluster_kernel(RefitParams p) {
  cg::cluster_group cluster = cg::this_cluster();
  const int rank = (int)cluster.block_rank();
  const int s = blockIdx.x / kSelClusterSize;
  if (p.active != nullptr && p.active[s] == 0) return;      // uniform over the cluster
  extern __shared__ float sh[];           // [groups][HA] partials, [HA] CTA sums, [HA] mean, [HA] sigma
  const int HA = p.H * p.A;
  const int groups = kRefitThreads / HA > 0 ? kRefitThreads / HA : 1;
  float* part = sh;
  float* cta_sum = part + groups * HA;
  float* mean = cta_sum + HA;
  float* sig = mean + HA;
  int* eoff = reinterpret_cast<int*>(sig + HA);   // [per]
  const int tid = threadIdx.x;
  const float* acts = p.actions + (long)s * p.N * HA;
  const int* elite = p.elite + (long)s * p.K;
  const float kf = (float)p.K;
  const int per = (p.K + kSelClusterSize - 1) / kSelClusterSize;
  const int k_lo = min(p.K, rank * per), k_hi = min(p.K, k_lo + per);
  const int c = tid % HA, grp = tid / HA;
  if (p.regen) {
    // population sharding: this CTA's elite rows that other ranks sampled are recomputed into the action
    // buffer first (same counters, same mu / sigma => bit-identical); only this CTA reads them back
    const int JB = (HA + 3) >> 2;
    for (int idx = tid; idx < (k_hi - k_lo) * JB; idx += kRefitThreads) {
      const int e = elite[k_lo + idx / JB];
      if (!sampled_here(p.sample, e)) sample_block_to(p.sample, s, e, idx % JB, p.actions);
    }
    __syncthreads();
  }

  // this CTA's elite rows as 32-bit element offsets in shared memory: the gathers below then cost one
  // shared-memory read and one add per element instead of a dependent global index load and 64-bit
  // index arithmetic (which made up half of the kernel's instructions)
  const int n_mine = k_hi - k_lo;
  for (int k = tid; k < n_mine; k += kRefitThreads) eoff[k] = elite[k_lo + k] * HA;
  __syncthreads();

  for (int pass = 0; pass < 2; ++pass) {
    if (grp < groups) {
      float acc = 0.0f;
      const float m = pass ? mean[c] : 0.0f;
      const float* col = acts + c;
      int k = grp;
      for (; k + 7 * groups < n_mine; k += 8 * groups) {
        float v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) v[u] = col[eoff[k + u * groups]];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          if (pass) { const float d = __fsub_rn(v[u], m); acc = __fadd_rn(acc, __fmul_rn(d, d)); }
          else acc = __fadd_rn(acc, v[u]);
        }
      }
      for (; k < n_mine; k += groups) {
        const float v = col[eoff[k]];
        if (pass) { const float d = __fsub_rn(v, m); acc = __fadd_rn(acc, __fmul_rn(d, d)); }
        else acc = __fadd_rn(acc, v);
      }
      part[grp * HA + c] = acc;
    }
    __syncthreads();
    for (int cc = tid; cc < HA; cc += kRefitThreads) {
      float t = 0.0f;
      for (int gI = 0; gI < groups; ++gI) t = __fadd_rn(t, part[gI * HA + cc]);
      cta_sum[cc] = t;
    }
    cluster.sync();                            // every CTA's column sums of this pass are visible
    for (int cc = tid; cc < HA; cc += kRefitThreads) {
      float t = 0.0f;
      for (int r = 0; r < kSelClusterSize; ++r) t = __fadd_rn(t, cluster.map_shared_rank(cta_sum, r)[cc]);
      const float r_ = __fdiv_rn(t, kf);
      if (pass == 0) mean[cc] = r_;
      else {
        const float sd = sqrtf(r_);                                       // cem_mpc.py:63
        const float mu_new = __fadd_rn(__fmul_rn(p.smoothing, p.mu[s * HA + cc]),
                                       __fmul_rn(p.one_minus_smoothing, mean[cc]));
        const float sg_new = __fadd_rn(__fmul_rn(p.smoothing, p.sigma[s * HA + cc]),
                                       __fmul_rn(p.one_minus_smoothing, sd));
        sig[cc] = sg_new;
        mean[cc] = mu_new;
      }
    }
    cluster.sync();                            // remote reads of cta_sum are done before it is rewritten
  }
  if (rank == 0) {
    // mu / sigma are read by every CTA above and written only here, after the last barrier
    for (int cc = tid; cc < HA; cc += kRefitThreads) {
      p.mu[s * HA + cc] = mean[cc];                                       // cem_mpc.py:64-65
      p.sigma[s * HA + cc] = sig[cc];
    }
    if (tid == 0) {
      float t = 0.0f;
      for (int cc = 0; cc < HA; ++cc) t = __fadd_rn(t, sig[cc]);
      if (p.iterations_run != nullptr) p.iterations_run[s] += 1;
      if (p.active != nullptr && __fdiv_rn(t, (float)HA) <= p.stddev_threshold)  // cem_mpc.py:66-67
        p.active[s] = 0;
    }
  }
}

cudaError_t launch_refit(const RefitParams& p_in, cudaStream_t st) {
  RefitParams p = p_in;
  const int HA = p.H * p.A;
  const int groups = kRefitThreads / HA > 0 ? kRefitThreads / HA : 1;
  p.groups = groups;
  if (p.K >= 2048) {
    if ((long)p.N * HA > 0x7fffffffL) return cudaErrorInvalidValue;   // 32-bit element offsets in the kernel
    const size_t smem = (size_t)(groups * HA + 3 * HA) * sizeof(float) +
                        (size_t)((p.K + kSelClusterSize - 1) / kSelClusterSize) * sizeof(int);
    return launch_kernel(refit_cluster_kernel, p.S * kSelClusterSize, kRefitThreads, smem, st, kSelClusterSize, false, p);
  }
  const size_t smem = (size_t)(groups * HA + 2 * HA) * sizeof(float);
  refit_kernel<<<p.S, kRefitThreads, smem, st>>>(p);
  return cudaGetLastError();
}

// =============================================================================================
// k11  final noise — simba/policies/cem_mpc.py:68 : best + z * noise_stddev (not re-clipped)
// =============================================================================================
// z * noise_stddev of element idx = s * A + a of the [S, A] action
__device__ __forceinline__ float final_noise(const FinalizeParams& p, int idx) {
  const int s = idx / p.A, a = idx - s * p.A;
  float z;
  if (p.z != nullptr) z = p.z[idx];
  else {
    const float4 n = philox_normals<false>(p.seed_ptr ? *p.seed_ptr : p.seed, kStreamFinal, (uint32_t)s, 0u, 0u, 0u,
                                           (uint32_t)(a >> 2));
    const float zz[4] = {n.x, n.y, n.z, n.w};
    z = zz[a & 3];
  }
  return __fadd_rn(__fmul_rn(z, p.noise_stddev), 0.0f);
}

__device__ __forceinline__ void finalize_element(const FinalizeParams& p, int idx) {
  p.out[idx] = __fadd_rn(p.best[idx], final_noise(p, idx));
}

__global__ void finalize_kernel(FinalizeParams p) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= p.S * p.A) return;
  finalize_element(p, idx);
}

cudaError_t launch_finalize(const FinalizeParams& p, cudaStream_t st) {
  const int n = p.S * p.A;
  finalize_kernel<<<(n + 127) / 128, 128, 0, st>>>(p);
  return cudaGetLastError();
}

// =============================================================================================
// Fused CEM update for small populations (one rank, N <= 1024): k8 + k9 + k10 of this iteration,
// then k1 of the NEXT iteration (or k11 + the plan outputs after the last one), one CTA per state.
// Same device functions and the same arithmetic order as the separate kernels (bit-identical
// results); what it removes is 3-4 kernel boundaries per iteration on the latency-bound C1 plan.
// Selection is rank-by-counting: thread i owns candidate i and counts the keys that beat it.
// =============================================================================================
#ifdef SIMBA_TC_TIMELINE
#define UTL(k) do { if (u.timeline != nullptr && blockIdx.x == 0 && threadIdx.x == 0) { u.timeline[k] = clock64(); \
    unsigned long long gt_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt_)); u.timeline[32 + (k)] = (long long)gt_; } } while (0)
#else
#define UTL(k) do { } while (0)
#endif
// Particles gq, gq + G, ... of candidate i: per-step counts of set mask bits in byte lanes, W words of four
// steps each (fully unrolled), added to the candidate's shared counters cnt_sm[i * ld + w], w < W4
template <int W>
__device__ __forceinline__ void count_steps(const unsigned long long* st_mask, uint32_t* cnt_sm, int i, int gq, int G,
                                            int P, int N, int W4, int ld) {
  uint32_t acc[W];
#pragma unroll
  for (int w = 0; w < W; ++w) acc[w] = 0u;
  for (int q = gq; q < P; q += G) {
    const unsigned long long m = st_mask[q * N + i];
    const uint32_t lo = (uint32_t)m, hi = (uint32_t)(m >> 32);
#pragma unroll
    for (int w = 0; w < W; ++w)
      acc[w] += ((((w < 8 ? lo : hi) >> (4 * (w & 7))) & 0xfu) * 0x00204081u) & 0x01010101u;
  }
#pragma unroll
  for (int w = 0; w < W; ++w)
    if (w < W4 && acc[w] != 0u) atomicAdd(&cnt_sm[i * ld + w], acc[w]);
}

// Shared-memory staging of the fused update kernel (u.stage != 0), behind the elite list, 16-byte aligned:
//   [W][rows] u64 cost-mask planes, [rows] returns, [rows] cost sums   (rows = P * N: the rollout's per-row
//   outputs, W = cmask_planes(H)), [N * HA] this state's current actions, [N * JB * 4] the next iteration's
//   N(0,1) draws, [N] per-candidate maximum step count, [N] per-candidate rank, the per-element action bounds,
//   [N][max(16, ceil(H / 4))] per-step particle counters
__host__ __device__ inline size_t update_stage_bytes(int P, int N, int H, int HA) {
  const size_t rows = (size_t)P * N, JB = (size_t)(HA + 3) / 4;
  const size_t W = (size_t)cmask_planes(H), W4 = (size_t)(H + 3) / 4;
  return rows * (8 * W + 8) + (size_t)N * HA * 4 + (size_t)N * JB * 16 + (size_t)N * 8 + (size_t)(HA + 4) * 8 +
         (size_t)N * 4 * (W4 > 16 ? W4 : 16) + 96;
}

// STAGED is a template parameter so that the kernel a single plan runs carries none of the fallback code
// (measured +0.1 %: the kernel is bound by the latency of its serial path, of which dead branches were a small part).
template <bool STAGED>
__global__ void __launch_bounds__(kRefitThreads) cem_update_kernel(UpdateParams u) {
  UTL(0);
  // PDL: the next rollout may start its prologue (TMEM allocation, barrier init) now.
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  // The kernel is one dependent chain on a single SM (measured: 31 k cycles per iteration before this
  // layout, a fifth of a C1 plan), so it is written for latency:
  //   * it is resident long before the rollout it follows has finished, so everything that does not depend
  //     on that rollout — the next iteration's N(0,1) draws: Philox + the accurate Box-Muller, 7 k cycles of
  //     instruction issue on one SM — happens BEFORE the dependency wait, into shared memory;
  //   * after the wait every global load is issued at once (one L2 round trip, ~2 k cycles here): the
  //     rollout's per-row outputs and the state's current actions are staged in shared memory;
  //   * the per-candidate work is spread over all 1024 threads (150 candidate threads were issue-latency
  //     bound): per-step particle counts by (candidate, step), ranks by (candidate, key chunk), combined
  //     with integer shared-memory atomics — exact, order-free;
  //   * the refit gathers from the staged actions and the next actions are clip(z sigma + mu) from shared
  //     copies. Floating-point arithmetic and its order are those of the separate kernels.
  const int s = blockIdx.x;
  const int tid = threadIdx.x;
  // refit scratch, then keys / elite list, then the staging area. All pointers are `sh + index` (no integer
  // round trips), so the compiler keeps them in the shared address space: with generic pointers every
  // staging store was a generic ST.E that serialised the global loads behind it (eight round trips).
  extern __shared__ __align__(16) float sh[];
  const int HA = u.refit.H * u.refit.A;
  const int groups = u.refit.groups;
  const int N = u.select.N, K = u.select.K;
  const int P = u.reduce.P;
  const int rows = P * N;
  const int JB = (HA + 3) >> 2;
  const int n_planes = cmask_planes(u.reduce.H);                        // 64-step planes of the cost masks
  const int o_keys = (groups + 2) * HA + ((groups + 2) * HA & 1);       // float index, 8-byte aligned
  const int o_elite = o_keys + 2 * N;
  const int o_mask = (o_elite + K + 3) & ~3;                            // 16-byte aligned from here on
  const int o_ret = o_mask + 2 * rows * n_planes;
  const int o_csum = o_ret + rows;
  const int o_act = (o_csum + rows + 3) & ~3;
  const int o_z = (o_act + N * HA + 3) & ~3;
  const int o_maxc = o_z + N * JB * 4;
  unsigned long long* keys = reinterpret_cast<unsigned long long*>(sh + o_keys);
  int* elite_sh = reinterpret_cast<int*>(sh + o_elite);
  unsigned long long* st_mask = reinterpret_cast<unsigned long long*>(sh + o_mask);
  float* st_ret = sh + o_ret;
  float* st_csum = sh + o_csum;
  float* act_sm = sh + o_act;
  float* z_sm = sh + o_z;
  int* maxc_sm = reinterpret_cast<int*>(sh + o_maxc);
  int* rank_sm = maxc_sm + N;
  const int o_lb = (o_maxc + 2 * N + 3) & ~3;
  const int HA4 = (HA + 3) & ~3;
  float* lb_sm = sh + o_lb;                                             // per-element action bounds [HA4] each
  float* ub_sm = lb_sm + HA4;
  const int W4 = (u.reduce.H + 3) >> 2;                                  // 32-bit words of four byte-wide step counters
  uint32_t* cnt_sm = reinterpret_cast<uint32_t*>(ub_sm + HA4);           // [N][W4] particle counts per step
  const float inv_JB = u.inv_JB, inv_N = u.inv_N;
  __shared__ int warp_sums[32];
  __shared__ int sh_total;
  __shared__ int sh_stopped;
  constexpr bool staged = STAGED;
  const bool presample = staged && !u.last;           // Philox draws, or the externally supplied ones (parity mode)
  // the plan's seed is uploaded before the plan's first kernel, which is a full dependency of everything here
  const uint64_t seed_now = u.sample.seed_ptr ? *u.sample.seed_ptr : u.sample.seed;
  if (presample) {
    for (int idx = tid; idx < N * JB; idx += kRefitThreads) {
      const int i = div_small(idx, JB, inv_JB);
      float z[4];
      sample_draws4(u.sample, seed_now, s, i, idx - i * JB, z);
      *reinterpret_cast<float4*>(z_sm + 4 * idx) = make_float4(z[0], z[1], z[2], z[3]);
    }
  }
  if (staged) {
    for (int i = tid; i < 2 * N; i += kRefitThreads) maxc_sm[i] = 0;          // maxc_sm and rank_sm
    for (int i = tid; i < N * W4; i += kRefitThreads) cnt_sm[i] = 0u;
    for (int e = tid; e < HA4; e += kRefitThreads) {                          // bounds of element e (action dim e % A)
      lb_sm[e] = e < HA ? u.sample.lb[e % u.sample.A] : 0.0f;
      ub_sm[e] = e < HA ? u.sample.ub[e % u.sample.A] : 0.0f;
    }
  }
  if (tid == 0) sh_stopped = 0;
  UTL(7);
  // this kernel needs the previous rollout's row outputs (and the update before it): wait for that grid
  asm volatile("griddepcontrol.wait;" ::: "memory");
  UTL(1);
#ifdef SIMBA_TC_TIMELINE
  if (threadIdx.x == 0) s_rtl_ptr = u.timeline;       // only thread 0 reads it back
#endif
  // ---- every load whose address is known, unconditionally and at once --------------------------------
  const bool active = u.refit.active == nullptr || u.refit.active[s] != 0;
  const float best_prev = u.select.best_score[s];
  const bool refit_one = staged && K <= groups;       // refit_single: its mu / sigma / counter loads ride along here
  float mu_old = 0.0f, sg_old = 0.0f;
  int iters_old = 0;
  if (refit_one && tid < HA) { mu_old = u.refit.mu[s * HA + tid]; sg_old = u.refit.sigma[s * HA + tid]; }
  if (refit_one && tid == 0 && u.refit.iterations_run != nullptr) iters_old = u.refit.iterations_run[s];
  if (staged) {
    // batches of four elements per thread and array: all loads of a batch are in flight before the first store
    const float* gret = u.reduce.row_return + (long)s * rows;
    const uint64_t* gmask = u.reduce.row_costmask + (long)s * rows;
    const float* gcsum = u.reduce.row_costsum + (long)s * rows;
    const float* gact = u.select.actions + (long)s * N * HA;
    const int n_act = N * HA;
    if (((rows | n_act) & 3) == 0) {
      // 16-byte loads: rows / 4 + rows / 4 + rows / 2 + n_act / 4 of them, a handful per thread, all in flight together
      const int n1 = rows >> 2, n2 = rows >> 1, n3 = n_act >> 2;
      const float4* g1 = reinterpret_cast<const float4*>(gret);
      const float4* g2 = reinterpret_cast<const float4*>(gcsum);
      const float4* g3 = reinterpret_cast<const float4*>(gmask);
      const float4* g4 = reinterpret_cast<const float4*>(gact);
      float4* d1 = reinterpret_cast<float4*>(st_ret);
      float4* d2 = reinterpret_cast<float4*>(st_csum);
      float4* d3 = reinterpret_cast<float4*>(st_mask);
      float4* d4 = reinterpret_cast<float4*>(act_sm);
      for (int b0 = 0; b0 < n2 || b0 < n3; b0 += 2 * kRefitThreads) {
        float4 v1[2], v2[2], v3[2], v4[2];
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          const int idx = b0 + q * kRefitThreads + tid;
          if (idx < n1) { v1[q] = g1[idx]; v2[q] = g2[idx]; }
          if (idx < n2) v3[q] = g3[idx];
          if (idx < n3) v4[q] = g4[idx];
        }
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          const int idx = b0 + q * kRefitThreads + tid;
          if (idx < n1) { d1[idx] = v1[q]; d2[idx] = v2[q]; }
          if (idx < n2) d3[idx] = v3[q];
          if (idx < n3) d4[idx] = v4[q];
        }
      }
    } else
    for (int b0 = 0; b0 < rows || b0 < n_act; b0 += 4 * kRefitThreads) {
      float r[4], c[4], av[4];
      uint64_t m[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int idx = b0 + q * kRefitThreads + tid;
        if (idx < rows) { r[q] = gret[idx]; m[q] = gmask[idx]; c[q] = gcsum[idx]; }
        if (idx < n_act) av[q] = gact[idx];
      }
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int idx = b0 + q * kRefitThreads + tid;
        if (idx < rows) { st_ret[idx] = r[q]; st_mask[idx] = m[q]; st_csum[idx] = c[q]; }
        if (idx < n_act) act_sm[idx] = av[q];
      }
    }
    if (n_planes > 1) {
      // H > 64: the later planes of the cost masks (global plane stride S * rows: one rank, N_local = N)
#pragma unroll 1
      for (int idx = tid; idx < (n_planes - 1) * rows; idx += kRefitThreads) {
        const int w = 1 + idx / rows, r = idx - (w - 1) * rows;
        st_mask[w * rows + r] = gmask[(long)w * u.reduce.S * rows + r];
      }
    }
  }
  __syncthreads();                                    // staged; everyone has read active[s] before refit clears it
  UTL(8);

  if (active) {
    // ---- k8: (return, cost) of candidate tid --------------------------------------------------
    float2 pr = make_float2(0.0f, 0.0f);
    unsigned long long key = 0ull;
    const int objective = u.reduce.objective;
    if (staged) {
      const bool counts = objective != SIMBA_OBJ_LEAST_COST && objective != SIMBA_OBJ_REWARD;
      if (counts) {
        // Number of particles whose done-masked cost bit is set, per step (safe_cem_mpc.py:110-120): every mask
        // is read once. Thread (i, gq) takes particles gq, gq + G, ... of candidate i and spreads each nibble
        // of the mask into four byte lanes (n * 0x00204081 & 0x01010101 puts bit k of n into byte k), so one
        // 32-bit add counts four steps; the G partial words per candidate are combined with shared-memory
        // atomics (bytes cannot overflow: P <= 255, checked at planner creation). Integer arithmetic: exact and
        // order-free.
        const int G = u.chunks;
        const int gq = div_small(tid, N, inv_N), i = tid - gq * N;
        if (gq < G) {
          if (W4 <= 4) count_steps<4>(st_mask, cnt_sm, i, gq, G, P, N, W4, W4);        // H <= 16
          else if (W4 <= 8) count_steps<8>(st_mask, cnt_sm, i, gq, G, P, N, W4, W4);   // H <= 32
          else                                                                      // 64 steps per plane
#pragma unroll 1
            for (int w = 0; w < n_planes; ++w)
              count_steps<16>(st_mask + w * rows, cnt_sm + 16 * w, i, gq, G, P, N, min(16, W4 - 16 * w), W4);
        }
      }
      float ret = 0.0f, csum = 0.0f;
      if (tid < N) {
#pragma unroll 4
        for (int q = 0; q < P; ++q) {                   // fixed order (p ascending), as reduce_rows
          ret = __fadd_rn(ret, st_ret[q * N + tid]);
          csum = __fadd_rn(csum, st_csum[q * N + tid]);
        }
      }
      __syncthreads();
      if (tid < N) {
        float cost = 0.0f;
        if (objective == SIMBA_OBJ_LEAST_COST) cost = __fdiv_rn(csum, (float)P);
        else if (counts) {
          uint32_t mx = 0u;                                   // max over the byte lanes (steps >= H are never set)
          for (int w = 0; w < W4; ++w) {
            const uint32_t c4 = cnt_sm[tid * W4 + w];
            mx = max(max(mx, c4 & 0xffu), max((c4 >> 8) & 0xffu, max((c4 >> 16) & 0xffu, c4 >> 24)));
          }
          cost = (float)mx;
        }
        pr = make_float2(__fdiv_rn(ret, (float)P), cost);
      }
    } else if (tid < N) {
      pr = reduce_candidate(u.reduce, s, tid);
    }
    if (tid < N) {
      if (u.reduce.out_pairs != nullptr) reinterpret_cast<float2*>(u.reduce.out_pairs)[(long)s * N + tid] = pr;
      key = pair_key(u.select.objective, pr.x, pr.y, u.select.c_max);
      // Rank key: the order key with the index folded in (lower index wins ties), so that one 64-bit compare
      // decides "j beats i": class bit 63 -> bit 50, bits 32..39 (violations, FEASIBLE_FIRST) -> 42..49, the
      // ordered score -> bits 10..41, 1023 - index in the low ten bits (N <= 1024 on this path).
      if (staged)
        key = ((key >> 63) << 50) | (((key >> 32) & 0xffull) << 42) | ((key & 0xffffffffull) << 10) |
              (unsigned long long)(1023 - tid);
      keys[tid] = key;
    }
    UTL(9);
    __syncthreads();
    UTL(2);
    // ---- k9: rank by counting (ties -> lower index), ordered compaction, best-so-far ------------
    int rank = 0;
    const int chunks = u.chunks;                        // key chunks per candidate: kRefitThreads / N
    if (staged && chunks > 1) {
      const int ch = div_small(tid, N, inv_N), i = tid - ch * N;
      if (ch < chunks) {
        const int per = u.per;
        const int j0 = ch * per, j1 = min(N, j0 + per);
        const unsigned long long ki = keys[i];
        int cnt = 0;
#pragma unroll 5
        for (int jn = j0; jn < j1; ++jn) cnt += keys[jn] > ki ? 1 : 0;      // rank keys are unique
        if (cnt > 0) atomicAdd(&rank_sm[i], cnt);
      }
      __syncthreads();
      if (tid < N) rank = rank_sm[tid];
    } else if (tid < N) {
#pragma unroll 8
      for (int jn = 0; jn < N; ++jn) {
        const unsigned long long kj = keys[jn];
        rank += (kj > key || (kj == key && jn < tid)) ? 1 : 0;   // also right for rank keys (never equal)
      }
    }
    const int sel = (tid < N && rank < K) ? 1 : 0;
    UTL(3);
    const int pos = block_exclusive_scan<kRefitThreads>(sel, warp_sums, &sh_total);
    if (sel) {
      elite_sh[pos] = tid;
      u.select.out_elite[(long)s * K + pos] = tid;
    }
    if (tid < N && u.select.out_scores != nullptr)
      u.select.out_scores[(long)s * N + tid] = pair_score(u.select.objective, pr.x, pr.y, u.select.c_max);
    if (tid < N && rank == 0) {                                   // argmax, first max
      const float top_score = pair_score(u.select.objective, pr.x, pr.y, u.select.c_max);
      if (top_score > best_prev) {                                // cem_mpc.py:58 strict '>'
        const float* arow = staged ? act_sm + tid * HA : u.select.actions + ((long)s * N + tid) * HA;
        for (int a = 0; a < u.select.A; ++a) u.select.best_action[s * u.select.A + a] = arow[a];
        u.select.best_score[s] = top_score;
      }
    }
    __syncthreads();
    UTL(4);
    // ---- k10: refit (also clears active[s] when the stddev threshold is met) --------------------
    if (refit_one) refit_single(u.refit, s, elite_sh, act_sm, sh, sh + groups * HA, sh + (groups + 1) * HA, &sh_stopped,
                                mu_old, sg_old, iters_old);
    else refit_body(u.refit, s, elite_sh, sh, &sh_stopped, staged ? act_sm : nullptr);
    __syncthreads();
    UTL(5);
  }
  if (!u.last) {
    // ---- k1 of the next iteration (skipped for states that just stopped, like the early break) --
    if (active && sh_stopped == 0) {
      const float* mu_s = sh + groups * HA;            // refit_body left mu_new / sigma_new of this state here
      const float* sigma_s = sh + (groups + 1) * HA;
      for (int idx = tid; idx < N * JB; idx += kRefitThreads) {
        const int i = div_small(idx, JB, inv_JB), j = idx - i * JB;
        float z[4], out[4];
        if (staged) {                                     // draws made before the dependency wait
          const float4 zz = *reinterpret_cast<const float4*>(z_sm + 4 * idx);
          z[0] = zz.x; z[1] = zz.y; z[2] = zz.z; z[3] = zz.w;
        } else {
          sample_draws4(u.sample, seed_now, s, i, j, z);
        }
        if (staged && (HA & 3) == 0) {
          // sample_apply4 on 16-byte shared-memory reads: mu, sigma and the per-element bounds of elements 4 j .. 4 j + 3
          const float4 m4 = *reinterpret_cast<const float4*>(mu_s + 4 * j), s4 = *reinterpret_cast<const float4*>(sigma_s + 4 * j);
          const float4 l4 = *reinterpret_cast<const float4*>(lb_sm + 4 * j), u4 = *reinterpret_cast<const float4*>(ub_sm + 4 * j);
          out[0] = fminf(fmaxf(__fadd_rn(__fmul_rn(z[0], s4.x), m4.x), l4.x), u4.x);
          out[1] = fminf(fmaxf(__fadd_rn(__fmul_rn(z[1], s4.y), m4.y), l4.y), u4.y);
          out[2] = fminf(fmaxf(__fadd_rn(__fmul_rn(z[2], s4.z), m4.z), l4.z), u4.z);
          out[3] = fminf(fmaxf(__fadd_rn(__fmul_rn(z[3], s4.w), m4.w), l4.w), u4.w);
        } else if (staged) {
          // sample_apply4 with the per-element bounds from shared memory (no e % A, no indexed constant loads)
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const int e = 4 * j + q;                    // < HA4: the tables are padded
            const float v = __fadd_rn(__fmul_rn(z[q], sigma_s[e < HA ? e : 0]), mu_s[e < HA ? e : 0]);
            out[q] = e < HA ? fminf(fmaxf(v, lb_sm[e]), ub_sm[e]) : 0.0f;
          }
        } else {
          sample_apply4(u.sample, mu_s, sigma_s, z, j, out);
        }
        store_block4(u.sample, s, i, j, out, u.sample.out);
      }
    }
  } else {
    // ---- k11 + plan outputs ----------------------------------------------------------------------
    __threadfence_block();
    __syncthreads();
    if (tid < u.finalize.A) finalize_element(u.finalize, s * u.finalize.A + tid);
    if (tid == 0) {
      u.out_score[s] = u.select.best_score[s];
      if (u.out_iters != nullptr) u.out_iters[s] = u.refit.iterations_run[s];
    }
  }
  UTL(6);
}

size_t cem_update_smem_bytes(int P, int N, int K, int H, int A, bool* staged) {
  const int HA = H * A;
  const int groups = kRefitThreads / HA > 0 ? kRefitThreads / HA : 1;
  size_t smem = (size_t)((groups + 2) * HA + 1) * sizeof(float);
  smem = (smem + 7) / 8 * 8 + (size_t)N * 8 + (size_t)K * 4 + 16;
  // the staging area (rows, actions, draws; see update_stage_bytes), when it fits
  const size_t stage = update_stage_bytes(P, N, H, HA);
  *staged = smem + stage + 1024 <= 200 * 1024 && N <= kRefitThreads;
  return *staged ? smem + stage : smem;
}

cudaError_t launch_cem_update(const UpdateParams& u_in, cudaStream_t st) {
  UpdateParams u = u_in;
  const int HA = u.refit.H * u.refit.A;
  u.refit.groups = kRefitThreads / HA > 0 ? kRefitThreads / HA : 1;
  u.chunks = kRefitThreads / u.select.N > 0 ? kRefitThreads / u.select.N : 1;
  u.per = (u.select.N + u.chunks - 1) / u.chunks;
  u.inv_N = 1.0f / (float)u.select.N;
  u.inv_JB = 1.0f / (float)((HA + 3) / 4);
  bool staged = false;
  const size_t smem = cem_update_smem_bytes(u.reduce.P, u.select.N, u.select.K, u.refit.H, u.refit.A, &staged);
  u.stage = staged ? 1 : 0;
  return launch_kernel(u.stage ? cem_update_kernel<true> : cem_update_kernel<false>, u.refit.S, kRefitThreads, smem, st,
                       1, u.pdl != 0, u);
}

// =============================================================================================
// MPPI update — Williams et al., "Information theoretic MPC for model-based reinforcement learning"
// (ICRA 2017), the update PDDM (Nagabandi et al., 2019) plans with: every candidate contributes to the
// new mean, weighted by exp((score - max score) / temperature); sigma stays fixed. Sampling, rollout,
// scoring and the final noise are CEM's code. Both sums of the weighted mean run in one fixed order on
// every path: ascending within blocks of 32 candidates, blocks folded in ascending order into
// superblocks of 1024 candidates, superblocks folded in ascending order. The fused kernel (N <= 1024,
// one superblock) and the separate refit kernel therefore give the same bits.
// =============================================================================================
constexpr int kMppiThreads = 1024;
constexpr int kMppiSuper = 1024;          // candidates per superblock
constexpr int kMppiBlock = 32;            // candidates per block
constexpr int kMppiClusterSize = 8;       // CTAs per state of the refit when N > kMppiSuper

// weight of a score against the largest non-NaN score m; a NaN score (a diverged rollout) weighs 0
__device__ __forceinline__ float mppi_weight(float score, float m, float temperature) {
  return score != score ? 0.0f : expf(__fdiv_rn(__fsub_rn(score, m), temperature));
}

// order key of the best candidate: larger score first, the lower index among ties. A key whose upper half is 0
// belongs to a NaN score, so a maximum of 0 means every score was NaN.
__device__ __forceinline__ unsigned long long mppi_key(float score, int i) {
  return ((unsigned long long)ordered_u32(score) << 32) | (unsigned long long)(0xffffffffu - (uint32_t)i);
}
__device__ __forceinline__ int mppi_key_index(unsigned long long k) { return (int)(0xffffffffu - (uint32_t)k); }
__device__ __forceinline__ float mppi_key_score(unsigned long long k) {     // inverse of ordered_u32 (-0 reads +0)
  const uint32_t u = (uint32_t)(k >> 32);
  return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u);
}

// the largest key over the CTA, returned to every thread; called once per kernel (slot: a shared word)
__device__ __forceinline__ unsigned long long mppi_block_max(unsigned long long k, unsigned long long* slot) {
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) {
    const unsigned long long o = __shfl_xor_sync(0xffffffffu, k, d);
    k = o > k ? o : k;
  }
  if (threadIdx.x == 0) *slot = 0ull;
  __syncthreads();
  if ((threadIdx.x & 31) == 0) atomicMax(slot, k);
  __syncthreads();
  return *slot;
}

// One superblock's column sums: out[c] = sum_i w[i] * acts[i * HA + c] for c < HA and out[HA] = sum_i w[i], over
// i < n <= kMppiSuper, in the fixed block order. acts: global or shared memory. blk: [ceil(n / 32)][HA + 1] shared
// partials. Called by all kMppiThreads threads; ends with a CTA barrier.
__device__ __forceinline__ void mppi_superblock(const float* w, const float* acts, int n, int HA, float* blk,
                                                float* out) {
  const int C = HA + 1, nb = (n + kMppiBlock - 1) / kMppiBlock;
  for (int it = threadIdx.x; it < nb * C; it += kMppiThreads) {
    const int b = it / C, c = it - b * C;
    const int i0 = b * kMppiBlock, i1 = min(n, i0 + kMppiBlock);
    float acc = 0.0f;
    if (c < HA) {
#pragma unroll 8
      for (int i = i0; i < i1; ++i) acc = __fadd_rn(acc, __fmul_rn(w[i], acts[(long)i * HA + c]));
    } else {
      for (int i = i0; i < i1; ++i) acc = __fadd_rn(acc, w[i]);
    }
    blk[it] = acc;
  }
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += kMppiThreads) {
    float acc = blk[c];
    for (int b = 1; b < nb; ++b) acc = __fadd_rn(acc, blk[b * C + c]);
    out[c] = acc;
  }
  __syncthreads();
}

// mu <- smoothing mu + (1 - smoothing) tot[c] / tot[HA], in the CEM refit's operation order; left unchanged when
// every score was NaN. Best-so-far with strict '>' from the top key (acts_top: that candidate's row), and one more
// iteration run. mu_sm (or null) receives this state's mean after the update. Called by every thread of one CTA.
__device__ __forceinline__ void mppi_finish(const MppiParams& p, int s, unsigned long long top, const float* tot,
                                            const float* acts_top, float* mu_sm) {
  const int HA = p.H * p.A;
  const bool valid = (top >> 32) != 0ull;
  const float best_prev = p.best_score[s];
  for (int c = threadIdx.x; c < HA; c += kMppiThreads) {
    float v = p.mu[s * HA + c];
    if (valid) {
      v = __fadd_rn(__fmul_rn(p.smoothing, v), __fmul_rn(p.one_minus_smoothing, __fdiv_rn(tot[c], tot[HA])));
      p.mu[s * HA + c] = v;
    }
    if (mu_sm != nullptr) mu_sm[c] = v;
  }
  __syncthreads();                                     // best_score[s] has been read by every thread
  const float top_score = mppi_key_score(top);
  if (valid && top_score > best_prev) {                // cem_mpc.py:58 strict '>'
    if (threadIdx.x < p.A) p.best_action[s * p.A + threadIdx.x] = acts_top[threadIdx.x];
    if (threadIdx.x == 0) p.best_score[s] = top_score;
  }
  if (threadIdx.x == 0 && p.iterations_run != nullptr) p.iterations_run[s] += 1;
}

// The separate refit: `ctas` CTAs per state (a cluster of kMppiClusterSize when N > kMppiSuper, one CTA otherwise),
// CTA r taking superblocks [r per, r per + per). The maximum is combined over the cluster (exact); rank 0 folds every
// superblock's sums in ascending order through distributed shared memory.
__global__ void __launch_bounds__(kMppiThreads) mppi_refit_kernel(MppiParams p, int ctas, int per) {
  const int s = blockIdx.x / ctas, rank = blockIdx.x - s * ctas;
  if (p.active != nullptr && p.active[s] == 0) return;      // uniform over the cluster
  extern __shared__ __align__(16) float sh[];
  const int HA = p.H * p.A, C = HA + 1, N = p.N;
  float* w = sh;                                             // [kMppiSuper] weights of one superblock
  float* blk = w + kMppiSuper;                               // [32][C] block partials
  float* sbp = blk + kMppiBlock * C;                         // [per][C] this CTA's superblock sums
  float* tot = sbp + per * C;                                // [C]
  __shared__ unsigned long long sh_key;
  const float2* pairs = reinterpret_cast<const float2*>(p.pairs) + (long)s * N;
  const int lo = min(N, rank * per * kMppiSuper), hi = min(N, lo + per * kMppiSuper);
  unsigned long long k = 0ull;
  for (int i = lo + threadIdx.x; i < hi; i += kMppiThreads) {
    const float2 pr = pairs[i];
    const unsigned long long ki = mppi_key(pair_score(p.objective, pr.x, pr.y, p.c_max), i);
    k = ki > k ? ki : k;
  }
  unsigned long long top = mppi_block_max(k, &sh_key);
  cg::cluster_group cluster = cg::this_cluster();
  if (ctas > 1) {
    cluster.sync();                                          // every CTA's maximum is in its sh_key
    for (int r = 0; r < ctas; ++r) {
      const unsigned long long o = *cluster.map_shared_rank(&sh_key, r);
      top = o > top ? o : top;
    }
  }
  const float m = mppi_key_score(top);
  const float* acts = p.actions + (long)s * N * HA;
  for (int q = 0; lo + q * kMppiSuper < hi; ++q) {
    const int i0 = lo + q * kMppiSuper, n = min(kMppiSuper, hi - i0);
    for (int j = threadIdx.x; j < n; j += kMppiThreads) {
      const float2 pr = pairs[i0 + j];
      w[j] = mppi_weight(pair_score(p.objective, pr.x, pr.y, p.c_max), m, p.temperature);
    }
    __syncthreads();
    mppi_superblock(w, acts + (long)i0 * HA, n, HA, blk, sbp + q * C);
  }
  if (ctas > 1) cluster.sync();                              // every superblock's sums are complete
  if (rank == 0) {
    const int n_super = (N + kMppiSuper - 1) / kMppiSuper;
    for (int c = threadIdx.x; c < C; c += kMppiThreads) {
      float acc = sbp[c];
#pragma unroll 8
      for (int g = 1; g < n_super; ++g) {
        const int r = g / per;
        const float* src = r == 0 ? sbp : cluster.map_shared_rank(sbp, r);
        acc = __fadd_rn(acc, src[(g - r * per) * C + c]);
      }
      tot[c] = acc;
    }
    __syncthreads();
    mppi_finish(p, s, top, tot, acts + (long)mppi_key_index(top) * HA, nullptr);
  }
  if (ctas > 1) cluster.sync();                              // no CTA exits while rank 0 reads its shared memory
}

static void mppi_refit_geometry(int N, int* ctas, int* per) {
  const int n_super = (N + kMppiSuper - 1) / kMppiSuper;
  *ctas = n_super > 1 ? kMppiClusterSize : 1;
  *per = (n_super + *ctas - 1) / *ctas;
}

size_t mppi_refit_smem_bytes(int N, int H, int A) {
  int ctas = 1, per = 1;
  mppi_refit_geometry(N, &ctas, &per);
  const size_t C = (size_t)H * A + 1;
  return (kMppiSuper + (kMppiBlock + per + 1) * C) * sizeof(float);
}

cudaError_t launch_mppi_refit(const MppiParams& p, cudaStream_t st) {
  int ctas = 1, per = 1;
  mppi_refit_geometry(p.N, &ctas, &per);
  return launch_kernel(mppi_refit_kernel, p.S * ctas, kMppiThreads, mppi_refit_smem_bytes(p.N, p.H, p.A), st, ctas,
                       false, p, ctas, per);
}

// Fused MPPI update for one rank's population of at most 1024 candidates, one CTA per state: k8 of this iteration
// (the rows staged in shared memory when they fit, reduced by reduce_rows), the update, then k1 of the NEXT iteration
// from the new mean, or k11 on mu[s, 0, :] and the plan outputs after the last one. Launched behind the rollout as a
// programmatic dependent, like cem_update_kernel. The same device functions as score_reduce_kernel, mppi_refit_kernel,
// sample_actions_kernel and finalize_kernel: the same bits.
template <bool STAGED>
__global__ void __launch_bounds__(kMppiThreads) mppi_update_kernel(MppiUpdateParams u) {
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  asm volatile("griddepcontrol.wait;" ::: "memory");
  const MppiParams& p = u.mppi;
  const int s = blockIdx.x, tid = threadIdx.x;
  const int HA = p.H * p.A, C = HA + 1, N = p.N, P = u.reduce.P, rows = P * N;
  const int n_planes = cmask_planes(u.reduce.H);
  extern __shared__ __align__(16) float sh[];
  float* w = sh;                                             // [N] weights
  float* blk = w + kMppiSuper;                               // [32][C] block partials
  float* tot = blk + kMppiBlock * C;                         // [C]
  float* mu_sm = tot + C;                                    // [HA] the new mean
  float* sg_sm = mu_sm + HA;                                 // [HA] sigma
  const int o_stage = (kMppiSuper + (kMppiBlock + 1) * C + 2 * HA + 3) & ~3;
  uint64_t* st_mask = reinterpret_cast<uint64_t*>(sh + o_stage);             // [W][rows]
  float* st_ret = sh + o_stage + 2 * n_planes * rows;        // [rows]
  float* st_csum = st_ret + rows;                            // [rows]
  float* act_sm = st_csum + rows;                            // [N][HA]
  __shared__ unsigned long long sh_key;
  const bool active = p.active == nullptr || p.active[s] != 0;
  if (active) {
    if (STAGED) {
      const float* gret = u.reduce.row_return + (long)s * rows;
      const float* gcsum = u.reduce.row_costsum + (long)s * rows;
      const uint64_t* gmask = u.reduce.row_costmask + (long)s * rows;
      const float* gact = p.actions + (long)s * N * HA;
      for (int idx = tid; idx < rows; idx += kMppiThreads) { st_ret[idx] = gret[idx]; st_csum[idx] = gcsum[idx]; }
      for (int idx = tid; idx < n_planes * rows; idx += kMppiThreads) {   // plane stride S * rows in global memory
        const int pl = idx / rows;
        st_mask[idx] = gmask[(long)pl * u.reduce.S * rows + (idx - pl * rows)];
      }
      for (int idx = tid; idx < N * HA; idx += kMppiThreads) act_sm[idx] = gact[idx];
      __syncthreads();
    }
    float score = 0.0f;
    unsigned long long k = 0ull;
    if (tid < N) {
      const float2 pr = STAGED ? reduce_rows(st_ret, st_mask, st_csum, tid, N, P, u.reduce.H, rows, u.reduce.objective)
                               : reduce_candidate(u.reduce, s, tid);
      if (u.reduce.out_pairs != nullptr) reinterpret_cast<float2*>(u.reduce.out_pairs)[(long)s * N + tid] = pr;
      score = pair_score(p.objective, pr.x, pr.y, p.c_max);
      k = mppi_key(score, tid);
    }
    const unsigned long long top = mppi_block_max(k, &sh_key);
    if (tid < N) w[tid] = mppi_weight(score, mppi_key_score(top), p.temperature);
    __syncthreads();
    const float* acts = STAGED ? act_sm : p.actions + (long)s * N * HA;
    mppi_superblock(w, acts, N, HA, blk, tot);
    mppi_finish(p, s, top, tot, acts + (long)mppi_key_index(top) * HA, mu_sm);
    __syncthreads();
  }
  if (!u.last) {
    if (active) {                                            // k1 of the next iteration, from the new mean
      for (int c = tid; c < HA; c += kMppiThreads) sg_sm[c] = u.sample.sigma[s * HA + c];
      __syncthreads();
      const uint64_t seed = u.sample.seed_ptr ? *u.sample.seed_ptr : u.sample.seed;
      const int JB = (HA + 3) >> 2;
      for (int idx = tid; idx < N * JB; idx += kMppiThreads) {
        const int i = idx / JB, j = idx - i * JB;
        float out[4];
        sample_values4_from(u.sample, mu_sm, sg_sm, seed, s, i, j, out);
        store_block4(u.sample, s, i, j, out, u.sample.out);
      }
    }
  } else {
    // ---- k11 on mu[s, 0, :] + plan outputs ----------------------------------------------------------
    __threadfence_block();
    __syncthreads();
    if (tid < u.finalize.A) {
      const int idx = s * u.finalize.A + tid;
      u.finalize.out[idx] = __fadd_rn(mu_sm[tid], final_noise(u.finalize, idx));     // mu[s, 0, a] + noise
    }
    if (tid == 0) {
      u.out_score[s] = p.best_score[s];
      if (u.out_iters != nullptr) u.out_iters[s] = p.iterations_run[s];
    }
  }
}

// k11 of an MPPI plan: mu[s, 0, :] + noise (p.best = mu [S, H, A])
__global__ void mppi_finalize_kernel(FinalizeParams p, int HA) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= p.S * p.A) return;
  const int s = idx / p.A;
  p.out[idx] = __fadd_rn(p.best[s * HA + (idx - s * p.A)], final_noise(p, idx));
}

cudaError_t launch_mppi_finalize(const FinalizeParams& p, int HA, cudaStream_t st) {
  const int n = p.S * p.A;
  mppi_finalize_kernel<<<(n + 127) / 128, 128, 0, st>>>(p, HA);
  return cudaGetLastError();
}

size_t mppi_update_smem_bytes(int P, int N, int H, int A, bool* staged) {
  const int HA = H * A, C = HA + 1;
  const size_t base = (size_t)((kMppiSuper + (kMppiBlock + 1) * C + 2 * HA + 3) & ~3) * sizeof(float);
  const size_t rows = (size_t)P * N;
  const size_t stage = rows * (8 * (size_t)cmask_planes(H) + 8) + (size_t)N * HA * 4;
  *staged = base + stage + 1024 <= 200 * 1024;
  return *staged ? base + stage : base;
}

cudaError_t launch_mppi_update(const MppiUpdateParams& u_in, cudaStream_t st) {
  MppiUpdateParams u = u_in;
  if (u.mppi.N > kMppiSuper) return cudaErrorInvalidValue;
  bool staged = false;
  const size_t smem = mppi_update_smem_bytes(u.reduce.P, u.mppi.N, u.mppi.H, u.mppi.A, &staged);
  u.stage = staged ? 1 : 0;
  return launch_kernel(staged ? mppi_update_kernel<true> : mppi_update_kernel<false>, u.mppi.S, kMppiThreads, smem, st,
                       1, u.pdl != 0, u);
}

// plan bookkeeping: reset mu/sigma/best/active at the start of a plan (cem_mpc.py:36-42)
__global__ void plan_init_kernel(PlanInitParams p) {
  const int HA = p.H * p.A;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx < p.S * HA) {
    const int a = (idx % HA) % p.A;
    p.mu[idx] = p.init_mean[a];
    p.sigma[idx] = p.init_stddev[a];
  }
  if (idx < p.S * p.A) p.best_action[idx] = 0.0f;
  if (idx < p.S) {
    p.best_score[idx] = -INFINITY;
    p.active[idx] = 1;
    p.iterations_run[idx] = 0;
  }
}

// plan_init + the first iteration's sampling in one launch (the fused single-rank plan): mu / sigma of iteration 0
// are the initial mean / stddev per action dimension, so no thread has to read what another one initialises
__global__ void __launch_bounds__(256) plan_begin_kernel(PlanInitParams ip, SampleParams sp) {
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");   // the first rollout's prologue may start
  __shared__ float mu0[1024], sg0[1024];                            // H * A <= 1024 (checked at creation)
  const int HA = ip.H * ip.A;
  for (int e = threadIdx.x; e < HA; e += blockDim.x) {
    mu0[e] = ip.init_mean[e % ip.A];
    sg0[e] = ip.init_stddev[e % ip.A];
  }
  const long gtid = blockIdx.x * (long)blockDim.x + threadIdx.x, gsize = (long)gridDim.x * blockDim.x;
  for (long idx = gtid; idx < (long)ip.S * HA; idx += gsize) {
    const int a = (int)(idx % HA) % ip.A;
    ip.mu[idx] = ip.init_mean[a];
    ip.sigma[idx] = ip.init_stddev[a];
  }
  for (long idx = gtid; idx < (long)ip.S * ip.A; idx += gsize) ip.best_action[idx] = 0.0f;
  for (long idx = gtid; idx < ip.S; idx += gsize) {
    ip.best_score[idx] = -INFINITY;
    ip.active[idx] = 1;
    ip.iterations_run[idx] = 0;
  }
  __syncthreads();
  const uint64_t seed = sp.seed_ptr ? *sp.seed_ptr : sp.seed;
  const int JB = (HA + 3) >> 2;
  const long total = (long)sp.S * sp.N * JB;
  for (long idx = gtid; idx < total; idx += gsize) {
    const int j = (int)(idx % JB);
    const long si = idx / JB;
    const int s = (int)(si / sp.N), i = (int)(si - (long)s * sp.N);
    float out[4];
    sample_values4_from(sp, mu0, sg0, seed, s, i, j, out);
    store_block4(sp, s, i, j, out, sp.out);
  }
}

cudaError_t launch_plan_begin(const PlanInitParams& ip, const SampleParams& sp, cudaStream_t st) {
  const long total = (long)sp.S * sp.N * ((sp.H * sp.A + 3) / 4);
  int blocks = (int)((total + 255) / 256);
  if (blocks > 148 * 8) blocks = 148 * 8;
  if (blocks < 1) blocks = 1;
  plan_begin_kernel<<<blocks, 256, 0, st>>>(ip, sp);
  return cudaGetLastError();
}

cudaError_t launch_plan_init(const PlanInitParams& p, cudaStream_t st) {
  const int n = p.S * p.H * p.A;
  plan_init_kernel<<<(n + 255) / 256, 256, 0, st>>>(p);
  return cudaGetLastError();
}

__global__ void plan_output_kernel(const float* best_score, const int32_t* iterations_run,
                                   float* out_score, int32_t* out_iters, int S) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx < S) {
    out_score[idx] = best_score[idx];
    if (out_iters != nullptr) out_iters[idx] = iterations_run[idx];
  }
}

cudaError_t launch_plan_output(const float* best_score, const int32_t* iterations_run,
                               float* out_score, int32_t* out_iters, int S, cudaStream_t st) {
  plan_output_kernel<<<(S + 127) / 128, 128, 0, st>>>(best_score, iterations_run, out_score,
                                                       out_iters, S);
  return cudaGetLastError();
}

// =============================================================================================
// Batch versions of the reference's public helper methods
// =============================================================================================
// TransitionModel.scale — simba/models/transition_model.py:79-87
__global__ void scale_kernel(const float* x, const float* smin, const float* sdelta, int scale_on,
                             long total, int IN, float* out) {
  const long idx = blockIdx.x * (long)blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int k = (int)(idx % IN);
  out[idx] = scale_on ? __fdiv_rn(__fsub_rn(x[idx], smin[k]), sdelta[k]) : x[idx];
}

cudaError_t launch_scale(const float* x, const float* smin, const float* sdelta, int scale_on,
                         long batch, int IN, float* out, cudaStream_t st) {
  const long total = batch * IN;
  scale_kernel<<<(int)((total + 255) / 256), 256, 0, st>>>(x, smin, sdelta, scale_on, total, IN, out);
  return cudaGetLastError();
}

// SafetyGymStateScorer.reward / .cost — simba/environment_utils/safety_gym.py:110-166
__global__ void scorer_eval_kernel(simba_scorer_t sc, const float* obs, const float* next_obs,
                                   int batch, int O, float* out_reward, int32_t* out_done,
                                   float* out_cost) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= batch) return;
  const float* a = obs + (long)r * O;
  auto lda = [&](int b) { return a[b]; };
  if (out_cost != nullptr) out_cost[r] = state_cost(sc, lda);
  if (out_reward != nullptr && next_obs != nullptr) {
    const float* n = next_obs + (long)r * O;
    const float d0 = goal_distance(sc, lda);
    const float d1 = goal_distance(sc, [&](int b) { return n[b]; });
    const bool goal = d0 <= sc.goal_threshold;
    out_reward[r] = step_reward(sc, d0, d1, goal);
    if (out_done != nullptr) out_done[r] = goal ? 1 : 0;
  }
}

cudaError_t launch_scorer_eval(const simba_scorer_t& sc, const float* obs, const float* next_obs,
                               int batch, int O, float* out_reward, int32_t* out_done,
                               float* out_cost, cudaStream_t st) {
  scorer_eval_kernel<<<(batch + 127) / 128, 128, 0, st>>>(sc, obs, next_obs, batch, O, out_reward,
                                                           out_done, out_cost);
  return cudaGetLastError();
}

// per-row part of compute_objective on materialised trajectories [rows, H+1, O]
// (simba/policies/mpc_policy.py:30-37, simba/policies/safe_cem_mpc.py:82-93)
__global__ void score_traj_rows_kernel(simba_scorer_t sc, const float* traj, int rows, int H, int O,
                                       int objective, float* row_return, uint64_t* row_costmask,
                                       float* row_costsum) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= rows) return;
  const float* base = traj + (long)r * (H + 1) * O;
  RowScore rs;
  row_score_init(rs, sc, [&](int b) { return base[b]; });
  const bool done_first = objective_done_first(objective);
  for (int t = 0; t < H; ++t) {
    const float* nx = base + (long)(t + 1) * O;
    row_score_step(rs, sc, done_first, t, [&](int b) { return nx[b]; });
    if (cmask_word_ends(t, H)) {                       // planes [W, rows]
      row_costmask[(long)(t >> 6) * rows + r] = rs.cmask;
      rs.cmask = 0ull;
    }
  }
  row_return[r] = rs.cum;
  row_costmask[(long)((H - 1) >> 6) * rows + r] = rs.cmask;
  row_costsum[r] = rs.costsum;
}

cudaError_t launch_score_traj_rows(const simba_scorer_t& sc, const float* traj, int rows, int H,
                                   int O, int objective, float* row_return, uint64_t* row_costmask,
                                   float* row_costsum, cudaStream_t st) {
  score_traj_rows_kernel<<<(rows + 127) / 128, 128, 0, st>>>(sc, traj, rows, H, O, objective,
                                                             row_return, row_costmask, row_costsum);
  return cudaGetLastError();
}

__global__ void pairs_to_scores_kernel(const float* pairs, int n, int objective, float c_max,
                                       float* out_scores) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float2 pr = reinterpret_cast<const float2*>(pairs)[i];
  out_scores[i] = pair_score(objective, pr.x, pr.y, c_max);
}

cudaError_t launch_pairs_to_scores(const float* pairs, int n, int objective, float c_max,
                                   float* out_scores, cudaStream_t st) {
  pairs_to_scores_kernel<<<(n + 255) / 256, 256, 0, st>>>(pairs, n, objective, c_max, out_scores);
  return cudaGetLastError();
}

// =============================================================================================
// RNG contract probes
// =============================================================================================
__global__ void philox_raw_kernel(uint4 ctr, uint2 key, uint32_t* out) {
  const uint4 r = philox4x32_10(ctr, key);
  out[0] = r.x; out[1] = r.y; out[2] = r.z; out[3] = r.w;
}

cudaError_t launch_philox_raw(const uint32_t ctr[4], const uint32_t key[2], uint32_t* out_dev,
                              cudaStream_t st) {
  philox_raw_kernel<<<1, 1, 0, st>>>(make_uint4(ctr[0], ctr[1], ctr[2], ctr[3]),
                                     make_uint2(key[0], key[1]), out_dev);
  return cudaGetLastError();
}

template <bool kFast>
__global__ void philox_normals_kernel(uint64_t seed, uint32_t stream, uint32_t iteration,
                                      uint32_t t, uint32_t s, uint32_t first_row, int n_rows,
                                      int n_elems, float* out) {
  const int per = (stream == kStreamNoise) ? 8 : 4;       // NOISE: 8 normals per block (16-bit uniforms)
  const int JB = (n_elems + per - 1) / per;
  const long idx = blockIdx.x * (long)blockDim.x + threadIdx.x;
  if (idx >= (long)n_rows * JB) return;
  const int row = (int)(idx / JB), j = (int)(idx % JB);
  float z[8];
  if (stream == kStreamNoise) {
    philox_noise8<kFast>(seed, s, iteration, t, first_row + row, (uint32_t)j, z);
  } else {
    const float4 n = philox_normals<kFast>(seed, stream, s, iteration, t, first_row + row, (uint32_t)j);
    z[0] = n.x; z[1] = n.y; z[2] = n.z; z[3] = n.w;
  }
  for (int q = 0; q < per; ++q)
    if (per * j + q < n_elems) out[(long)row * n_elems + per * j + q] = z[q];
}

cudaError_t launch_philox_normals(uint64_t seed, int stream, int iteration, int t, int s,
                                  int first_row, int n_rows, int n_elems, int fast, float* out,
                                  cudaStream_t st) {
  const int per = (stream == (int)kStreamNoise) ? 8 : 4;
  const long total = (long)n_rows * ((n_elems + per - 1) / per);
  const int blocks = (int)((total + 255) / 256);
  if (fast)
    philox_normals_kernel<true><<<blocks, 256, 0, st>>>(seed, stream, iteration, t, s, first_row,
                                                        n_rows, n_elems, out);
  else
    philox_normals_kernel<false><<<blocks, 256, 0, st>>>(seed, stream, iteration, t, s, first_row,
                                                         n_rows, n_elems, out);
  return cudaGetLastError();
}

}  // namespace simba

// knn_refine.cuh — steps 3 and 4 of K4 (knn_tc3.cuh): refine the filter's survivors on their approximate
// values, re-score the few that remain with the reference's EXACT sequential fp32 arithmetic (the same
// mac<FMA> / cosine_tail K1 uses; reference call site rag_search_engine/utils/semantic_search.py:254-261),
// sort by the vec0 emit-order key and emit the packed candidates K1+K2 would emit.
#pragma once
#include "select.cuh"
#include "tc_common.cuh"

namespace rse {

// ---------------------------------------------------------------- refine + exact re-score + finish
// One CTA per query.
//   (a) second-level refinement on the approximate values the filter kept: with s_K = the K'-th
//       largest dot~/|a| among the survivors (= among ALL rows, because every row above the filter
//       threshold survived), only rows with s >= s_K - 2*eps*|q| can be in the exact top-K'
//       (same argument as the filter bound, now with the exact K'-th approximate value);
//   (b) those few rows (K' plus the 2*eps band) are re-computed with the EXACT sequential fp32
//       arithmetic of K1 (mac<FMA>, cosine_tail), lane-per-row straight from global memory;
//   (c) the exact emit-order keys are sorted and the first K' emitted as packed candidates.
// status[q] = 1 (host re-runs the query through K1/K2) when the survivor list or the refined
// list overflowed, or fewer than K' rows survived (a corpus/query the bound does not cover: fewer
// than K' valid rows, zero or non-finite query norm).  `normalized`: the survivor values are cos~
// (knn_tc3, unit-norm operands) instead of dot~/|a| (knn_tc / knn_tc2), so the band is not scaled by |q|.
// smem: kRefineSmemBytes = 80 KB (the pairs, cap * 8 <= 64 KB; later the row staging area, or the keys of the slow
// path) + 8 KB (keys of the fast path).
// 16-byte asynchronous copy global -> shared, L2 only (the staged rows are read once)
__device__ __forceinline__ void cp_async16_cg(uint32_t smem_dst, const void* gmem_src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_dst), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

constexpr int kRefineFastKeys = 512;                                  // the staged path sorts up to this many keys
constexpr int kRefineChunkFloats = 32;                                // one 128-byte line per row per stage
constexpr int kRefineStageBytes = 32 * kRefineChunkFloats * 4;        // 32 rows of a warp: 4 KB
constexpr int kRefineStagingBytes = 20 * kRefineStageBytes;           // 80 KB: the pairs (cap * 8 = 64 KB), later 20 stages
constexpr int kRefineSmemBytes = kRefineStagingBytes + 2 * kRefineFastKeys * 8;   // + keys and rank-sorted keys
static_assert(kTcCandCap * 8 <= kRefineStagingBytes, "the survivor pairs must fit the staging region");

// The exact dot product of the warp's 32 rows (lane l owns row `myrow` of lane l) with the query in s_q, rows STAGED
// through shared memory: each 128-byte line of a row arrives as one coalesced request (8 lanes x 16 B, cp.async, L2
// only) instead of 32 lanes pulling 16 B each from 32 different rows (r02 timeline: lane-per-row loads made this phase
// 42 of the kernel's 64 us on the isotropic corpus — 39 k random rows per launch at 1.4 TB/s; staged: 13 us with two
// stages).  Lane l then walks ITS row in order from shared memory (the reference's sequential sum); float4 j of row r
// sits at slot j ^ (r & 7), so the 8 lanes of a quarter-warp hit 8 different 16-byte bank groups.  STAGES - 1 lines
// are in flight while one is summed.  D = the row width, a multiple of 64.
template <bool FMA, int STAGES, int D>
__device__ __forceinline__ float staged_row_dot(const float* __restrict__ emb, uint32_t myrow, const float* s_q,
                                                unsigned char* wbuf, int lane) {
  constexpr int kChunks = D / kRefineChunkFloats;                          // 384 wide: 12
  const uint32_t wbuf_s = smem_u32(wbuf);
  auto issue = [&](int k) {
    if (k < kChunks) {
#pragma unroll
      for (int it = 0; it < 8; ++it) {
        const int r = 4 * it + (lane >> 3);
        const uint32_t row = __shfl_sync(0xFFFFFFFFu, myrow, r);
        cp_async16_cg(wbuf_s + (k % STAGES) * kRefineStageBytes + r * 128 + (((lane & 7) ^ (r & 7)) << 4),
                      emb + static_cast<int64_t>(row) * D + k * kRefineChunkFloats + (lane & 7) * 4);
      }
    }
    cp_async_commit();                                                     // (an empty group past the last line)
  };
#pragma unroll
  for (int k = 0; k < STAGES - 1; ++k) issue(k);
  float acc = 0.0f;
#pragma unroll 1
  for (int k = 0; k < kChunks; ++k) {
    issue(k + STAGES - 1);
    cp_async_wait<STAGES - 1>();
    __syncwarp();
    const unsigned char* rb = wbuf + (k % STAGES) * kRefineStageBytes + lane * 128;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float4 a = *reinterpret_cast<const float4*>(rb + ((j ^ (lane & 7)) << 4));
      const float4 qv = *reinterpret_cast<const float4*>(s_q + k * kRefineChunkFloats + 4 * j);
      acc = mac<FMA>(acc, a.x, qv.x);
      acc = mac<FMA>(acc, a.y, qv.y);
      acc = mac<FMA>(acc, a.z, qv.z);
      acc = mac<FMA>(acc, a.w, qv.w);
    }
    __syncwarp();                                                          // the stage is free for line k + STAGES
  }
  cp_async_wait<0>();
  return acc;
}

#ifdef RSE_REFINE_TIMING
__device__ unsigned long long g_refine_ns[8 * 4096];
#define RT_STAMP(k) do { if (threadIdx.x == 0 && blockIdx.x < 4096) { unsigned long long t_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_)); g_refine_ns[blockIdx.x * 8 + (k)] = t_; } } while (0)
#define RT_SYNC() __syncthreads()
#else
#define RT_STAMP(k)
#define RT_SYNC()
#endif

// KB = D / 64 (the row width of knn_tc3_kernel<MODE, KB>); the exact re-score is the sequential sum over all D.
template <bool FMA, int KB>
__global__ void __launch_bounds__(kSelThreads, 2)
knn_refine_kernel(const float* __restrict__ emb, const float* __restrict__ amag, const float* __restrict__ q,
                  const double* __restrict__ sb, const uint2* __restrict__ cand_pairs,
                  unsigned int* __restrict__ cand_count, int cap, int kprime, uint64_t pos_base,
                  const int64_t* __restrict__ rowid, const int32_t* __restrict__ movie_idx,
                  long long* __restrict__ cand, int* __restrict__ status, int normalized,
                  const float* __restrict__ thr2, const unsigned int* __restrict__ gate,
                  unsigned long long* __restrict__ counters, float* __restrict__ thr2_out,
                  unsigned int* __restrict__ gate_out, const float* __restrict__ tverify) {
  constexpr int D = KB * 64;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  uint2* pairs = reinterpret_cast<uint2*>(smem_raw);                       // [cap]
  __shared__ float s_q[D];
  __shared__ unsigned int s_hist[256];
  __shared__ unsigned int s_prefix, s_need, s_m, s_digit, s_before;
  __shared__ unsigned int s_warp[8];
  __shared__ uint32_t s_and[kSelThreads / 32], s_or[kSelThreads / 32];
  __shared__ uint32_t s_rows[kTcRefineCap];
  const int qi = blockIdx.x;
  if (thr2 == nullptr) RT_STAMP(0);
  // second-chance pass: only the queries the second threshold kernel re-armed (thr2 finite), and only if any
  if (thr2 != nullptr && (gate[qi >> 8] == 0u || status[qi] == 0 || !(thr2[qi] < __int_as_float(0x7F800000)))) return;
  const unsigned int cnt = cand_count[qi];
  long long* out = cand + static_cast<int64_t>(qi) * kprime * 3;
  // Survivor overflow (count > cap: the sample's K'-th value was a poor bound — a dense neighbourhood on a
  // clustered corpus).  First pass with thr2_out: ARM THE SECOND CHANCE instead of giving up — the `cap` survivors
  // that were kept are K'+ rows with known cos~, so their K'-th largest value s' is a valid lower bound of the
  // K'-th largest cos~ overall and thr2 = s' - 2 eps keeps every row of the exact top-K' by the same argument as
  // the first bound, only much tighter.  The filter and this kernel are enqueued a second time, gated on *gate_out.
  const bool overflow = cnt > static_cast<unsigned int>(cap);
  const bool arm = overflow && thr2_out != nullptr && kprime <= cap;
  if (thr2_out != nullptr && threadIdx.x == 0) thr2_out[qi] = __int_as_float(0x7F800000);   // default: keep nothing
  if (overflow && !arm) {
    if (threadIdx.x == 0) status[qi] = 1;
    for (int i = threadIdx.x; i < kprime * 3; i += blockDim.x) out[i] = -1ll;
    return;
  }
  const int n = overflow ? cap : static_cast<int>(cnt);
  // (knn_tc3 never emits an empty slot or a zero row: its thresholds are positive and those rows read cos~ = 0;
  //  knn_tc / knn_tc2 check |a|^2 in their epilogues)
  // the bits every survivor's key shares (AND == OR) need no histogram pass: cos~ of the survivors sits in a narrow
  // range above the threshold, so the sign/exponent byte is constant and the first radix pass — 2300 shared-memory
  // atomics on ONE bin — is skipped
  uint32_t k_and = 0xFFFFFFFFu, k_or = 0u;
  // (eight loads in flight per thread: a load -> store loop is one HBM round trip per 256 pairs, 6 us of the kernel)
  for (int i0 = threadIdx.x; i0 < n; i0 += 8 * kSelThreads) {
    uint2 pr[8];
#pragma unroll
    for (int u = 0; u < 8; ++u)
      if (i0 + u * kSelThreads < n) pr[u] = cand_pairs[static_cast<int64_t>(qi) * cap + i0 + u * kSelThreads];
#pragma unroll
    for (int u = 0; u < 8; ++u)
      if (i0 + u * kSelThreads < n) {
        pairs[i0 + u * kSelThreads] = pr[u];
        const uint32_t key = ~f32_orderable(pr[u].y);
        k_and &= key; k_or |= key;
      }
  }
  for (int i = threadIdx.x; i < D; i += blockDim.x) s_q[i] = q[static_cast<int64_t>(qi) * D + i];
  k_and = __reduce_and_sync(0xFFFFFFFFu, k_and);
  k_or = __reduce_or_sync(0xFFFFFFFFu, k_or);
  if ((threadIdx.x & 31) == 0) { s_and[threadIdx.x >> 5] = k_and; s_or[threadIdx.x >> 5] = k_or; }
  if (threadIdx.x == 0) { s_prefix = 0u; s_need = static_cast<unsigned int>(kprime < n ? kprime : n); s_m = 0u; }
  __syncthreads();
#pragma unroll
  for (int w = 0; w < kSelThreads / 32; ++w) { k_and &= s_and[w]; k_or |= s_or[w]; }
  const uint32_t same_bits = ~(k_and ^ k_or);                             // 1 = the bit is identical in every key
  RT_STAMP(1);

  // ---- (a) K'-th largest approximate value: MSD radix select (4 x 8 bits) on ~orderable(s)
  //      (descending s == ascending ~orderable)
  uint32_t resolved_mask = 0u;
  const bool select = n > kprime || (tverify != nullptr && n == kprime);   // (the verified path needs s_K even then)
  if (select) {
    // Three passes resolve the top 24 bits of the K'-th key; the low byte is left at its largest value, i.e. s_K is
    // UNDER-estimated by at most 2^-15 of its magnitude (4e-6 against the 5e-3 band): the cut only moves down, the
    // kept set stays a superset of the exact top-K' (the same holds for the second-chance bound s' below).
    for (int pass = 0; pass < 3; ++pass) {
      const int shift = 24 - 8 * pass;
      if (((same_bits >> shift) & 0xFFu) == 0xFFu) {                       // block-uniform: every key has this byte
        if (threadIdx.x == 0) s_prefix = s_prefix | (k_and & (0xFFu << shift));
        resolved_mask |= 0xFFu << shift;
        __syncthreads();
        continue;
      }
      for (int i = threadIdx.x; i < 256; i += blockDim.x) s_hist[i] = 0u;
      __syncthreads();
      const uint32_t prefix = s_prefix;
      for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const uint32_t key = ~f32_orderable(pairs[i].y);
        if ((key & resolved_mask) == prefix) atomicAdd(&s_hist[(key >> shift) & 0xFFu], 1u);
      }
      __syncthreads();
      block_pick_digit(s_hist, s_need, s_warp, &s_digit, &s_before);     // a thread-0 loop over the bins cost 10 % of the kernel
      if (threadIdx.x == 0) {
        s_prefix = prefix | ((s_digit & 0xFFu) << shift);
        s_need = s_need - s_before;
      }
      resolved_mask |= 0xFFu << shift;
      __syncthreads();
    }
  }
  if (select) {
    if (threadIdx.x == 0) s_prefix = s_prefix | 0xFFu;
    __syncthreads();
  }
  RT_STAMP(2);
  // Sample path (tverify): the filter's cut came from the probe's j-th best sample value T, j << K' — tight, but
  // only valid if at least K' rows reach T, i.e. if s_K >= T (then every row of the exact top-K', cos~ >= s_K - 2 eps,
  // passed the filter's cut T - 2 eps - 1e-6; the 1e-7 absorbs the rounding of T = 1 - (1 - cos~)).  s_K here is a
  // lower bound of the true value (low byte unresolved), so the test is conservative.  When it fails, s_K IS still
  // the K'-th largest cos~ overall (everything above the filter's cut is in the list), so the second chance runs
  // with the exact bound s_K - 2 eps.
  const bool reverify = !overflow && select && tverify != nullptr && thr2_out != nullptr &&
                        !(__uint_as_float(f32_from_orderable(~s_prefix)) >= tverify[qi] - 1e-7f);
  if (arm || reverify) {                                                   // (arm: n = cap > K', s_prefix is s' of the kept survivors)
    if (threadIdx.x == 0) {
      const float s_k = __uint_as_float(f32_from_orderable(~s_prefix));
      const float cut2 = s_k - 2.0f * kTcEps - 1e-6f;
      if (cut2 > 1e-6f) {
        thr2_out[qi] = cut2;
        cand_count[qi] = 0u;
        atomicAdd(&gate_out[qi >> 8], 1u);                      // one gate per 256-query block
      }
      status[qi] = 1;
    }
    for (int i = threadIdx.x; i < kprime * 3; i += blockDim.x) out[i] = -1ll;
    return;
  }
  // s_K (exact K'-th largest approximate value), cut = s_K - 2 eps |q|  (slack for f32 rounding)
  float cut = -__int_as_float(0x7F800000);
  if (select) {
    const float s_k = __uint_as_float(f32_from_orderable(~s_prefix));
    const float qn = normalized ? 1.0f : static_cast<float>(sb[qi]);
    cut = s_k - (2.0f * kTcEps + 1e-6f) * qn - 1e-30f;
  }
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const uint2 pr = pairs[i];
    if (__uint_as_float(pr.y) >= cut && pr.y != 0xFF800000u) {
      const unsigned int slot = atomicAdd(&s_m, 1u);
      if (slot < kTcRefineCap) s_rows[slot] = pr.x;
    }
  }
  __syncthreads();
  const unsigned int m = s_m;
  RT_STAMP(3);
  if (m > kTcRefineCap || m < static_cast<unsigned int>(kprime)) {         // refined list overflow (mass ties) / too few rows
    if (threadIdx.x == 0) status[qi] = 1;
    for (int i = threadIdx.x; i < kprime * 3; i += blockDim.x) out[i] = -1ll;
    return;
  }
  if (threadIdx.x == 0) {
    status[qi] = 0;
    if (thr2 != nullptr && counters) atomicAdd(&counters[3], 1ull);      // answered by the second-chance pass
  }

  // ---- (b) exact distances: one lane per row, the reference's sequential fp32 sum
  const double sbq = sb[qi];
  const bool fast = m <= static_cast<unsigned int>(kRefineFastKeys);
  // fast path keys live AFTER the pairs region, which becomes the staging area; the slow path (a refined list above
  // 512 rows: mass ties, second-chance leftovers) keeps the r01 layout — keys over the dead pairs, lane-per-row loads
  unsigned long long* keys = fast ? reinterpret_cast<unsigned long long*>(smem_raw + kRefineStagingBytes)
                                  : reinterpret_cast<unsigned long long*>(smem_raw);
  __syncthreads();                                                         // pairs are dead
  int m2 = 2;
  while (m2 < static_cast<int>(m)) m2 <<= 1;
  if (fast) {
    // 20 stages of 4 KB are shared out among the warps that own rows: 4 per warp up to 160 rows (the usual K' + band),
    // 3 up to 192, 2 beyond
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n_active = m >= static_cast<unsigned int>(kSelThreads) ? kSelThreads / 32 : static_cast<int>((m + 31u) >> 5);
    const int per_warp = (kRefineStagingBytes / kRefineStageBytes) / n_active;
    const int stages = per_warp >= 4 ? 4 : per_warp;                       // 8 warps -> 2
    unsigned char* wbuf = smem_raw + warp * stages * kRefineStageBytes;
    for (int base = warp * 32; base < static_cast<int>(m); base += kSelThreads) {
      const int i = base + lane;
      const uint32_t myrow = s_rows[i < static_cast<int>(m) ? i : static_cast<int>(m) - 1];
      float acc;
      if (stages == 4) acc = staged_row_dot<FMA, 4, D>(emb, myrow, s_q, wbuf, lane);
      else if (stages == 3) acc = staged_row_dot<FMA, 3, D>(emb, myrow, s_q, wbuf, lane);
      else acc = staged_row_dot<FMA, 2, D>(emb, myrow, s_q, wbuf, lane);
      if (i < static_cast<int>(m)) {
        const float d = cosine_tail(acc, sqrt(static_cast<double>(__ldg(amag + myrow))), sbq);
        keys[i] = knn_key(f32_orderable(__float_as_uint(d)), pos_base + static_cast<uint64_t>(myrow));
      }
    }
  } else {
    for (int i = threadIdx.x; i < m2; i += blockDim.x) {
      unsigned long long key = ~0ull;
      if (i < static_cast<int>(m)) {
        const uint32_t row = s_rows[i];
        const float4* rp = reinterpret_cast<const float4*>(emb + static_cast<int64_t>(row) * D);
        float acc = 0.0f;
        // 24 float4 in flight per step; when D / 4 is not a multiple of 24 (every width but 192 and 384) the last
        // step is a partial one, still summed in index order
        constexpr bool kTail = (D / 4) % 24 != 0;
#pragma unroll 1
        for (int c0 = 0; c0 < D / 4; c0 += 24) {
          float4 a[24];
#pragma unroll
          for (int c = 0; c < 24; ++c)
            if (!kTail || c0 + c < D / 4) a[c] = __ldg(rp + c0 + c);
#pragma unroll
          for (int c = 0; c < 24; ++c) {
            if (kTail && c0 + c >= D / 4) break;
            acc = mac<FMA>(acc, a[c].x, s_q[4 * (c0 + c) + 0]);
            acc = mac<FMA>(acc, a[c].y, s_q[4 * (c0 + c) + 1]);
            acc = mac<FMA>(acc, a[c].z, s_q[4 * (c0 + c) + 2]);
            acc = mac<FMA>(acc, a[c].w, s_q[4 * (c0 + c) + 3]);
          }
        }
        const float d = cosine_tail(acc, sqrt(static_cast<double>(__ldg(amag + row))), sbq);
        key = knn_key(f32_orderable(__float_as_uint(d)), pos_base + static_cast<uint64_t>(row));
      }
      keys[i] = key;
    }
  }
  RT_SYNC();
  RT_STAMP(4);
  // ---- (c) sort the keys (all distinct: the position is part of the key), emit the first K'
  const unsigned long long* sorted = keys;
  if (fast) {
    // rank counting: every key is compared with all the others straight from shared memory (broadcast reads), no
    // barrier per stage — K' plus a thin band is a few hundred keys
    unsigned long long* dst = keys + kRefineFastKeys;
    __syncthreads();
    for (int i = threadIdx.x; i < static_cast<int>(m); i += blockDim.x) {
      const unsigned long long me = keys[i];
      int rank = 0;
      for (int j = 0; j < static_cast<int>(m); ++j) rank += keys[j] < me ? 1 : 0;
      dst[rank] = me;
    }
    sorted = dst;
  } else {
    for (int size = 2; size <= m2; size <<= 1) {
      for (int stride = size >> 1; stride > 0; stride >>= 1) {
        __syncthreads();
        for (int t = threadIdx.x; t < (m2 >> 1); t += blockDim.x) {
          const int lo = 2 * t - (t & (stride - 1));
          const int hi = lo + stride;
          const bool up = ((lo & size) == 0);
          const unsigned long long a = keys[lo], b = keys[hi];
          if ((a > b) == up) { keys[lo] = b; keys[hi] = a; }
        }
      }
    }
  }
  __syncthreads();
  RT_STAMP(5);
  for (int i = threadIdx.x; i < kprime; i += blockDim.x) {
    long long* c = out + static_cast<int64_t>(i) * 3;
    if (i < static_cast<int>(m)) {
      const uint64_t key = sorted[i];
      const uint64_t pos = knn_key_pos(key);
      const int64_t local = static_cast<int64_t>(pos - pos_base);
      c[0] = static_cast<long long>(key);
      c[1] = rowid ? rowid[local] : static_cast<long long>(pos);
      c[2] = movie_idx ? movie_idx[local] : -1;
    } else {
      c[0] = -1ll; c[1] = -1ll; c[2] = -1ll;
    }
  }
  RT_SYNC();
  RT_STAMP(6);
#ifdef RSE_REFINE_TIMING
  if (threadIdx.x == 0 && blockIdx.x < 4096) g_refine_ns[blockIdx.x * 8 + 7] = m;
#endif
}

// Host fallback of the tensor-core path (rse.cu knn_local_finish): the flagged queries of a batch are gathered into
// one contiguous group so that ONE exact scan pass serves up to 16 of them (r01 ran one pass per contiguous run
// of flagged queries — scattered flags cost a 1 ms pass each), and their candidates scattered back afterwards.
__global__ void knn_gather_queries_kernel(const float* __restrict__ q, const double* __restrict__ sb,
                                          const int* __restrict__ list, int dim, float* __restrict__ q_out,
                                          double* __restrict__ sb_out) {
  const int src = list[blockIdx.x];
  for (int i = threadIdx.x; i < dim; i += blockDim.x)
    q_out[static_cast<int64_t>(blockIdx.x) * dim + i] = q[static_cast<int64_t>(src) * dim + i];
  if (threadIdx.x == 0) sb_out[blockIdx.x] = sb[src];
}
__global__ void knn_scatter_cand_kernel(const long long* __restrict__ src, const int* __restrict__ list, int per_query,
                                        long long* __restrict__ dst) {
  const int q = list[blockIdx.x];
  for (int i = threadIdx.x; i < per_query; i += blockDim.x)
    dst[static_cast<int64_t>(q) * per_query + i] = src[static_cast<int64_t>(blockIdx.x) * per_query + i];
}

// *out += the number of queries whose status flag is set (rse_knn_flags_dev: the count rides along with the
// results of a row-sharded step instead of a host round trip per step)
__global__ void knn_flag_count_kernel(const int* __restrict__ status, int n, int* __restrict__ out) {
  int c = 0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) c += status[i] != 0 ? 1 : 0;
  c = __reduce_add_sync(0xFFFFFFFFu, c);
  if ((threadIdx.x & 31) == 0 && c) atomicAdd(out, c);
}

}  // namespace rse

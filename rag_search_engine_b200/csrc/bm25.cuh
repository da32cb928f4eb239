// bm25.cuh — K6/K7: BM25 scoring over CSR postings and top-k with the reference's
// tie order.  Replaces the Python/SQLite loop of KeywordSearch.search
// (rag_search_engine/utils/keyword_search.py:196-250).
//
// Bit-exactness: every score is the reference's own IEEE-double expression,
//   denom = tf + k1*(1.0 - b + b*(dl/avgdl))            (:241)
//   add   = idf*(tf*(k1 + 1.0)/denom)                   (:242)
//   score = scores.get(doc, 0.0) + add                  (:244)
// evaluated with explicit round-to-nearest intrinsics (never contracted), and a
// document's adds happen in query-token order because the token passes are
// separated by a CTA barrier and a document appears at most once per posting
// list — so no atomics are needed and the sum order is the reference's.
// idf (:224) is computed on the host with the same libm `log` CPython uses.
//
// B200 mapping (HBM/L2 gather bound, 8 B/posting + 8 B gathered norm):
//   * documents are cut into ranges of kBmRange = 7168; one CTA owns one
//     (query, range) pair with the range's fp64 accumulators (56 KB) and
//     first-token bytes (7 KB) in shared memory — 3 CTAs/SM;
//   * a per-term range-offset table built at load time gives each CTA its slice
//     of every posting list without searching; slices are read as coalesced
//     8-byte (doc, tf) pairs;
//   * k1*(1 - b + b*dl/avgdl) depends only on the document, so it is cached per
//     (k1, b) as normk[M] (same expression, same bits) and gathered from L2;
//   * the CTA emits its range's top-k under the key
//     (score desc, first-token asc, doc asc) = sorted(..., reverse=True) on a
//     dict in insertion order (:250); a per-query k-way merge finishes.
#pragma once
#include "common.cuh"

namespace rse {

constexpr int kBmRange = 7168;   // 7 x 1024: 63 KB of accumulators + first-token bytes → 3 CTAs per SM
constexpr int kBmThreads = 256;
constexpr int kBmMaxTokens = 255;
constexpr int kBmDocsPerThread = kBmRange / kBmThreads;   // 32
constexpr unsigned int kBmCandCap = 192;                    // survivors of the threshold pass kept in smem
constexpr int kBmGeneralMaxK = 256;                         // bm25_score_kernel; bm25_deep_score_kernel above it
constexpr int kBmDeepMaxK = 512;                            // = RSE_MAX_BM25_K

struct Key128 {
  unsigned long long hi;   // ~orderable(score): ascending hi == descending score
  unsigned long long lo;   // (first_token << 32) | doc
};
__device__ __forceinline__ bool key_less(const Key128& a, const Key128& b) {
  return a.hi < b.hi || (a.hi == b.hi && a.lo < b.lo);
}
__device__ __forceinline__ Key128 key_inf() { return Key128{~0ull, ~0ull}; }

// normk[d] = k1 * (1.0 - b + b * (dl[d] / avgdl))   — keyword_search.py:241
__global__ void bm25_norm_kernel(const uint32_t* __restrict__ dl, int64_t n_docs, double k1, double b,
                                 double avgdl, double* __restrict__ normk) {
  int64_t d = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (d >= n_docs) return;
  const double ratio = __ddiv_rn(static_cast<double>(dl[d]), avgdl);
  const double inner = __dadd_rn(__dsub_rn(1.0, b), __dmul_rn(b, ratio));
  normk[d] = __dmul_rn(k1, inner);
}

// Range-offset table: roff[t*(NR+1) + r] = number of postings of term t with
// doc < r*kBmRange.  One thread per (term, boundary) binary-searches the posting
// list (load time only).
__global__ void bm25_range_offsets_by_term_kernel(const int64_t* __restrict__ indptr,
                                                  const uint2* __restrict__ post, int64_t n_terms, int nr,
                                                  uint32_t* __restrict__ roff) {
  const int64_t gid = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const int64_t total = n_terms * (nr + 1);
  if (gid >= total) return;
  const int64_t t = gid / (nr + 1);
  const int r = static_cast<int>(gid - t * (nr + 1));
  const int64_t lo0 = indptr[t], hi0 = indptr[t + 1];
  const uint32_t bound = static_cast<uint32_t>(static_cast<int64_t>(r) * kBmRange > 0xFFFFFFFFll
                                                   ? 0xFFFFFFFFu
                                                   : static_cast<uint32_t>(r) * kBmRange);
  int64_t lo = lo0, hi = hi0;   // first posting with doc >= bound
  if (r == nr) {
    lo = hi0;
  } else {
    while (lo < hi) {
      const int64_t mid = (lo + hi) >> 1;
      if (post[mid].x < bound) lo = mid + 1; else hi = mid;
    }
  }
  roff[gid] = static_cast<uint32_t>(lo - lo0);
}

// Block-wide arg-min of per-thread Key128 values.  Returns the winning key to all
// threads and the winning thread id through *winner.  s_k / s_w are smem scratch
// of 8 entries (one per warp).
__device__ __forceinline__ Key128 block_argmin(Key128 mine, Key128* s_k, int* s_w, int* winner) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  Key128 best = mine;
  int who = threadIdx.x;
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    Key128 o;
    o.hi = __shfl_xor_sync(0xFFFFFFFFu, best.hi, off);
    o.lo = __shfl_xor_sync(0xFFFFFFFFu, best.lo, off);
    int ow = __shfl_xor_sync(0xFFFFFFFFu, who, off);
    if (key_less(o, best)) { best = o; who = ow; }
  }
  __syncthreads();   // protect scratch from the previous round's readers
  if (lane == 0) { s_k[warp] = best; s_w[warp] = who; }
  __syncthreads();
  const int nw = blockDim.x >> 5;
  Key128 r = s_k[0];
  int rw = s_w[0];
  for (int w = 1; w < nw; ++w) {
    Key128 o = s_k[w];
    if (key_less(o, r)) { r = o; rw = s_w[w]; }
  }
  *winner = rw;
  return r;
}

// K6: one CTA per (range, query).
//   cand_hi/lo: [nq][nr][k]; cand_cnt: [nq][nr]
// kDeep (k > kBmGeneralMaxK): the range's k best are found by a radix selection instead of k barrier rounds.
template <bool kDeep>
__device__ __forceinline__ void
bm25_score_one(const int64_t* __restrict__ indptr, const uint2* __restrict__ post,
               const uint32_t* __restrict__ roff, const double* __restrict__ normk, int nr,
               int64_t n_docs, const int32_t* __restrict__ tok_indptr, const int32_t* __restrict__ term_rows,
               const double* __restrict__ tok_idf, int q, int k, double k1p1,
               unsigned long long* __restrict__ cand_hi, unsigned long long* __restrict__ cand_lo,
               int* __restrict__ cand_cnt) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double* acc = reinterpret_cast<double*>(smem_raw);                       // [kBmRange]
  unsigned char* first = reinterpret_cast<unsigned char*>(acc + kBmRange); // [kBmRange]
  // token tables (scoring phase) and selection scratch (afterwards) share one buffer
  constexpr int kTokBytes = (kBmMaxTokens + 1) * (8 + 8 + 4);
  constexpr int kSelBytes = kDeep ? 256 * 4 + kBmDeepMaxK * static_cast<int>(sizeof(Key128))
                                  : (256 + static_cast<int>(kBmCandCap)) * static_cast<int>(sizeof(Key128));
  __shared__ __align__(16) unsigned char s_cand_mem[kTokBytes > kSelBytes ? kTokBytes : kSelBytes];
  long long* s_lo = reinterpret_cast<long long*>(s_cand_mem);
  double* s_idf = reinterpret_cast<double*>(s_cand_mem + (kBmMaxTokens + 1) * 8);
  unsigned int* s_n = reinterpret_cast<unsigned int*>(s_cand_mem + (kBmMaxTokens + 1) * 16);
  __shared__ Key128 s_k[kBmThreads / 32];
  __shared__ int s_w[kBmThreads / 32];
  __shared__ unsigned int s_total;
  __shared__ unsigned int s_ncand;
  __shared__ Key128 s_tau;

  const int r = blockIdx.x;
  const int t0 = tok_indptr[q], t1 = tok_indptr[q + 1];
  const int ntok = t1 - t0;
  const int64_t cbase = (static_cast<int64_t>(q) * nr + r);

  __syncthreads();                                        // a previous query of this CTA may still be reading the scratch
  if (threadIdx.x == 0) s_total = 0u;
  __syncthreads();
  for (int t = threadIdx.x; t < ntok; t += blockDim.x) {
    const int term = term_rows[t0 + t];
    long long lo = 0;
    unsigned int n = 0;
    if (term >= 0) {
      const uint32_t* ro = roff + static_cast<int64_t>(term) * (nr + 1) + r;
      const uint32_t a = ro[0], bnd = ro[1];
      lo = indptr[term] + a;
      n = bnd - a;
    }
    s_lo[t] = lo; s_n[t] = n; s_idf[t] = tok_idf[t0 + t];
    if (n) atomicAdd(&s_total, n);
  }
  __syncthreads();
  if (s_total == 0u) {
    if (threadIdx.x == 0) cand_cnt[cbase] = 0;
    return;
  }

  {
    uint4* a4 = reinterpret_cast<uint4*>(acc);                 // 64 KB of +0.0
    for (int i = threadIdx.x; i < kBmRange / 2; i += blockDim.x) a4[i] = make_uint4(0u, 0u, 0u, 0u);
    uint4* f4 = reinterpret_cast<uint4*>(first);               // 8 KB of 0xFF
    for (int i = threadIdx.x; i < kBmRange / 16; i += blockDim.x) f4[i] = make_uint4(~0u, ~0u, ~0u, ~0u);
  }
  __syncthreads();

  const uint32_t doc_base = static_cast<uint32_t>(r) * kBmRange;
  for (int t = 0; t < ntok; ++t) {
    const unsigned int n = s_n[t];
    if (n == 0u) continue;            // uniform across the CTA
    const uint2* p = post + s_lo[t];
    const double idf = s_idf[t];
    // 4 postings per thread per trip: all posting loads first, then all norm gathers, then the
    // arithmetic — two dependent global loads per posting otherwise leave the warp on the long
    // scoreboard (r01 ncu).  A document occurs once per list, so the 4 smem updates never alias.
    for (unsigned int i0 = threadIdx.x; i0 < n; i0 += 4 * kBmThreads) {
      uint2 e[4];
      double nk[4];
      bool ok[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const unsigned int i = i0 + j * kBmThreads;
        ok[j] = i < n;
        e[j] = ok[j] ? __ldg(p + i) : make_uint2(doc_base, 1u);
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) nk[j] = ok[j] ? __ldg(normk + e[j].x) : 1.0;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        if (!ok[j]) continue;
        const double tfd = static_cast<double>(e[j].y);
        const double denom = __dadd_rn(tfd, nk[j]);
        const double add = __dmul_rn(idf, __ddiv_rn(__dmul_rn(tfd, k1p1), denom));
        const uint32_t l = e[j].x - doc_base;
        if (first[l] == 0xFF) first[l] = static_cast<unsigned char>(t);
        acc[l] = __dadd_rn(acc[l], add);          // first touch is 0.0 + add
      }
    }
    __syncthreads();
  }

  __syncthreads();   // the token tables are dead from here on: their storage becomes selection scratch

  // ---- K7 (range part): the range's top-k under (score desc, first token asc, doc asc).
  auto make_key = [&](int l) -> Key128 {
    Key128 kk;
    kk.hi = ~f64_orderable(static_cast<uint64_t>(__double_as_longlong(acc[l])));
    kk.lo = (static_cast<unsigned long long>(first[l]) << 32) | (doc_base + static_cast<uint32_t>(l));
    return kk;
  };
  if constexpr (kDeep) {
    // Radix selection over the key (score desc, first token asc, doc asc), one byte per pass: the 8 bytes of the
    // orderable score, the first token, then the document's offset in the range (13 bits: two passes).  Thread t
    // owns documents t + 256 i: bit i of `live` (still tied with the threshold prefix) and of `taken` (strictly
    // better than it).  The keys are distinct, so exactly min(k, touched) documents end up taken; they are
    // collected and ordered by rank counting.
    unsigned int* s_hist = reinterpret_cast<unsigned int*>(s_cand_mem);              // [256]
    Key128* s_sel = reinterpret_cast<Key128*>(s_cand_mem + 256 * 4);                // [kBmDeepMaxK]
    __shared__ unsigned int s_warp[kBmThreads / 32], s_digit, s_before, s_touched;
    auto digit = [&](int pass, int l) -> unsigned int {
      if (pass < 8) {
        const uint64_t hi = ~f64_orderable(static_cast<uint64_t>(__double_as_longlong(acc[l])));
        return static_cast<unsigned int>(hi >> (56 - 8 * pass)) & 0xFFu;
      }
      if (pass == 8) return first[l];
      return pass == 9 ? static_cast<unsigned int>(l) >> 8 : static_cast<unsigned int>(l) & 0xFFu;
    };
    uint32_t live = 0u, taken = 0u;
#pragma unroll 4
    for (int i = 0; i < kBmDocsPerThread; ++i)
      if (first[threadIdx.x + i * kBmThreads] != 0xFF) live |= 1u << i;
    if (threadIdx.x == 0) s_touched = 0u;
    __syncthreads();
    if (live) atomicAdd(&s_touched, static_cast<unsigned int>(__popc(live)));
    __syncthreads();
    unsigned int need = static_cast<unsigned int>(k);
    if (s_touched <= need) {
      taken = live;
    } else {
      for (int pass = 0; pass < 11; ++pass) {
        s_hist[threadIdx.x] = 0u;
        __syncthreads();
        for (uint32_t m = live; m; m &= m - 1u)
          atomicAdd(&s_hist[digit(pass, threadIdx.x + (__ffs(m) - 1) * kBmThreads)], 1u);
        __syncthreads();
        block_pick_digit(s_hist, need, s_warp, &s_digit, &s_before);
        const unsigned int d = s_digit, in_bin = s_hist[d];
        need -= s_before;
        for (uint32_t m = live; m; m &= m - 1u) {
          const int i = __ffs(m) - 1;
          const unsigned int g = digit(pass, threadIdx.x + i * kBmThreads);
          if (g < d) taken |= 1u << i;
          if (g != d) live &= ~(1u << i);
        }
        if (in_bin == need) { taken |= live; break; }                 // the whole bin is in: uniform
        __syncthreads();                                              // s_hist / s_digit are read before the reset
      }
    }
    __syncthreads();
    if (threadIdx.x == 0) s_touched = 0u;
    __syncthreads();
    for (uint32_t m = taken; m; m &= m - 1u) {
      const int l = threadIdx.x + (__ffs(m) - 1) * kBmThreads;
      s_sel[atomicAdd(&s_touched, 1u)] = make_key(l);
    }
    __syncthreads();
    const int nc = static_cast<int>(s_touched);
    for (int i = threadIdx.x; i < nc; i += kBmThreads) {
      const Key128 me = s_sel[i];
      int rank = 0;
      for (int j = 0; j < nc; ++j) rank += key_less(s_sel[j], me) ? 1 : 0;
      cand_hi[cbase * k + rank] = me.hi;
      cand_lo[cbase * k + rank] = me.lo;
    }
    if (threadIdx.x == 0) cand_cnt[cbase] = nc;
    return;
  }
  if (k <= 32) {
    // Fast path.  (1) every thread finds the best of its 32 documents; (2) each warp sorts its 32
    // thread-bests with shuffles; (3) warp 0 merges the 8 sorted lists to the k-th best overall — a
    // valid threshold because the thread-bests are distinct documents; (4) one collect pass keeps the
    // documents at least that good (≥ k of them, usually barely more); (5) rank counting orders them.
    Key128 mine = key_inf();
#pragma unroll 4
    for (int i = 0; i < kBmDocsPerThread; ++i) {
      const int l = threadIdx.x + i * kBmThreads;
      if (first[l] == 0xFF) continue;
      const Key128 kk = make_key(l);
      if (key_less(kk, mine)) mine = kk;
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // warp bitonic sort, ascending (best first)
#pragma unroll
    for (int size = 2; size <= 32; size <<= 1) {
#pragma unroll
      for (int stride = size >> 1; stride > 0; stride >>= 1) {
        Key128 o;
        o.hi = __shfl_xor_sync(0xFFFFFFFFu, mine.hi, stride);
        o.lo = __shfl_xor_sync(0xFFFFFFFFu, mine.lo, stride);
        const bool up = ((lane & size) == 0);
        const bool lower = ((lane & stride) == 0);
        const bool take_min = (up == lower);
        const bool o_less = key_less(o, mine);
        if (take_min ? o_less : !o_less) mine = o;
      }
    }
    Key128* s_wb = reinterpret_cast<Key128*>(s_cand_mem);        // [8][32]
    s_wb[warp * 32 + lane] = mine;
    __syncthreads();
    if (warp == 0) {
      // 8-way merge: lane w < 8 owns list w
      int head = 0;
      Key128 cur = (lane < kBmThreads / 32) ? s_wb[lane * 32] : key_inf();
      Key128 tau = key_inf();
      for (int round = 0; round < k; ++round) {
        Key128 best = cur;
        int who = lane;
#pragma unroll
        for (int off = 4; off > 0; off >>= 1) {
          Key128 o;
          o.hi = __shfl_xor_sync(0xFFFFFFFFu, best.hi, off);
          o.lo = __shfl_xor_sync(0xFFFFFFFFu, best.lo, off);
          const int ow = __shfl_xor_sync(0xFFFFFFFFu, who, off);
          if (key_less(o, best)) { best = o; who = ow; }
        }
        best.hi = __shfl_sync(0xFFFFFFFFu, best.hi, 0);
        best.lo = __shfl_sync(0xFFFFFFFFu, best.lo, 0);
        who = __shfl_sync(0xFFFFFFFFu, who, 0);
        tau = best;
        if (best.hi == ~0ull && best.lo == ~0ull) break;         // fewer than k touched documents
        if (lane == who) {
          ++head;
          cur = (head < 32) ? s_wb[lane * 32 + head] : key_inf();
        }
      }
      if (lane == 0) { s_tau = tau; s_ncand = 0u; }
    }
    __syncthreads();
    const Key128 tau = s_tau;
    Key128* s_cand = reinterpret_cast<Key128*>(s_cand_mem) + 256;  // [kBmCandCap], after the warp lists
#pragma unroll 4
    for (int i = 0; i < kBmDocsPerThread; ++i) {
      const int l = threadIdx.x + i * kBmThreads;
      if (first[l] == 0xFF) continue;
      const Key128 kk = make_key(l);
      if (!key_less(tau, kk)) {                                  // kk <= tau
        const unsigned int slot = atomicAdd(&s_ncand, 1u);
        if (slot < kBmCandCap) s_cand[slot] = kk;
      }
    }
    __syncthreads();
    const unsigned int nc = s_ncand;
    if (nc <= kBmCandCap) {
      const int emitted = static_cast<int>(nc) < k ? static_cast<int>(nc) : k;
      if (threadIdx.x < nc) {
        const Key128 me = s_cand[threadIdx.x];
        int rank = 0;
        for (unsigned int j = 0; j < nc; ++j) rank += key_less(s_cand[j], me) ? 1 : 0;
        if (rank < k) {
          cand_hi[cbase * k + rank] = me.hi;
          cand_lo[cbase * k + rank] = me.lo;
        }
      }
      if (threadIdx.x == 0) cand_cnt[cbase] = emitted;
      return;
    }
    // survivor overflow (mass ties at the threshold): fall through to the general path
    __syncthreads();
  }

  // General path (k > 32, or overflow): k rounds of block arg-min over per-thread cached bests.
  auto scan_best = [&](const Key128& after, bool have_after) -> Key128 {
    Key128 best = key_inf();
#pragma unroll 4
    for (int i = 0; i < kBmDocsPerThread; ++i) {
      const int l = threadIdx.x + i * kBmThreads;
      if (first[l] == 0xFF) continue;
      const Key128 kk = make_key(l);
      if (have_after && !key_less(after, kk)) continue;   // already emitted (kk <= after)
      if (key_less(kk, best)) best = kk;
    }
    return best;
  };
  Key128 mine = scan_best(key_inf(), false);
  int emitted = 0;
  for (int round = 0; round < k; ++round) {
    int winner;
    const Key128 w = block_argmin(mine, s_k, s_w, &winner);
    if (w.hi == ~0ull && w.lo == ~0ull) break;            // range exhausted
    if (threadIdx.x == winner) {
      cand_hi[cbase * k + round] = w.hi;
      cand_lo[cbase * k + round] = w.lo;
      mine = scan_best(w, true);
    }
    ++emitted;
  }
  if (threadIdx.x == 0) cand_cnt[cbase] = emitted;
}

// flagged == nullptr: grid (nr, nq), CTA (r, j) scores query q0 + j.
// flagged != nullptr (second launch after bm25_stream_kernel): grid (nr, few); the CTAs walk the compacted list of
// the queries the streaming path flagged (flagged[0] = count, flagged[1..] = query indices) — usually empty, so
// the launch costs a few microseconds instead of one early-exit CTA per (range, query).
__global__ void __launch_bounds__(kBmThreads)
bm25_score_kernel(const int64_t* __restrict__ indptr, const uint2* __restrict__ post,
                  const uint32_t* __restrict__ roff, const double* __restrict__ normk, int nr,
                  int64_t n_docs, const int32_t* __restrict__ tok_indptr, const int32_t* __restrict__ term_rows,
                  const double* __restrict__ tok_idf, int q0, int k, double k1p1,
                  unsigned long long* __restrict__ cand_hi, unsigned long long* __restrict__ cand_lo,
                  int* __restrict__ cand_cnt, const int* __restrict__ flagged) {
  if (!flagged) {
    bm25_score_one<false>(indptr, post, roff, normk, nr, n_docs, tok_indptr, term_rows, tok_idf, q0 + blockIdx.y, k, k1p1, cand_hi,
                   cand_lo, cand_cnt);
    return;
  }
  const int n = flagged[0];
  for (int j = blockIdx.y; j < n; j += gridDim.y)
    bm25_score_one<false>(indptr, post, roff, normk, nr, n_docs, tok_indptr, term_rows, tok_idf, flagged[1 + j], k, k1p1, cand_hi,
                   cand_lo, cand_cnt);
}

// k > kBmGeneralMaxK: grid (nr, nq), CTA (r, j) scores query q0 + j; the per-range lists go through bm25_merge_kernel.
__global__ void __launch_bounds__(kBmThreads)
bm25_deep_score_kernel(const int64_t* __restrict__ indptr, const uint2* __restrict__ post,
                       const uint32_t* __restrict__ roff, const double* __restrict__ normk, int nr,
                       int64_t n_docs, const int32_t* __restrict__ tok_indptr, const int32_t* __restrict__ term_rows,
                       const double* __restrict__ tok_idf, int q0, int k, double k1p1,
                       unsigned long long* __restrict__ cand_hi, unsigned long long* __restrict__ cand_lo,
                       int* __restrict__ cand_cnt) {
  bm25_score_one<true>(indptr, post, roff, normk, nr, n_docs, tok_indptr, term_rows, tok_idf, q0 + blockIdx.y, k, k1p1,
                       cand_hi, cand_lo, cand_cnt);
}

// flagged[0] = number of queries in [q0, q0 + nc) with status != 0, flagged[1..] = those queries (ascending)
// counters (optional): [0] += the number of flagged queries — the BM25 counterpart of tc_fallback_queries
__global__ void bm25_flag_compact_kernel(const int* __restrict__ status, int q0, int nc, int* __restrict__ flagged,
                                         unsigned long long* __restrict__ counters) {
  __shared__ int s_n;
  if (threadIdx.x == 0) s_n = 0;
  __syncthreads();
  for (int base = 0; base < nc; base += blockDim.x) {      // one CTA; order inside the list does not matter
    const int j = base + threadIdx.x;
    if (j < nc && status[q0 + j] != 0) flagged[1 + atomicAdd(&s_n, 1)] = q0 + j;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    flagged[0] = s_n;
    if (counters && s_n) atomicAdd(&counters[0], static_cast<unsigned long long>(s_n));
  }
}

// ---------------------------------------------------------------------------------------------
// K6' + K7': streaming BM25 (the default path for k <= 32 and <= 16 query tokens).
//
// r01 ncu of bm25_score_kernel: 21.5 k CTAs (one per 7168-document range and query), each paying a
// chain of dependent global loads for its token slices, a gathered norm per posting, a 64 KB clear and
// a full top-k (thread bests, 8 warp sorts, a serial 8-way merge, a collect pass) for ~3.6 k postings
// of real work: 0.9 ms per 256-query step, 36 k cycles per CTA.  Here
//   * the per-posting weight w = tf*(k1+1)/(tf + k1*(1-b+b*dl/avgdl)) — keyword_search.py:241-242 up to
//     the multiplication by idf, in the reference's association — is precomputed per (k1, b) next to
//     the document index (16 B postings), so a posting costs one coalesced 16 B load, DMUL, DADD and
//     a shared-memory update: no gather, no division at query time;
//   * one CTA owns a QUERY and a GROUP of consecutive ranges; the range offsets of its tokens are read
//     once into shared memory, the accumulator array is reused range after range (cleared by the scan
//     that reads it);
//   * top-k is a running threshold: the first non-empty range establishes theta = k-th largest of the
//     256 per-thread maxima (distinct documents, so a valid lower bound of the k-th best score); every
//     later range only collects documents with score >= theta (a handful), and theta is tightened
//     whenever the candidate list is compacted.  Ties are resolved at the very end, for the <= k + ties
//     finalists only: the first query token whose posting list holds the document is found by binary
//     search instead of being tracked per posting.
// The emitted per-group lists have the format of bm25_score_kernel's per-range lists and go through the
// same bm25_merge_kernel.  A query the kernel cannot finish (more than 16 tokens, candidate overflow
// from mass ties) is flagged in status[] and re-scored by bm25_score_kernel — no host round trip.
struct __align__(16) Post16 {
  uint32_t doc;
  uint32_t tf;
  double w;        // tf*(k1+1) / (tf + normk[doc])
};

constexpr int kBsWideThreads = 896;               // bm25_fx_kernel underneath the filter (see there)
constexpr int kBsThreads = 512;                   // 16 warps x 3 CTAs per SM: the kernel is issue-latency-bound, TLP is what it needs
constexpr int kBsPerTrip = 2;                     // postings per thread per trip
constexpr int kBsDocsPerThread = kBmRange / kBsThreads;   // 14
constexpr int kBsMaxTok = 16;
constexpr int kBsMaxRpg = 128;                    // ranges per group (bounds the offset table in shared memory)
constexpr unsigned int kBsCandCap = 256;
constexpr unsigned int kBsCompactAt = 128;
constexpr int kBsMaxGroups = 32;                  // groups per query bm25_fx_finish_kernel merges
constexpr unsigned int kBsRangeCap = 256;         // documents that may cross theta inside one range
constexpr int kBsFinalCap = 64;                   // finalists (k + ties) ranked exactly

// out4 (optional): the 4-byte stream bm25_fx_kernel reads, (doc % kBmRange) | round(w * wq4_scale) << 13 — see the
// K6'' header
__global__ void bm25_weight_kernel(const uint2* __restrict__ post, const double* __restrict__ normk, int64_t n,
                                   double k1p1, Post16* __restrict__ out, uint32_t* __restrict__ out4, double wq4_scale) {
  const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint2 e = post[i];
  const double tfd = static_cast<double>(e.y);
  Post16 o;
  o.doc = e.x; o.tf = e.y;
  o.w = __ddiv_rn(__dmul_rn(tfd, k1p1), __dadd_rn(tfd, normk[e.x]));
  out[i] = o;
  if (out4) {
    unsigned int wq = __double2uint_rn(__dmul_rn(o.w, wq4_scale));
    if (wq > 0x7FFFFu) wq = 0x7FFFFu;                      // (k1+1) * wq4_scale <= 2^19: only a weight at the very top clamps
    if (wq == 0u && o.w > 0.0) wq = 1u;                    // a weight word of 0 adds nothing: a posting that counts must not round to it
    out4[i] = (e.x % static_cast<uint32_t>(kBmRange)) | (wq << 13);
  }
}

constexpr int bs_smem_bytes() {
  return kBmRange * 8 + kBsMaxTok * (kBsMaxRpg + 1) * 4 + 2 * static_cast<int>(kBsCandCap) * 16;
}

__global__ void __launch_bounds__(kBsThreads, 3)
bm25_stream_kernel(const int64_t* __restrict__ indptr, const Post16* __restrict__ post, const uint32_t* __restrict__ roff,
                   int nr, const int32_t* __restrict__ tok_indptr, const int32_t* __restrict__ term_rows,
                   const double* __restrict__ tok_idf, int q0, int k, int rpg, int ng,
                   unsigned long long* __restrict__ cand_hi, unsigned long long* __restrict__ cand_lo,
                   int* __restrict__ cand_cnt, int* __restrict__ status) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double* acc = reinterpret_cast<double*>(smem_raw);                                   // [kBmRange]
  uint32_t* s_off = reinterpret_cast<uint32_t*>(acc + kBmRange);                       // [kBsMaxTok][rpg + 1]
  double2* s_cand0 = reinterpret_cast<double2*>(s_off + kBsMaxTok * (kBsMaxRpg + 1));  // {score, doc as double bits}
  double2* s_cand1 = s_cand0 + kBsCandCap;
  __shared__ long long s_base[kBsMaxTok];
  __shared__ double s_idf[kBsMaxTok];
  __shared__ int s_term[kBsMaxTok];
  __shared__ unsigned int s_ncand, s_nkept, s_nrc;
  __shared__ unsigned short s_rc[kBsRangeCap];
  __shared__ unsigned long long s_min_bits;
  __shared__ unsigned long long s_tw[kBsThreads / 32];

  const int g = blockIdx.x;
  const int q = q0 + blockIdx.y;
  const int t0 = tok_indptr[q], ntok = tok_indptr[q + 1] - t0;
  const int64_t cbase = static_cast<int64_t>(q) * ng + g;
  if (ntok > kBsMaxTok) {                                 // uniform: the whole query goes to the general kernel
    if (threadIdx.x == 0) { cand_cnt[cbase] = 0; if (g == 0) status[q] = 1; }
    return;
  }
  const int r0 = g * rpg, r1 = min(nr, r0 + rpg);
  const int nrg = r1 - r0;
  if (threadIdx.x < ntok) {
    const int term = term_rows[t0 + threadIdx.x];
    s_term[threadIdx.x] = term;
    s_base[threadIdx.x] = term >= 0 ? indptr[term] : 0;
    s_idf[threadIdx.x] = tok_idf[t0 + threadIdx.x];
  }
  if (threadIdx.x == 0) { s_ncand = 0u; s_nrc = 0u; }
  __syncthreads();
  for (int i = threadIdx.x; i < ntok * (nrg + 1); i += blockDim.x) {
    const int t = i / (nrg + 1), j = i - t * (nrg + 1);
    const int term = s_term[t];
    s_off[t * (kBsMaxRpg + 1) + j] = term >= 0 ? roff[static_cast<int64_t>(term) * (nr + 1) + r0 + j] : 0u;
  }
  {
    uint4* a4 = reinterpret_cast<uint4*>(acc);
    for (int i = threadIdx.x; i < kBmRange / 2; i += blockDim.x) a4[i] = make_uint4(0u, 0u, 0u, 0u);
  }
  __syncthreads();

  double2* cand = s_cand0;
  double2* cand_alt = s_cand1;
  double theta = 0.0;                                     // 0 = not established: every touched document qualifies
  bool established = false;

  // keep the documents that fewer than k others beat on score (ties at the boundary stay), tighten theta
  auto compact = [&]() {
    const unsigned int n = s_ncand;                       // uniform (read after a barrier)
    if (n < static_cast<unsigned int>(k)) return;
    if (threadIdx.x == 0) { s_nkept = 0u; s_min_bits = ~0ull; }
    __syncthreads();
    if (threadIdx.x < n) {
      const double2 me = cand[threadIdx.x];
      unsigned int greater = 0u;
      for (unsigned int j = 0; j < n; ++j) greater += cand[j].x > me.x ? 1u : 0u;
      if (greater < static_cast<unsigned int>(k)) {
        cand_alt[atomicAdd(&s_nkept, 1u)] = me;
        atomicMin(&s_min_bits, static_cast<unsigned long long>(__double_as_longlong(me.x)));   // scores are > 0: bit order = value order
      }
    }
    __syncthreads();
    double2* tmp = cand; cand = cand_alt; cand_alt = tmp;
    theta = __longlong_as_double(static_cast<long long>(s_min_bits));
    established = true;
    __syncthreads();
    if (threadIdx.x == 0) s_ncand = s_nkept;
    __syncthreads();
  };

  for (int r = r0; r < r1; ++r) {
    const int j = r - r0;
    unsigned int total = 0u;
    for (int t = 0; t < ntok; ++t) total += s_off[t * (kBsMaxRpg + 1) + j + 1] - s_off[t * (kBsMaxRpg + 1) + j];
    if (total == 0u) continue;                            // uniform
    const uint32_t doc_base = static_cast<uint32_t>(r) * kBmRange;
    // once theta is established the candidates of a range are the documents whose sum CROSSES theta while the
    // postings are applied — no scan over the 7168 accumulators (r01 ncu: the scan was 26 % of the instructions)
    const bool crossing = established;
    const double cross = crossing ? theta : __longlong_as_double(0x7FF0000000000000ll);
    for (int t = 0; t < ntok; ++t) {
      const uint32_t a = s_off[t * (kBsMaxRpg + 1) + j];
      const unsigned int n = s_off[t * (kBsMaxRpg + 1) + j + 1] - a;
      if (n == 0u) continue;                              // uniform
      const Post16* p = post + s_base[t] + a;
      const double idf = s_idf[t];
      for (unsigned int i0 = threadIdx.x; i0 < n; i0 += kBsPerTrip * kBsThreads) {
        uint4 e[kBsPerTrip];
        bool ok[kBsPerTrip];
#pragma unroll
        for (int u = 0; u < kBsPerTrip; ++u) {
          const unsigned int i = i0 + u * kBsThreads;
          ok[u] = i < n;
          e[u] = ok[u] ? __ldg(reinterpret_cast<const uint4*>(p + i)) : make_uint4(doc_base, 0u, 0u, 0u);
        }
#pragma unroll
        for (int u = 0; u < kBsPerTrip; ++u) {
          if (!ok[u]) continue;
          const double w = __hiloint2double(static_cast<int>(e[u].w), static_cast<int>(e[u].z));
          const uint32_t l = e[u].x - doc_base;
          const double old = acc[l];
          const double nw = __dadd_rn(old, __dmul_rn(idf, w));   // first touch is 0.0 + add (keyword_search.py:244)
          acc[l] = nw;
          if (nw >= cross && old < cross) {               // the document just reached theta (scores only grow): note it once
            const unsigned int slot = atomicAdd(&s_nrc, 1u);
            if (slot < kBsRangeCap) s_rc[slot] = static_cast<unsigned short>(l);
          }
        }
      }
      __syncthreads();
    }
    if (crossing) {
      // (the barrier after the last token pass has been taken) the noted documents now hold their final sums
      const unsigned int nrc = s_nrc;
      if (nrc > kBsRangeCap) {                            // uniform
        if (threadIdx.x == 0) { status[q] = 1; cand_cnt[cbase] = 0; }
        return;
      }
      if (threadIdx.x < nrc) {
        const uint32_t l = s_rc[threadIdx.x];
        const unsigned int slot = atomicAdd(&s_ncand, 1u);
        if (slot < kBsCandCap) cand[slot] = make_double2(acc[l], __longlong_as_double(static_cast<long long>(doc_base + l)));
      }
      __syncthreads();
      uint4* a4 = reinterpret_cast<uint4*>(acc);
#pragma unroll
      for (int i = 0; i < kBmRange / 2 / kBsThreads; ++i) a4[threadIdx.x + i * kBsThreads] = make_uint4(0u, 0u, 0u, 0u);
      if (threadIdx.x == 0) s_nrc = 0u;
    } else {
      // theta = the k-th largest of the warps' best thread maxima (m = ceil(k/16) per warp): maxima of distinct
      // threads are distinct documents, so k of them at or above theta make it a lower bound of the k-th best score
      double mx = 0.0;
#pragma unroll 2
      for (int i = 0; i < kBsDocsPerThread; ++i) mx = fmax(mx, acc[threadIdx.x + i * kBsThreads]);
      unsigned long long mine = static_cast<unsigned long long>(__double_as_longlong(mx));
      const int lane = threadIdx.x & 31;
      const int m = (k + kBsThreads / 32 - 1) / (kBsThreads / 32);        // 1 or 2
      unsigned long long* s_top = reinterpret_cast<unsigned long long*>(cand_alt);
      for (int round = 0; round < m; ++round) {
        unsigned long long wm = mine;
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) wm = max(wm, __shfl_xor_sync(0xFFFFFFFFu, wm, off));
        const unsigned int holders = __ballot_sync(0xFFFFFFFFu, mine == wm);
        if (lane == __ffs(holders) - 1) { s_top[(threadIdx.x >> 5) * m + round] = wm; mine = 0ull; }
      }
      if (threadIdx.x == 0) s_tw[0] = 0ull;
      __syncthreads();
      const int nv = (kBsThreads / 32) * m;                                // 16 or 32
      if (static_cast<int>(threadIdx.x) < nv) {
        const unsigned long long me = s_top[threadIdx.x];
        int r2 = 0;
        for (int jj = 0; jj < nv; ++jj) {
          const unsigned long long o = s_top[jj];
          r2 += (o > me || (o == me && jj < static_cast<int>(threadIdx.x))) ? 1 : 0;
        }
        if (r2 == k - 1) s_tw[0] = me;                     // 0 when fewer than k threads saw a document
      }
      __syncthreads();
      const unsigned long long tb = s_tw[0];
      if (tb != 0ull) { theta = __longlong_as_double(static_cast<long long>(tb)); established = true; }
      // scan + clear: collect the documents at or above theta
#pragma unroll 2
      for (int i = 0; i < kBsDocsPerThread; ++i) {
        const int l = threadIdx.x + i * kBsThreads;
        const double sc = acc[l];
        if (sc != 0.0) {
          acc[l] = 0.0;
          if (sc >= theta) {
            const unsigned int slot = atomicAdd(&s_ncand, 1u);
            if (slot < kBsCandCap) cand[slot] = make_double2(sc, __longlong_as_double(static_cast<long long>(doc_base + l)));
          }
        }
      }
    }
    __syncthreads();
    if (s_ncand > kBsCandCap) {                           // uniform: mass ties → the general kernel re-scores the query
      if (threadIdx.x == 0) { status[q] = 1; cand_cnt[cbase] = 0; }
      return;
    }
    if (s_ncand >= kBsCompactAt) compact();
  }
  compact();
  const unsigned int n = s_ncand;
  if (n > static_cast<unsigned int>(kBsFinalCap)) {
    if (threadIdx.x == 0) { status[q] = 1; cand_cnt[cbase] = 0; }
    return;
  }
  // finalists: first query token whose posting list holds the document, then the exact key order
  Key128* s_keys = reinterpret_cast<Key128*>(cand_alt);
  if (threadIdx.x < n) {
    const double2 me = cand[threadIdx.x];
    const uint32_t doc = static_cast<uint32_t>(__double_as_longlong(me.y));
    const int r = static_cast<int>(doc / kBmRange);
    unsigned int first = 0xFFu;
    for (int t = 0; t < ntok && first == 0xFFu; ++t) {
      const uint32_t a = s_off[t * (kBsMaxRpg + 1) + (r - r0)], b = s_off[t * (kBsMaxRpg + 1) + (r - r0) + 1];
      const Post16* p = post + s_base[t];
      uint32_t lo = a, hi = b;
      while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (__ldg(&p[mid].doc) < doc) lo = mid + 1; else hi = mid;
      }
      if (lo < b && __ldg(&p[lo].doc) == doc) first = static_cast<unsigned int>(t);
    }
    Key128 kk;
    kk.hi = ~f64_orderable(static_cast<uint64_t>(__double_as_longlong(me.x)));
    kk.lo = (static_cast<unsigned long long>(first) << 32) | doc;
    s_keys[threadIdx.x] = kk;
  }
  __syncthreads();
  if (threadIdx.x < n) {
    const Key128 me = s_keys[threadIdx.x];
    int rank = 0;
    for (unsigned int j = 0; j < n; ++j) rank += key_less(s_keys[j], me) ? 1 : 0;
    if (rank < k) {
      cand_hi[cbase * k + rank] = me.hi;
      cand_lo[cbase * k + rank] = me.lo;
    }
  }
  if (threadIdx.x == 0) cand_cnt[cbase] = static_cast<int>(n) < k ? static_cast<int>(n) : k;
}

// ---------------------------------------------------------------------------------------------
// K6'' + K7'': fixed-point streaming BM25 — selection on an order-free sum, exact re-score of the finalists.
//
// bm25_stream_kernel keeps the reference's summation order with a CTA barrier after every (range, token) slice;
// the median slice holds ~150 postings, so its 16 warps mostly wait at barriers (r01 ncu: barrier 8.7 + long
// scoreboard 5.9 stall cycles per issue, 0.43 ms per 256-query step whatever is done about load latency).
// The order only matters for the low bits of a sum.  This kernel accumulates idf*w in 32-bit FIXED POINT with
// native shared-memory integer atomics (ATOMS.ADD; 64-bit and double shared atomics are CAS loops on sm_100).  The
// scale is the largest power of two that keeps (k1+1)*log(N+2)*16 below 2^31 (2^21 for the default k1: steps of
// 4.8e-7).  The kernel is HBM-bound on the posting stream (in a hybrid step it shares the HBM with the tensor-core
// filter), so it reads a 4-BYTE posting instead of the 16-byte {doc, tf, double w}: 13 bits of document offset
// inside its range (the range is known from the slice being read) and a 19-bit weight, wq = round(w * wq4_scale)
// with wq4_scale the largest power of two keeping (k1+1) * wq4_scale <= 2^19.  0 is a sentinel twice over — a weight
// word of 0 adds nothing, a sum of 0 is an untouched document — so a posting with w > 0 is stored as wq >= 1, and a
// contribution is ROUNDED UP, ceil(idfx * wq) >= 1: every document a query touches keeps a non-zero sum.  A weight is
// known to +-1 unit of wq (0.5 from its rounding, the clamp at the top, the raise from 0 to 1), i.e. +-idfx units of
// the sum (idfx = idf * scale / wq4_scale), and rounding up adds [0, 1) unit: a document's sum lies within
// [-idfx_t, idfx_t + 1) per term of its exact value, so the sums of two documents disagree with their exact order by
// less than sum_t (2 * idfx_t + 1).  The sum is exact in that format and independent of the order, so all the token
// slices of a range are cut into 128-posting items (a lane loads one aligned 16-byte QUAD) that the warps take round
// robin with NO barrier between tokens.  Everything decided on these sums compares two of them with a margin of
// 2 * sum_t (idfx_t + 0.5) + 8 units PER QUERY, at least kFxMargin (~1e-3 in score units for a 16-token query with
// the default k1); the finalists (k plus whatever lies within the margin of the k-th) are RE-SCORED in
// bm25_fx_finish_kernel with the reference's own expression in query-token order — one thread per (document, token)
// finds the posting by binary search — which also yields the reference's tie key (first token holding the
// document).  Scores, order and ties are therefore bit-identical to the general kernel; queries it cannot finish
// are flagged for it exactly like before.  (r02: the first version read an 8-byte {doc, wq} posting with a 31-bit
// weight and a constant margin; the 4-byte stream halves the bytes and pays the per-item token lookup half as
// often, at the price of a few more finalists for the exact finish kernel.)
constexpr unsigned int kFxMargin = 40u;               // floor of the per-query margin
constexpr int kFxFinalCap = 48;
constexpr int kFxRescoreCap = 96;

__host__ __device__ constexpr int fx_smem_bytes(int rpg) {
  return kBmRange * 4 + ((kBsMaxTok * (rpg + 1) * 4 + 15) & ~15) + 2 * static_cast<int>(kBsCandCap) * 8;
}

// fin: [nq][ng][kFxFinalCap] {fixed-point sum, doc}; fin_cnt: [nq][ng]
// 4 CTAs per SM = 32 registers per thread: that is also what lets ONE of these CTAs sit beside the tensor-core
// filter's CTA in a hybrid step — at 40 registers the pair overflows a scheduler's 16 K registers and BM25 silently
// waits for the filter to finish.  THREADS = 512 is the stand-alone shape (4 CTAs per SM); THREADS = kBsWideThreads
// is the shape of the CTA that runs UNDERNEATH the filter: the filter's 10 warps put 3 on two of the four
// schedulers (3 x 32 x 96 registers = 9216 of 16384), which leaves room for exactly 7 warps of 32 registers per
// scheduler — 28 warps instead of 16.  (A 768-thread shape does NOT fit: its launch bound lets ptxas take 39
// registers.)  r02 measurements, all on one box: stand-alone the kernel is thread-parallelism-bound (4 / 3 / 2 / 1
// CTAs per SM, set by padding the shared memory: 0.31 / 0.34 / 0.42 / 0.69 ms), but beside the filter it runs at
// ~14 % of the stand-alone rate whatever its shape — 28 warps instead of 16 finish 8 us earlier (step 1.078 -> 1.070
// ms), and a 55-register variant with four posting loads in flight per lane was slower overall (1.13 ms: only two
// of those fit an SM once the filter is gone).
// What it competes for there is the memory system: the filter streams the shadow at 4.9 TB/s of the 6.5 the HBM gives.
// The grid is (queries, groups): the CTAs that are resident together work on the SAME ranges for different queries,
// so the slices of the hot posting lists they share are read within microseconds of each other.
template <int THREADS, int DEPTH>
__device__ __forceinline__ void
bm25_fx_body(const int64_t* __restrict__ indptr, const uint32_t* __restrict__ post4, const uint32_t* __restrict__ roff,
             int nr, const int32_t* __restrict__ tok_indptr, const int32_t* __restrict__ term_rows,
             const double* __restrict__ tok_idf, double scale, int q0, int k, int rpg, int ng,
             uint2* __restrict__ fin, int* __restrict__ fin_cnt, int* __restrict__ status) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  uint32_t* acc = reinterpret_cast<uint32_t*>(smem_raw);                               // [kBmRange] fixed-point sums
  uint32_t* s_off = acc + kBmRange;                                                    // [kBsMaxTok][rpg + 1]
  const int ostride = rpg + 1;
  uint2* s_cand0 = reinterpret_cast<uint2*>(smem_raw + kBmRange * 4 + ((kBsMaxTok * ostride * 4 + 15) & ~15));
  uint2* s_cand1 = s_cand0 + kBsCandCap;                                               // {sum, doc}
  __shared__ long long s_base[kBsMaxTok];
  __shared__ double s_idfx[kBsMaxTok];                                                 // idf * scale / wq4_scale (exact: powers of two)
  __shared__ int s_term[kBsMaxTok];
  __shared__ unsigned int s_ncand, s_nkept;
  __shared__ unsigned int s_min, s_tw, s_margin;

  const int g = blockIdx.y;
  const int q = q0 + blockIdx.x;
  const int t0 = tok_indptr[q], ntok = tok_indptr[q + 1] - t0;
  const int64_t cbase = static_cast<int64_t>(q) * ng + g;
  if (ntok > kBsMaxTok) {                                 // uniform: the whole query goes to the general kernel
    if (threadIdx.x == 0) { fin_cnt[cbase] = 0; if (g == 0) status[q] = 1; }
    return;
  }
  const int r0 = g * rpg, r1 = min(nr, r0 + rpg);
  const int nrg = r1 - r0;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x < ntok) {
    const int term = term_rows[t0 + threadIdx.x];
    s_term[threadIdx.x] = term;
    s_base[threadIdx.x] = term >= 0 ? indptr[term] : 0;
    s_idfx[threadIdx.x] = tok_idf[t0 + threadIdx.x] * scale;
  }
  if (threadIdx.x == 0) s_ncand = 0u;
  __syncthreads();
  for (int i = threadIdx.x; i < ntok * (nrg + 1); i += blockDim.x) {
    const int t = i / (nrg + 1), j = i - t * (nrg + 1);
    const int term = s_term[t];
    s_off[t * ostride + j] = term >= 0 ? roff[static_cast<int64_t>(term) * (nr + 1) + r0 + j] : 0u;
  }
  {
    uint4* a4 = reinterpret_cast<uint4*>(acc);
    for (int i = threadIdx.x; i < kBmRange / 4; i += blockDim.x) a4[i] = make_uint4(0u, 0u, 0u, 0u);
  }
  if (threadIdx.x == 0) {                         // the margin lives in shared memory: the kernel has no register to spare
    double m = 0.0;
    for (int t = 0; t < ntok; ++t) m += s_idfx[t] + 0.5;
    const unsigned int mq = 2u * static_cast<unsigned int>(ceil(m)) + 8u;
    s_margin = mq > kFxMargin ? mq : kFxMargin;
  }
  __syncthreads();

  uint2* cand = s_cand0;
  uint2* cand_alt = s_cand1;
  unsigned int theta = 0u;                        // 0 = not established: every touched document qualifies
  bool established = false;

  // keep the documents that fewer than k others beat beyond the margin; new theta = (smallest kept sum) - margin:
  // a later document below it has k documents above it by more than the margin, i.e. k exactly greater scores
  auto compact = [&]() {
    const unsigned int n = s_ncand;                       // uniform (read after a barrier)
    if (n < static_cast<unsigned int>(k)) return;
    if (threadIdx.x == 0) { s_nkept = 0u; s_min = ~0u; }
    __syncthreads();
    if (threadIdx.x < n) {
      const uint2 me = cand[threadIdx.x];
      const unsigned int bar = me.x + s_margin;
      unsigned int greater = 0u;
      for (unsigned int j = 0; j < n; ++j) greater += cand[j].x > bar ? 1u : 0u;
      if (greater < static_cast<unsigned int>(k)) {
        cand_alt[atomicAdd(&s_nkept, 1u)] = me;
        atomicMin(&s_min, me.x);
      }
    }
    __syncthreads();
    uint2* tmp = cand; cand = cand_alt; cand_alt = tmp;
    const unsigned int mn = s_min;
    theta = mn > s_margin ? mn - s_margin : 1u;
    established = true;
    __syncthreads();
    if (threadIdx.x == 0) s_ncand = s_nkept;
    __syncthreads();
  };

  constexpr unsigned int kW = THREADS / 32;
  constexpr int kVec = kBmRange / 4;                      // accumulators as uint4
  for (int r = r0; r < r1; ++r) {
    const int jr = r - r0;
    // Items of this range: slice t contributes items of 32 aligned posting QUADS (one 16-byte load per lane).
    // Every warp derives the same item prefix in registers (lane t owns token t): no shared item table, no
    // barrier before the postings — the two barriers of a range are "sums complete" and "accumulators cleared".
    long long sb = 0;
    unsigned int sn = 0u, c = 0u;
    if (lane < ntok) {
      const uint32_t a = s_off[lane * ostride + jr];
      sn = s_off[lane * ostride + jr + 1] - a;
      sb = s_base[lane] + a;
      c = sn ? (sn + static_cast<unsigned int>(sb & 3) + 127u) >> 7 : 0u;   // quads start at a multiple of 4
    }
    unsigned int incl = c;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
      const unsigned int o = __shfl_up_sync(0xFFFFFFFFu, incl, off);
      if (lane >= off) incl += o;
    }
    const unsigned int n_items = __shfl_sync(0xFFFFFFFFu, incl, 31);
    if (n_items == 0u) continue;                          // uniform (every warp computes the same prefix)
    const unsigned int pre = incl - c;                    // first item of token `lane`
    const unsigned int has = __ballot_sync(0xFFFFFFFFu, c != 0u);
    const uint32_t doc_base = static_cast<uint32_t>(r) * kBmRange;
    const int sb_lo = static_cast<int>(static_cast<unsigned long long>(sb) & 0xFFFFFFFFull);
    const int sb_hi = static_cast<int>(static_cast<unsigned long long>(sb) >> 32);

    auto item_load = [&](unsigned int item, uint4& e, double& idfx) {
      e = make_uint4(0u, 0u, 0u, 0u);                     // a zero word adds nothing
      idfx = 0.0;
      if (item >= n_items) return;                        // warp-uniform
      // token of the item: the highest lane holding items whose first item is <= item
      const unsigned int le = __ballot_sync(0xFFFFFFFFu, pre <= item) & has;
      const int t = 31 - __clz(static_cast<int>(le));
      const unsigned int chunk = item - __shfl_sync(0xFFFFFFFFu, pre, t);
      const long long tsb = static_cast<long long>(
          (static_cast<unsigned long long>(static_cast<unsigned int>(__shfl_sync(0xFFFFFFFFu, sb_hi, t))) << 32) |
          static_cast<unsigned int>(__shfl_sync(0xFFFFFFFFu, sb_lo, t)));
      const unsigned int tsn = __shfl_sync(0xFFFFFFFFu, sn, t);
      idfx = s_idfx[t];
      // four packed postings per lane; a word of 0 (weight 0) adds nothing, so that is also the "not mine" mark
      // (positions relative to the slice start, 32-bit: the kernel has no register to spare)
      const int len = static_cast<int>(tsn);
      const int rel = static_cast<int>(chunk * 128u + 4u * lane) - static_cast<int>(tsb & 3);   // of e.x; >= -3
      if (rel + 3 >= 0 && rel < len) {                    // the quad overlaps the slice (the stream is padded by one quad)
        e = __ldg(reinterpret_cast<const uint4*>(post4 + (tsb + rel)));
        if (rel < 0) e.x = 0u;
        if (rel + 1 < 0 || rel + 1 >= len) e.y = 0u;
        if (rel + 2 < 0 || rel + 2 >= len) e.z = 0u;
        if (rel + 3 >= len) e.w = 0u;
      }
    };
    auto item_apply = [&](const uint4& e, double idfx) {
      // sums only grow and nothing reads them before the barrier: plain reductions, no returned value to wait for.
      // Rounded UP, a contribution of a non-zero word is at least 1: a sum of 0 means "untouched" to the scan.
      const uint32_t w4[4] = {e.x, e.y, e.z, e.w};
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (w4[u] >> 13) atomicAdd(&acc[w4[u] & 0x1FFFu], __double2uint_ru(__dmul_rn(idfx, __uint2double_rn(w4[u] >> 13))));
    };
    {
      // DEPTH loads in flight per lane (a ring of named buffers: every index below is a compile-time constant)
      uint4 e[DEPTH];
      double f[DEPTH];
      unsigned int it = warp;
#pragma unroll
      for (int d = 0; d < DEPTH - 1; ++d) item_load(it + d * kW, e[d], f[d]);
      while (it < n_items) {
#pragma unroll
        for (int d = 0; d < DEPTH; ++d) {
          item_load(it + (DEPTH - 1) * kW, e[(d + DEPTH - 1) % DEPTH], f[(d + DEPTH - 1) % DEPTH]);
          item_apply(e[d], f[d]);
          it += kW;
          if (it >= n_items) break;
        }
      }
    }
    __syncthreads();                                      // the range's sums are complete

    uint4* a4 = reinterpret_cast<uint4*>(acc);
    if (!established) {
      // theta = (k-th largest of the warps' best thread maxima) - margin: maxima of distinct threads are distinct
      // documents, so k of them at or above it bound the k-th best exact score from below
      unsigned int mine = 0u;
      for (int v = threadIdx.x; v < kVec; v += THREADS) {
        const uint4 x = a4[v];
        mine = max(mine, max(max(x.x, x.y), max(x.z, x.w)));
      }
      const int m = (k + THREADS / 32 - 1) / (THREADS / 32);        // 1 or 2
      unsigned int* s_top = reinterpret_cast<unsigned int*>(cand_alt);
      for (int round = 0; round < m; ++round) {
        unsigned int wm = mine;
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) wm = max(wm, __shfl_xor_sync(0xFFFFFFFFu, wm, off));
        const unsigned int holders = __ballot_sync(0xFFFFFFFFu, mine == wm);
        if (lane == __ffs(holders) - 1) { s_top[warp * m + round] = wm; mine = 0u; }
      }
      if (threadIdx.x == 0) s_tw = 0u;
      __syncthreads();
      const int nv = (THREADS / 32) * m;                                // 16 or 32
      if (static_cast<int>(threadIdx.x) < nv) {
        const unsigned int me = s_top[threadIdx.x];
        int r2 = 0;
        for (int jj = 0; jj < nv; ++jj) {
          const unsigned int o = s_top[jj];
          r2 += (o > me || (o == me && jj < static_cast<int>(threadIdx.x))) ? 1 : 0;
        }
        if (r2 == k - 1) s_tw = me;                        // 0 when fewer than k threads saw a document
      }
      __syncthreads();
      const unsigned int tb = s_tw;
      if (tb != 0u) { theta = tb > s_margin ? tb - s_margin : 1u; established = true; }
    }
    // scan + clear: collect the documents at or above theta (theta = 0: every touched document)
    {
      const unsigned int bar = theta ? theta : 1u;
      for (int v = threadIdx.x; v < kVec; v += THREADS) {
        const uint4 x = a4[v];
        if ((x.x | x.y | x.z | x.w) == 0u) continue;
        a4[v] = make_uint4(0u, 0u, 0u, 0u);
        const unsigned int mx = max(max(x.x, x.y), max(x.z, x.w));
        if (mx < bar) continue;
        const unsigned int xs[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          if (xs[u] >= bar) {
            const unsigned int slot = atomicAdd(&s_ncand, 1u);
            if (slot < kBsCandCap) cand[slot] = make_uint2(xs[u], doc_base + static_cast<uint32_t>(v) * 4u + u);
          }
        }
      }
    }
    __syncthreads();                                      // accumulators are clear, the candidate count is final
    if (s_ncand > kBsCandCap) {                           // uniform: mass ties → the general kernel re-scores the query
      if (threadIdx.x == 0) { status[q] = 1; fin_cnt[cbase] = 0; }
      return;
    }
    if (s_ncand >= kBsCompactAt) compact();
  }
  __syncthreads();
  compact();
  const unsigned int n = s_ncand;
  if (n > static_cast<unsigned int>(kFxFinalCap)) {
    if (threadIdx.x == 0) { status[q] = 1; fin_cnt[cbase] = 0; }
    return;
  }
  if (threadIdx.x < n) fin[cbase * kFxFinalCap + threadIdx.x] = cand[threadIdx.x];
  if (threadIdx.x == 0) fin_cnt[cbase] = static_cast<int>(n);
}

template <int THREADS>
__global__ void __launch_bounds__(THREADS, (THREADS <= 512 ? 4 : 2))
bm25_fx_kernel(const int64_t* __restrict__ indptr, const uint32_t* __restrict__ post4, const uint32_t* __restrict__ roff,
               int nr, const int32_t* __restrict__ tok_indptr, const int32_t* __restrict__ term_rows,
               const double* __restrict__ tok_idf, double scale, int q0, int k, int rpg, int ng,
               uint2* __restrict__ fin, int* __restrict__ fin_cnt, int* __restrict__ status) {
  bm25_fx_body<THREADS, 2>(indptr, post4, roff, nr, tok_indptr, term_rows, tok_idf, scale, q0, k, rpg, ng, fin, fin_cnt, status);
}
// K7'': one CTA per query bm25_fx_kernel finished (see the header above).
__global__ void __launch_bounds__(kBmThreads)
bm25_fx_finish_kernel(const uint2* __restrict__ fin, const int* __restrict__ fin_cnt, int ng, int* __restrict__ status,
                      const int64_t* __restrict__ indptr, const Post16* __restrict__ post,
                      const uint32_t* __restrict__ roff, int nr, const int32_t* __restrict__ tok_indptr,
                      const int32_t* __restrict__ term_rows, const double* __restrict__ tok_idf, int q0, int k,
                      double* __restrict__ out_score, int* __restrict__ out_doc, int* __restrict__ out_count,
                      unsigned long long* __restrict__ counters, double idfx_scale) {
  __shared__ uint2 s_c[kBsMaxGroups * kFxFinalCap];       // 12 KB: the groups' candidates {sum, doc}
  __shared__ double s_w[kFxRescoreCap][kBsMaxTok];        // 12 KB: weight of (document, token), 0 = not in the list
  __shared__ uint32_t s_doc[kFxRescoreCap];
  __shared__ Key128 s_key[kFxRescoreCap];
  __shared__ unsigned int s_n, s_m;
  const int q = q0 + blockIdx.x;
  if (status[q] != 0) return;                             // the general path owns this query
  const int t0 = tok_indptr[q], ntok = tok_indptr[q + 1] - t0;
  unsigned int margin = kFxMargin;                        // the same per-query margin bm25_fx_body decided with
  {
    double m = 0.0;
    for (int t = 0; t < ntok; ++t) m += tok_idf[t0 + t] * idfx_scale + 0.5;
    const unsigned int mq = 2u * static_cast<unsigned int>(ceil(m)) + 8u;
    if (mq > margin) margin = mq;
  }
  if (threadIdx.x == 0) { s_n = 0u; s_m = 0u; }
  __syncthreads();
  for (int g = 0; g < ng; ++g) {
    const int64_t cb = static_cast<int64_t>(q) * ng + g;
    const int c = fin_cnt[cb];
    if (static_cast<int>(threadIdx.x) < c) s_c[atomicAdd(&s_n, 1u)] = fin[cb * kFxFinalCap + threadIdx.x];
  }
  __syncthreads();
  const unsigned int n = s_n;
  // documents that fewer than k others beat beyond the margin: the exact top-k is among them
  for (unsigned int e = threadIdx.x; e < n; e += blockDim.x) {
    const uint2 me = s_c[e];
    const unsigned int bar = me.x + margin;
    unsigned int greater = 0u;
    for (unsigned int j = 0; j < n; ++j) greater += s_c[j].x > bar ? 1u : 0u;
    if (greater < static_cast<unsigned int>(k)) {
      const unsigned int slot = atomicAdd(&s_m, 1u);
      if (slot < static_cast<unsigned int>(kFxRescoreCap)) s_doc[slot] = me.y;
    }
  }
  __syncthreads();
  if (s_m > static_cast<unsigned int>(kFxRescoreCap)) {   // a near-tie group at the k-th score larger than the cap:
    if (threadIdx.x == 0) status[q] = 1;                  // the general kernels run after this one and pick the query up
    return;
  }
  const unsigned int m = s_m;
  if (counters && threadIdx.x == 0) {                     // [1] finalists re-scored exactly, [2] candidates the groups handed over
    atomicAdd(&counters[1], static_cast<unsigned long long>(m));
    atomicAdd(&counters[2], static_cast<unsigned long long>(n));
  }
  // exact re-score, step 1: the posting of every (document, token) pair
  for (unsigned int pidx = threadIdx.x; pidx < m * static_cast<unsigned int>(ntok); pidx += blockDim.x) {
    const unsigned int d = pidx / ntok;
    const int t = static_cast<int>(pidx - d * ntok);
    const uint32_t doc = s_doc[d];
    const int term = term_rows[t0 + t];
    double w = 0.0;
    if (term >= 0) {
      const uint32_t* ro = roff + static_cast<int64_t>(term) * (nr + 1) + static_cast<int>(doc / kBmRange);
      const uint32_t a = ro[0], b = ro[1];
      const Post16* p = post + indptr[term];
      uint32_t lo = a, hi = b;
      while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (__ldg(&p[mid].doc) < doc) lo = mid + 1; else hi = mid;
      }
      if (lo < b && __ldg(&p[lo].doc) == doc) w = __ldg(&p[lo].w);
    }
    s_w[d][t] = w;
  }
  __syncthreads();
  // step 2: the reference's sum in query-token order (keyword_search.py:241-244) and the tie key
  if (threadIdx.x < m) {
    double score = 0.0;
    unsigned int first = 0xFFu;
    for (int t = 0; t < ntok; ++t) {
      const double w = s_w[threadIdx.x][t];
      if (w != 0.0) {
        score = __dadd_rn(score, __dmul_rn(tok_idf[t0 + t], w));
        if (first == 0xFFu) first = static_cast<unsigned int>(t);
      }
    }
    Key128 kk;
    kk.hi = ~f64_orderable(static_cast<uint64_t>(__double_as_longlong(score)));
    kk.lo = (static_cast<unsigned long long>(first) << 32) | s_doc[threadIdx.x];
    s_key[threadIdx.x] = kk;
  }
  __syncthreads();
  if (threadIdx.x < m) {
    const Key128 me = s_key[threadIdx.x];
    int rank = 0;
    for (unsigned int j = 0; j < m; ++j) rank += key_less(s_key[j], me) ? 1 : 0;
    if (rank < k) {
      const int64_t o = static_cast<int64_t>(q) * k + rank;
      const uint64_t ob = ~me.hi;
      const uint64_t bits = (ob & 0x8000000000000000ull) ? (ob & 0x7FFFFFFFFFFFFFFFull) : ~ob;
      out_score[o] = __longlong_as_double(static_cast<long long>(bits));
      out_doc[o] = static_cast<int>(static_cast<uint32_t>(me.lo));
    }
  }
  const int emitted = static_cast<int>(m) < k ? static_cast<int>(m) : k;
  if (threadIdx.x == 0) out_count[q] = emitted;
  for (int i = emitted + threadIdx.x; i < k; i += blockDim.x) {
    out_score[static_cast<int64_t>(q) * k + i] = 0.0;
    out_doc[static_cast<int64_t>(q) * k + i] = -1;
  }
}

// K7 (query part): k-way merge of the per-range sorted candidate lists.
// One CTA per query; thread j owns ranges j, j+blockDim, ...
__global__ void __launch_bounds__(kBmThreads)
bm25_merge_kernel(const unsigned long long* __restrict__ cand_hi, const unsigned long long* __restrict__ cand_lo,
                  const int* __restrict__ cand_cnt, int nr, int q0, int k, double* __restrict__ out_score,
                  int* __restrict__ out_doc, int* __restrict__ out_count,
                  const unsigned long long* __restrict__ alt_hi, const unsigned long long* __restrict__ alt_lo,
                  const int* __restrict__ alt_cnt, int alt_nr, const int* __restrict__ use_alt) {
  __shared__ Key128 s_k[kBmThreads / 32];
  __shared__ int s_w[kBmThreads / 32];
  const int q = q0 + blockIdx.x;
  // the streaming kernel's per-group lists unless it flagged the query (then the general kernel's per-range lists)
  if (use_alt && use_alt[q] == 0) {
    if (!alt_hi) return;                                  // bm25_fx_finish_kernel already wrote this query's results
    cand_hi = alt_hi; cand_lo = alt_lo; cand_cnt = alt_cnt; nr = alt_nr;
  }
  // per-thread heads (a thread may own several ranges when nr > blockDim; it keeps
  // the best head among them and re-scans its ranges after winning)
  constexpr int kMaxOwn = 8;                 // nr <= 2048 ranges = 14,680,064 docs
  int head[kMaxOwn];
#pragma unroll
  for (int i = 0; i < kMaxOwn; ++i) head[i] = 0;
  auto best_head = [&](int* which) -> Key128 {
    Key128 best = key_inf();
    *which = -1;
#pragma unroll
    for (int i = 0; i < kMaxOwn; ++i) {
      const int r = threadIdx.x + i * kBmThreads;
      if (r >= nr) break;
      const int64_t cb = static_cast<int64_t>(q) * nr + r;
      if (head[i] < cand_cnt[cb]) {
        Key128 kk{cand_hi[cb * k + head[i]], cand_lo[cb * k + head[i]]};
        if (key_less(kk, best)) { best = kk; *which = i; }
      }
    }
    return best;
  };
  int which;
  Key128 mine = best_head(&which);
  int emitted = 0;
  for (int round = 0; round < k; ++round) {
    int winner;
    const Key128 w = block_argmin(mine, s_k, s_w, &winner);
    if (w.hi == ~0ull && w.lo == ~0ull) break;
    if (threadIdx.x == winner) {
      const int64_t o = static_cast<int64_t>(q) * k + round;
      const uint64_t ob = ~w.hi;   // orderable(score)
      const uint64_t bits = (ob & 0x8000000000000000ull) ? (ob & 0x7FFFFFFFFFFFFFFFull) : ~ob;
      out_score[o] = __longlong_as_double(static_cast<long long>(bits));
      out_doc[o] = static_cast<int>(static_cast<uint32_t>(w.lo));
#pragma unroll
      for (int i = 0; i < kMaxOwn; ++i)
        if (i == which) head[i]++;
      mine = best_head(&which);
    }
    ++emitted;
  }
  if (threadIdx.x == 0) out_count[q] = emitted;
  for (int i = emitted + threadIdx.x; i < k; i += blockDim.x) {
    out_score[static_cast<int64_t>(q) * k + i] = 0.0;
    out_doc[static_cast<int64_t>(q) * k + i] = -1;
  }
}

}  // namespace rse

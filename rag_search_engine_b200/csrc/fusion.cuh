// fusion.cuh — K8/K9: weighted (min-max) and reciprocal-rank fusion.
// Replaces HybridSearch.weighted_search / rrf_search fusion cores
// (rag_search_engine/utils/hybrid_search.py:117-180 and :217-272,379) and
// min_max_norm / rrf_score (utils/utils.py:182-191, :205-206).
//
// All arithmetic is IEEE double with explicit round-to-nearest intrinsics in the
// reference's association.  The candidate order before the stable sort is the
// iteration order of the CPython set union (pyset.h) in RSE_TIE_REFERENCE mode,
// or ascending id in RSE_TIE_BY_ID mode; the stable descending sort is done by
// rank counting (rank = #greater + #equal-before).
//
// Latency-bound, ≤ 2*limit items per query.  Up to kFuseMaxLimit (every hybrid call of the serving loop, the
// fusion entry points and the cross-encoder rerank): one warp per query, lane 0 runs the serial set emulation in
// shared memory with the keys in the table slots, all lanes do the scoring / ranking.  Above it, up to
// kFuseDeepLimit (deep result lists for a reranker): one CTA of 256 threads per query; the sets hold 16-bit indices
// into the staged ids (8-byte slots for a 2048-id union would need 384 KB of shared memory, more than a block may
// have), and the ascending-id union, the scoring and the rank counting are spread over all eight warps.
#pragma once
#include "common.cuh"
#include "pyset.h"

namespace rse {

constexpr int kFuseMaxLimit = 128;
constexpr int kFuseDeepLimit = 1024;
constexpr int kFuseDeepThreads = 256;

__host__ __device__ inline int fuse_cap_side(int limit) { return pyset_capacity_for(limit); }
__host__ __device__ inline int fuse_cap_union(int limit) { return pyset_capacity_for(2 * limit); }
// smem bytes: ta + tb + tr + scratch (int64) + order[2L] i64 + score[2L] f64 + aux a/b [2L] f64 x2
__host__ __device__ inline size_t fuse_smem_bytes(int limit) {
  size_t tables = static_cast<size_t>(2 * fuse_cap_side(limit) + 2 * fuse_cap_union(limit)) * 8;
  return tables + static_cast<size_t>(2 * limit) * 8 * 4 + 64;
}
// deep kernel: order / score / a / b [2L] and the staged ids, scores, distances [L] x 2 (8 B each), then the four
// tables of 16-bit slots — 192 KB at limit 1024
__host__ __device__ inline size_t fuse_deep_smem_bytes(int limit) {
  size_t tables = static_cast<size_t>(2 * fuse_cap_side(limit) + 2 * fuse_cap_union(limit)) * 2;
  return static_cast<size_t>(2 * limit) * 8 * 6 + tables + 64;
}

template <int kThreads>
__device__ __forceinline__ void fuse_sync() {
  if constexpr (kThreads == 32) __syncwarp(); else __syncthreads();
}

struct FuseIn {
  const long long* bm25_id; const double* bm25_score; const int* bm25_count;   // [nq][limit]
  const long long* sem_id; const float* sem_dist; const int* sem_count;         // [nq][limit]
  const double* sem_dist64;   // when non-NULL used instead of sem_dist (Python floats from a plugged-in retriever)
  // fused hybrid path: the hits arrive as dense indices and are mapped to ids here (id = table[idx], -1 if out of
  // range) instead of by two separate gather launches; used when bm25_id / sem_id are NULL
  const int* bm25_idx = nullptr; const long long* bm25_table = nullptr; long long bm25_table_n = 0;
  const int* sem_idx = nullptr;  const long long* sem_table = nullptr;  long long sem_table_n = 0;
};

// mode 0 = rrf (param = k), mode 1 = weighted (param = alpha)
// inputs [nq][limit]; outputs [nq][out_w] (limit <= out_w <= 2 * limit): id, score, a, b  (rrf: a/b =
// bm25_rank/sem_rank as double, -1 = None; weighted: a/b = bm25_norm/sem_norm).  out_w = limit is the reference's
// [:limit]; out_w = 2 * limit keeps the whole union in fused order (what the cross-encoder rerank scores).
// The deep kernel's shared memory allows one CTA per SM anyway; saying so (min blocks 1) keeps ptxas from spilling
// the set emulation's loop state at 48 registers.
template <int kMaxLimit>
__global__ void __launch_bounds__(kMaxLimit > kFuseMaxLimit ? kFuseDeepThreads : 32, kMaxLimit > kFuseMaxLimit ? 1 : 0)
fuse_kernel(FuseIn in, int nq, int limit, int out_w, int mode, double param, int tie_mode, long long* __restrict__ out_id,
            double* __restrict__ out_score, double* __restrict__ out_a, double* __restrict__ out_b,
            int* __restrict__ out_count) {
  constexpr bool kDeep = kMaxLimit > kFuseMaxLimit;
  constexpr int kThreads = kDeep ? kFuseDeepThreads : 32;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int q = blockIdx.x;
  if (q >= nq) return;
  const int lane = threadIdx.x;
  const int cs = fuse_cap_side(limit), cu = fuse_cap_union(limit);
  int64_t *ta, *tb, *tr, *sc, *order;
  double *score, *va, *vb;
  long long *s_bid, *s_sid;
  double *s_bsc, *s_sds;
  uint16_t* t16 = nullptr;
  __shared__ int s_n;
  if constexpr (kDeep) {
    order = reinterpret_cast<int64_t*>(smem_raw);                 // [2*limit]
    score = reinterpret_cast<double*>(order + 2 * limit);
    va = score + 2 * limit;
    vb = va + 2 * limit;
    s_bid = reinterpret_cast<long long*>(vb + 2 * limit);         // [limit], s_sid right behind: the key array of
    s_sid = s_bid + limit;                                        // the index-slot sets (b's slots start at limit)
    s_bsc = reinterpret_cast<double*>(s_sid + limit);
    s_sds = s_bsc + limit;
    t16 = reinterpret_cast<uint16_t*>(s_sds + limit);             // ta, tb [cs], tr, scratch [cu]
    if (lane == 0) s_n = 0;
  } else {
    ta = reinterpret_cast<int64_t*>(smem_raw);
    tb = ta + cs;
    tr = tb + cs;
    sc = tr + cu;
    order = sc + cu;                                              // [2*limit]
    score = reinterpret_cast<double*>(order + 2 * limit);
    va = score + 2 * limit;
    vb = va + 2 * limit;
    // the two hit lists are staged in shared memory by the whole warp first: the set emulation below is a serial
    // walk by one lane, and every global load in it was a ~500-cycle round trip (23 us per 256-query batch)
    __shared__ long long s_bid_w[kFuseMaxLimit], s_sid_w[kFuseMaxLimit];
    __shared__ double s_bsc_w[kFuseMaxLimit], s_sds_w[kFuseMaxLimit];
    s_bid = s_bid_w; s_sid = s_sid_w; s_bsc = s_bsc_w; s_sds = s_sds_w;
  }
  int nb = in.bm25_count[q]; if (nb > limit) nb = limit; if (nb < 0) nb = 0;
  int ns = in.sem_count[q];  if (ns > limit) ns = limit; if (ns < 0) ns = 0;
  for (int i = lane; i < limit; i += kThreads) {
    const int64_t o = static_cast<int64_t>(q) * limit + i;
    long long b_id = -1ll, s_id = -1ll;
    if (i < nb) {
      if (in.bm25_id) b_id = in.bm25_id[o];
      else { const int v = in.bm25_idx[o]; b_id = (v >= 0 && v < in.bm25_table_n) ? in.bm25_table[v] : -1ll; }
    }
    if (i < ns) {
      if (in.sem_id) s_id = in.sem_id[o];
      else { const int v = in.sem_idx[o]; s_id = (v >= 0 && v < in.sem_table_n) ? in.sem_table[v] : -1ll; }
    }
    s_bid[i] = b_id;
    s_bsc[i] = i < nb ? in.bm25_score[o] : 0.0;
    s_sid[i] = s_id;
    s_sds[i] = i < ns ? (in.sem_dist64 ? in.sem_dist64[o] : static_cast<double>(in.sem_dist[o])) : 0.0;   // float(hit["distance"])
  }
  fuse_sync<kThreads>();
  const long long* bid = s_bid;
  const double* bsc = s_bsc;
  const long long* sid = s_sid;
  auto sem_d = [&](int i) -> double { return s_sds[i]; };

  if constexpr (kDeep) {
    if (tie_mode == 0) {
      if (lane == 0)
        s_n = pyset_union_order(PySetIndexedKeys{reinterpret_cast<const int64_t*>(bid), limit}, nb, ns, t16, cs,
                                t16 + cs, cs, t16 + 2 * cs, cu, t16 + 2 * cs + cu, cu, order);
    } else {
      // ascending-id union: member e of bid[0..nb) ++ sid[0..ns) is kept when no earlier member has its id, and
      // lands at the number of kept members with a smaller id
      unsigned char* kept = reinterpret_cast<unsigned char*>(t16);
      const int m = nb + ns;
      auto member = [&](int e) -> int64_t { return e < nb ? bid[e] : sid[e - nb]; };
      for (int e = lane; e < m; e += kThreads) {
        const int64_t v = member(e);
        bool first = true;
        for (int j = 0; j < e && first; ++j) first = member(j) != v;
        kept[e] = first;
      }
      __syncthreads();
      int mine = 0;
      for (int e = lane; e < m; e += kThreads) {
        if (!kept[e]) continue;
        const int64_t v = member(e);
        int pos = 0;
        for (int j = 0; j < m; ++j) pos += kept[j] && member(j) < v;
        order[pos] = v;
        ++mine;
      }
      if (mine) atomicAdd(&s_n, mine);
    }
  } else if (lane == 0) {
    int n;
    if (tie_mode == 0) {
      n = pyset_union_order(reinterpret_cast<const int64_t*>(bid), nb, reinterpret_cast<const int64_t*>(sid), ns,
                            ta, cs, tb, cs, tr, cu, sc, cu, order);
    } else {
      // ascending-id union (insertion sort of ≤ 2*limit ids, duplicates dropped)
      n = 0;
      for (int pass = 0; pass < 2; ++pass) {
        const long long* src = pass ? sid : bid;
        const int cnt = pass ? ns : nb;
        for (int i = 0; i < cnt; ++i) {
          const int64_t v = src[i];
          int p = 0;
          while (p < n && order[p] < v) ++p;
          if (p < n && order[p] == v) continue;
          for (int j = n; j > p; --j) order[j] = order[j - 1];
          order[p] = v; ++n;
        }
      }
    }
    s_n = n;
  }
  fuse_sync<kThreads>();
  const int n = s_n;
  if (n < 0) {   // cannot happen within kMaxLimit; keep the failure visible
    if (lane == 0) out_count[q] = -1;
    return;
  }

  // ---- per-side normalisation constants (weighted) -------------------------
  double bmin = 0.0, bmax = 0.0, smin = 0.0, smax = 0.0;
  if (mode == 1) {
    if (nb > 0) { bmin = bmax = bsc[0]; for (int i = 1; i < nb; ++i) { double v = bsc[i]; if (v < bmin) bmin = v; if (v > bmax) bmax = v; } }
    if (ns > 0) {
      smin = smax = __dsub_rn(1.0, sem_d(0));
      for (int i = 1; i < ns; ++i) { double v = __dsub_rn(1.0, sem_d(i)); if (v < smin) smin = v; if (v > smax) smax = v; }
    }
  }

  // ---- score every union member -------------------------------------------
  for (int i = lane; i < n; i += kThreads) {
    const int64_t id = order[i];
    int rb = -1, rs = -1;
    for (int j = 0; j < nb; ++j) if (bid[j] == id) rb = j;      // dict: last assignment wins
    for (int j = 0; j < ns; ++j) if (sid[j] == id) rs = j;
    double s, a, b;
    if (mode == 0) {
      // ranks: lists arrive already sorted (stable re-sort at :220-224,:235-238 is the identity)
      const double kb = __dadd_rn(param, static_cast<double>(rb >= 0 ? rb : 99999));
      const double ks = __dadd_rn(param, static_cast<double>(rs >= 0 ? rs : 99999));
      s = __dadd_rn(__ddiv_rn(1.0, kb), __ddiv_rn(1.0, ks));    // :255, BM25 term first
      a = static_cast<double>(rb); b = static_cast<double>(rs);
    } else {
      a = 0.0; b = 0.0;                                          // :160-161 missing side → 0.0
      if (rb >= 0) a = (bmin == bmax) ? 1.0 : __ddiv_rn(__dsub_rn(bsc[rb], bmin), __dsub_rn(bmax, bmin));
      if (rs >= 0) {
        const double sim = __dsub_rn(1.0, sem_d(rs));                     // :134
        b = (smin == smax) ? 1.0 : __ddiv_rn(__dsub_rn(sim, smin), __dsub_rn(smax, smin));
      }
      s = __dadd_rn(__dmul_rn(param, a), __dmul_rn(__dsub_rn(1.0, param), b));               // :163
    }
    score[i] = s; va[i] = a; vb[i] = b;
  }
  fuse_sync<kThreads>();

  // ---- stable descending sort by rank counting, then [:out_w] ---------------
  const int n_out = n < out_w ? n : out_w;
  for (int i = lane; i < n; i += kThreads) {
    const double si = score[i];
    int rank = 0;
    for (int j = 0; j < n; ++j) {
      const double sj = score[j];
      rank += (sj > si) || (sj == si && j < i);
    }
    if (rank < out_w) {
      const int64_t o = static_cast<int64_t>(q) * out_w + rank;
      out_id[o] = order[i]; out_score[o] = si; out_a[o] = va[i]; out_b[o] = vb[i];
    }
  }
  for (int i = n_out + lane; i < out_w; i += kThreads) {
    const int64_t o = static_cast<int64_t>(q) * out_w + i;
    out_id[o] = -1; out_score[o] = 0.0; out_a[o] = -1.0; out_b[o] = -1.0;
  }
  if (lane == 0) out_count[q] = n_out;
}

}  // namespace rse

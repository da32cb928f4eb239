// rerank.cuh — the cross-encoder rerank of a fused hybrid batch (HybridSearch.rrf_search(...,
// rerank_method="cross_encoder"), hybrid_search.py:279-312) around the encoder of encoder.cuh.
//
// The fusion kernel hands over the whole RRF union of every query in fused order ([nq][W], W = 2 * limit).  Every
// union member becomes one (query, document) pair
//     [CLS] q[:a] [SEP] d[:b] [SEP]      token types 0 for the first a + 2 tokens, 1 for the last b + 1
// with q the query's token ids and d the document's (the cross-encoder tokenizer's ids of f"{title} - {description}",
// special tokens stripped) taken from a CSR store in HBM, and (a, b) from HF fast tokenizers' longest_first rule
// (pair_truncate).  The pairs are packed back to back in (query, fused position) order for the encoder, whose
// logits the order kernel turns into the reference's ranking: a stable descending sort on
// (cross_encoder_score, rrf_score), then [:limit].
//
// Three launches assemble the packed batch: rerank_len_kernel (store lookup, truncation, per-query pair / token
// totals), rerank_scan_kernel (exclusive scans over the queries) and rerank_pack_kernel (cu_seqlens, ids, type_ids).
#pragma once
#include <climits>

#include "common.cuh"

namespace rse {

constexpr int kRrThreads = 256;      // one thread per member of a query's union (<= 2 * kFuseMaxLimit)
constexpr int kRrScanThreads = 1024;

// HF fast tokenizers, truncation=True (longest_first), for a pair of n1 + n2 tokens and M = max_length - 3 slots:
// how many tokens of each side stay.  Ties (n1 == n2) give the first input the "shorter" share.
__host__ __device__ inline void pair_truncate(int n1, int n2, int M, int* a, int* b) {
  if (n1 + n2 <= M) { *a = n1; *b = n2; return; }
  int s = n1 < n2 ? n1 : n2, l = n1 < n2 ? n2 : n1;
  l = s > M ? s : (s > M - s ? s : M - s);
  if (s + l > M) { s = M / 2; l = s + M % 2; }
  if (n1 <= n2) { *a = s; *b = l; } else { *a = l; *b = s; }
}

// exclusive prefix sum of v over the first blockDim.x threads (Hillis-Steele in shared memory); returns the total
__device__ __forceinline__ int rr_block_exscan(int v, int* buf, int* out) {
  const int t = threadIdx.x;
  buf[t] = v;
  __syncthreads();
  for (int d = 1; d < blockDim.x; d <<= 1) {
    const int x = t >= d ? buf[t - d] : 0;
    __syncthreads();
    buf[t] += x;
    __syncthreads();
  }
  *out = buf[t] - v;
  const int total = buf[blockDim.x - 1];
  __syncthreads();
  return total;
}

// meta[0] = ids missing from the store, meta[1] = smallest flat index (q * W + j) of such an id (as unsigned, reset
// to UINT_MAX by the host), meta[2] = pairs, meta[3] = tokens, meta[4 ..] = cu_seqlens of the packed pairs
constexpr int kRrMetaHead = 4;

// one CTA per query, one thread per union member: row in the store, (a, b), pair length; CTA totals
__global__ void __launch_bounds__(kRrThreads)
rerank_len_kernel(const long long* __restrict__ fid, const int* __restrict__ fcnt, int W,
                  const long long* __restrict__ doc_ids, long long n_docs, const long long* __restrict__ doc_indptr,
                  const int* __restrict__ q_indptr, int M, int* __restrict__ pair_row, int2* __restrict__ pair_ab,
                  int* __restrict__ q_np, int* __restrict__ q_nt, int* __restrict__ meta) {
  __shared__ int s_buf[kRrThreads];
  const int q = blockIdx.x, j = threadIdx.x;
  int n = fcnt[q];
  n = n < 0 ? 0 : (n > W ? W : n);
  const int n1 = q_indptr[q + 1] - q_indptr[q];
  int len = 0;
  if (j < n) {
    const int64_t o = static_cast<int64_t>(q) * W + j;
    const long long id = fid[o];
    long long lo = 0, hi = n_docs;                        // first row with doc_ids[row] >= id
    while (lo < hi) {
      const long long mid = (lo + hi) >> 1;
      if (doc_ids[mid] < id) lo = mid + 1; else hi = mid;
    }
    int a = 0, b = 0, row = -1;
    if (lo < n_docs && doc_ids[lo] == id) {
      row = static_cast<int>(lo);
      pair_truncate(n1, static_cast<int>(doc_indptr[lo + 1] - doc_indptr[lo]), M, &a, &b);
      len = a + b + 3;
    } else {
      atomicAdd(&meta[0], 1);
      atomicMin(reinterpret_cast<unsigned int*>(&meta[1]), static_cast<unsigned int>(o));
    }
    pair_row[o] = row;
    pair_ab[o] = make_int2(a, b);
  }
  int ex;
  const int tot = rr_block_exscan(len, s_buf, &ex);
  if (j == 0) { q_np[q] = n; q_nt[q] = tot; }
}

// one CTA: exclusive scans of the per-query pair and token counts -> q_pb / q_tb [nq + 1]; totals into meta[2..3]
__global__ void __launch_bounds__(kRrScanThreads)
rerank_scan_kernel(const int* __restrict__ q_np, const int* __restrict__ q_nt, int nq, int* __restrict__ q_pb,
                   int* __restrict__ q_tb, int* __restrict__ meta) {
  __shared__ int s_buf[kRrScanThreads];
  const int t = threadIdx.x;
  const int per = (nq + kRrScanThreads - 1) / kRrScanThreads;
  const int lo = min(nq, t * per), hi = min(nq, lo + per);
  int sp = 0, st = 0;
  for (int i = lo; i < hi; ++i) { sp += q_np[i]; st += q_nt[i]; }
  int bp, bt;
  const int tp = rr_block_exscan(sp, s_buf, &bp);
  const int tt = rr_block_exscan(st, s_buf, &bt);
  for (int i = lo; i < hi; ++i) {
    q_pb[i] = bp; q_tb[i] = bt;
    bp += q_np[i]; bt += q_nt[i];
  }
  if (t == 0) { q_pb[nq] = tp; q_tb[nq] = tt; meta[2] = tp; meta[3] = tt; }
}

// one CTA per query: cu_seqlens of its pairs, then one warp per pair writes ids / type_ids (lanes stride over the
// tokens: the document's tokens are read as contiguous runs)
__global__ void __launch_bounds__(kRrThreads)
rerank_pack_kernel(const int* __restrict__ fcnt, int W, const int* __restrict__ pair_row,
                   const int2* __restrict__ pair_ab, const int* __restrict__ q_pb, const int* __restrict__ q_tb,
                   const int* __restrict__ q_indptr, const int* __restrict__ q_tok,
                   const long long* __restrict__ doc_indptr, const int* __restrict__ doc_tok, int cls_id, int sep_id,
                   int* __restrict__ cu, int* __restrict__ ids, int* __restrict__ types) {
  __shared__ int s_buf[kRrThreads];
  __shared__ int s_off[kRrThreads];
  __shared__ int2 s_ab[kRrThreads];
  __shared__ int s_row[kRrThreads];
  const int q = blockIdx.x, j = threadIdx.x;
  int n = fcnt[q];
  n = n < 0 ? 0 : (n > W ? W : n);
  const int64_t o = static_cast<int64_t>(q) * W + j;
  int2 ab = make_int2(0, 0);
  int row = -1;
  if (j < n) { ab = pair_ab[o]; row = pair_row[o]; }
  const int len = j < n ? ab.x + ab.y + 3 : 0;
  int ex;
  rr_block_exscan(len, s_buf, &ex);
  const int pb = q_pb[q], tb = q_tb[q];
  if (j < n) cu[pb + j] = tb + ex;
  if (j == 0) cu[q_pb[q + 1]] = q_tb[q + 1];             // the next query's first entry (same value) or the total
  s_off[j] = tb + ex; s_ab[j] = ab; s_row[j] = row;
  __syncthreads();
  const int lane = j & 31, warp = j >> 5;
  const int* qt = q_tok + q_indptr[q];
  for (int p = warp; p < n; p += kRrThreads / 32) {
    const int a = s_ab[p].x, b = s_ab[p].y, off = s_off[p];
    const int* dt = doc_tok + (s_row[p] >= 0 ? doc_indptr[s_row[p]] : 0);
    const int L = a + b + 3;
    for (int t = lane; t < L; t += 32) {
      int v;
      if (t == 0) v = cls_id;
      else if (t <= a) v = qt[t - 1];
      else if (t == a + 1 || t == L - 1) v = sep_id;
      else v = dt[t - a - 2];
      ids[off + t] = v;
      types[off + t] = t < a + 2 ? 0 : 1;
    }
  }
}

// cu_seqlens of the pairs [p0, p0 + n) relative to their first token (the encoder's input for one slice)
__global__ void rerank_rebase_kernel(const int* __restrict__ cu, int p0, int n, int* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i <= n) out[i] = cu[p0 + i] - cu[p0];
}

// one CTA per query: activation, then the reference's stable descending sort on (score, rrf score) by rank counting
// (rank = #greater + #equal-before), [:limit].  Outputs [nq][limit]: id, rrf score, ce score, bm25_rank, sem_rank
// (-1 = None), rrf_rank (1-based fused position); count [nq].
__global__ void __launch_bounds__(kRrThreads)
rerank_order_kernel(const long long* __restrict__ fid, const double* __restrict__ fsc, const double* __restrict__ fa,
                    const double* __restrict__ fb, const int* __restrict__ fcnt, int W, const int* __restrict__ q_pb,
                    const float* __restrict__ logit, int activation, int limit, long long* __restrict__ o_id,
                    double* __restrict__ o_sc, float* __restrict__ o_ce, int* __restrict__ o_bm25,
                    int* __restrict__ o_sem, int* __restrict__ o_rrf, int* __restrict__ o_cnt) {
  __shared__ float s_ce[kRrThreads];
  __shared__ double s_rrf[kRrThreads];
  const int q = blockIdx.x, j = threadIdx.x;
  int n = fcnt[q];
  n = n < 0 ? 0 : (n > W ? W : n);
  const int64_t o = static_cast<int64_t>(q) * W + j;
  float ce = 0.0f;
  double r = 0.0;
  if (j < n) {
    ce = logit[q_pb[q] + j];
    // GpuCrossEncoder.predict_ids: float32(1 / (1 + exp(-logit))) evaluated in fp64
    if (activation == 1) ce = static_cast<float>(__ddiv_rn(1.0, __dadd_rn(1.0, exp(-static_cast<double>(ce)))));
    r = fsc[o];
  }
  s_ce[j] = ce; s_rrf[j] = r;
  __syncthreads();
  if (j < n) {
    int rank = 0;
    for (int i = 0; i < n; ++i) {
      const float c = s_ce[i];
      const double ri = s_rrf[i];
      rank += (c > ce) || (c == ce && (ri > r || (ri == r && i < j)));
    }
    if (rank < limit) {
      const int64_t w = static_cast<int64_t>(q) * limit + rank;
      o_id[w] = fid[o]; o_sc[w] = r; o_ce[w] = ce;
      o_bm25[w] = static_cast<int>(fa[o]); o_sem[w] = static_cast<int>(fb[o]); o_rrf[w] = j + 1;
    }
  }
  const int n_out = n < limit ? n : limit;
  for (int i = n_out + j; i < limit; i += kRrThreads) {
    const int64_t w = static_cast<int64_t>(q) * limit + i;
    o_id[w] = -1; o_sc[w] = 0.0; o_ce[w] = 0.0f; o_bm25[w] = -1; o_sem[w] = -1; o_rrf[w] = -1;
  }
  if (j == 0) o_cnt[q] = n_out;
}

}  // namespace rse

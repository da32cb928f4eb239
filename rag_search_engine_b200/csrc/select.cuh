// select.cuh — K2/K3/K5: exact top-K' selection under the vec0 emit order, decode,
// and best-chunk-per-movie aggregation.
//
// Replaces sqlite-vec's per-chunk `min_idx` + `merge_sorted_lists` (reached from
// semantic_search.py:254-261), SQLite's `ORDER BY knn.distance` (:262-279) and
// the Python aggregation loop (semantic_search.py:285-317).
//
// Selection is an MSD radix select on the 64-bit key
//   (orderable f32 distance << 32) | (global_pos ^ 1023)
// whose ascending order IS (distance asc, block asc, slot desc).  All keys are
// distinct, so the K' smallest are a unique set and the result is
// deterministic.  The distance array (4 B/row, 0.26 % of the scan's traffic)
// is L2-resident for the passes.  Passes after the distance bits are resolved
// only run when the K'-th distance is tied across rows.
#pragma once
#include "common.cuh"

namespace rse {

constexpr int kSelBins = 2048;
constexpr int kSelThreads = 256;

struct SelState {
  unsigned long long prefix;   // resolved high bits of the K'-th key
  unsigned long long mask;     // which bits are resolved
  unsigned int need;           // how many keys still to take inside the prefix bucket
  unsigned int done;
  unsigned int out_count;
  unsigned int ticket;
  unsigned int total;          // number of keys <= threshold (min(K', valid rows))
  unsigned int pad;
};

__global__ void select_init_kernel(SelState* st, int nq, unsigned int kprime) {
  int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= nq) return;
  SelState s;
  s.prefix = 0ull; s.mask = 0ull; s.need = kprime; s.done = 0u; s.out_count = 0u; s.ticket = 0u;
  s.total = 0u; s.pad = 0u;
  st[q] = s;
}

// The histogram -> digit step of one radix pass, shared by select_pass_kernel (keys derived
// from distances) and select_keys_pass_kernel (stored keys, knn_movies_exact.cuh): merge
// this CTA's histogram h into the query's global one gh, and let the last CTA of the
// query locate the digit holding the `need`-th smallest key.
__device__ __forceinline__ void select_pass_pick(const SelState s, SelState* __restrict__ st, int q,
                                                 unsigned int* __restrict__ h, unsigned int* __restrict__ gh,
                                                 unsigned int* s_part, int* s_last, int shift, unsigned int dmask) {
  for (int i = threadIdx.x; i < kSelBins; i += blockDim.x)
    if (h[i]) atomicAdd(&gh[i], h[i]);
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned int t = atomicAdd(&st[q].ticket, 1u);
    *s_last = (t == gridDim.x - 1);
  }
  __syncthreads();
  if (!*s_last) return;
  __threadfence();

  // ---- last CTA of this query: locate the digit that contains the need-th key
  constexpr int per = kSelBins / kSelThreads;   // 8 consecutive bins per thread
  unsigned int loc[per];
  unsigned int mysum = 0u;
#pragma unroll
  for (int i = 0; i < per; ++i) {
    loc[i] = __ldcg(&gh[threadIdx.x * per + i]);
    mysum += loc[i];
  }
  s_part[threadIdx.x] = mysum;
  __syncthreads();
  // exclusive prefix over 256 partial sums (Hillis-Steele in smem; once per pass)
  for (int off = 1; off < kSelThreads; off <<= 1) {
    unsigned int v = (threadIdx.x >= off) ? s_part[threadIdx.x - off] : 0u;
    __syncthreads();
    s_part[threadIdx.x] += v;
    __syncthreads();
  }
  const unsigned int incl = s_part[threadIdx.x];
  const unsigned int excl = incl - mysum;
  const unsigned int total = s_part[kSelThreads - 1];
  if (total < s.need) {
    // fewer matching keys than requested (only possible before any bit is
    // resolved: fewer valid rows than K') → take everything.
    if (threadIdx.x == 0) {
      st[q].done = 1u; st[q].mask = 0ull; st[q].prefix = 0ull;
      st[q].total = total; st[q].ticket = 0u;
    }
  } else if (excl < s.need && s.need <= incl) {   // exactly one thread owns the crossing
    unsigned int run = excl, below = 0u, in_bucket = 0u;
    int digit = -1;
#pragma unroll
    for (int i = 0; i < per; ++i) {
      if (digit < 0) {
        if (run + loc[i] >= s.need) { digit = threadIdx.x * per + i; below = run; in_bucket = loc[i]; }
        else run += loc[i];
      }
    }
    const unsigned int need2 = s.need - below;
    st[q].prefix = s.prefix | (static_cast<unsigned long long>(digit) << shift);
    st[q].mask = s.mask | (static_cast<unsigned long long>(dmask) << shift);
    st[q].need = need2;
    st[q].ticket = 0u;
    if (in_bucket == need2 || shift == 0) st[q].done = 1u;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < kSelBins; i += blockDim.x) gh[i] = 0u;
}

// One radix pass: histogram the digit [shift, shift+bits) of every key that matches
// the resolved prefix; the last CTA of each query picks the digit holding the
// `need`-th smallest key and refines the state.  `hist` is [nq][kSelBins], zero on
// entry and left zero on exit.
__global__ void __launch_bounds__(kSelThreads)
select_pass_kernel(const uint32_t* __restrict__ dist, int64_t ld, int64_t n_rows, uint64_t pos_base,
                   SelState* __restrict__ st, unsigned int* __restrict__ hist, int shift, int bits) {
  const int q = blockIdx.y;
  __shared__ unsigned int h[kSelBins];
  __shared__ unsigned int s_part[kSelThreads];
  __shared__ int s_last;
  const SelState s = st[q];
  if (s.done) return;
  for (int i = threadIdx.x; i < kSelBins; i += blockDim.x) h[i] = 0u;
  __syncthreads();

  const unsigned int dmask = (1u << bits) - 1u;
  const uint32_t* d = dist + static_cast<int64_t>(q) * ld;   // raw f32 bits: integer-typed so the
  // compiler cannot lower the sign-bit OR to a NaN-canonicalising FADD (it did, see DESIGN.md)
  unsigned int run_digit = 0xFFFFFFFFu, run_cnt = 0u;
  auto visit = [&](uint32_t bits32, int64_t row) {
    const uint32_t okey = f32_orderable(bits32);
    if (okey == kInvalidOKey) return;
    const uint64_t key = knn_key(okey, pos_base + static_cast<uint64_t>(row));
    if ((key & s.mask) != s.prefix) return;
    const unsigned int digit = static_cast<unsigned int>(key >> shift) & dmask;
    if (digit == run_digit) {
      ++run_cnt;
    } else {
      if (run_cnt) atomicAdd(&h[run_digit], run_cnt);
      run_digit = digit; run_cnt = 1u;
    }
  };
  // 128-bit loads, two in flight per thread (ld is a multiple of 32 rows, so d is 16 B aligned)
  const int64_t n4 = n_rows >> 2;
  const uint4* d4 = reinterpret_cast<const uint4*>(d);
  const int64_t gstride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  for (; i + gstride < n4; i += 2 * gstride) {
    const uint4 v0 = __ldcg(d4 + i);
    const uint4 v1 = __ldcg(d4 + i + gstride);
    visit(v0.x, 4 * i); visit(v0.y, 4 * i + 1); visit(v0.z, 4 * i + 2); visit(v0.w, 4 * i + 3);
    const int64_t i1 = i + gstride;
    visit(v1.x, 4 * i1); visit(v1.y, 4 * i1 + 1); visit(v1.z, 4 * i1 + 2); visit(v1.w, 4 * i1 + 3);
  }
  if (i < n4) {
    const uint4 v0 = __ldcg(d4 + i);
    visit(v0.x, 4 * i); visit(v0.y, 4 * i + 1); visit(v0.z, 4 * i + 2); visit(v0.w, 4 * i + 3);
  }
  if (blockIdx.x == 0 && threadIdx.x < (n_rows & 3)) {
    const int64_t row = (n4 << 2) + threadIdx.x;
    visit(__ldcg(d + row), row);
  }
  if (run_cnt) atomicAdd(&h[run_digit], run_cnt);
  __syncthreads();
  select_pass_pick(s, st, q, h, hist + static_cast<int64_t>(q) * kSelBins, s_part, &s_last, shift, dmask);
}

// Gather the selected keys: everything whose resolved bits are <= the threshold prefix.
__global__ void __launch_bounds__(kSelThreads)
select_collect_kernel(const uint32_t* __restrict__ dist, int64_t ld, int64_t n_rows, uint64_t pos_base,
                      SelState* __restrict__ st, unsigned long long* __restrict__ out_keys, int kprime) {
  const int q = blockIdx.y;
  const unsigned long long prefix = st[q].prefix, mask = st[q].mask;
  const uint32_t* d = dist + static_cast<int64_t>(q) * ld;
  auto visit = [&](uint32_t bits32, int64_t row) {
    const uint32_t okey = f32_orderable(bits32);
    if (okey == kInvalidOKey) return;
    const uint64_t key = knn_key(okey, pos_base + static_cast<uint64_t>(row));
    if ((key & mask) <= prefix) {
      unsigned int slot = atomicAdd(&st[q].out_count, 1u);
      if (slot < static_cast<unsigned int>(kprime)) out_keys[static_cast<int64_t>(q) * kprime + slot] = key;
    }
  };
  const int64_t n4 = n_rows >> 2;
  const uint4* d4 = reinterpret_cast<const uint4*>(d);
  const int64_t gstride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  for (; i + gstride < n4; i += 2 * gstride) {
    const uint4 v0 = __ldcg(d4 + i);
    const uint4 v1 = __ldcg(d4 + i + gstride);
    visit(v0.x, 4 * i); visit(v0.y, 4 * i + 1); visit(v0.z, 4 * i + 2); visit(v0.w, 4 * i + 3);
    const int64_t i1 = i + gstride;
    visit(v1.x, 4 * i1); visit(v1.y, 4 * i1 + 1); visit(v1.z, 4 * i1 + 2); visit(v1.w, 4 * i1 + 3);
  }
  if (i < n4) {
    const uint4 v0 = __ldcg(d4 + i);
    visit(v0.x, 4 * i); visit(v0.y, 4 * i + 1); visit(v0.z, 4 * i + 2); visit(v0.w, 4 * i + 3);
  }
  if (blockIdx.x == 0 && threadIdx.x < (n_rows & 3)) {
    const int64_t row = (n4 << 2) + threadIdx.x;
    visit(__ldcg(d + row), row);
  }
}

// Sort the ≤K' selected keys of each query (one CTA per query) and emit packed
// candidates {key, rowid, movie_idx}; unused tail entries get key = ~0.
// smem: keys[kp2] u64 + vals[kp2] u32.
__global__ void __launch_bounds__(kSelThreads)
select_finish_kernel(const unsigned long long* __restrict__ keys_in, const SelState* __restrict__ st,
                     int kprime, int kp2, uint64_t pos_base, const int64_t* __restrict__ rowid,
                     const int32_t* __restrict__ movie_idx, long long* __restrict__ cand) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  unsigned long long* keys = reinterpret_cast<unsigned long long*>(smem_raw);
  unsigned int* vals = reinterpret_cast<unsigned int*>(keys + kp2);
  const int q = blockIdx.x;
  unsigned int n = st[q].out_count;
  if (n > static_cast<unsigned int>(kprime)) n = kprime;
  for (int i = threadIdx.x; i < kp2; i += blockDim.x) {
    keys[i] = (i < static_cast<int>(n)) ? keys_in[static_cast<int64_t>(q) * kprime + i] : ~0ull;
    vals[i] = i;
  }
  block_bitonic_sort(keys, vals, kp2);
  for (int i = threadIdx.x; i < kprime; i += blockDim.x) {
    long long* c = cand + (static_cast<int64_t>(q) * kprime + i) * 3;
    if (i < static_cast<int>(n)) {
      const uint64_t key = keys[i];
      const uint64_t pos = knn_key_pos(key);
      const int64_t local = static_cast<int64_t>(pos - pos_base);
      c[0] = static_cast<long long>(key);
      c[1] = rowid ? rowid[local] : static_cast<long long>(pos);
      c[2] = movie_idx ? movie_idx[local] : -1;
    } else {
      c[0] = -1ll; c[1] = -1ll; c[2] = -1ll;
    }
  }
}

// Merge n_lists candidate lists per query (layout [n_lists][nq][kprime][3]) and keep
// the kprime smallest keys: the row-sharded multi-GPU exchange step (SURVEY §8e).
// smem: keys[n2] u64 + vals[n2] u32, n2 = pow2 >= n_lists*kprime.
__global__ void __launch_bounds__(kSelThreads)
knn_merge_kernel(const long long* __restrict__ gathered, int n_lists, int nq, int kprime, int n2,
                 long long* __restrict__ cand) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  unsigned long long* keys = reinterpret_cast<unsigned long long*>(smem_raw);
  unsigned int* vals = reinterpret_cast<unsigned int*>(keys + n2);
  const int q = blockIdx.x;
  const int n = n_lists * kprime;
  for (int i = threadIdx.x; i < n2; i += blockDim.x) {
    if (i < n) {
      const int l = i / kprime, j = i - l * kprime;
      const long long* c = gathered + ((static_cast<int64_t>(l) * nq + q) * kprime + j) * 3;
      keys[i] = static_cast<unsigned long long>(c[0]);
    } else {
      keys[i] = ~0ull;
    }
    vals[i] = i;
  }
  block_bitonic_sort(keys, vals, n2);
  for (int i = threadIdx.x; i < kprime; i += blockDim.x) {
    long long* o = cand + (static_cast<int64_t>(q) * kprime + i) * 3;
    if (i < n && keys[i] != ~0ull) {
      const int src = vals[i];
      const int l = src / kprime, j = src - l * kprime;
      const long long* c = gathered + ((static_cast<int64_t>(l) * nq + q) * kprime + j) * 3;
      o[0] = c[0]; o[1] = c[1]; o[2] = c[2];
    } else {
      o[0] = -1ll; o[1] = -1ll; o[2] = -1ll;
    }
  }
}

// Unpack candidates to the plain KNN outputs.
__global__ void knn_unpack_kernel(const long long* __restrict__ cand, int nq, int kprime,
                                  float* __restrict__ out_dist, long long* __restrict__ out_pos,
                                  long long* __restrict__ out_rowid, int* __restrict__ out_movie,
                                  int* __restrict__ out_count) {
  const int q = blockIdx.x;
  __shared__ int s_cnt;
  if (threadIdx.x == 0) s_cnt = 0;
  __syncthreads();
  int local = 0;
  for (int i = threadIdx.x; i < kprime; i += blockDim.x) {
    const long long* c = cand + (static_cast<int64_t>(q) * kprime + i) * 3;
    const unsigned long long key = static_cast<unsigned long long>(c[0]);
    const bool ok = key != ~0ull;
    const int64_t o = static_cast<int64_t>(q) * kprime + i;
    out_dist[o] = ok ? __uint_as_float(f32_from_orderable(static_cast<uint32_t>(key >> 32))) : 0.0f;
    if (out_pos) out_pos[o] = ok ? static_cast<long long>(knn_key_pos(key)) : -1ll;
    if (out_rowid) out_rowid[o] = ok ? c[1] : -1ll;
    if (out_movie) out_movie[o] = ok ? static_cast<int>(c[2]) : -1;
    local += ok ? 1 : 0;
  }
  atomicAdd(&s_cnt, local);
  __syncthreads();
  if (threadIdx.x == 0) out_count[q] = s_cnt;
}

// K5: best chunk per movie (semantic_search.py:285-317).  Input rows are already in
// emit order, so "replace only on strictly smaller distance" (:301) never fires
// and the first row of each movie wins; the stable sort by distance (:314-317)
// keeps that order.  Rows whose movie_idx is -1 are the ones the reference's
// inner JOINs (:262-276) drop.  smem: movie[kprime] i32 + keep[kprime] u16-as-int.
__global__ void __launch_bounds__(kSelThreads)
knn_aggregate_kernel(const long long* __restrict__ cand, int nq, int kprime, int k,
                     float* __restrict__ out_dist, long long* __restrict__ out_rowid,
                     int* __restrict__ out_movie, int* __restrict__ out_count) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  int* movie = reinterpret_cast<int*>(smem_raw);
  int* keep = movie + kprime;
  const int q = blockIdx.x;
  const long long* cq = cand + static_cast<int64_t>(q) * kprime * 3;
  for (int i = threadIdx.x; i < kprime; i += blockDim.x) {
    const bool ok = static_cast<unsigned long long>(cq[i * 3]) != ~0ull;
    movie[i] = ok ? static_cast<int>(cq[i * 3 + 2]) : -1;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < kprime; i += blockDim.x) {
    const int m = movie[i];
    int kp = (m >= 0) ? 1 : 0;
    for (int j = 0; j < i && kp; ++j)
      if (movie[j] == m) kp = 0;
    keep[i] = kp;
  }
  __syncthreads();
  // serial compaction by one thread: ≤ K' flags, once per query
  if (threadIdx.x == 0) {
    int n = 0;
    for (int i = 0; i < kprime; ++i) {
      if (keep[i] && n < k) keep[i] = ++n; else keep[i] = 0;
    }
    out_count[q] = n;
  }
  __syncthreads();
  const int n = out_count[q];
  for (int i = threadIdx.x; i < kprime; i += blockDim.x) {
    const int slot = keep[i];
    if (slot >= 1 && slot <= n) {
      const int64_t o = static_cast<int64_t>(q) * k + (slot - 1);
      const unsigned long long key = static_cast<unsigned long long>(cq[i * 3]);
      out_dist[o] = __uint_as_float(f32_from_orderable(static_cast<uint32_t>(key >> 32)));
      out_rowid[o] = cq[i * 3 + 1];
      out_movie[o] = movie[i];
    }
  }
  for (int i = n + threadIdx.x; i < k; i += blockDim.x) {
    const int64_t o = static_cast<int64_t>(q) * k + i;
    out_dist[o] = 0.0f; out_rowid[o] = -1ll; out_movie[o] = -1;
  }
}

}  // namespace rse

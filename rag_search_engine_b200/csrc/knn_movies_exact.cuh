// knn_movies_exact.cuh — exact movie-level KNN: the k nearest movies by best chunk over EVERY row
// (rse_knn_movies_exact, DESIGN §11).
//
// A movie's best chunk is its row with the smallest vec0 key (select.cuh); movies are ordered by that key.  The
// distances come from the exact scan of knn_scan.cuh, unchanged: the scan writes a [QB][n_rows] f32 distance tile
// exactly as it does for rse_knn, so every distance here is the one rse_knn reports for that row, in both FMA modes
// and at every width.  This header adds what comes after the scan:
//   * movies_layout_kernel / movies_layout_join_kernel: once per corpus, whether the rows that compete (valid, and
//     movie_idx >= 0) have non-decreasing movie_idx by position, and n_movie_slots = max(movie_idx) + 1;
//   * movies_segmin_kernel: one pass over the distance tile that folds each movie's run of rows into one key per
//     (query, movie) — a segmented minimum inside each warp, then one 64-bit atomicMin per run and warp, which also
//     joins runs that cross a warp or CTA boundary.  On a corpus whose movie_idx is not sorted, every row does its
//     own atomicMin (RUNS = false): slower, same result;
//   * the movie-level top k: the radix passes of select.cuh over the stored per-movie keys
//     (select_keys_pass_kernel / select_keys_collect_kernel), then select_finish_kernel and knn_unpack_kernel as is.
#pragma once
#include "common.cuh"
#include "select.cuh"

namespace rse {

// The first stage asks rse_knn_movies for the top K' = 10 k chunks (SemanticSearch's default knn_multiplier); it
// runs only when the tensor-core filter serves that K' (K' <= 2048), i.e. for k <= 204 (DESIGN §11).
constexpr int kMoviesExactStageMult = 10;
constexpr int kLayoutRowsPerThread = 4096;
constexpr int kSegThreads = 256;

// One thread per span of kLayoutRowsPerThread rows: the span's first and last competing movie_idx (-1 when it has
// none) and whether it is sorted inside; n_slots (zero on entry) gets max(movie_idx) + 1.  A row competes when its
// squared norm is not the -1 of an empty vec0 slot (amag, knn_row_sqmag_kernel) and its movie_idx is >= 0.
__global__ void movies_layout_kernel(const int32_t* __restrict__ movie_idx, const float* __restrict__ amag,
                                     int64_t n_rows, int n_spans, int4* __restrict__ span,
                                     unsigned int* __restrict__ n_slots) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_spans) return;
  const int64_t r0 = static_cast<int64_t>(s) * kLayoutRowsPerThread;
  const int64_t r1 = min(n_rows, r0 + kLayoutRowsPerThread);
  int first = -1, last = -1, top = -1, sorted = 1;
#pragma unroll 8
  for (int64_t r = r0; r < r1; ++r) {
    const int m = __ldg(movie_idx + r);
    if (m < 0 || __ldg(amag + r) < 0.0f) continue;
    if (first < 0) first = m;
    if (m < last) sorted = 0;
    last = m;
    top = max(top, m);
  }
  span[s] = make_int4(first, last, sorted, 0);
  if (top >= 0) atomicMax(n_slots, static_cast<unsigned int>(top) + 1u);
}

// One thread joins the spans in order: out = 1 when the competing rows are sorted over the whole corpus, else 0.
// Once per loaded corpus: n_rows / 4096 dependent steps.
__global__ void movies_layout_join_kernel(const int4* __restrict__ span, int n_spans, int* __restrict__ out) {
  int sorted = 1, last = -1;
  for (int s = 0; s < n_spans && sorted; ++s) {
    const int4 v = span[s];
    if (v.x < 0) continue;
    if (!v.z || v.x < last) sorted = 0;
    last = v.y;
  }
  *out = sorted;
}

// Fold the distance tile dist[nq][ld] (rows [0, n_rows)) into best[nq][n_slots] (all ones on entry): best[q][m] =
// the smallest key (orderable distance << 32 | pos ^ 1023) among the competing rows of movie m.  Rows the scan marks
// empty (okey = kInvalidOKey) and rows with movie_idx -1 never compete.  grid = (row blocks, nq).
//
// RUNS: a sorted layout puts each movie in a contiguous run, so a warp first folds each run with a segmented
// minimum over its 32 lanes (a lane only ever takes a key of its own movie), and the first lane of each run in the
// warp does the atomicMin.  Rows with movie_idx -1 between two rows of one movie split the run; both pieces still
// reach best[q][m] through the atomic.
template <bool RUNS>
__global__ void __launch_bounds__(kSegThreads)
movies_segmin_kernel(const uint32_t* __restrict__ dist, int64_t ld, int64_t n_rows, uint64_t pos_base,
                     const int32_t* __restrict__ movie_idx, int64_t n_slots, unsigned long long* __restrict__ best) {
  const int q = blockIdx.y;
  const uint32_t* d = dist + static_cast<int64_t>(q) * ld;
  unsigned long long* bq = best + static_cast<int64_t>(q) * n_slots;
  const int lane = threadIdx.x & 31;
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  // every lane of a warp walks the same iterations (the bound is rounded up to whole warps) so the shuffles see
  // the full warp
  const int64_t n_iter = ((n_rows + 31) / 32) * 32;
  for (int64_t r = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; r < n_iter; r += stride) {
    int m = -1;
    unsigned long long key = ~0ull;
    if (r < n_rows) {
      m = __ldg(movie_idx + r);
      const uint32_t okey = f32_orderable(__ldcs(d + r));
      if (m >= 0 && okey != kInvalidOKey) key = knn_key(okey, pos_base + static_cast<uint64_t>(r));
      else m = -1;
    }
    if constexpr (RUNS) {
#pragma unroll
      for (int off = 1; off < 32; off <<= 1) {
        const unsigned long long ok = __shfl_down_sync(0xFFFFFFFFu, key, off);
        const int om = __shfl_down_sync(0xFFFFFFFFu, m, off);
        if (lane + off < 32 && om == m && ok < key) key = ok;
      }
      const int pm = __shfl_up_sync(0xFFFFFFFFu, m, 1);
      if (m >= 0 && (lane == 0 || pm != m)) atomicMin(bq + m, key);
    } else {
      if (m >= 0) atomicMin(bq + m, key);
    }
  }
}

// select_pass_kernel over stored keys keys[q][0..n) (ld apart): an all-ones entry is an empty movie slot.
__global__ void __launch_bounds__(kSelThreads)
select_keys_pass_kernel(const unsigned long long* __restrict__ keys, int64_t ld, int64_t n, SelState* __restrict__ st,
                        unsigned int* __restrict__ hist, int shift, int bits) {
  const int q = blockIdx.y;
  __shared__ unsigned int h[kSelBins];
  __shared__ unsigned int s_part[kSelThreads];
  __shared__ int s_last;
  const SelState s = st[q];
  if (s.done) return;
  for (int i = threadIdx.x; i < kSelBins; i += blockDim.x) h[i] = 0u;
  __syncthreads();
  const unsigned int dmask = (1u << bits) - 1u;
  const unsigned long long* kq = keys + static_cast<int64_t>(q) * ld;
  const int64_t gstride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  // a thread's keys share their high digits (movie keys differ mostly in the low distance bits), so equal digits in
  // a row are counted in a register and added once, as select_pass_kernel does
  unsigned int run_digit = 0xFFFFFFFFu, run_cnt = 0u;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += gstride) {
    const unsigned long long key = __ldcg(kq + i);
    if (key == ~0ull || (key & s.mask) != s.prefix) continue;
    const unsigned int digit = static_cast<unsigned int>(key >> shift) & dmask;
    if (digit == run_digit) {
      ++run_cnt;
    } else {
      if (run_cnt) atomicAdd(&h[run_digit], run_cnt);
      run_digit = digit; run_cnt = 1u;
    }
  }
  if (run_cnt) atomicAdd(&h[run_digit], run_cnt);
  __syncthreads();
  select_pass_pick(s, st, q, h, hist + static_cast<int64_t>(q) * kSelBins, s_part, &s_last, shift, dmask);
}

// select_collect_kernel over stored keys: everything whose resolved bits are <= the threshold prefix.
__global__ void __launch_bounds__(kSelThreads)
select_keys_collect_kernel(const unsigned long long* __restrict__ keys, int64_t ld, int64_t n,
                           SelState* __restrict__ st, unsigned long long* __restrict__ out_keys, int kprime) {
  const int q = blockIdx.y;
  const unsigned long long prefix = st[q].prefix, mask = st[q].mask;
  const unsigned long long* kq = keys + static_cast<int64_t>(q) * ld;
  const int64_t gstride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += gstride) {
    const unsigned long long key = __ldcg(kq + i);
    if (key == ~0ull || (key & mask) > prefix) continue;
    const unsigned int slot = atomicAdd(&st[q].out_count, 1u);
    if (slot < static_cast<unsigned int>(kprime)) out_keys[static_cast<int64_t>(q) * kprime + slot] = key;
  }
}

// Scatter the [n, k] results of the gathered queries back to their rows list[i] of the [nq, k] outputs.
__global__ void movies_scatter_kernel(const float* __restrict__ s_dist, const long long* __restrict__ s_rowid,
                                      const int* __restrict__ s_movie, const int* __restrict__ s_count,
                                      const int* __restrict__ list, int k, float* __restrict__ dist,
                                      long long* __restrict__ rowid, int* __restrict__ movie, int* __restrict__ count) {
  const int64_t src = blockIdx.x, dst = list[blockIdx.x];
  for (int i = threadIdx.x; i < k; i += blockDim.x) {
    dist[dst * k + i] = s_dist[src * k + i];
    rowid[dst * k + i] = s_rowid[src * k + i];
    movie[dst * k + i] = s_movie[src * k + i];
  }
  if (threadIdx.x == 0) count[dst] = s_count[src];
}

}  // namespace rse

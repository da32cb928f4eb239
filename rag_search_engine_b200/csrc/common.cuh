// common.cuh — shared helpers for the sm_100a kernels of librse.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace rse {

constexpr int kVec0Block = 1024;          // sqlite-vec default chunk_size
constexpr uint32_t kInvalidOKey = 0xFFFFFFFFu;

// Monotone map float -> uint32 (ascending float == ascending uint).  The KNN
// orders by the f32 distance first (vec0 stores/compares f32 distances).
__host__ __device__ __forceinline__ uint32_t f32_orderable(uint32_t bits) {
  return (bits & 0x80000000u) ? ~bits : (bits | 0x80000000u);
}
__host__ __device__ __forceinline__ uint32_t f32_from_orderable(uint32_t o) {
  return (o & 0x80000000u) ? (o & 0x7FFFFFFFu) : ~o;
}
// Monotone map double -> uint64.
__host__ __device__ __forceinline__ uint64_t f64_orderable(uint64_t bits) {
  return (bits & 0x8000000000000000ull) ? ~bits : (bits | 0x8000000000000000ull);
}

// vec0 emit order (distance asc, block asc, slot desc) as ONE ascending 64-bit
// key: high word = orderable distance, low word = global position with the slot
// bits inverted (pos ^ 1023)  — SURVEY App. A.2.
__host__ __device__ __forceinline__ uint64_t knn_key(uint32_t okey, uint64_t global_pos) {
  return (static_cast<uint64_t>(okey) << 32) | static_cast<uint32_t>(global_pos ^ (kVec0Block - 1));
}
__host__ __device__ __forceinline__ uint64_t knn_key_pos(uint64_t key) {
  return static_cast<uint32_t>(key) ^ static_cast<uint32_t>(kVec0Block - 1);
}

// In-shared-memory bitonic sort of (key, payload) pairs, ascending by key.
// n must be a power of two; all threads of the block participate.
template <typename K, typename V>
__device__ __forceinline__ void block_bitonic_sort(K* keys, V* vals, int n) {
  for (int size = 2; size <= n; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      __syncthreads();
      for (int t = threadIdx.x; t < (n >> 1); t += blockDim.x) {
        int lo = 2 * t - (t & (stride - 1));
        int hi = lo + stride;
        bool up = ((lo & size) == 0);
        K a = keys[lo], b = keys[hi];
        if ((a > b) == up) {
          keys[lo] = b; keys[hi] = a;
          V va = vals[lo]; vals[lo] = vals[hi]; vals[hi] = va;
        }
      }
    }
  }
  __syncthreads();
}

__host__ __device__ __forceinline__ int next_pow2(int x) {
  int p = 1;
  while (p < x) p <<= 1;
  return p;
}

// 256 threads, 256 histogram bins (one per thread): the digit d with  sum(hist[0..d-1]) < need <= sum(hist[0..d]).
// The thread that owns d writes *out_digit = d and *out_before = sum(hist[0..d-1]); *out_digit stays 256 when
// the histogram holds fewer than `need` entries.  s_warp: 8 words of scratch.  Ends with a barrier.
__device__ __forceinline__ void block_pick_digit(const unsigned int* s_hist, unsigned int need, unsigned int* s_warp,
                                                 unsigned int* out_digit, unsigned int* out_before) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const unsigned int c = s_hist[threadIdx.x];
  unsigned int incl = c;
#pragma unroll
  for (int off = 1; off < 32; off <<= 1) {
    const unsigned int o = __shfl_up_sync(0xFFFFFFFFu, incl, off);
    if (lane >= off) incl += o;
  }
  if (lane == 31) s_warp[warp] = incl;
  if (threadIdx.x == 0) *out_digit = 256u;
  __syncthreads();
  unsigned int base = 0u;
#pragma unroll
  for (int w = 0; w < 8; ++w) base += (w < warp) ? s_warp[w] : 0u;
  incl += base;
  if (incl >= need && incl - c < need) { *out_digit = threadIdx.x; *out_before = incl - c; }
  __syncthreads();
}

}  // namespace rse

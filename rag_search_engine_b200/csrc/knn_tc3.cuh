// knn_tc3.cuh — K4, third mapping: the probe/filter GEMM over an fp16 NORMALISED SHADOW of the corpus.
//
// Same job as knn_tc_kernel (knn_tc.cuh): an approximate cosine for every (row, query) pair whose only
// use is to discard rows that cannot be in the exact top-K'; the rows that survive are re-computed
// with the reference's exact sequential fp32 arithmetic (knn_refine_kernel), so results stay
// bit-identical to K1+K2 (reference call site rag_search_engine/utils/semantic_search.py:254-261).
//
// Why a shadow.  r01 ncu of the TF32 kernels: with 256 queries per pass the TF32 GEMM needs 0.84 ms of
// tensor pipe and 1.13 ms of HBM per pass over S-600k, and the 393 KB fp32 query block does not fit in
// shared memory, so it either re-streams from L2 (knn_tc_kernel: 2x the rows through TMA, 2.1 ms) or
// lives in TMEM as the A operand with tiny N (knn_tc2: 2.9 ms).  The filter does not need fp32 inputs:
//   shadow[r][i] = fp16_rn( a[r][i] / ||a_r|| )      (built once per corpus, 768 B/row)
//   q16[q][i]    = fp16_rn( q[q][i] / ||q|| )
// halves the bytes per pass (768 B/row, nothing else streamed), doubles the tensor rate (kind::f16),
// and the 256 queries (196 KB) now FIT in the shared memory of a CTA pair (98 KB each, the A operand
// of a cta_group::2 UMMA) so they are loaded once per launch.  The accumulator is cos~ directly.
//
// Widths: every kernel here is instantiated for KB = D / 64 = 1..8 k-blocks of 64 halves (D = 64..512; the
// sentence-transformers 384 is KB = 6, CLIP's 512 is KB = 8).  Only the k-loops, the resident-query block (16 KB per
// k-block per CTA: 128 KB at KB = 8, 210,224 B of shared memory in all) and the shadow layout depend on KB; tile,
// UMMA shape, ring, epilogue, probe and survivor queues do not.  768 wide would need 192 KB of resident queries plus
// the ring: more than a CTA may have (a 64-query tile is the way there).
//
// Error bound (eps = kTcEps = 2.5e-3 is kept; the fp16 shadow is TIGHTER than TF32 truncation), for a row width
// D = 64 KB <= 512:
//   |a^_i| <= 1, so fp16_rn has relative error <= 2^-11 above 2^-14 and absolute error <= 2^-25 below;
//   |cos~ - cos| <= (2^-10 + 2^-22) * sum|a^_i q^_i| + 2^-25 * (sum|a^_i| + sum|q^_i|) + D * 2^-23 (truncating adds)
//     sum|a^_i q^_i| <= 1 (Cauchy-Schwarz, unit vectors): 9.77e-4 at every D;
//     sum|a^_i| <= sqrt(D) for a unit vector: 2^-25 * 2 sqrt(D) = 2^-24 sqrt(D) <= 1.35e-6 (384: 1.17e-6);
//     D fp32 adds, truncating: D * 2^-23 <= 6.10e-5 (384: 4.58e-5);
//   together <= 1.04e-3 at D = 512 (1.02e-3 at 384), plus D * 2^-24 <= 3.05e-5 (384: 2.29e-5) for the reference's
//   own fp32 rounding of dot: <= 1.07e-3, less than half of eps at every width K4 serves.
//
// Mapping: cluster of 2 CTAs (one TPC) x 74, persistent over 256-row tiles.
//   UMMA 256x256x16 kind::f16 cta_group::2:  A = the queries (M = 256: 128 per CTA, resident),
//   B = the tile's rows (N = 256: each CTA streams 128 of them), D[128 lanes = queries x 256 columns = rows]
//   f32 per CTA, two D buffers = the 512 TMEM columns.  Lane = query means a thread's threshold lives in
//   a register and "does any of these 32 rows survive" is a 3-input-max tree + one compare: 17
//   instructions per 32 elements (the first version had lane = row, read the 256 thresholds from shared
//   memory and chained 32 dependent FSETPs on one warp per scheduler: 2.0 ms per pass, issue-latency-bound).
//   warp 0   : TMA producer — 4-stage ring of 16 KB k-blocks (128 rows x 64 halves, SWIZZLE_128B), each
//              one contiguous block of the tiled shadow (tc3_shadow_kernel); the loads of BOTH CTAs
//              complete on the leader's mbarrier (cp.async.bulk.tensor...cta_group::2)
//   warp 1   : leader CTA only — single-thread tcgen05.mma issuer; tcgen05.commit multicast frees the
//              stage / publishes the accumulator in both CTAs
//   warps 2-9: epilogue, two warps per TMEM lane quarter (128 columns each) so every scheduler has two
//              warps to alternate between.  A lane that saw a survivor pushes {row, q, cos~} into its
//              warp's shared-memory queue; the queue is flushed with one global atomicAdd per entry
//              issued by 32 lanes IN PARALLEL (global atomics inside the per-lane loop serialised
//              ~1.5 us of latency per survivor).
#pragma once
#include <cuda_fp16.h>

#include "knn_refine.cuh"

namespace rse {

constexpr int kT3TileRows = 256;                          // UMMA M (CTA pair)
constexpr int kT3HalfRows = 128;                          // rows each CTA streams per tile = queries each CTA holds
constexpr int kT3BK = 64;                                 // halves per k-block: one 128-byte swizzle atom
constexpr int kT3MaxKBlocks = 8;                          // KB = D / 64 k-blocks per row, 1..8 (D = 64..512; 384: KB = 6)
constexpr int kT3StageBytes = kT3HalfRows * kT3BK * 2;    // 16,384
constexpr int kT3Stages = 4;                              // 64 KB of rows in flight per SM.  3..7 stages measure the same
                                                          // (0.81-0.85 ms, r01): the pass is not fill-bound, and the
                                                          // smaller footprint (178 KB; 90 registers since the epilogue
                                                          // reads 32 columns at a time) leaves room for ONE BM25 CTA per SM
                                                          // to run underneath it (rse.cu, hybrid step; 896 threads, r02).
                                                          // Room for two (3 stages, r01) was worse: the filter slowed
                                                          // from 0.86 to 0.99 ms and the step from 1.28 to 1.40 ms
constexpr int kT3ProbeTop = 8;                            // MODE 2: sample values kept per thread
constexpr int kT3QueueCap = 128;                          // per-warp survivor queue (entries of 12 B)
constexpr int kT3QueueFlush = 32;                         // flushed to global memory once this full
constexpr int kT3EpiWarps = 8;                            // two per TMEM lane quarter
constexpr int kT3Threads = 64 + 32 * kT3EpiWarps;         // 320
// this CTA's 128 resident queries: KB k-blocks of 16 KB (384 wide: 98,304)
__host__ __device__ constexpr int t3_qbytes(int kb) { return kb * kT3StageBytes; }
// 384 wide: 177,456 B; 512 wide (KB = 8): 210,224 B of the 232,448 a CTA may have
__host__ __device__ constexpr int t3_smem_bytes(int kb) {
  return t3_qbytes(kb) + kT3Stages * kT3StageBytes + kT3EpiWarps * (kT3QueueCap * 12 + 4) + 32 * 8 + 16 + 1024;
}
// kind::f16: D = f32 (bit 4), A = B = f16 (format 0), both K-major, N = 256 rows, M = 256 queries (pair)
constexpr uint32_t kT3Idesc = (1u << 4) | ((kT3TileRows >> 3) << 17) | ((kTcBN >> 4) << 24);

// TMA load whose completion bytes land on an mbarrier of the LEADER CTA (both CTAs of the pair fill
// their own shared memory, one barrier in CTA 0 collects both halves of a stage).
__device__ __forceinline__ void tma_load_2d_2sm(void* smem_dst, const CUtensorMap* tmap, int c0, int c1,
                                                uint32_t leader_bar_addr) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::
          "r"(smem_u32(smem_dst)),
      "l"(tmap), "r"(leader_bar_addr), "r"(c0), "r"(c1)
      : "memory");
}
// The same load with an L2 eviction policy.  The shadow is a read-once 3.7 GB stream through a 126 MB L2 that the
// BM25 kernels of the hybrid step share (their hot posting lists are re-read by many queries of a batch): marked
// evict-first, the stream stops pushing them out.
__device__ __forceinline__ void tma_load_2d_2sm_hint(void* smem_dst, const CUtensorMap* tmap, int c0, int c1,
                                                     uint32_t leader_bar_addr, uint64_t policy) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3, %4}], [%2], %5;" ::"r"(smem_u32(smem_dst)),
      "l"(tmap), "r"(leader_bar_addr), "r"(c0), "r"(c1), "l"(policy)
      : "memory");
}
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ uint32_t map_to_rank(const void* local, uint32_t rank) {
  uint32_t raddr;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(raddr) : "r"(smem_u32(local)), "r"(rank));
  return raddr;
}
__device__ __forceinline__ void tc3_mma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}


// 3-input max (FMNMX3 on sm_100)
__device__ __forceinline__ float fmax3(float a, float b, float c) {
  float d;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
  return d;
}
// remote mbarrier arrive without the cluster-scope release fence of mbar_arrive_remote (knn_tc2.cuh): the
// epilogue's TMEM reads are ordered by tcgen05.fence::before_thread_sync, nothing else is published.
// (r01 ncu: the .release.cluster form lowered to MEMBAR.ALL.GPU + ERRBAR + CGAERRBAR, 9 % of the stall
// samples of the peer CTA's epilogue.)
__device__ __forceinline__ void mbar_arrive_remote_relaxed(uint64_t* local_bar, uint32_t target_rank) {
  uint32_t raddr;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(raddr) : "r"(smem_u32(local_bar)), "r"(target_rank));
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(raddr) : "memory");
}

// Per-warp survivor queue in shared memory (filter epilogue).
struct T3Queue {
  uint32_t* row;      // [kT3QueueCap]
  uint32_t* val;      // [kT3QueueCap] cos~ bits
  uint32_t* qid;      // [kT3QueueCap]
  uint32_t* count;    // [1]
};
__device__ __forceinline__ void t3_emit(uint2* __restrict__ cand_pairs, unsigned int* __restrict__ cand_count, int cap,
                                        uint32_t q, uint32_t row, uint32_t val) {
  const unsigned int slot = atomicAdd(&cand_count[q], 1u);
  if (slot < static_cast<unsigned int>(cap)) cand_pairs[static_cast<int64_t>(q) * cap + slot] = make_uint2(row, val);
}
// all 32 lanes: drain the queue, one entry per lane per round (the global atomics overlap)
__device__ __forceinline__ void t3_flush(const T3Queue& qu, int lane, uint2* __restrict__ cand_pairs,
                                         unsigned int* __restrict__ cand_count, int cap) {
  __syncwarp();
  const uint32_t n = min(*qu.count, static_cast<uint32_t>(kT3QueueCap));
  for (uint32_t i = lane; i < n; i += 32) t3_emit(cand_pairs, cand_count, cap, qu.qid[i], qu.row[i], qu.val[i]);
  __syncwarp();
  if (lane == 0) *qu.count = 0u;
  __syncwarp();
}
// one survivor → the warp's queue (straight to global memory if the queue is full); kept out of line:
// it is called from 32 sites per chunk and must not bloat the hot loop's instruction footprint
__device__ __noinline__ void t3_push(uint32_t* qrow, uint32_t* qcount, uint32_t row, uint32_t val, uint32_t q,
                                     uint2* __restrict__ cand_pairs, unsigned int* __restrict__ cand_count, int cap) {
  const uint32_t pos = atomicAdd(qcount, 1u);
  if (pos < static_cast<uint32_t>(kT3QueueCap)) {
    qrow[pos] = row; qrow[kT3QueueCap + pos] = val; qrow[2 * kT3QueueCap + pos] = q;
  } else {
    t3_emit(cand_pairs, cand_count, cap, q, row, val);
  }
}

// max of a thread's 32 accumulator columns: 16 instructions, depth 4
__device__ __forceinline__ float t3_max32(const uint32_t* v) {
  float m[10];
#pragma unroll
  for (int i = 0; i < 10; ++i)
    m[i] = fmax3(__uint_as_float(v[3 * i]), __uint_as_float(v[3 * i + 1]), __uint_as_float(v[3 * i + 2]));
  const float a = fmax3(m[0], m[1], m[2]), b = fmax3(m[3], m[4], m[5]), c = fmax3(m[6], m[7], m[8]);
  const float d = fmax3(m[9], __uint_as_float(v[30]), __uint_as_float(v[31]));
  return fmaxf(fmax3(a, b, c), d);
}

// One thread (= one query), 32 accumulator columns (= 32 rows): max tree (16 instructions, depth 4) and one
// compare; only when the maximum reaches the threshold is the tree walked back down to the element(s)
// that did (≈ 10 compares for one survivor instead of 32).  Returns whether anything was pushed.
struct T3Sink {
  uint32_t* qrow; uint32_t* qcount; uint32_t q; uint2* cand_pairs; unsigned int* cand_count; int cap;
  __device__ __forceinline__ void push(uint32_t row, uint32_t val) const {
    t3_push(qrow, qcount, row, val, q, cand_pairs, cand_count, cap);
  }
};
__device__ __forceinline__ bool t3_scan32(const uint32_t* v, float thr, uint32_t row0, const T3Sink& sink) {
  float m[10];
#pragma unroll
  for (int i = 0; i < 10; ++i)
    m[i] = fmax3(__uint_as_float(v[3 * i]), __uint_as_float(v[3 * i + 1]), __uint_as_float(v[3 * i + 2]));
  float g[4];
  g[0] = fmax3(m[0], m[1], m[2]); g[1] = fmax3(m[3], m[4], m[5]); g[2] = fmax3(m[6], m[7], m[8]);
  g[3] = fmax3(m[9], __uint_as_float(v[30]), __uint_as_float(v[31]));
  if (!(fmaxf(fmax3(g[0], g[1], g[2]), g[3]) >= thr)) return false;
#pragma unroll
  for (int gi = 0; gi < 4; ++gi) {
    if (g[gi] >= thr) {
#pragma unroll
      for (int ti = 3 * gi; ti < 3 * gi + 3 && ti < 10; ++ti) {
        if (m[ti] >= thr) {
#pragma unroll
          for (int j = 3 * ti; j < 3 * ti + 3; ++j)
            if (__uint_as_float(v[j]) >= thr) sink.push(row0 + static_cast<uint32_t>(j), v[j]);
        }
      }
      if (gi == 3) {
        if (__uint_as_float(v[30]) >= thr) sink.push(row0 + 30u, v[30]);
        if (__uint_as_float(v[31]) >= thr) sink.push(row0 + 31u, v[31]);
      }
    }
  }
  return true;
}

// Probe epilogue: offer a thread's 32 accumulator columns to its running top-8 (sorted descending).  Same max tree
// as t3_scan32 with the list's 8th value as the (moving) threshold: only sub-trees that still hold a candidate are
// walked.  (r01 ran a flat 32-step compare-and-insert loop whenever the group's maximum qualified — and some lane
// of the warp almost always had a candidate, so nearly every group paid 640 instructions: the probe's epilogue was
// as slow as its MMAs.  Offering only the group MAXIMUM instead — any subset of the sample is a valid sample — was
// 3 % faster on isotropic rows and 70 % slower on the clustered corpus: a movie's chunks are adjacent rows, the
// sample's best rows DO share groups, and the weaker bound tripled the survivors.)
__device__ __forceinline__ void t3_top_insert(float (&top)[kT3ProbeTop], float x) {
  top[kT3ProbeTop - 1] = x;
#pragma unroll
  for (int i = kT3ProbeTop - 1; i > 0; --i) {
    const float hi = fmaxf(top[i - 1], top[i]), lo = fminf(top[i - 1], top[i]);
    top[i - 1] = hi; top[i] = lo;
  }
}
__device__ __forceinline__ void t3_probe32(const uint32_t* v, float (&top)[kT3ProbeTop]) {
  float m[10];
#pragma unroll
  for (int i = 0; i < 10; ++i)
    m[i] = fmax3(__uint_as_float(v[3 * i]), __uint_as_float(v[3 * i + 1]), __uint_as_float(v[3 * i + 2]));
  float g[4];
  g[0] = fmax3(m[0], m[1], m[2]); g[1] = fmax3(m[3], m[4], m[5]); g[2] = fmax3(m[6], m[7], m[8]);
  g[3] = fmax3(m[9], __uint_as_float(v[30]), __uint_as_float(v[31]));
  if (!(fmaxf(fmax3(g[0], g[1], g[2]), g[3]) > top[kT3ProbeTop - 1])) return;
#pragma unroll
  for (int gi = 0; gi < 4; ++gi) {
    if (g[gi] > top[kT3ProbeTop - 1]) {
#pragma unroll
      for (int ti = 3 * gi; ti < 3 * gi + 3 && ti < 10; ++ti) {
        if (m[ti] > top[kT3ProbeTop - 1]) {
#pragma unroll
          for (int j = 3 * ti; j < 3 * ti + 3; ++j)
            if (__uint_as_float(v[j]) > top[kT3ProbeTop - 1]) t3_top_insert(top, __uint_as_float(v[j]));
        }
      }
      if (gi == 3) {
        if (__uint_as_float(v[30]) > top[kT3ProbeTop - 1]) t3_top_insert(top, __uint_as_float(v[30]));
        if (__uint_as_float(v[31]) > top[kT3ProbeTop - 1]) t3_top_insert(top, __uint_as_float(v[31]));
      }
    }
  }
}

// two back-to-back 32-column loads, one wait (the register-lean variant of tc_ld128)
__device__ __forceinline__ void tc_ld64(uint32_t taddr, uint32_t (&v)[64]) {
#pragma unroll
  for (int c = 0; c < 2; ++c) {
    uint32_t* w = v + 32 * c;
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
        : "=r"(w[0]), "=r"(w[1]), "=r"(w[2]), "=r"(w[3]), "=r"(w[4]), "=r"(w[5]), "=r"(w[6]), "=r"(w[7]), "=r"(w[8]),
          "=r"(w[9]), "=r"(w[10]), "=r"(w[11]), "=r"(w[12]), "=r"(w[13]), "=r"(w[14]), "=r"(w[15]), "=r"(w[16]),
          "=r"(w[17]), "=r"(w[18]), "=r"(w[19]), "=r"(w[20]), "=r"(w[21]), "=r"(w[22]), "=r"(w[23]), "=r"(w[24]),
          "=r"(w[25]), "=r"(w[26]), "=r"(w[27]), "=r"(w[28]), "=r"(w[29]), "=r"(w[30]), "=r"(w[31])
        : "r"(taddr + static_cast<uint32_t>(32 * c))
        : "memory");
  }
#pragma unroll
  for (int c = 0; c < 2; ++c) {
    uint32_t* w = v + 32 * c;
    asm volatile("tcgen05.wait::ld.sync.aligned;\n"
                 : "+r"(w[0]), "+r"(w[1]), "+r"(w[2]), "+r"(w[3]), "+r"(w[4]), "+r"(w[5]), "+r"(w[6]), "+r"(w[7]),
                   "+r"(w[8]), "+r"(w[9]), "+r"(w[10]), "+r"(w[11]), "+r"(w[12]), "+r"(w[13]), "+r"(w[14]), "+r"(w[15]),
                   "+r"(w[16]), "+r"(w[17]), "+r"(w[18]), "+r"(w[19]), "+r"(w[20]), "+r"(w[21]), "+r"(w[22]), "+r"(w[23]),
                   "+r"(w[24]), "+r"(w[25]), "+r"(w[26]), "+r"(w[27]), "+r"(w[28]), "+r"(w[29]), "+r"(w[30]), "+r"(w[31])
                 :
                 : "memory");
  }
}

// four back-to-back 32-column loads (128 accumulator columns of this thread's lane), one wait
__device__ __forceinline__ void tc_ld128(uint32_t taddr, uint32_t (&v)[128]) {
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    uint32_t* w = v + 32 * c;
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
        : "=r"(w[0]), "=r"(w[1]), "=r"(w[2]), "=r"(w[3]), "=r"(w[4]), "=r"(w[5]), "=r"(w[6]), "=r"(w[7]), "=r"(w[8]),
          "=r"(w[9]), "=r"(w[10]), "=r"(w[11]), "=r"(w[12]), "=r"(w[13]), "=r"(w[14]), "=r"(w[15]), "=r"(w[16]),
          "=r"(w[17]), "=r"(w[18]), "=r"(w[19]), "=r"(w[20]), "=r"(w[21]), "=r"(w[22]), "=r"(w[23]), "=r"(w[24]),
          "=r"(w[25]), "=r"(w[26]), "=r"(w[27]), "=r"(w[28]), "=r"(w[29]), "=r"(w[30]), "=r"(w[31])
        : "r"(taddr + static_cast<uint32_t>(32 * c))
        : "memory");
  }
  // the wait names every destination register so that no use can be scheduled above it
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    uint32_t* w = v + 32 * c;
    asm volatile("tcgen05.wait::ld.sync.aligned;\n"
                 : "+r"(w[0]), "+r"(w[1]), "+r"(w[2]), "+r"(w[3]), "+r"(w[4]), "+r"(w[5]), "+r"(w[6]), "+r"(w[7]),
                   "+r"(w[8]), "+r"(w[9]), "+r"(w[10]), "+r"(w[11]), "+r"(w[12]), "+r"(w[13]), "+r"(w[14]), "+r"(w[15]),
                   "+r"(w[16]), "+r"(w[17]), "+r"(w[18]), "+r"(w[19]), "+r"(w[20]), "+r"(w[21]), "+r"(w[22]), "+r"(w[23]),
                   "+r"(w[24]), "+r"(w[25]), "+r"(w[26]), "+r"(w[27]), "+r"(w[28]), "+r"(w[29]), "+r"(w[30]), "+r"(w[31])
                 :
                 : "memory");
  }
}

// ---------------------------------------------------------------- shadow / query preparation
// One warp per row: shadow row r = fp16_rn(a[r] / ||a_r||) with ||a_r|| = sqrt(amag[r]) (the same sequential
// fp32 sum K1 uses).  Empty vec0 slots (amag < 0) become zero rows.  A zero or non-finite amag makes
// the exact distance NaN, which the bound cannot cover: such rows are counted in *bad and the host
// keeps the whole index on the exact scan (MiniLM embeddings are unit-norm; this is a guard).
//
// Layout: the shadow is private to the probe/filter GEMM, so it is stored the way the GEMM consumes it —
// [row / 128][k-block 0..KB-1][row % 128][64 halves]: every pipeline stage (128 rows x one 128-byte k-block)
// is ONE contiguous 16 KB block of HBM.  (A row-major shadow made each stage 128 separate 128-byte
// pieces 768 B apart; the filter pass then stalled on TMA data at 4.5 TB/s, r01 ncu.)  The buffer is
// padded with zero rows to a multiple of 256 rows.
// A warp converts 128 floats (32 float4) per step; at D = 64, 192, 320 and 448 (KB odd) the last step is a half
// step: lanes 0..15 hold its 16 float4.
template <int KB>
__device__ __forceinline__ int64_t t3_shadow_offset(int64_t row, int kb) {      // in halves
  return (((row >> 7) * KB + kb) * kT3HalfRows + (row & 127)) * kT3BK;
}
template <int KB>
__device__ __forceinline__ void t3_shadow_row(const float* __restrict__ emb, const float* __restrict__ amag, int64_t r,
                                              int lane, __half* __restrict__ shadow, unsigned int* __restrict__ bad) {
  const float am = __ldg(amag + r);
  float inv = 0.0f;
  if (am > 0.0f && am < __int_as_float(0x7F800000)) inv = static_cast<float>(1.0 / sqrt(static_cast<double>(am)));
  else if (!(am < 0.0f) && lane == 0) atomicAdd(bad, 1u);              // 0, +inf or NaN
  const float4* src = reinterpret_cast<const float4*>(emb + r * (KB * kT3BK));
#pragma unroll
  for (int j = 0; j < (KB + 1) / 2; ++j) {
    if (KB % 2 != 0 && j == KB / 2 && lane >= 16) break;                // the half step
    const int f4 = j * 32 + lane;                                       // float4 index inside the row: 0..16 KB - 1
    const float4 f = __ldg(src + f4);
    const __half2 lo = __floats2half2_rn(__fmul_rn(f.x, inv), __fmul_rn(f.y, inv));
    const __half2 hi = __floats2half2_rn(__fmul_rn(f.z, inv), __fmul_rn(f.w, inv));
    uint2 o;
    o.x = *reinterpret_cast<const uint32_t*>(&lo);
    o.y = *reinterpret_cast<const uint32_t*>(&hi);
    const int kb = f4 >> 4, within = f4 & 15;                           // 16 float4 (= 64 halves) per k-block
    reinterpret_cast<uint2*>(shadow + t3_shadow_offset<KB>(r, kb))[within] = o;
  }
}
template <int KB>
__global__ void __launch_bounds__(256)
tc3_shadow_kernel(const float* __restrict__ emb, const float* __restrict__ amag, int64_t n_rows,
                  __half* __restrict__ shadow, unsigned int* __restrict__ bad) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = (static_cast<int64_t>(gridDim.x) * blockDim.x) >> 5;
  if (KB == 2) {
#pragma unroll 1                                                        // (unrolled, this loop spills at KB = 2)
    for (int64_t r = warp0; r < n_rows; r += n_warps) t3_shadow_row<KB>(emb, amag, r, lane, shadow, bad);
  } else {
    for (int64_t r = warp0; r < n_rows; r += n_warps) t3_shadow_row<KB>(emb, amag, r, lane, shadow, bad);
  }
}

// The probe's SAMPLE (r02): sample row i is one row of the group [i*stride, (i+1)*stride) of corpus rows, at a
// hashed offset that depends on i only — a stratified sample, independent of the data, stored as its own small
// shadow in the same tiled layout (n_rows / stride rows, zero-padded to whole tiles).  Because the choice is
// independent of the data, the number X of sample rows among ANY K' rows (the exact top-K' of a query) is a sum of
// independent Bernoulli draws with mean K'/stride, whose upper tail is bounded by Binomial(K', 1/stride)
// (Hoeffding 1956).  rse.cu turns that into the probe's order statistic; the result is VERIFIED in the refine
// kernel, so the tail only costs a second filter pass, never a wrong answer.
__device__ __forceinline__ int64_t t3_sample_source(int64_t i, int stride, int64_t n_rows) {
  uint32_t x = static_cast<uint32_t>(i) * 0x9E3779B1u;
  x ^= x >> 15; x *= 0x85EBCA77u; x ^= x >> 13; x *= 0xC2B2AE3Du; x ^= x >> 16;
  const int64_t g = i * stride;
  const int64_t gs = n_rows - g < stride ? n_rows - g : stride;
  return g + static_cast<int64_t>(x % static_cast<uint32_t>(gs));
}
template <int KB>
__global__ void __launch_bounds__(256)
tc3_sample_kernel(const float* __restrict__ emb, const float* __restrict__ amag, int64_t n_rows, int stride,
                  int64_t n_sample, __half* __restrict__ sample) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = (static_cast<int64_t>(gridDim.x) * blockDim.x) >> 5;
  for (int64_t i = warp0; i < n_sample; i += n_warps) {
    const int64_t r = t3_sample_source(i, stride, n_rows);
    const float am = __ldg(amag + r);
    float inv = 0.0f;                                                    // empty slots stay zero rows
    if (am > 0.0f && am < __int_as_float(0x7F800000)) inv = static_cast<float>(1.0 / sqrt(static_cast<double>(am)));
    const float4* src = reinterpret_cast<const float4*>(emb + r * (KB * kT3BK));
#pragma unroll
    for (int j = 0; j < (KB + 1) / 2; ++j) {
      if (KB % 2 != 0 && j == KB / 2 && lane >= 16) break;              // the half step
      const int f4 = j * 32 + lane;
      const float4 f = __ldg(src + f4);
      const __half2 lo = __floats2half2_rn(__fmul_rn(f.x, inv), __fmul_rn(f.y, inv));
      const __half2 hi = __floats2half2_rn(__fmul_rn(f.z, inv), __fmul_rn(f.w, inv));
      uint2 o;
      o.x = *reinterpret_cast<const uint32_t*>(&lo);
      o.y = *reinterpret_cast<const uint32_t*>(&hi);
      const int kb = f4 >> 4, within = f4 & 15;
      reinterpret_cast<uint2*>(sample + t3_shadow_offset<KB>(i, kb))[within] = o;
    }
  }
}

// q16[q] = fp16_rn(q / ||q||) for q < nq (||q|| = sb[q], the K1 factor), zero rows for the padding and
// for queries whose norm is zero / non-finite (those get thr = +inf and are re-run exactly).  One thread per float4:
// 16 KB threads per query (384 wide: 96).
template <int KB>
__global__ void __launch_bounds__(16 * KB)
tc3_query_prep_kernel(const float* __restrict__ q, const double* __restrict__ sb, int nq, __half* __restrict__ q16) {
  const int qi = blockIdx.x;
  float inv = 0.0f;
  if (qi < nq) {
    const double s = sb[qi];
    if (s > 0.0 && s < 1e300) inv = static_cast<float>(1.0 / s);
  }
  float4 f = make_float4(0.f, 0.f, 0.f, 0.f);
  if (qi < nq) f = __ldg(reinterpret_cast<const float4*>(q + static_cast<int64_t>(qi) * (KB * kT3BK)) + threadIdx.x);
  const __half2 lo = __floats2half2_rn(__fmul_rn(f.x, inv), __fmul_rn(f.y, inv));
  const __half2 hi = __floats2half2_rn(__fmul_rn(f.z, inv), __fmul_rn(f.w, inv));
  uint2 o;
  o.x = *reinterpret_cast<const uint32_t*>(&lo);
  o.y = *reinterpret_cast<const uint32_t*>(&hi);
  reinterpret_cast<uint2*>(q16 + static_cast<int64_t>(qi) * (KB * kT3BK))[threadIdx.x] = o;
}

// thr[q] = 1 - tau_s - 2 eps (compared against cos~); +inf — nothing survives, the refine step then hands
// the query to the exact scan — for padding queries, unusable norms, a sample without K' rows, and a
// bound that is not positive (the filter relies on thr > 0: zero rows of the shadow never pass, and a
// query that would keep half the corpus overflows its survivor list anyway).
__global__ void tc3_threshold_kernel(const SelState* __restrict__ st, const double* __restrict__ sb, int nq,
                                     float* __restrict__ thr) {
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= kTcBN) return;
  float t = __int_as_float(0x7F800000);
  if (q < nq && sb[q] > 0.0 && sb[q] < 1e300) {
    const SelState s = st[q];
    const unsigned long long hi_mask = s.mask >> 32, hi_pref = s.prefix >> 32;
    if (s.mask != 0ull) {
      const uint32_t okey = static_cast<uint32_t>(hi_pref | (~hi_mask & 0xFFFFFFFFull));
      const float tau = __uint_as_float(f32_from_orderable(okey));
      const float cut = 1.0f - tau - 2.0f * kTcEps - 1e-6f;
      if (cut > 1e-6f) t = cut;
    }
  }
  thr[q] = t;
}

// Sparse probe → thresholds in one launch: one CTA per query finds the K'-th smallest of its <= 2048 probe
// values (MSD radix select, 4 x 8 bits, in shared memory) and writes thr[q] like tc3_threshold_kernel.
// (select_init + three select passes + the threshold kernel were five launches and 35 us for 1184 values.)
constexpr int kT3SelMax = 2048;
__global__ void __launch_bounds__(256)
tc3_probe_threshold_kernel(const uint32_t* __restrict__ dist, int64_t ld, int nq, int kprime,
                           const double* __restrict__ sb, float* __restrict__ thr, float* __restrict__ tver) {
  __shared__ uint32_t s_key[kT3SelMax];
  __shared__ unsigned int s_hist[256];
  __shared__ unsigned int s_prefix, s_need, s_fail, s_digit, s_before;
  __shared__ unsigned int s_warp[8];
  const int q = blockIdx.x;                        // grid = the padded query count (a multiple of 256)
  const float inf = __int_as_float(0x7F800000);
  if (q >= nq || !(sb[q] > 0.0 && sb[q] < 1e300)) {
    if (threadIdx.x == 0) { thr[q] = inf; if (tver) tver[q] = inf; }
    return;
  }
  const int n = static_cast<int>(ld);
  for (int i = threadIdx.x; i < n; i += blockDim.x) s_key[i] = f32_orderable(dist[static_cast<int64_t>(q) * ld + i]);
  if (threadIdx.x == 0) { s_prefix = 0u; s_need = static_cast<unsigned int>(kprime); s_fail = n < kprime ? 1u : 0u; }
  __syncthreads();
  uint32_t resolved = 0u;
  for (int pass = 0; pass < 4 && s_fail == 0u; ++pass) {
    const int shift = 24 - 8 * pass;
    s_hist[threadIdx.x] = 0u;
    __syncthreads();
    const uint32_t prefix = s_prefix;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
      const uint32_t key = s_key[i];
      if ((key & resolved) == prefix) atomicAdd(&s_hist[(key >> shift) & 0xFFu], 1u);
    }
    __syncthreads();
    block_pick_digit(s_hist, s_need, s_warp, &s_digit, &s_before);
    if (threadIdx.x == 0) {
      s_prefix = prefix | ((s_digit & 0xFFu) << shift);
      s_need = s_need - s_before;
    }
    resolved |= 0xFFu << shift;
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    float t = inf;
    if (s_fail == 0u) {
      const float tau = __uint_as_float(f32_from_orderable(s_prefix));   // K'-th smallest d~ (NaN if it is a sentinel)
      const float cut = 1.0f - tau - 2.0f * kTcEps - 1e-6f;
      if (cut > 1e-6f) t = cut;
      // the un-banded bound the refine kernel verifies (sample path: kprime here is the probe's order statistic j,
      // and "the K'-th largest cos~ of the survivors >= 1 - tau" is what makes the cut valid)
      if (tver) tver[q] = cut > 1e-6f ? 1.0f - tau : inf;
    } else if (tver) {
      tver[q] = inf;
    }
    thr[q] = t;
  }
}

// ---------------------------------------------------------------- the GEMM
// MODE 0 (probe) : tiles t = 0..n_tiles-1 map to the 256-row tile t*tile_stride; d~ = 1 - cos~ is stored to
//                  dist[q*ld + t*256 + r].  Empty slots / rows past the end are zero rows of the shadow:
//                  they read d~ = 1, which can only matter when tau_s >= 1 - 2 eps — and then the query is
//                  handed to the exact scan anyway (tc3_threshold_kernel).
// MODE 2 (probe, K' <= 256): same tiles as MODE 0, but nothing dense is stored: every epilogue thread keeps the
//                  8 largest cos~ of the (query, rows) pairs it sees in registers and writes them at the end —
//                  dist[q*ld + (cluster*2 + half)*8 + i], ld = n_clusters*16.  The K'-th smallest d~ of that
//                  union is the K'-th smallest of a SUBSET of the sample: still an upper bound of the K'-th
//                  exact distance (+eps), and equal to the dense answer unless one thread holds more than 8 of
//                  the sample's best K' (148 threads share them).  The dense probe wrote 182 MB per 256-query
//                  batch and its three radix-select passes cost 0.19 ms; this one writes 1.2 MB.
// MODE 1 (filter): all tiles; survivors appended to cand_pairs[q*cap + slot] = {local row, cos~}.  thr > 0
//                  for every query (or +inf), so zero rows never survive.
// QUERY BLOCKS (r02): one launch serves n_qblocks blocks of 256 queries — q16 / thr / dist / cand_* are indexed by
//                  the global query qb*256 + q.  The CTA pair loops over the blocks: the producer reloads the
//                  resident queries once the MMAs of the previous block have retired (qfree, a multicast commit),
//                  the tile ring, the two accumulator buffers and their phases simply run on.  (r01 launched the
//                  whole probe / threshold / filter / refine chain once per block from a host loop: a 2048-query
//                  step on a shard was 40 launches, each paying launch latency, TMEM allocation and the pipeline
//                  fill of a 0.1 ms pass.)  MODE 0 is only used with one block.
// gate (MODE 1, second-chance pass): gate[qb] == 0 -> block qb is skipped by every role; all zero -> the kernel
//                  returns before any barrier / TMEM allocation (enqueued unconditionally, rse.cu).
// KB = D / 64: k-blocks per row and per resident query (every k-loop, the resident-query block and the shadow layout).
// grid = 2 * n_clusters (<= 148), cluster = 2.
template <int MODE, int KB>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kT3Threads, 1)
knn_tc3_kernel(const __grid_constant__ CUtensorMap tmap_rows, const __grid_constant__ CUtensorMap tmap_q,
               int64_t n_tiles, int64_t tile_stride, int nq, int n_qblocks, const float* __restrict__ thr,
               uint32_t* __restrict__ dist, int64_t ld, uint2* __restrict__ cand_pairs,
               unsigned int* __restrict__ cand_count, int cap, const unsigned int* __restrict__ gate) {
  static_assert(KB >= 1 && KB <= kT3MaxKBlocks, "knn_tc3: 64 to 512 halves per row");
  static_assert(t3_smem_bytes(KB) <= 232448, "knn_tc3: shared memory budget");
  constexpr int kT3KBlocks = KB;
  constexpr int kT3QBytes = t3_qbytes(KB);
  if (gate != nullptr) {
    bool any = false;
    for (int b = 0; b < n_qblocks; ++b) any |= gate[b] != 0u;
    if (!any) return;                              // uniform over the grid
  }
  extern __shared__ unsigned char smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  unsigned char* smem = smem_raw + (base - smem_u32(smem_raw));
  unsigned char* ring = smem + kT3QBytes;
  uint32_t* s_queue = reinterpret_cast<uint32_t*>(ring + kT3Stages * kT3StageBytes);   // [8 warps][3][cap] + [8] counts
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_queue + kT3EpiWarps * 3 * kT3QueueCap + kT3EpiWarps);
  uint64_t* full = bars;                          // [S] leader: both CTAs' halves of the stage landed
  uint64_t* empty = bars + kT3Stages;             // [S] both CTAs: the MMAs reading the stage retired
  uint64_t* tfull = bars + 2 * kT3Stages;         // [2] both CTAs: accumulator buffer complete
  uint64_t* tempty = bars + 2 * kT3Stages + 2;    // [2] leader: both CTAs' epilogues drained the buffer
  uint64_t* qfull = bars + 2 * kT3Stages + 4;     // [1] leader: both CTAs' query halves landed
  uint64_t* qfree = bars + 2 * kT3Stages + 5;     // [1] both CTAs: the MMAs that read the resident queries retired
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kT3Stages + 6);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int64_t cluster_id = blockIdx.x >> 1;
  const int64_t n_clusters = gridDim.x >> 1;

  if (threadIdx.x < kT3EpiWarps) s_queue[kT3EpiWarps * 3 * kT3QueueCap + threadIdx.x] = 0u;
  if (threadIdx.x == 0) {
    for (int s = 0; s < kT3Stages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(&tfull[b], 1); mbar_init(&tempty[b], 2 * kT3EpiWarps); }
    mbar_init(qfull, 1);
    mbar_init(qfree, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"(512u)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();                              // barriers of both CTAs initialised before any remote use
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===================== TMA producer (both CTAs) =====================
    if (lane == 0) {
      asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_rows) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_q) : "memory");
      const uint32_t lq = map_to_rank(qfull, 0u);
      const uint64_t stream_policy = l2_policy_evict_first();
      int stage = 0;
      uint32_t phase = 0;
      uint32_t nb = 0;                             // query blocks processed so far (skipped ones do not count)
      // (An L2 prefetch 6-18 stages ahead of the fill — cp.async.bulk.prefetch.tensor — changed nothing:
      // with every MMA but one per stage removed the same ring streams at 7.4 TB/s; the pass is bound by
      // the tensor pipe + TMEM reads, not by the fill.  r01 experiments, DESIGN.md §5.)
      const int64_t my_tiles = (n_tiles - cluster_id + n_clusters - 1) / n_clusters;
      const int64_t my_stages = my_tiles * kT3KBlocks;
      for (int qb = 0; qb < n_qblocks; ++qb) {
        if (gate != nullptr && gate[qb] == 0u) continue;
        // my 128 queries of this block (the previous block's MMAs must have retired: they read this memory)
        if (nb > 0) mbar_wait(qfree, (nb - 1u) & 1u);
        if (leader) mbar_arrive_expect_tx(qfull, 2 * kT3QBytes);
#pragma unroll
        for (int kb = 0; kb < kT3KBlocks; ++kb)
          tma_load_2d_2sm(smem + kb * kT3StageBytes, &tmap_q, kb * kT3BK,
                          qb * kTcBN + static_cast<int>(rank) * kT3HalfRows, lq);
        for (int64_t g = 0; g < my_stages; ++g) {
          // my 128 rows of the tile = 6 contiguous 16 KB blocks of the tiled shadow (one per k-block)
          const int64_t t = cluster_id + (g / kT3KBlocks) * n_clusters;
          const int line = static_cast<int>(((t * tile_stride * 2 + rank) * kT3KBlocks + g % kT3KBlocks) * kT3HalfRows);
          mbar_wait(&empty[stage], phase ^ 1u);
          if (leader) mbar_arrive_expect_tx(&full[stage], 2 * kT3StageBytes);
          tma_load_2d_2sm_hint(ring + stage * kT3StageBytes, &tmap_rows, 0, line, map_to_rank(&full[stage], 0u), stream_policy);
          if (++stage == kT3Stages) { stage = 0; phase ^= 1u; }
        }
        ++nb;
      }
    }
    __syncwarp();                                  // reconverge before the aligned cluster barrier below
  } else if (warp == 1) {
    // ===================== MMA issuer (leader CTA only) =====================
    if (lane == 0 && leader) {
      int stage = 0;
      uint32_t phase = 0;
      uint32_t it = 0, nb = 0;
      for (int qb = 0; qb < n_qblocks; ++qb) {
        if (gate != nullptr && gate[qb] == 0u) continue;
        mbar_wait(qfull, nb & 1u);
        tc_fence_after();
        for (int64_t t = cluster_id; t < n_tiles; t += n_clusters, ++it) {
          const uint32_t buf = it & 1u, use = it >> 1;
          mbar_wait(&tempty[buf], (use & 1u) ^ 1u);  // both epilogues drained this buffer
          tc_fence_after();
          const uint32_t d_addr = tmem_base + buf * kT3TileRows;
          for (int kb = 0; kb < kT3KBlocks; ++kb) {
            mbar_wait(&full[stage], phase);
            tc_fence_after();
            const uint64_t adesc = tc_smem_desc(base + kb * kT3StageBytes);                      // queries
            const uint64_t bdesc = tc_smem_desc(base + kT3QBytes + stage * kT3StageBytes);       // rows
#pragma unroll
            for (int k = 0; k < kT3BK / 16; ++k) {
              // advance 16 halves = 32 B inside the swizzle atom: +2 in the (>>4) start-address field
              tc3_mma_f16(d_addr, adesc + static_cast<uint64_t>(2 * k), bdesc + static_cast<uint64_t>(2 * k), kT3Idesc,
                          (kb | k) != 0 ? 1u : 0u);
            }
            tc2_commit_mc(&empty[stage]);            // both CTAs may refill this stage
            if (++stage == kT3Stages) { stage = 0; phase ^= 1u; }
          }
          tc2_commit_mc(&tfull[buf]);                // accumulator complete in both CTAs
        }
        tc2_commit_mc(qfree);                        // every MMA that reads this block's queries has been issued: the
        ++nb;                                        // barrier flips in both CTAs when they retire
      }
    }
    __syncwarp();
  } else {
    // ===================== epilogue (warps 2..9): one thread = one query, 128 of the tile's 256 rows =====================
    const int ew = warp - 2;                       // 0..7
    const int quarter = warp & 3;                  // TMEM lanes [32*quarter, +32) belong to this warp
    const int col_half = ew >> 2;                  // which 128 columns (rows of the tile)
    const int qi0 = static_cast<int>(rank) * kT3HalfRows + quarter * 32 + lane;   // my query inside a block
    uint32_t* qrow = s_queue + ew * 3 * kT3QueueCap;
    uint32_t* qcount = s_queue + kT3EpiWarps * 3 * kT3QueueCap + ew;
    T3Queue qu;
    qu.row = qrow; qu.val = qrow + kT3QueueCap; qu.qid = qrow + 2 * kT3QueueCap; qu.count = qcount;
    uint32_t it = 0;
    for (int qb = 0; qb < n_qblocks; ++qb) {
    if (gate != nullptr && gate[qb] == 0u) continue;
    const int qi = qb * kTcBN + qi0;               // global query
    const float my_thr = (MODE == 1) ? __ldg(thr + qi) : 0.0f;
    const T3Sink sink{qrow, qcount, static_cast<uint32_t>(qi), cand_pairs, cand_count, cap};
    float top[kT3ProbeTop];
#pragma unroll
    for (int i = 0; i < kT3ProbeTop; ++i) top[i] = -3.0f;                    // below any cosine
    for (int64_t t = cluster_id; t < n_tiles; t += n_clusters, ++it) {
      const uint32_t buf = it & 1u, use = it >> 1;
      mbar_wait(&tfull[buf], use & 1u);
      tc_fence_after();
      const uint32_t taddr0 = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + buf * kT3TileRows +
                              static_cast<uint32_t>(col_half * 128);
      if (MODE == 0) {
        // d~ of the sample: 32 consecutive rows per thread per load, written as 8 x 16 B
        uint32_t* drow = dist + static_cast<int64_t>(qi) * ld + t * kT3TileRows + col_half * 128;
#pragma unroll 1
        for (int c0 = 0; c0 < 128; c0 += 32) {
          uint32_t v[32];
          tc_ld32(taddr0 + static_cast<uint32_t>(c0), v);
          if (qi < nq) {
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              uint4 o;
              o.x = __float_as_uint(1.0f - __uint_as_float(v[j + 0]));
              o.y = __float_as_uint(1.0f - __uint_as_float(v[j + 1]));
              o.z = __float_as_uint(1.0f - __uint_as_float(v[j + 2]));
              o.w = __float_as_uint(1.0f - __uint_as_float(v[j + 3]));
              *reinterpret_cast<uint4*>(drow + c0 + j) = o;
            }
          }
        }
      } else if (MODE == 2) {
        // running top-8 of this thread's share of the sample (registers, sorted descending)
#pragma unroll 1
        for (int c = 0; c < 4; ++c) {
          uint32_t v[32];
          tc_ld32(taddr0 + static_cast<uint32_t>(32 * c), v);
          t3_probe32(v, top);
        }
      } else {
        const uint32_t row_base = static_cast<uint32_t>(t * kT3TileRows + col_half * 128);
        bool pushed = false;                       // rare per lane: ≈ K'·stride + band survivors per query per pass
#pragma unroll 1
        for (int hcol = 0; hcol < 128; hcol += 32) {     // 32 columns per tcgen05.ld: 90 registers (64: 118, 128: 168), same
          uint32_t v[32];                                // speed — and 96 allocated registers are what lets a 28-warp BM25
          tc_ld32(taddr0 + static_cast<uint32_t>(hcol), v);   // CTA share the SM (bm25.cuh, bm25_fx_kernel)
          pushed |= t3_scan32(v, my_thr, row_base + static_cast<uint32_t>(hcol), sink);
        }
        if (__any_sync(0xFFFFFFFFu, pushed)) {
          __syncwarp();
          if (*qcount >= static_cast<uint32_t>(kT3QueueFlush)) t3_flush(qu, lane, cand_pairs, cand_count, cap);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (leader) mbar_arrive(&tempty[buf]); else mbar_arrive_remote_relaxed(&tempty[buf], 0u);
      }
    }
    if (MODE == 1) t3_flush(qu, lane, cand_pairs, cand_count, cap);
    if (MODE == 2 && qi < nq) {
      // d~ of this thread's best 8 sample rows; unused slots carry the invalid sentinel
      uint32_t* o = dist + static_cast<int64_t>(qi) * ld + (cluster_id * 2 + col_half) * kT3ProbeTop;
#pragma unroll
      for (int i = 0; i < kT3ProbeTop; ++i)
        o[i] = top[i] > -2.0f ? __float_as_uint(1.0f - top[i]) : 0x7FFFFFFFu;
    }
    }                                              // query blocks
  }

  tc_fence_before();
  cluster_sync_all();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
  }
}

}  // namespace rse

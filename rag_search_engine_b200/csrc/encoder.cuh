// encoder.cuh — §8(f2)/(f3): the BERT-family text encoders of the reference on the same GPU as the index.
//
//   head 0: SentenceTransformer("all-MiniLM-L6-v2") — the QUERY ENCODER of the semantic path
//           (rag_search_engine/utils/semantic_search.py:45, :211-222): BertModel (6 layers, hidden 384, 12 heads,
//           intermediate 1536) -> mean pooling over the attention mask -> L2 normalise;
//   head 1: CrossEncoder("cross-encoder/ms-marco-TinyBERT-L2-v2") — the rerank step right after fusion
//           (rag_search_engine/utils/hybrid_search.py:279-312): BertModel (2 layers, hidden 128, 2 heads,
//           intermediate 512) -> BERT pooler (tanh(dense([CLS]))) -> linear classifier -> one logit per pair.
//
// Both are the same graph with different sizes, so there is ONE implementation, driven by a config.  The model is
// the HuggingFace BertModel: embeddings (word + position + token type) -> LayerNorm; per layer: fused QKV
// projection, scaled-dot-product attention with a key padding mask, output projection + residual + LayerNorm,
// GELU(erf) feed-forward + residual + LayerNorm.
//
// Numerics.  The bar for this row is the fp32 PyTorch model to <= 1e-5 relative on the pooled vector, so every
// matrix product accumulates in fp32 with fused multiply-adds (fmaf, explicit: the library is built with
// --fmad=false), softmax / LayerNorm / GELU are fp32 with expf / erff / rsqrtf-free sqrt, and nothing is stored
// in reduced precision.  A TF32 tensor-core GEMM would be ~1e-3 off and fail that bar; the tcgen05 route to fp32
// accuracy is a 3-pass split (hi*hi + lo*hi + hi*lo), see DESIGN.md §10.
//
// Layout: PACKED tokens — the sequences of a batch are concatenated, [T, hidden] row-major, with cu_seqlens
// [n_seq + 1] (queries are 3-20 tokens: padding to the longest would waste half the GEMM rows); position ids are
// the index inside the sequence; attention and pooling work per sequence from cu_seqlens.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>

#include "tc_common.cuh"

namespace rse {

constexpr int kEncMaxHidden = 1024;

// tf32 split of an fp32 value (see the tensor-core GEMM at the end of this file): hi = tf32(x), lo = tf32(x - hi)
__device__ __forceinline__ float tf32_rna(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}
__device__ __forceinline__ void tf32_split(float x, float& hi, float& lo) {
  hi = tf32_rna(x);
  lo = tf32_rna(x - hi);                                        // x - hi is exact in fp32
}

// ---------------------------------------------------------------- embeddings + LayerNorm / residual + LayerNorm
// one warp per token; two-pass mean / variance in registers (torch.nn.LayerNorm: biased variance, eps inside sqrt)
template <int MAX_PER_LANE>
__device__ __forceinline__ void warp_layernorm(float (&v)[MAX_PER_LANE], int per_lane, int hidden, float eps,
                                               const float* __restrict__ gamma, const float* __restrict__ beta,
                                               float* __restrict__ out_row, int lane,
                                               float* __restrict__ hi_row = nullptr, float* __restrict__ lo_row = nullptr) {
  float s = 0.0f;
#pragma unroll
  for (int i = 0; i < MAX_PER_LANE; ++i) if (i < per_lane) s += v[i];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xFFFFFFFFu, s, o);
  const float mean = s / static_cast<float>(hidden);
  float q = 0.0f;
#pragma unroll
  for (int i = 0; i < MAX_PER_LANE; ++i) if (i < per_lane) { const float d = v[i] - mean; q = fmaf(d, d, q); }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xFFFFFFFFu, q, o);
  const float rstd = 1.0f / sqrtf(q / static_cast<float>(hidden) + eps);
#pragma unroll
  for (int i = 0; i < MAX_PER_LANE; ++i)
    if (i < per_lane) {
      const int c = i * 32 + lane;
      const float y = fmaf((v[i] - mean) * rstd, gamma[c], beta[c]);
      out_row[c] = y;
      if (hi_row) { float h, l; tf32_split(y, h, l); hi_row[c] = h; lo_row[c] = l; }
    }
}

__global__ void __launch_bounds__(128)
enc_embed_ln_kernel(const int32_t* __restrict__ ids, const int32_t* __restrict__ type_ids,
                    const int32_t* __restrict__ pos_of_token, int n_tokens, int hidden, int vocab, int max_pos,
                    int type_vocab, const float* __restrict__ word, const float* __restrict__ pos,
                    const float* __restrict__ type, const float* __restrict__ gamma, const float* __restrict__ beta,
                    float eps, float* __restrict__ out, float* __restrict__ out_hi, float* __restrict__ out_lo) {
  const int lane = threadIdx.x & 31;
  const int t = blockIdx.x * 4 + (threadIdx.x >> 5);
  if (t >= n_tokens) return;
  int id = ids[t]; id = id < 0 ? 0 : (id >= vocab ? vocab - 1 : id);
  int p = pos_of_token[t]; p = p >= max_pos ? max_pos - 1 : p;
  int tt = type_ids ? type_ids[t] : 0; tt = tt < 0 ? 0 : (tt >= type_vocab ? type_vocab - 1 : tt);
  const int per_lane = hidden / 32;
  float v[kEncMaxHidden / 32];
#pragma unroll
  for (int i = 0; i < kEncMaxHidden / 32; ++i)
    if (i < per_lane) {
      const int c = i * 32 + lane;
      // BertEmbeddings.forward: (inputs_embeds + token_type_embeddings) + position_embeddings
      v[i] = (word[static_cast<int64_t>(id) * hidden + c] + type[static_cast<int64_t>(tt) * hidden + c]) +
             pos[static_cast<int64_t>(p) * hidden + c];
    }
  const int64_t ro = static_cast<int64_t>(t) * hidden;
  warp_layernorm(v, per_lane, hidden, eps, gamma, beta, out + ro, lane, out_hi ? out_hi + ro : nullptr,
                 out_hi ? out_lo + ro : nullptr);
}

// out = LayerNorm(x + residual)
__global__ void __launch_bounds__(128)
enc_add_ln_kernel(const float* __restrict__ x, const float* __restrict__ residual, int n_tokens, int hidden,
                  const float* __restrict__ gamma, const float* __restrict__ beta, float eps, float* __restrict__ out,
                  float* __restrict__ out_hi, float* __restrict__ out_lo) {
  const int lane = threadIdx.x & 31;
  const int t = blockIdx.x * 4 + (threadIdx.x >> 5);
  if (t >= n_tokens) return;
  const int per_lane = hidden / 32;
  float v[kEncMaxHidden / 32];
#pragma unroll
  for (int i = 0; i < kEncMaxHidden / 32; ++i)
    if (i < per_lane) {
      const int64_t o = static_cast<int64_t>(t) * hidden + i * 32 + lane;
      v[i] = x[o] + residual[o];
    }
  const int64_t ro = static_cast<int64_t>(t) * hidden;
  warp_layernorm(v, per_lane, hidden, eps, gamma, beta, out + ro, lane, out_hi ? out_hi + ro : nullptr,
                 out_hi ? out_lo + ro : nullptr);
}

// ---------------------------------------------------------------- GEMM: C[M, N] = A[M, K] . W[N, K]^T + bias
// (torch.nn.Linear layout: both operands K-contiguous.)  fp32 SIMT, fmaf accumulation: 128 x 128 x 16 tiles, 256
// threads, 8 x 8 outputs per thread as two 4-wide groups in each dimension (conflict-free float4 reads of the
// k-major shared tiles), register-prefetched double buffering.  K % 16 == 0.  EPI: 0 = bias, 1 = bias + GELU(erf),
// 2 = bias + quick_gelu (CLIP, clip.cuh).
constexpr int kGemmBM = 128, kGemmBN = 128, kGemmBK = 16, kGemmPad = 4;

__device__ __forceinline__ float gelu_erf(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f)); }
// transformers' QuickGELUActivation: x * sigmoid(1.702 x)
__device__ __forceinline__ float quick_gelu(float x) { return x * (1.0f / (1.0f + expf(-1.702f * x))); }

template <int EPI>
__global__ void __launch_bounds__(256, 2)
enc_gemm_kernel(const float* __restrict__ A, const float* __restrict__ W, const float* __restrict__ bias,
                float* __restrict__ C, int M, int N, int K) {
  __shared__ __align__(16) float As[2][kGemmBK][kGemmBM + kGemmPad];
  __shared__ __align__(16) float Ws[2][kGemmBK][kGemmBN + kGemmPad];
  const int tid = threadIdx.x;
  const int m0 = blockIdx.y * kGemmBM, n0 = blockIdx.x * kGemmBN;
  const int ty = tid >> 4, tx = tid & 15;                 // 16 x 16 threads
  // global -> register staging: 2 float4 of A and 2 of W per thread per k-block (row = idx / 4, k-quad = idx % 4)
  float4 ra[2], rw[2];
  auto load_tiles = [&](int k0) {
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const int idx = tid + 256 * j, row = idx >> 2, kq = idx & 3;
      const int gm = m0 + row, gn = n0 + row;
      ra[j] = gm < M ? *reinterpret_cast<const float4*>(A + static_cast<int64_t>(gm) * K + k0 + kq * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
      rw[j] = gn < N ? *reinterpret_cast<const float4*>(W + static_cast<int64_t>(gn) * K + k0 + kq * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  };
  auto store_tiles = [&](int buf) {
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const int idx = tid + 256 * j, row = idx >> 2, kq = idx & 3;
      As[buf][kq * 4 + 0][row] = ra[j].x; As[buf][kq * 4 + 1][row] = ra[j].y;
      As[buf][kq * 4 + 2][row] = ra[j].z; As[buf][kq * 4 + 3][row] = ra[j].w;
      Ws[buf][kq * 4 + 0][row] = rw[j].x; Ws[buf][kq * 4 + 1][row] = rw[j].y;
      Ws[buf][kq * 4 + 2][row] = rw[j].z; Ws[buf][kq * 4 + 3][row] = rw[j].w;
    }
  };
  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.0f;
  load_tiles(0);
  store_tiles(0);
  __syncthreads();
  const int nk = K / kGemmBK;
  for (int kb = 0; kb < nk; ++kb) {
    const int buf = kb & 1;
    if (kb + 1 < nk) load_tiles((kb + 1) * kGemmBK);
#pragma unroll
    for (int k = 0; k < kGemmBK; ++k) {
      const float4 a0 = *reinterpret_cast<const float4*>(&As[buf][k][ty * 4]);
      const float4 a1 = *reinterpret_cast<const float4*>(&As[buf][k][64 + ty * 4]);
      const float4 b0 = *reinterpret_cast<const float4*>(&Ws[buf][k][tx * 4]);
      const float4 b1 = *reinterpret_cast<const float4*>(&Ws[buf][k][64 + tx * 4]);
      const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      const float b[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    if (kb + 1 < nk) {
      store_tiles(buf ^ 1);
      __syncthreads();
    }
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int gm = m0 + (i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4));
    if (gm >= M) continue;
#pragma unroll
    for (int jg = 0; jg < 2; ++jg) {
      const int gn = n0 + (jg == 0 ? tx * 4 : 64 + tx * 4);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        if (gn + j < N) {
          float v = acc[i][jg * 4 + j] + bias[gn + j];
          if (EPI == 1) v = gelu_erf(v);
          if (EPI == 2) v = quick_gelu(v);
          C[static_cast<int64_t>(gm) * N + gn + j] = v;
        }
      }
    }
  }
}

// ---------------------------------------------------------------- attention
// qkv: packed [T, 3*hidden] rows = [q | k | v], head h at columns h*HD.  One CTA per (sequence, head) of 32..256 threads (the
// longest sequence of the batch, rse.cu): thread t owns query row t (+blockDim, ... for longer sequences), keys / values stream through shared memory 64 at a time;
// online softmax (running max / sum), fp32, expf.  Keys beyond the sequence do not exist in the packed layout, which
// IS the reference's padding mask (BertModel's extended attention mask adds -inf to padded keys).  CAUSAL (the CLIP
// text tower): query i of a sequence attends to its keys j <= i only.
template <int HD, bool CAUSAL = false>
__global__ void __launch_bounds__(256)
enc_attention_kernel(const float* __restrict__ qkv, const int32_t* __restrict__ cu_seqlens, int hidden,
                     float* __restrict__ ctx, float* __restrict__ ctx_lo) {   // ctx_lo != NULL: ctx <- hi, ctx_lo <- lo
  constexpr int KB = 64;
  __shared__ __align__(16) float sK[KB][HD];
  __shared__ __align__(16) float sV[KB][HD];
  const int seq = blockIdx.x, head = blockIdx.y;
  const int t0 = cu_seqlens[seq], len = cu_seqlens[seq + 1] - t0;
  const int ld = 3 * hidden;
  const float scale = 1.0f / sqrtf(static_cast<float>(HD));
  for (int q0 = 0; q0 < len; q0 += blockDim.x) {
    const int qi = q0 + threadIdx.x;
    const bool active = qi < len;
    float q[HD], acc[HD];
#pragma unroll
    for (int d = 0; d < HD; ++d) { q[d] = 0.0f; acc[d] = 0.0f; }
    if (active) {
      const float4* qp = reinterpret_cast<const float4*>(qkv + static_cast<int64_t>(t0 + qi) * ld + head * HD);
#pragma unroll
      for (int d = 0; d < HD / 4; ++d) { const float4 f = qp[d]; q[4 * d] = f.x; q[4 * d + 1] = f.y; q[4 * d + 2] = f.z; q[4 * d + 3] = f.w; }
    }
    float m = -__int_as_float(0x7F800000), l = 0.0f;
    for (int k0 = 0; k0 < len; k0 += KB) {
      const int nk = min(KB, len - k0);
      __syncthreads();
      for (int i = threadIdx.x; i < nk * (HD / 4); i += blockDim.x) {
        const int r = i / (HD / 4), c = i % (HD / 4);
        const float* row = qkv + static_cast<int64_t>(t0 + k0 + r) * ld + head * HD;
        reinterpret_cast<float4*>(&sK[r][0])[c] = reinterpret_cast<const float4*>(row + hidden)[c];
        reinterpret_cast<float4*>(&sV[r][0])[c] = reinterpret_cast<const float4*>(row + 2 * hidden)[c];
      }
      __syncthreads();
      if (active) {
        const int jn = CAUSAL ? min(nk, qi - k0 + 1) : nk;
        for (int j = 0; j < jn; ++j) {
          float s = 0.0f;
#pragma unroll
          for (int d = 0; d < HD; ++d) s = fmaf(q[d], sK[j][d], s);
          s *= scale;
          const float m_new = fmaxf(m, s);
          const float corr = expf(m - m_new);            // exp(-inf) = 0 on the first key
          const float p = expf(s - m_new);
          l = fmaf(l, corr, p);
#pragma unroll
          for (int d = 0; d < HD; ++d) acc[d] = fmaf(acc[d], corr, p * sV[j][d]);
          m = m_new;
        }
      }
    }
    if (active) {
      const float inv = 1.0f / l;
      const int64_t off = static_cast<int64_t>(t0 + qi) * hidden + head * HD;
      float4* op = reinterpret_cast<float4*>(ctx + off);
      float4* ol = ctx_lo ? reinterpret_cast<float4*>(ctx_lo + off) : nullptr;
#pragma unroll
      for (int d = 0; d < HD / 4; ++d) {
        float y[4] = {acc[4 * d] * inv, acc[4 * d + 1] * inv, acc[4 * d + 2] * inv, acc[4 * d + 3] * inv};
        if (ol) {
          float h[4], l[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) tf32_split(y[e], h[e], l[e]);
          op[d] = make_float4(h[0], h[1], h[2], h[3]);
          ol[d] = make_float4(l[0], l[1], l[2], l[3]);
        } else {
          op[d] = make_float4(y[0], y[1], y[2], y[3]);
        }
      }
    }
  }
}

// ---------------------------------------------------------------- heads
// head 0 (sentence-transformers Pooling(mean) + Normalize): mean over the sequence's tokens (sum / clamp(len, 1e-9)),
// then x / max(||x||_2, 1e-12).  One CTA per sequence, one thread per column.
__global__ void enc_pool_mean_norm_kernel(const float* __restrict__ x, const int32_t* __restrict__ cu_seqlens, int hidden,
                                          float* __restrict__ out) {
  __shared__ float s_part[32];
  const int seq = blockIdx.x;
  const int t0 = cu_seqlens[seq], len = cu_seqlens[seq + 1] - t0;
  float sq = 0.0f;
  float mean_c[kEncMaxHidden / 128];                     // blockDim = 128: columns c = threadIdx.x + 128*i
  const int per = (hidden + 127) / 128;
#pragma unroll
  for (int i = 0; i < kEncMaxHidden / 128; ++i) {
    mean_c[i] = 0.0f;
    const int c = threadIdx.x + 128 * i;
    if (i < per && c < hidden) {
      float s = 0.0f;
      for (int t = 0; t < len; ++t) s += x[static_cast<int64_t>(t0 + t) * hidden + c];
      const float mval = s / fmaxf(static_cast<float>(len), 1e-9f);
      mean_c[i] = mval;
      sq = fmaf(mval, mval, sq);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(0xFFFFFFFFu, sq, o);
  if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = sq;
  __syncthreads();
  float tot = 0.0f;
  for (int w = 0; w < (blockDim.x >> 5); ++w) tot += s_part[w];
  const float inv = 1.0f / fmaxf(sqrtf(tot), 1e-12f);
#pragma unroll
  for (int i = 0; i < kEncMaxHidden / 128; ++i) {
    const int c = threadIdx.x + 128 * i;
    if (i < per && c < hidden) out[static_cast<int64_t>(seq) * hidden + c] = mean_c[i] * inv;
  }
}

// head 1 (BertPooler + classifier, num_labels = 1): logit = w_c . tanh(W_p . h[CLS] + b_p) + b_c.  One CTA per
// sequence, one thread per pooler output row.
__global__ void enc_cls_head_kernel(const float* __restrict__ x, const int32_t* __restrict__ cu_seqlens, int hidden,
                                    const float* __restrict__ pool_w, const float* __restrict__ pool_b,
                                    const float* __restrict__ cls_w, const float* __restrict__ cls_b,
                                    float* __restrict__ out) {
  extern __shared__ float s_h[];                         // [hidden] h[CLS], then [32] partial sums
  float* s_part = s_h + hidden;
  const int seq = blockIdx.x;
  const float* h = x + static_cast<int64_t>(cu_seqlens[seq]) * hidden;
  for (int c = threadIdx.x; c < hidden; c += blockDim.x) s_h[c] = h[c];
  __syncthreads();
  float part = 0.0f;
  for (int r = threadIdx.x; r < hidden; r += blockDim.x) {
    float s = 0.0f;
    const float* w = pool_w + static_cast<int64_t>(r) * hidden;
    for (int c = 0; c < hidden; ++c) s = fmaf(w[c], s_h[c], s);
    part = fmaf(cls_w[r], tanhf(s + pool_b[r]), part);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xFFFFFFFFu, part, o);
  if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = part;
  __syncthreads();
  if (threadIdx.x == 0) {
    float tot = 0.0f;
    for (int w = 0; w < (blockDim.x >> 5); ++w) tot += s_part[w];
    out[seq] = tot + cls_b[0];
  }
}

// position of every token inside its sequence (cu_seqlens -> pos_of_token), one thread per token via binary search
__global__ void enc_positions_kernel(const int32_t* __restrict__ cu_seqlens, int n_seq, int n_tokens,
                                     int32_t* __restrict__ pos_of_token) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_tokens) return;
  int lo = 0, hi = n_seq;                                // last s with cu[s] <= t
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (cu_seqlens[mid] <= t) lo = mid; else hi = mid;
  }
  pos_of_token[t] = t - cu_seqlens[lo];
}

// ================================================================ tensor-core GEMM with fp32 accuracy (3 x TF32)
// The SIMT GEMM above is exact-ish but runs at ~19 TFLOP/s (r02 bench: 2.8 ms for a 256-query batch).  The
// tensor cores have no fp32 mode; kind::tf32 keeps 10 mantissa bits of each operand, which alone is ~1e-3 off and
// fails the 1e-5 bar.  The remedy (Ootomo & Yokota, "Recovering single precision accuracy from Tensor Cores"):
//   (1) split every operand into hi = tf32(x) and lo = tf32(x - hi) and compute hi*hi + lo*hi + hi*lo (the dropped
//       lo*lo term is 2^-22 relative);
//   (2) do NOT accumulate everything in the tensor core: its fp32 accumulator is updated with truncation, a
//       one-sided error that grows LINEARLY with the number of accumulation steps — the first version of this
//       kernel (all 3*K/8 MMAs of a tile into one TMEM accumulator) was 2.2e-5 off the PyTorch fp32 model after 6
//       layers, 20x worse than the SIMT kernel (9e-7).  So the dominant hi*hi products are accumulated in TMEM only
//       over K-CHUNKS of 128 (16 MMAs), each chunk from zero into one of two chunk buffers, and the epilogue warps
//       add the chunk sums into fp32 REGISTER accumulators (round-to-nearest, CUDA cores) while the next chunk is
//       being computed; the two correction products, 2^-11 smaller, accumulate in a third TMEM buffer over the
//       whole K (their truncation error is below 2^-30 relative).
//   * weights are split once at load (enc_split_kernel), activations by the kernel that produces them
//     (LayerNorm / attention / GELU epilogue write hi and lo next to or instead of the fp32 value).  (Tried in r02:
//     loading the plain fp32 boxes and splitting them IN SHARED MEMORY with the epilogue warps — half the operand
//     traffic, no hi/lo copies — was 10 % SLOWER, 1.22 vs 1.11 ms per 256-query batch: the tile is bound by the
//     latency of a 3-stage ring per CTA and by wave quantisation, not by L2 bandwidth, and the split adds a hop
//     to every stage.)
//   * one 128 x 64 output tile per CTA (cta_group::1): warp 0 = TMA producer (2-stage ring, per stage two
//     128 x 32-float boxes A_hi, A_lo and two 64 x 32-float boxes W_hi, W_lo, SWIZZLE_128B), warp 1 = single-thread
//     tcgen05.mma issuer (12 MMAs of 128x64x8 per k-block: 4 k-steps x 3 products), warps 2-5 = epilogue
//     (tcgen05.ld 32x32b, one TMEM lane = one token row per thread, 64 accumulators in registers): bias (+ GELU +
//     split), 128-byte stores.
// The tile is 64 wide, not 128, because a 128-wide tiling leaves most SMs idle (MiniLM's N = 384 projections on a
// 2.5 k-token batch: 60 tiles for 148 SMs; 120 with 64-wide tiles), and the 64-wide tile fits TWICE on an SM (96 KB
// of shared memory, 256 TMEM columns, 132 registers x 192 threads each): four stages in flight per SM and one CTA's
// prologue / epilogue under the other's main loop.
constexpr int kEgBM = 128, kEgBN = 64, kEgBK = 32;
constexpr int kEgStages = 2;
constexpr int kEgBox = kEgBM * kEgBK * 4;                       // 16,384 B: one 128-row operand box
constexpr int kEgWBox = kEgBN * kEgBK * 4;                      // 8,192 B: one 64-row weight box
constexpr int kEgThreads = 192;
constexpr int kEgChunkKB = 4;                                   // k-blocks per hi*hi accumulation chunk (K = 128)
constexpr int kEgStageBytes = 2 * kEgBox + 2 * kEgWBox;
constexpr int kEgSmemBytes = kEgStages * kEgStageBytes + 16 * 8 + 16 + 1024;
// kind::tf32: D = f32 (bit 4), A = B = tf32 (format 2), both K-major, N = kEgBN, M = 128
constexpr uint32_t kEgIdesc = (1u << 4) | (2u << 7) | (2u << 10) | ((static_cast<uint32_t>(kEgBN) >> 3) << 17) | ((kEgBM >> 4) << 24);

__global__ void enc_split_kernel(const float* __restrict__ x, int64_t n, float* __restrict__ hi, float* __restrict__ lo) {
  const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float h, l;
  tf32_split(x[i], h, l);
  hi[i] = h; lo[i] = l;
}

__device__ __forceinline__ void eg_tma_load_2d(void* smem_dst, const CUtensorMap* tmap, int c0, int c1, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::
          "r"(smem_u32(smem_dst)),
      "l"(tmap), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void eg_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void eg_mma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}

// EPI 0: C = acc + bias (fp32).  EPI 1: g = GELU(acc + bias) -> C_hi / C_lo (the operand of the next GEMM).
// EPI 2: the same with quick_gelu (CLIP).
template <int EPI>
__global__ void __launch_bounds__(kEgThreads, 2)
enc_gemm_tc_kernel(const __grid_constant__ CUtensorMap tmap_a_hi, const __grid_constant__ CUtensorMap tmap_a_lo,
                   const __grid_constant__ CUtensorMap tmap_w_hi, const __grid_constant__ CUtensorMap tmap_w_lo,
                   const float* __restrict__ bias, float* __restrict__ C, float* __restrict__ C_lo, int M, int N, int K) {
  extern __shared__ unsigned char smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  unsigned char* smem = smem_raw + (base - smem_u32(smem_raw));
  constexpr uint32_t kTmemCols = 256u;                          // 3 x kEgBN columns, rounded up to a power of two
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kEgStages * kEgStageBytes);
  uint64_t* full = bars;                       // [stages]
  uint64_t* empty = bars + kEgStages;          // [stages]
  uint64_t* cfull = bars + 2 * kEgStages;      // [2] hi*hi chunk buffer complete
  uint64_t* cempty = bars + 2 * kEgStages + 2; // [2] the four epilogue warps drained it
  uint64_t* sfull = bars + 2 * kEgStages + 4;  // [1] correction accumulator complete (= every MMA retired)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kEgStages + 5);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m0 = blockIdx.y * kEgBM, n0 = blockIdx.x * kEgBN;
  const int nkb = K / kEgBK;
  const int nchunks = nkb / kEgChunkKB;        // K % 128 == 0 (checked on the host)

  if (threadIdx.x == 0) {
    for (int s = 0; s < kEgStages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(&cfull[b], 1); mbar_init(&cempty[b], 4); }
    mbar_init(sfull, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(kTmemCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;       // columns [0,BN): corrections, [BN,2BN) / [2BN,3BN): hi*hi chunks (BN = kEgBN)

  if (warp == 0) {
    if (lane == 0) {
      asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_a_hi) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_a_lo) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_w_hi) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_w_lo) : "memory");
      int stage = 0;
      uint32_t phase = 0;
      for (int kb = 0; kb < nkb; ++kb) {
        mbar_wait(&empty[stage], phase ^ 1u);
        mbar_arrive_expect_tx(&full[stage], kEgStageBytes);
        unsigned char* st = smem + stage * kEgStageBytes;
        eg_tma_load_2d(st, &tmap_a_hi, kb * kEgBK, m0, &full[stage]);            // rows past M are zero-filled
        eg_tma_load_2d(st + kEgBox, &tmap_a_lo, kb * kEgBK, m0, &full[stage]);
        eg_tma_load_2d(st + 2 * kEgBox, &tmap_w_hi, kb * kEgBK, n0, &full[stage]);
        eg_tma_load_2d(st + 2 * kEgBox + kEgWBox, &tmap_w_lo, kb * kEgBK, n0, &full[stage]);
        if (++stage == kEgStages) { stage = 0; phase ^= 1u; }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int c = 0; c < nchunks; ++c) {
        const uint32_t buf = c & 1, use = c >> 1;
        mbar_wait(&cempty[buf], (use & 1u) ^ 1u);               // the epilogue has read this chunk buffer's last sums
        tc_fence_after();
        const uint32_t d_main = tmem_base + static_cast<uint32_t>(kEgBN) * (1u + buf);
        for (int kc = 0; kc < kEgChunkKB; ++kc) {
          mbar_wait(&full[stage], phase);
          tc_fence_after();
          const uint32_t st = base + stage * kEgStageBytes;
          const uint64_t a_hi = tc_smem_desc(st), a_lo = tc_smem_desc(st + kEgBox);
          const uint64_t w_hi = tc_smem_desc(st + 2 * kEgBox), w_lo = tc_smem_desc(st + 2 * kEgBox + kEgWBox);
#pragma unroll
          for (int k = 0; k < kEgBK / 8; ++k) {
            const uint64_t o = static_cast<uint64_t>(2 * k);    // 8 tf32 = 32 B inside the swizzle atom
            eg_mma_tf32(tmem_base, a_lo + o, w_hi + o, kEgIdesc, (c | kc | k) != 0 ? 1u : 0u);
            eg_mma_tf32(tmem_base, a_hi + o, w_lo + o, kEgIdesc, 1u);
            eg_mma_tf32(d_main, a_hi + o, w_hi + o, kEgIdesc, (kc | k) != 0 ? 1u : 0u);
          }
          eg_commit(&empty[stage]);
          if (++stage == kEgStages) { stage = 0; phase ^= 1u; }
        }
        eg_commit(&cfull[buf]);
      }
      eg_commit(sfull);
    }
    __syncwarp();
  } else {
    const int quarter = warp & 3;                               // TMEM lanes [32*quarter, +32) belong to this warp
    const int row = m0 + quarter * 32 + lane;
    const uint32_t lane_addr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16);
    float acc[kEgBN];
#pragma unroll
    for (int j = 0; j < kEgBN; ++j) acc[j] = 0.0f;
    for (int c = 0; c < nchunks; ++c) {
      const uint32_t buf = c & 1, use = c >> 1;
      mbar_wait(&cfull[buf], use & 1u);
      tc_fence_after();
#pragma unroll
      for (int c0 = 0; c0 < kEgBN; c0 += 32) {
        uint32_t v[32];
        tc_ld32(lane_addr + static_cast<uint32_t>(kEgBN) * (1u + buf) + static_cast<uint32_t>(c0), v);
#pragma unroll
        for (int j = 0; j < 32; ++j) acc[c0 + j] += __uint_as_float(v[j]);      // fp32 add, round to nearest
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&cempty[buf]);
    }
    mbar_wait(sfull, 0u);
    tc_fence_after();
#pragma unroll
    for (int c0 = 0; c0 < kEgBN; c0 += 32) {
      uint32_t v[32];
      tc_ld32(lane_addr + static_cast<uint32_t>(c0), v);
      if (row < M) {
        const int col = n0 + c0;
        float* dst = C + static_cast<int64_t>(row) * N + col;
        float* dst_lo = (EPI != 0) ? C_lo + static_cast<int64_t>(row) * N + col : nullptr;
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
          float o[4], l[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            float x = (acc[c0 + j + e] + __uint_as_float(v[j + e])) + (col + j + e < N ? __ldg(bias + col + j + e) : 0.0f);
            if (EPI == 1) { x = gelu_erf(x); tf32_split(x, o[e], l[e]); }
            else if (EPI == 2) { x = quick_gelu(x); tf32_split(x, o[e], l[e]); }
            else { o[e] = x; }
          }
          if (col + j + 3 < N) {
            *reinterpret_cast<float4*>(dst + j) = make_float4(o[0], o[1], o[2], o[3]);
            if (EPI != 0) *reinterpret_cast<float4*>(dst_lo + j) = make_float4(l[0], l[1], l[2], l[3]);
          } else {
#pragma unroll
            for (int e = 0; e < 4; ++e)
              if (col + j + e < N) { dst[j + e] = o[e]; if (EPI != 0) dst_lo[j + e] = l[e]; }
          }
        }
      }
    }
    tc_fence_before();
  }
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols) : "memory");
  }
}

}  // namespace rse

// clip.cuh — §10 f4: the CLIP image and text towers of the image search on the same GPU as the index.
//
// The reference's MultimodalSearch (llm/multimodal.py) runs SentenceTransformer("clip-ViT-B-32"): every document's
// "title: description" is encoded once by the text tower, every query image by the vision tower.  What
// sentence-transformers calls is the HuggingFace CLIPModel's get_text_features / get_image_features, i.e. the
// forward of CLIPTextModelWithProjection / CLIPVisionModelWithProjection, in fp32, not normalised.
//
// Both towers are pre-LN transformers of the kind encoder.cuh already runs, so the GEMMs (3xTF32 tcgen05 and fp32
// SIMT), the packed-token attention and the weight split are encoder.cuh's; what is CLIP's own lives here:
//   vision: pixel_values [n, 3, S, S] -> patch rows [n*G*G, 3*P*P] (clip_patchify_kernel) -> patch GEMM (conv
//           without bias) -> tokens [class | patches] + position_embedding -> pre_layrnorm (clip_vision_embed_kernel);
//   text:   token_embedding[id] + position_embedding[pos] (clip_text_embed_kernel), no LayerNorm;
//   layer:  y = LN1(x); qkv = y.Wqkv; attention (text: causal); x += ctx.Wo; y = LN2(x); x += quick_gelu(y.W1).W2
//           — the residual stream x and the GEMM operand y are separate buffers (BERT's post-LN writes one);
//           each residual add is fused with the LayerNorm that follows it (clip_residual_ln_kernel);
//   heads:  post_layernorm of the class token / final_layer_norm of the pooled token, then the projection
//           (clip_head_kernel).
// Numerics as in encoder.cuh: fp32 storage, explicit fmaf (the library is built with --fmad=false), expf.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>

#include "encoder.cuh"

namespace rse {

// pixel_values [n, 3, S, S] (NCHW) -> rows [n*G*G, Kp], column (c, ky, kx) = the flattened conv weight
// [hidden, 3, P, P], columns 3*P*P .. Kp-1 zero (Kp = 3*P*P rounded up to the GEMMs' K granule); patch (py, px) of
// image i is row i*G*G + py*G + px.  One thread per output element: a row's P consecutive kx are P consecutive
// pixels of one image row, so reads and writes are both coalesced.
// hi != NULL: the tf32 hi / lo split for the tensor-core GEMM instead of the fp32 value.
__global__ void clip_patchify_kernel(const float* __restrict__ px, int64_t n_elem, int S, int P, int G, int Kp,
                                     float* __restrict__ out, float* __restrict__ hi, float* __restrict__ lo) {
  const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n_elem) return;
  const int64_t row = i / Kp;
  const int col = static_cast<int>(i - row * Kp);
  float v = 0.0f;
  if (col < 3 * P * P) {
    const int64_t img = row / (G * G);
    const int p = static_cast<int>(row - img * G * G);
    const int py = p / G, pxi = p - py * G;
    const int c = col / (P * P), r = col - c * P * P;
    const int ky = r / P, kx = r - ky * P;
    v = px[((img * 3 + c) * S + py * P + ky) * static_cast<int64_t>(S) + pxi * P + kx];
  }
  if (hi) { float h, l; tf32_split(v, h, l); hi[i] = h; lo[i] = l; }
  else out[i] = v;
}

// vision tokens: token 0 of image i = class_embedding, token 1+p = patch GEMM row i*G*G + p; + position_embedding
// [token]; x = pre_layrnorm(.) (the residual stream); y = layer 0's layer_norm1(x) (+ hi / lo).  One warp per token.
__global__ void __launch_bounds__(128)
clip_vision_embed_kernel(const float* __restrict__ patch_out, int n_tokens, int L, int hidden,
                         const float* __restrict__ cls, const float* __restrict__ pos,
                         const float* __restrict__ pre_g, const float* __restrict__ pre_b,
                         const float* __restrict__ ln1_g, const float* __restrict__ ln1_b, float eps,
                         float* __restrict__ x, float* __restrict__ y, float* __restrict__ y_hi, float* __restrict__ y_lo) {
  const int lane = threadIdx.x & 31;
  const int t = blockIdx.x * 4 + (threadIdx.x >> 5);
  if (t >= n_tokens) return;
  const int img = t / L, tok = t - img * L;
  const int per_lane = hidden / 32;
  const float* src = tok == 0 ? cls : patch_out + (static_cast<int64_t>(img) * (L - 1) + tok - 1) * hidden;
  float v[kEncMaxHidden / 32];
#pragma unroll
  for (int i = 0; i < kEncMaxHidden / 32; ++i)
    if (i < per_lane) {
      const int c = i * 32 + lane;
      v[i] = src[c] + pos[static_cast<int64_t>(tok) * hidden + c];
    }
  const int64_t ro = static_cast<int64_t>(t) * hidden;
  warp_layernorm(v, per_lane, hidden, eps, pre_g, pre_b, x + ro, lane);
#pragma unroll
  for (int i = 0; i < kEncMaxHidden / 32; ++i)
    if (i < per_lane) v[i] = x[ro + i * 32 + lane];            // this lane's own stores
  warp_layernorm(v, per_lane, hidden, eps, ln1_g, ln1_b, y + ro, lane, y_hi ? y_hi + ro : nullptr,
                 y_hi ? y_lo + ro : nullptr);
}

// text tokens: x = token_embedding[id] + position_embedding[pos] (CLIPTextEmbeddings: no LayerNorm);
// y = layer 0's layer_norm1(x) (+ hi / lo).  One warp per token.
__global__ void __launch_bounds__(128)
clip_text_embed_kernel(const int32_t* __restrict__ ids, const int32_t* __restrict__ pos_of_token, int n_tokens,
                       int hidden, int vocab, int max_pos, const float* __restrict__ tok_emb,
                       const float* __restrict__ pos, const float* __restrict__ ln1_g,
                       const float* __restrict__ ln1_b, float eps, float* __restrict__ x, float* __restrict__ y,
                       float* __restrict__ y_hi, float* __restrict__ y_lo) {
  const int lane = threadIdx.x & 31;
  const int t = blockIdx.x * 4 + (threadIdx.x >> 5);
  if (t >= n_tokens) return;
  int id = ids[t]; id = id < 0 ? 0 : (id >= vocab ? vocab - 1 : id);
  int p = pos_of_token[t]; p = p >= max_pos ? max_pos - 1 : p;
  const int per_lane = hidden / 32;
  const int64_t ro = static_cast<int64_t>(t) * hidden;
  float v[kEncMaxHidden / 32];
#pragma unroll
  for (int i = 0; i < kEncMaxHidden / 32; ++i)
    if (i < per_lane) {
      const int c = i * 32 + lane;
      v[i] = tok_emb[static_cast<int64_t>(id) * hidden + c] + pos[static_cast<int64_t>(p) * hidden + c];
      x[ro + c] = v[i];
    }
  warp_layernorm(v, per_lane, hidden, eps, ln1_g, ln1_b, y + ro, lane, y_hi ? y_hi + ro : nullptr,
                 y_hi ? y_lo + ro : nullptr);
}

// x += delta; y = LayerNorm(x) (+ hi / lo).  gamma == NULL (after the last layer): the add alone.
__global__ void __launch_bounds__(128)
clip_residual_ln_kernel(float* __restrict__ x, const float* __restrict__ delta, int n_tokens, int hidden,
                        const float* __restrict__ gamma, const float* __restrict__ beta, float eps,
                        float* __restrict__ y, float* __restrict__ y_hi, float* __restrict__ y_lo) {
  const int lane = threadIdx.x & 31;
  const int t = blockIdx.x * 4 + (threadIdx.x >> 5);
  if (t >= n_tokens) return;
  const int per_lane = hidden / 32;
  const int64_t ro = static_cast<int64_t>(t) * hidden;
  float v[kEncMaxHidden / 32];
#pragma unroll
  for (int i = 0; i < kEncMaxHidden / 32; ++i)
    if (i < per_lane) {
      const int64_t o = ro + i * 32 + lane;
      v[i] = x[o] + delta[o];
      x[o] = v[i];
    }
  if (!gamma) return;
  warp_layernorm(v, per_lane, hidden, eps, gamma, beta, y + ro, lane, y_hi ? y_hi + ro : nullptr,
                 y_hi ? y_lo + ro : nullptr);
}

// cu_seqlens of n images of L tokens each
__global__ void clip_fixed_cu_kernel(int n, int L, int32_t* __restrict__ cu) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i <= n) cu[i] = i * L;
}

// heads: out[seq] = proj . LayerNorm(x[pooled row]), proj [P, hidden] (no bias).  One CTA of 128 threads per
// sequence.  The pooled row: ids == NULL (vision) the sequence's first token (the class token); otherwise
// transformers' CLIPTextTransformer rule — eos_token_id == 2 (legacy configs): the first argmax of the sequence's
// ids; else the first position whose id is eos_token_id, position 0 if there is none.  Warp 0 finds the row and
// normalises it into shared memory; then one warp per output row, lanes across the hidden dimension.
__global__ void __launch_bounds__(128)
clip_head_kernel(const float* __restrict__ x, const int32_t* __restrict__ cu_seqlens, const int32_t* __restrict__ ids,
                 int eos, int hidden, const float* __restrict__ gamma, const float* __restrict__ beta, float eps,
                 const float* __restrict__ proj, int P, float* __restrict__ out) {
  __shared__ __align__(16) float s_h[kEncMaxHidden];
  const int seq = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (warp == 0) {
    const int t0 = cu_seqlens[seq], len = cu_seqlens[seq + 1] - t0;
    int best = 0;
    if (ids) {
      if (eos == 2) {                                      // first argmax: largest id, ties to the smaller position
        int bv = -2147483647 - 1, bp = 0x7FFFFFFF;
        for (int j = lane; j < len; j += 32) { const int v = ids[t0 + j]; if (v > bv) { bv = v; bp = j; } }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          const int ov = __shfl_xor_sync(0xFFFFFFFFu, bv, o), op = __shfl_xor_sync(0xFFFFFFFFu, bp, o);
          if (ov > bv || (ov == bv && op < bp)) { bv = ov; bp = op; }
        }
        best = bp;
      } else {                                             // first eos position, else 0
        int bp = 0x7FFFFFFF;
        for (int j = lane; j < len; j += 32) if (ids[t0 + j] == eos) { bp = j; break; }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) bp = min(bp, __shfl_xor_sync(0xFFFFFFFFu, bp, o));
        best = bp == 0x7FFFFFFF ? 0 : bp;
      }
    }
    const int per_lane = hidden / 32;
    const float* row = x + static_cast<int64_t>(t0 + best) * hidden;
    float v[kEncMaxHidden / 32];
#pragma unroll
    for (int i = 0; i < kEncMaxHidden / 32; ++i)
      if (i < per_lane) v[i] = row[i * 32 + lane];
    warp_layernorm(v, per_lane, hidden, eps, gamma, beta, s_h, lane);
  }
  __syncthreads();
  for (int r0 = warp * 32; r0 < P; r0 += 128) {          // 32 rows per warp, lane j keeps row r0 + j: one 128-byte store
    float mine = 0.0f;
    for (int j = 0; j < 32 && r0 + j < P; ++j) {
      const float* w = proj + static_cast<int64_t>(r0 + j) * hidden;
      float s = 0.0f;
      for (int c = lane; c < hidden; c += 32) s = fmaf(w[c], s_h[c], s);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xFFFFFFFFu, s, o);
      if (lane == j) mine = s;
    }
    if (r0 + lane < P) out[static_cast<int64_t>(seq) * P + r0 + lane] = mine;
  }
}

}  // namespace rse

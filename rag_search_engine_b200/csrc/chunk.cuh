// chunk.cuh — the semantic index's sentence chunking on the device, byte for byte store.plan_chunks /
// textutil.sentence_chunks (the reference's chunk / semantic_chunk, semantic_search.py:164-188):
//
//   chunk 0      the title, verbatim (not stripped)
//   chunk w + 1  window w of the description's sentences, their bytes joined without a separator
//
// The description is stripped of Python's whitespace (str.strip / re's \s: the 29 code points of chunk_ws) and split
// at every maximal whitespace run whose preceding code point is '.', '!' or '?' ((?<=[.!?])\s+); an empty stripped
// description is one empty sentence.  With carry = overlap if 0 < overlap < size else 0 and fresh = size - carry,
// window 0 is sentences [0, min(size, n)) and window w >= 1 is [size + (w - 1) fresh - carry, min(size + w fresh, n)).
//
// Movie m's title is text[offs[2m], offs[2m + 1]) and its description text[offs[2m + 1], offs[2m + 2]) (valid UTF-8,
// as Python encodes a str).  One thread per movie walks its description (a few hundred bytes to a few KB: the per-byte
// work is a UTF-8 decode and a compare, like the tokenizer's walk of the same texts).  Two launches of the same walk,
// as in wordpiece.cuh: the count pass (chunks and chunk bytes per movie), a one-CTA scan of each (wp_scan_kernel), and
// the write pass into the chunk CSR.  A window is re-walked from its first sentence, whose start the previous window
// kept, so the work is the bytes written.
#pragma once
#include <climits>
#include <cstdint>

#include "common.cuh"

namespace rse {

constexpr int kChunkThreads = 128;
// meta (u64): [0] movies whose chunk bytes exceed INT_MAX, [1] the first of them
constexpr int kChunkMeta = 2;

__device__ __forceinline__ bool chunk_ws(uint32_t c) {
  return (c >= 0x09 && c <= 0x0D) || (c >= 0x1C && c <= 0x20) || c == 0x85 || c == 0xA0 || c == 0x1680 ||
         (c >= 0x2000 && c <= 0x200A) || c == 0x2028 || c == 0x2029 || c == 0x202F || c == 0x205F || c == 0x3000;
}

// the code point at p < e and its length in bytes (well-formed UTF-8; a sequence cut by e reads as one byte that is
// neither whitespace nor punctuation, so a malformed text never makes the walk leave [.., e))
__device__ __forceinline__ uint32_t chunk_cp(const uint8_t* __restrict__ t, int64_t p, int64_t e, int* len) {
  const uint32_t b = t[p];
  const int need = b < 0x80 ? 1 : b < 0xE0 ? 2 : b < 0xF0 ? 3 : 4;
  if (b < 0x80 || p + need > e) { *len = 1; return b; }
  if (b < 0xE0) { *len = 2; return (b & 0x1F) << 6 | (t[p + 1] & 0x3F); }
  if (b < 0xF0) { *len = 3; return (b & 0x0F) << 12 | (t[p + 1] & 0x3F) << 6 | (t[p + 2] & 0x3F); }
  *len = 4;
  return (b & 0x07) << 18 | (t[p + 1] & 0x3F) << 12 | (t[p + 2] & 0x3F) << 6 | (t[p + 3] & 0x3F);
}

// the description without its leading and trailing whitespace: [*s, *e)
__device__ __forceinline__ void chunk_strip(const uint8_t* __restrict__ t, int64_t a, int64_t b, int64_t* s, int64_t* e) {
  int len;
  while (a < b && chunk_ws(chunk_cp(t, a, b, &len))) a += len;
  while (b > a) {
    int64_t q = b - 1;
    while (q > a && (t[q] & 0xC0) == 0x80) --q;
    if (!chunk_ws(chunk_cp(t, q, b, &len))) break;
    b = q;
  }
  *s = a;
  *e = b;
}

// the sentence that starts at p (< e): it ends at *end; the next one starts at *next (e when it was the last)
__device__ __forceinline__ void chunk_sentence(const uint8_t* __restrict__ t, int64_t p, int64_t e, int64_t* end,
                                               int64_t* next) {
  uint32_t prev = 0;
  while (p < e) {
    int len;
    const uint32_t c = chunk_cp(t, p, e, &len);
    if (chunk_ws(c) && (prev == '.' || prev == '!' || prev == '?')) {
      *end = p;
      while (p < e && chunk_ws(chunk_cp(t, p, e, &len))) p += len;
      *next = p;
      return;
    }
    prev = c;
    p += len;
  }
  *end = e;
  *next = e;
}

// movie m: its chunk count and chunk bytes (count pass), or also its chunk texts written at out, their offsets
// (byte_base + position in out) at offs_out[0 ..) and each chunk's movie row / chunk_index (write pass)
template <bool WRITE>
__device__ void chunk_movie(const uint8_t* __restrict__ t, const int64_t* __restrict__ offs, int m, int size, int carry,
                            int* n_chunks, int64_t* n_bytes, uint8_t* __restrict__ out, int64_t byte_base,
                            int64_t* __restrict__ offs_out, int32_t* __restrict__ movie_out,
                            int32_t* __restrict__ index_out, int movie_row) {
  const int64_t t0 = offs[2 * m], t1 = offs[2 * m + 1], d1 = offs[2 * m + 2];
  int64_t s, e;
  chunk_strip(t, t1, d1, &s, &e);
  int n = 1;                                  // sentences
  if (s < e) {
    n = 0;
    for (int64_t p = s; p < e; ++n) {
      int64_t end;
      chunk_sentence(t, p, e, &end, &p);
    }
  }
  const int fresh = size - carry;
  const int n_win = n > size ? 1 + (n - size + fresh - 1) / fresh : 1;
  int64_t at = 0;                             // bytes written so far
  if (WRITE) {
    for (int64_t i = t0; i < t1; ++i) out[i - t0] = t[i];
    offs_out[0] = byte_base;
    movie_out[0] = movie_row;
    index_out[0] = 0;
  }
  at += t1 - t0;
  int64_t start = s;                          // byte position of the current window's first sentence
  for (int w = 0; w < n_win; ++w) {
    const int first = w == 0 ? 0 : size + (w - 1) * fresh - carry;
    const int last = min(w == 0 ? size : size + w * fresh, n);   // exclusive
    const int next_first = size + w * fresh - carry;               // the next window's first sentence
    if (WRITE) {
      offs_out[w + 1] = byte_base + at;
      movie_out[w + 1] = movie_row;
      index_out[w + 1] = w + 1;
    }
    int64_t p = start, next_start = e;
    for (int j = first; j < last; ++j) {
      if (j == next_first) next_start = p;
      int64_t end = e, next = e;
      if (p < e) chunk_sentence(t, p, e, &end, &next);
      if (WRITE)
        for (int64_t i = p; i < end; ++i) out[at + (i - p)] = t[i];
      at += end - p;
      p = next;
    }
    if (last <= next_first) next_start = p;   // no carry: the next window starts where this one stopped
    start = next_start;
  }
  *n_chunks = 1 + n_win;
  *n_bytes = at;
}

// count pass: chunks[m] and bytes[m] of movies [0, n)
__global__ void __launch_bounds__(kChunkThreads)
chunk_count_kernel(const uint8_t* __restrict__ t, const int64_t* __restrict__ offs, int n, int size, int carry,
                   int32_t* __restrict__ chunks, int32_t* __restrict__ bytes, unsigned long long* __restrict__ meta) {
  const int m = blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= n) return;
  int nc;
  int64_t nb;
  chunk_movie<false>(t, offs, m, size, carry, &nc, &nb, nullptr, 0, nullptr, nullptr, nullptr, 0);
  if (nb > INT_MAX) {
    atomicAdd(&meta[0], 1ull);
    atomicMin(&meta[1], static_cast<unsigned long long>(m));
    nb = 0;
  }
  chunks[m] = nc;
  bytes[m] = static_cast<int32_t>(nb);
}

// write pass: movie m's chunks at chunk_cu[m] .., their bytes at byte_cu[m] ..; offs_out[chunk_cu[n]] = the total
__global__ void __launch_bounds__(kChunkThreads)
chunk_write_kernel(const uint8_t* __restrict__ t, const int64_t* __restrict__ offs, int n, int size, int carry,
                   const int64_t* __restrict__ chunk_cu, const int64_t* __restrict__ byte_cu, int movie_base,
                   uint8_t* __restrict__ out, int64_t* __restrict__ offs_out, int32_t* __restrict__ movie_out,
                   int32_t* __restrict__ index_out) {
  const int m = blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= n) return;
  const int64_t c0 = chunk_cu[m], b0 = byte_cu[m];
  int nc;
  int64_t nb;
  chunk_movie<true>(t, offs, m, size, carry, &nc, &nb, out + b0, b0, offs_out + c0, movie_out + c0, index_out + c0,
                    movie_base + m);
  if (m == n - 1) offs_out[c0 + nc] = b0 + nb;
}

// offsets[0 .. n] into a device text buffer of `bytes` bytes: *bad = the first i where offs[i] is outside [0, bytes]
// or below offs[i - 1] (left at ~0 when they are well formed).  They need not start at 0: a part of a larger buffer
// is addressed through its own slice of the offsets.
__global__ void dev_offsets_check_kernel(const int64_t* __restrict__ offs, int64_t n, int64_t bytes,
                                         unsigned long long* __restrict__ bad) {
  const int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (i > n) return;
  const int64_t v = offs[i];
  if (v < 0 || v > bytes || (i > 0 && v < offs[i - 1]))
    atomicMin(bad, static_cast<unsigned long long>(i));
}

}  // namespace rse

// wordpiece.cuh — BERT WordPiece tokenisation on the device, bit-identical to the HuggingFace fast tokenizer
// (tokenizers: AddedVocabulary -> BertNormalizer -> BertPreTokenizer -> WordPiece -> BertProcessing).
//
// The tables come from rag_search_engine_b200/wordpiece.py, probed through the tokenizer's own components:
//   map[cp]    the 0-3 code points BertNormalizer makes of cp (bits 0-20: the code point, or a row of extra[][3] when
//              there are two or three; bits 21-22: the count; bit 23: the output keeps a combining mark that NFD's
//              canonical reordering could move, see below)
//   cls[cp]    how BertPreTokenizer treats cp: other / whitespace (splits, dropped) / punctuation (a word of its own)
//   two tries over code points: node 0 roots the word-initial pieces, node 1 the continuation pieces ("##" removed);
//              node_first[n] .. node_first[n + 1] are node n's edges sorted by edge_cp, node_id[n] the piece ending there
//   the added tokens (the special tokens, matched literally in the raw text before normalisation, leftmost-longest)
//
// Joining the per-code-point outputs of the normaliser equals normalising the whole text, except where NFD would
// reorder combining marks: marks that survive the accent stripping (canonical class != 0, not Mn) of two different
// code points of one text.  Such a text is counted and refused (the caller tokenizes it on the host); a single code
// point's own decomposition is already in canonical order.
//
// One thread per text walks its UTF-8 bytes once: the words of a short query and the ~200 words of a 1 KB document
// alike.  Two launches of the same walk: the count pass (pieces per text, malformed UTF-8, reorder flags, largest
// id) and, after a one-CTA scan of the counts, the write pass into the CSR ids.  Truncation keeps the first `cap`
// pieces; words past the cut are not matched, but their bytes are still validated.
#pragma once
#include <climits>
#include <cstdint>

#include "common.cuh"

namespace rse {

constexpr int kWpCodePoints = 0x110000;
constexpr int kWpMaxWordChars = 256;  // the largest max_input_chars_per_word (a per-thread word buffer)
constexpr int kWpMaxAdded = 32;
constexpr int kWpThreads = 128;
constexpr int kWpScanThreads = 1024;
constexpr uint32_t kWpCpMask = 0x1FFFFFu;
constexpr uint32_t kWpReorder = 1u << 23;
constexpr uint8_t kWpOther = 0, kWpSpace = 1, kWpPunct = 2;
// meta (u64): [0] texts with malformed UTF-8, [1] the first of them, [2] texts NFD could reorder, [3] the first of
// them, [4] ids in all, [5] longest sequence, [6] largest id kept
constexpr int kWpMeta = 7;

struct WpTables {
  const uint32_t* map;
  const uint32_t* extra;
  const uint8_t* cls;
  const int32_t* node_first;
  const int32_t* node_id;
  const int32_t* edge_cp;
  const int32_t* edge_child;
  const uint8_t* added_bytes;
  const int32_t* added_off;  // [n_added + 1]
  const int32_t* added_id;
  int n_added;
  uint32_t added_first[8];   // bit b: some added token starts with byte b
  int unk, cls_id, sep_id, max_chars;
};

__device__ __forceinline__ int wp_child(const WpTables& t, int node, int cp) {
  const int end = t.node_first[node + 1];
  int lo = t.node_first[node], hi = end;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (t.edge_cp[mid] < cp) lo = mid + 1; else hi = mid;
  }
  return lo < end && t.edge_cp[lo] == cp ? t.edge_child[lo] : -1;
}

// well-formed UTF-8 (Unicode Table 3-7): the bytes used at s[p], or 0 when the sequence there is malformed
__device__ __forceinline__ int wp_utf8(const uint8_t* s, int64_t p, int64_t e, uint32_t* cp) {
  const uint32_t b0 = s[p];
  if (b0 < 0x80) { *cp = b0; return 1; }
  int n;
  uint32_t c, lo = 0x80, hi = 0xBF;
  if (b0 >= 0xC2 && b0 <= 0xDF) { n = 2; c = b0 & 0x1F; }
  else if (b0 >= 0xE0 && b0 <= 0xEF) { n = 3; c = b0 & 0x0F; if (b0 == 0xE0) lo = 0xA0; else if (b0 == 0xED) hi = 0x9F; }
  else if (b0 >= 0xF0 && b0 <= 0xF4) { n = 4; c = b0 & 0x07; if (b0 == 0xF0) lo = 0x90; else if (b0 == 0xF4) hi = 0x8F; }
  else return 0;
  if (p + n > e) return 0;
  for (int i = 1; i < n; ++i) {
    const uint32_t b = s[p + i];
    if (b < lo || b > hi) return 0;
    lo = 0x80; hi = 0xBF;
    c = (c << 6) | (b & 0x3F);
  }
  *cp = c;
  return n;
}

// The pieces of one text (special tokens not included): kept pieces go to out[0 .. cap) when WRITE.  Returns
// min(pieces, cap), or -1 for malformed UTF-8.  *max_id: the largest kept id; *reorder: code points with map bit 23.
template <bool WRITE>
__device__ int wp_text(const WpTables& t, const uint8_t* __restrict__ s, int64_t p, int64_t e, int cap,
                       int32_t* __restrict__ out, int* max_id, int* reorder) {
  int w[kWpMaxWordChars];
  int wl = 0, np = 0, mx = -1, nre = 0;
  auto emit = [&](int id) {
    if (np < cap) {
      if (WRITE) out[np] = id;
      mx = max(mx, id);
    }
    ++np;
  };
  // greedy longest match of w[0 .. wl) (tokenizers' WordPiece::tokenize), emitting the pieces when `commit`;
  // false when some position matches no piece
  auto walk = [&](bool commit) {
    int start = 0;
    while (start < wl) {
      int node = start == 0 ? 0 : 1, best = -1, bend = start;
      for (int i = start; i < wl; ++i) {
        node = wp_child(t, node, w[i]);
        if (node < 0) break;
        const int id = t.node_id[node];
        if (id >= 0) { best = id; bend = i + 1; }
      }
      if (best < 0) return false;
      if (commit) emit(best);
      start = bend;
    }
    return true;
  };
  // a word longer than max_chars, or with a position no piece matches, is one [UNK].  The write pass checks the word
  // before it writes: pieces written ahead of a failure could land past the text's last id, in the next text's ids.
  auto flush = [&]() {
    if (wl == 0) return;
    const int np0 = np, mx0 = mx;
    if (wl > t.max_chars || (WRITE && !walk(false)) || !walk(true)) {
      np = np0; mx = mx0;
      emit(t.unk);
    }
    wl = 0;
  };
  while (p < e) {
    const uint32_t b0 = s[p];
    if ((t.added_first[b0 >> 5] >> (b0 & 31)) & 1u) {
      int best = -1, blen = 0;
      for (int a = 0; a < t.n_added; ++a) {
        const int o = t.added_off[a], L = t.added_off[a + 1] - o;
        if (L <= blen || p + L > e) continue;
        int k = 0;
        while (k < L && s[p + k] == t.added_bytes[o + k]) ++k;
        if (k == L) { best = t.added_id[a]; blen = L; }
      }
      if (best >= 0) {
        flush();
        emit(best);
        p += blen;
        continue;
      }
    }
    uint32_t cp;
    const int nb = wp_utf8(s, p, e, &cp);
    if (nb == 0) return -1;
    p += nb;
    const uint32_t m = t.map[cp];
    nre += (m & kWpReorder) != 0;
    const int cnt = (m >> 21) & 3;
    for (int k = 0; k < cnt; ++k) {
      const uint32_t o = cnt == 1 ? (m & kWpCpMask) : t.extra[3 * (m & kWpCpMask) + k];
      const uint8_t c = t.cls[o];
      if (c == kWpOther) {
        if (np < cap) {                                    // past the cut a word adds nothing
          if (wl < kWpMaxWordChars) w[wl] = static_cast<int>(o);
          ++wl;
        }
      } else {
        flush();
        if (c == kWpPunct && np < cap) { w[0] = static_cast<int>(o); wl = 1; flush(); }
      }
    }
  }
  flush();
  *max_id = mx;
  *reorder = nre;
  return min(np, cap);
}

// count pass: count[i] = ids of text i (specials included); meta as above
__global__ void __launch_bounds__(kWpThreads)
wp_count_kernel(WpTables t, const uint8_t* __restrict__ text, const int64_t* __restrict__ offs, int n, int special,
                int cap, int32_t* __restrict__ count, unsigned long long* __restrict__ meta) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int mx = -1, nre = 0;
  int np = wp_text<false>(t, text, offs[i], offs[i + 1], cap, nullptr, &mx, &nre);
  if (np < 0) {
    atomicAdd(&meta[0], 1ull);
    atomicMin(&meta[1], static_cast<unsigned long long>(i));
    np = 0;
  } else if (nre >= 2) {
    atomicAdd(&meta[2], 1ull);
    atomicMin(&meta[3], static_cast<unsigned long long>(i));
  }
  if (special) mx = max(mx, max(t.cls_id, t.sep_id));
  if (mx >= 0) atomicMax(&meta[6], static_cast<unsigned long long>(mx));
  count[i] = np + 2 * special;
}

// write pass: text i's ids at ids[cu[i] ..), [CLS] ... [SEP] when special
__global__ void __launch_bounds__(kWpThreads)
wp_write_kernel(WpTables t, const uint8_t* __restrict__ text, const int64_t* __restrict__ offs, int n, int special,
                int cap, const int64_t* __restrict__ cu, int32_t* __restrict__ ids) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int32_t* out = ids + cu[i];
  int mx, nre;
  const int np = wp_text<true>(t, text, offs[i], offs[i + 1], cap, out + special, &mx, &nre);
  if (special) {
    out[0] = t.cls_id;
    out[1 + max(np, 0)] = t.sep_id;
  }
}

// one CTA: cu64[0 .. n] = exclusive prefix sums of count (cu32 the same in int32 when it fits, checked by the
// host against meta[4]); meta[4] = total, meta[5] = longest
__global__ void __launch_bounds__(kWpScanThreads)
wp_scan_kernel(const int32_t* __restrict__ count, int n, int64_t* __restrict__ cu64, int32_t* __restrict__ cu32,
               unsigned long long* __restrict__ meta) {
  __shared__ long long s_sum[kWpScanThreads];
  __shared__ int s_max[kWpScanThreads];
  const int tid = threadIdx.x;
  const long long per = (n + kWpScanThreads - 1ll) / kWpScanThreads;
  const int lo = static_cast<int>(min(static_cast<long long>(n), tid * per));
  const int hi = static_cast<int>(min(static_cast<long long>(n), lo + per));
  long long sum = 0;
  int mx = 0;
  for (int i = lo; i < hi; ++i) { sum += count[i]; mx = max(mx, count[i]); }
  s_sum[tid] = sum;
  s_max[tid] = mx;
  __syncthreads();
  for (int d = 1; d < kWpScanThreads; d <<= 1) {
    const long long x = tid >= d ? s_sum[tid - d] : 0;
    const int y = tid >= d ? s_max[tid - d] : 0;
    __syncthreads();
    s_sum[tid] += x;
    s_max[tid] = max(s_max[tid], y);
    __syncthreads();
  }
  long long run = s_sum[tid] - sum;
  for (int i = lo; i < hi; ++i) {
    cu64[i] = run;
    cu32[i] = static_cast<int32_t>(run);
    run += count[i];
  }
  if (tid == kWpScanThreads - 1) {
    cu64[n] = s_sum[tid];
    cu32[n] = static_cast<int32_t>(s_sum[tid]);
    meta[4] = static_cast<unsigned long long>(s_sum[tid]);
    meta[5] = static_cast<unsigned long long>(s_max[tid]);
  }
}

}  // namespace rse

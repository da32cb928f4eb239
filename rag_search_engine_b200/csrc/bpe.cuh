// bpe.cuh — CLIP's byte-level BPE tokenisation on the device, bit-identical to the HuggingFace fast tokenizer
// (tokenizers: AddedVocabulary -> NFC / Replace(\s+ -> " ") / Lowercase -> Split(CLIP pattern) + ByteLevel -> BPE
// with the "</w>" suffix -> RobertaProcessing).
//
// The tables come from rag_search_engine_b200/bpe.py, probed through the tokenizer's own components:
//   map[cp]     the 0-3 code points the normaliser makes of cp (as in wordpiece.cuh: bits 0-20 the code point or a row
//               of extra[][3], bits 21-22 the count) and bit 23: cp needs the host (NFC could join or reorder it with
//               its neighbours, so the per-code-point map is exact only for texts without such code points)
//   cls[cp]     how the Split pattern sees cp: other / whitespace / \p{L} / \p{N}
//   byte_id[b]  the initial symbol of byte b inside a piece, byte_id[256 + b] as a piece's last byte ("</w>"), unk
//               where the vocab lacks the symbol
//   merges      (left, right) -> (rank, merged) in an open-addressing table, linear probing from bpe_hash
//   the added tokens (the two special tokens, matched literally in the raw text before normalisation, leftmost-longest)
//
// Pieces follow the CLIP pattern's leftmost-first alternation at every match start: the literals "<|startoftext|>" /
// "<|endoftext|>" (reached only through the lowercasing, e.g. "<|ENDOFTEXT|>"), the contractions 's 't 're 've 'm 'll
// 'd, a run of letters, one number, a run of anything else but whitespace.  ByteLevel's own GPT-2 pattern leaves each
// such piece whole except a literal, which it cuts into "<|", the word, "|>".  A piece's bytes become symbols and
// merge like HF's heap: the adjacent pair of lowest rank first, the leftmost of equal ranks (an entry of the heap
// whose pair has changed is skipped there, so its order is exactly this one).
//
// One thread per text: document texts stop at max_length - 2 (75) ids, so a text's work is bounded by the cut and
// not by its length, and a batch of them (600 k movie texts) fills the GPU thread by thread.  The text's tail past
// the cut is only validated (UTF-8, host-route code points), never tokenized.  Count pass, one-CTA scan
// (wordpiece.cuh's), write pass, as in wordpiece.cuh.  A piece longer than kBpeMaxWord bytes that is needed before
// the cut is reported (meta[2]), not truncated: the caller tokenizes that text on the host.
#pragma once
#include <climits>
#include <cstdint>

#include "common.cuh"
#include "wordpiece.cuh"

namespace rse {

constexpr int kBpeMaxWord = 256;     // bytes of one piece the per-thread merge buffer holds
constexpr int kBpeLook = 32;         // normalized code points of look-ahead (a literal is 15)
constexpr uint32_t kBpeRoute = 1u << 23;
constexpr uint8_t kBpeOther = 0, kBpeSpace = 1, kBpeLetter = 2, kBpeNumber = 3;

struct BpeTables {
  const uint32_t* map;
  const uint32_t* extra;
  const uint8_t* cls;
  const int32_t* byte_id;    // [512]
  const int4* merges;        // [merge_mask + 1]: {left, right, rank, merged}, left < 0 empty
  uint32_t merge_mask;
  const uint8_t* added_bytes;
  const int32_t* added_off;  // [n_added + 1]
  const int32_t* added_id;
  int n_added;
  uint32_t added_first[8];   // bit b: some added token starts with byte b
  int bos_id, eos_id;
};

__device__ __forceinline__ uint32_t bpe_hash(int a, int b, uint32_t mask) {
  const unsigned long long key = (static_cast<unsigned long long>(static_cast<uint32_t>(a)) << 32) | static_cast<uint32_t>(b);
  return static_cast<uint32_t>((key * 0x9E3779B97F4A7C15ull) >> 32) & mask;
}

// {rank, merged} of the pair (a, b), rank INT_MAX when it has no merge
__device__ __forceinline__ int2 bpe_merge(const BpeTables& t, int a, int b) {
  uint32_t s = bpe_hash(a, b, t.merge_mask);
  while (true) {
    const int4 m = __ldg(&t.merges[s]);
    if (m.x == a && m.y == b) return make_int2(m.z, m.w);
    if (m.x < 0) return make_int2(INT_MAX, -1);
    s = (s + 1) & t.merge_mask;
  }
}

// The normalized code points of one segment of raw text (between special tokens), with look-ahead.  peek(k) is the
// k-th code point from the current one, -1 past the segment's end; a malformed byte sets bad and ends the segment.
struct BpeStream {
  const BpeTables* t;
  const uint8_t* s;
  int64_t p, e;
  uint32_t q[kBpeLook];
  int head = 0, n = 0;
  bool bad = false;

  __device__ bool fill() {
    if (p >= e || bad || n + 3 > kBpeLook) return false;
    uint32_t cp;
    const int nb = wp_utf8(s, p, e, &cp);
    if (nb == 0) { bad = true; return false; }
    p += nb;
    const uint32_t m = t->map[cp];
    const int cnt = (m >> 21) & 3;
    for (int k = 0; k < cnt; ++k)
      q[(head + n++) & (kBpeLook - 1)] = cnt == 1 ? (m & kWpCpMask) : t->extra[3 * (m & kWpCpMask) + k];
    return true;
  }
  __device__ int peek(int k) {
    while (n <= k)
      if (!fill()) return -1;
    return static_cast<int>(q[(head + k) & (kBpeLook - 1)]);
  }
  __device__ void pop() { head = (head + 1) & (kBpeLook - 1); --n; }
};

__device__ __forceinline__ int bpe_utf8_put(uint32_t c, uint8_t* o) {
  if (c < 0x80) { o[0] = static_cast<uint8_t>(c); return 1; }
  if (c < 0x800) { o[0] = 0xC0 | (c >> 6); o[1] = 0x80 | (c & 0x3F); return 2; }
  if (c < 0x10000) { o[0] = 0xE0 | (c >> 12); o[1] = 0x80 | ((c >> 6) & 0x3F); o[2] = 0x80 | (c & 0x3F); return 3; }
  o[0] = 0xF0 | (c >> 18); o[1] = 0x80 | ((c >> 12) & 0x3F); o[2] = 0x80 | ((c >> 6) & 0x3F); o[3] = 0x80 | (c & 0x3F);
  return 4;
}

// The ids of one text (special tokens of the template not included): kept ids go to out[0 .. cap) when WRITE.
// Returns min(ids, cap), -1 for malformed UTF-8, -2 for a text the host must tokenize.  *max_id: the largest kept id.
template <bool WRITE>
__device__ int bpe_text(const BpeTables& t, const uint8_t* __restrict__ s, int64_t p, const int64_t e, int cap,
                        int32_t* __restrict__ out, int* max_id) {
  int sym[kBpeMaxWord];   // the piece's symbols, merged in place
  int rk[kBpeMaxWord];    // rk[i]: the rank of the pair (sym[i], sym[i + 1])
  int wl = 0, np = 0, mx = -1;
  bool refuse = false;
  auto emit = [&](int id) {
    if (np < cap) {
      if (WRITE) out[np] = id;
      mx = max(mx, id);
    }
    ++np;
  };
  // one more byte of the piece: its symbol as an inner byte; the piece's last one is re-read at flush
  uint8_t last = 0;
  auto add_byte = [&](uint8_t b) {
    if (wl < kBpeMaxWord) sym[wl] = t.byte_id[b];
    last = b;
    ++wl;
  };
  auto add_cp = [&](uint32_t c) {
    uint8_t u[4];
    const int k = bpe_utf8_put(c, u);
    for (int j = 0; j < k; ++j) add_byte(u[j]);
  };
  auto flush = [&]() {
    if (wl == 0) return;
    if (wl > kBpeMaxWord) { refuse = true; wl = 0; return; }
    const int n0 = wl;
    int n = n0;
    sym[n - 1] = t.byte_id[256 + last];
    for (int i = 0; i + 1 < n; ++i) rk[i] = bpe_merge(t, sym[i], sym[i + 1]).x;
    while (n > 1) {
      int best = INT_MAX, bi = -1;
      for (int i = 0; i + 1 < n; ++i)
        if (rk[i] < best) { best = rk[i]; bi = i; }
      if (bi < 0) break;
      sym[bi] = bpe_merge(t, sym[bi], sym[bi + 1]).y;
      for (int i = bi + 1; i + 1 < n; ++i) sym[i] = sym[i + 1];
      for (int i = bi + 1; i + 2 < n; ++i) rk[i] = rk[i + 1];
      --n;
      if (bi > 0) rk[bi - 1] = bpe_merge(t, sym[bi - 1], sym[bi]).x;
      if (bi + 1 < n) rk[bi] = bpe_merge(t, sym[bi], sym[bi + 1]).x;
    }
    for (int i = 0; i < n && np < cap; ++i) emit(sym[i]);
    wl = 0;
  };
  auto word = [&](const char* w) {
    for (; *w; ++w) add_byte(static_cast<uint8_t>(*w));
    flush();
  };
  const int64_t start = p;
  // pieces, segment by segment, until the cut
  while (p < e && np < cap && !refuse) {
    // the segment runs to the next special token (leftmost, then longest) or the end
    int64_t q = p;
    int sp_id = -1, sp_len = 0;
    for (; q < e; ++q) {
      const uint32_t b0 = s[q];
      if (!((t.added_first[b0 >> 5] >> (b0 & 31)) & 1u)) continue;
      for (int a = 0; a < t.n_added; ++a) {
        const int o = t.added_off[a], L = t.added_off[a + 1] - o;
        if (L <= sp_len || q + L > e) continue;
        int k = 0;
        while (k < L && s[q + k] == t.added_bytes[o + k]) ++k;
        if (k == L) { sp_id = t.added_id[a]; sp_len = L; }
      }
      if (sp_id >= 0) break;
    }
    BpeStream st{&t, s, p, q};
    int c;
    while (np < cap && !refuse && (c = st.peek(0)) >= 0) {
      const uint8_t k = t.cls[c];
      if (k == kBpeSpace) { st.pop(); continue; }
      if (k == kBpeLetter || k == kBpeNumber) {
        do { add_cp(static_cast<uint32_t>(c)); st.pop(); } while (k == kBpeLetter && (c = st.peek(0)) >= 0 && t.cls[c] == kBpeLetter);
        flush();
        continue;
      }
      if (c == '<') {                      // the pattern's literals, after lowercasing
        const char* lit[2] = {"<|startoftext|>", "<|endoftext|>"};
        const char* mid[2] = {"startoftext", "endoftext"};
        int hit = -1;
        for (int a = 0; a < 2 && hit < 0; ++a) {
          int j = 0;
          while (lit[a][j] && st.peek(j) == lit[a][j]) ++j;
          if (!lit[a][j]) hit = a;
        }
        if (hit >= 0) {
          for (int j = 0; lit[hit][j]; ++j) st.pop();
          word("<|");
          if (np < cap) word(mid[hit]);
          if (np < cap) word("|>");
          continue;
        }
      } else if (c == '\'') {              // 's 't 're 've 'm 'll 'd
        const int c1 = st.peek(1);
        int len = 0;
        if (c1 == 's' || c1 == 't' || c1 == 'm' || c1 == 'd') len = 2;
        else if ((c1 == 'r' || c1 == 'v') && st.peek(2) == 'e') len = 3;
        else if (c1 == 'l' && st.peek(2) == 'l') len = 3;
        if (len) {
          for (int j = 0; j < len; ++j) { add_cp(static_cast<uint32_t>(st.peek(0))); st.pop(); }
          flush();
          continue;
        }
      }
      do { add_cp(static_cast<uint32_t>(c)); st.pop(); } while ((c = st.peek(0)) >= 0 && t.cls[c] == kBpeOther);
      flush();
    }
    if (st.bad) return -1;
    if (np >= cap || refuse) { p = st.p; break; }
    p = q;
    if (sp_id >= 0) { emit(sp_id); p += sp_len; }
  }
  // the whole text is validated (and checked for host-route code points), tokenized or not
  bool route = false;
  for (int64_t r = start; r < e;) {
    uint32_t cp;
    const int nb = wp_utf8(s, r, e, &cp);
    if (nb == 0) return -1;
    r += nb;
    route |= (t.map[cp] & kBpeRoute) != 0;
  }
  *max_id = mx;
  if (route || refuse) return -2;
  return min(np, cap);
}

// count pass: count[i] = ids of text i (bos / eos included); meta as wordpiece.cuh's, [2] / [3] the texts the host
// must tokenize
__global__ void __launch_bounds__(kWpThreads)
bpe_count_kernel(BpeTables t, const uint8_t* __restrict__ text, const int64_t* __restrict__ offs, int n, int special,
                 int cap, int32_t* __restrict__ count, unsigned long long* __restrict__ meta) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int mx = -1;
  int np = bpe_text<false>(t, text, offs[i], offs[i + 1], cap, nullptr, &mx);
  if (np == -1) {
    atomicAdd(&meta[0], 1ull);
    atomicMin(&meta[1], static_cast<unsigned long long>(i));
    np = 0;
  } else if (np == -2) {
    atomicAdd(&meta[2], 1ull);
    atomicMin(&meta[3], static_cast<unsigned long long>(i));
    np = 0;
  }
  if (special) mx = max(mx, max(t.bos_id, t.eos_id));
  if (mx >= 0) atomicMax(&meta[6], static_cast<unsigned long long>(mx));
  count[i] = np + 2 * special;
}

// write pass: text i's ids at ids[cu[i] ..), bos ... eos when special
__global__ void __launch_bounds__(kWpThreads)
bpe_write_kernel(BpeTables t, const uint8_t* __restrict__ text, const int64_t* __restrict__ offs, int n, int special,
                 int cap, const int64_t* __restrict__ cu, int32_t* __restrict__ ids) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int32_t* out = ids + cu[i];
  int mx;
  const int np = bpe_text<true>(t, text, offs[i], offs[i + 1], cap, out + special, &mx);
  if (special) {
    out[0] = t.bos_id;
    out[1 + max(np, 0)] = t.eos_id;
  }
}

// cu[0 .. n] -> cu[k] - cu[0] for one slice of a CLIP text batch (its positions in the slice's own rows)
__global__ void bpe_rebase_kernel(const int32_t* __restrict__ cu, int n, int32_t* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i <= n) out[i] = cu[i] - cu[0];
}

}  // namespace rse

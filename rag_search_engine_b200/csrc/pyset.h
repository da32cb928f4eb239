// pyset.h — iteration-order emulation of CPython's `set` for int keys.
//
// Why this exists: the reference builds the fused candidate list by iterating
// `set(bm25.keys()) | set(sem.keys())` (rag_search_engine/utils/hybrid_search.py:148,
// :248) and then stable-sorts by score, so the order of equal-score results —
// and therefore WHICH ids survive the `[:limit]` cut — is the iteration order of
// that set (SURVEY App. A.5).  RRF ties are structural (a BM25-only doc at rank
// r and a semantic-only doc at rank r get the identical double), so bit-exact
// top-k parity needs this order.
//
// This is a restatement of the open-addressing scheme of CPython 3.11/3.12
// Objects/setobject.c (set_add_entry, set_insert_clean, set_table_resize,
// set_merge): 8 initial slots, slot = hash & mask, LINEAR_PROBES = 9, then
// i = i*5 + 1 + (perturb >>= 5); grow by 4x used when fill*5 >= mask*3;
// `a | b` = copy of a (an empty set merged with a) then merge(b) in b's TABLE
// order.  hash(int) = the value itself for |v| < 2**61-1 (-1 -> -2).
// No deletions ever happen on this path, so there are no dummy entries.
// Checked against the real CPython set, for both slot kinds below, in tests/test_host_cpu.py and
// tests/test_pyset_indexed.py (not GPU).
//
// Header-only, host + device (plain C++), no allocation: the caller provides
// the tables.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define RSE_HD __host__ __device__ __forceinline__
#else
#define RSE_HD inline
#endif

namespace rse {

constexpr int64_t kPySetEmpty = INT64_MIN;   // never a valid document id
constexpr int kPySetMinSize = 8;
constexpr int kPySetLinearProbes = 9;
constexpr int kPySetPerturbShift = 5;

// CPython long hash: value mod (2**61 - 1), sign preserved, -1 mapped to -2.
RSE_HD int64_t py_hash_int(int64_t v) {
  const uint64_t P = (1ull << 61) - 1ull;
  uint64_t mag = v < 0 ? (0ull - static_cast<uint64_t>(v)) : static_cast<uint64_t>(v);
  uint64_t m = mag < P ? mag : mag % P;        // ids are far below 2**61: skip the 64-bit division
  int64_t h = v < 0 ? -static_cast<int64_t>(m) : static_cast<int64_t>(m);
  if (h == -1) h = -2;
  return h;
}

// A table slot holds either the key itself (PySetKeys: 8-byte slots) or a 16-bit index into one staged key array
// (PySetIndexedKeys: a quarter of the storage, what lets the fusion kernel keep the sets of a 1024-deep union in
// shared memory).  Hashes and equality are always taken from the key, so both give CPython's iteration order.
// The policies also name the slot of the i-th key of operand a and of operand b.
struct PySetKeys {
  using Slot = int64_t;
  static constexpr Slot kEmpty = kPySetEmpty;
  const int64_t* a;
  const int64_t* b;
  RSE_HD int64_t key(Slot s) const { return s; }
  RSE_HD Slot a_slot(int i) const { return a[i]; }
  RSE_HD Slot b_slot(int i) const { return b[i]; }
};
struct PySetIndexedKeys {
  using Slot = uint16_t;
  static constexpr Slot kEmpty = 0xFFFF;     // keys[] holds fewer than 65535 entries
  const int64_t* keys;                       // operand a at keys[0 .. na), operand b at keys[b_off .. b_off + nb)
  int b_off;
  RSE_HD int64_t key(Slot s) const { return keys[s]; }
  RSE_HD Slot a_slot(int i) const { return static_cast<Slot>(i); }
  RSE_HD Slot b_slot(int i) const { return static_cast<Slot>(b_off + i); }
};

template <class K>
struct PySet {
  typename K::Slot* table;   // capacity `cap` entries, K::kEmpty = unused
  int cap;                   // storage capacity (power of two)
  int mask;                  // current table size - 1
  int used;                  // == fill (no dummies)
};

template <class K>
RSE_HD void pyset_init(PySet<K>* s, typename K::Slot* storage, int cap) {
  s->table = storage; s->cap = cap; s->mask = kPySetMinSize - 1; s->used = 0;
  for (int i = 0; i < kPySetMinSize; ++i) storage[i] = K::kEmpty;
}

// set_insert_clean: key known absent, table has no dummies.
template <class K>
RSE_HD void pyset_insert_clean(const K& k, typename K::Slot* table, uint64_t mask, typename K::Slot entry) {
  const uint64_t hash = static_cast<uint64_t>(py_hash_int(k.key(entry)));
  uint64_t perturb = hash;
  uint64_t i = hash & mask;
  while (true) {
    if (table[i] == K::kEmpty) { table[i] = entry; return; }
    if (i + kPySetLinearProbes <= mask) {
      for (int j = 1; j <= kPySetLinearProbes; ++j) {
        if (table[i + j] == K::kEmpty) { table[i + j] = entry; return; }
      }
    }
    perturb >>= kPySetPerturbShift;
    i = (i * 5 + 1 + perturb) & mask;
  }
}

// set_table_resize(so, minused) through `scratch` (capacity >= new size).
// Returns false when the new size exceeds the storage.
template <class K>
RSE_HD bool pyset_resize(const K& k, PySet<K>* s, int minused, typename K::Slot* scratch, int scratch_cap) {
  int newsize = kPySetMinSize;
  while (newsize <= minused) newsize <<= 1;
  if (newsize > s->cap || newsize > scratch_cap) return false;
  for (int i = 0; i < newsize; ++i) scratch[i] = K::kEmpty;
  const uint64_t newmask = static_cast<uint64_t>(newsize - 1);
  for (int i = 0; i <= s->mask; ++i)
    if (s->table[i] != K::kEmpty) pyset_insert_clean(k, scratch, newmask, s->table[i]);
  for (int i = 0; i < newsize; ++i) s->table[i] = scratch[i];
  s->mask = newsize - 1;
  return true;
}

// set_add_entry
template <class K>
RSE_HD bool pyset_add(const K& k, PySet<K>* s, typename K::Slot entry, typename K::Slot* scratch, int scratch_cap) {
  const int64_t key = k.key(entry);
  const uint64_t hash = static_cast<uint64_t>(py_hash_int(key));
  const uint64_t mask = static_cast<uint64_t>(s->mask);
  uint64_t perturb = hash;
  uint64_t i = hash & mask;
  while (true) {
    int probes = (i + kPySetLinearProbes <= mask) ? kPySetLinearProbes : 0;
    uint64_t e = i;
    bool placed = false;
    do {
      if (s->table[e] == K::kEmpty) { placed = true; break; }
      if (k.key(s->table[e]) == key) return true;   // found_active
      ++e;
    } while (probes--);
    if (placed) {
      s->table[e] = entry;
      s->used++;
      if (static_cast<uint64_t>(s->used) * 5 < mask * 3) return true;
      return pyset_resize(k, s, s->used > 50000 ? s->used * 2 : s->used * 4, scratch, scratch_cap);
    }
    perturb >>= kPySetPerturbShift;
    i = (i * 5 + 1 + perturb) & mask;
  }
}

// set_merge(so, other)
template <class K>
RSE_HD bool pyset_merge(const K& k, PySet<K>* so, const PySet<K>* other, typename K::Slot* scratch, int scratch_cap) {
  if (other->used == 0) return true;
  if (static_cast<uint64_t>(so->used + other->used) * 5 >= static_cast<uint64_t>(so->mask) * 3) {
    if (!pyset_resize(k, so, (so->used + other->used) * 2, scratch, scratch_cap)) return false;
  }
  if (so->used == 0 && so->mask == other->mask) {   // same size, empty target: copy slots verbatim
    for (int i = 0; i <= other->mask; ++i) so->table[i] = other->table[i];
    so->used = other->used;
    return true;
  }
  if (so->used == 0) {                               // empty target: insert_clean in other's table order
    so->used = other->used;
    for (int i = 0; i <= other->mask; ++i)
      if (other->table[i] != K::kEmpty)
        pyset_insert_clean(k, so->table, static_cast<uint64_t>(so->mask), other->table[i]);
    return true;
  }
  for (int i = 0; i <= other->mask; ++i)
    if (other->table[i] != K::kEmpty)
      if (!pyset_add(k, so, other->table[i], scratch, scratch_cap)) return false;
  return true;
}

// Storage needed (entries) for a set that will hold up to n keys via pyset_add /
// pyset_merge: the largest table CPython can reach is < 8*n (grow to > 4*used).
RSE_HD int pyset_capacity_for(int n) {
  int c = kPySetMinSize;
  while (c <= 4 * n) c <<= 1;
  return c;
}

// Iteration order of  set(a_keys) | set(b_keys)  where both operands are built by
// adding the keys in list order (hybrid_search.py:148, :248).  Writes the union
// to `out` (capacity na+nb) and returns its size, or -1 if storage was too small.
//   ta/tb/tr: storage for the three sets; scratch: resize buffer.
template <class K>
RSE_HD int pyset_union_order(const K& k, int na, int nb, typename K::Slot* ta, int cap_a, typename K::Slot* tb,
                             int cap_b, typename K::Slot* tr, int cap_r, typename K::Slot* scratch, int scratch_cap,
                             int64_t* out) {
  PySet<K> A, B, R;
  pyset_init(&A, ta, cap_a);
  pyset_init(&B, tb, cap_b);
  pyset_init(&R, tr, cap_r);
  for (int i = 0; i < na; ++i)
    if (!pyset_add(k, &A, k.a_slot(i), scratch, scratch_cap)) return -1;
  for (int i = 0; i < nb; ++i)
    if (!pyset_add(k, &B, k.b_slot(i), scratch, scratch_cap)) return -1;
  if (!pyset_merge(k, &R, &A, scratch, scratch_cap)) return -1;   // set_copy(A)
  if (!pyset_merge(k, &R, &B, scratch, scratch_cap)) return -1;   // |= B
  int n = 0;
  for (int i = 0; i <= R.mask; ++i)
    if (R.table[i] != K::kEmpty) out[n++] = k.key(R.table[i]);
  return n;
}

// The same on 8-byte key slots.
RSE_HD int pyset_union_order(const int64_t* a_keys, int na, const int64_t* b_keys, int nb, int64_t* ta,
                             int cap_a, int64_t* tb, int cap_b, int64_t* tr, int cap_r, int64_t* scratch,
                             int scratch_cap, int64_t* out) {
  return pyset_union_order(PySetKeys{a_keys, b_keys}, na, nb, ta, cap_a, tb, cap_b, tr, cap_r, scratch, scratch_cap,
                           out);
}

}  // namespace rse

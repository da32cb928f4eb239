// Host build of the 16-bit index-slot variant of csrc/pyset.h (the one the deep fusion kernel uses), next to the
// key-slot shim it extends (tests/test_pyset_indexed.py).
#include "pyset_shim.cpp"
extern "C" int pyset_shim_union_indexed(const int64_t* a, int na, const int64_t* b, int nb, int64_t* out) {
  std::vector<int64_t> keys(a, a + na);
  keys.insert(keys.end(), b, b + nb);
  int ca = rse::pyset_capacity_for(na), cb = rse::pyset_capacity_for(nb), cr = rse::pyset_capacity_for(na + nb);
  std::vector<uint16_t> ta(ca), tb(cb), tr(cr), sc(cr);
  return rse::pyset_union_order(rse::PySetIndexedKeys{keys.data(), na}, na, nb, ta.data(), ca, tb.data(), cb, tr.data(),
                                cr, sc.data(), cr, out);
}

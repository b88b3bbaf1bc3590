// TEST-ONLY host simulation of the per-thread body of k_miller_tables (csrc/miller_tables.cuh: miller_tables_item) for
// M = 1, 2, 4 pairs per item.  Used by tests/test_miller_tables_hostsim.py.
#include "../../sylow_b200/csrc/miller_tables.cuh"

#include <cstring>
#include <vector>

using namespace sylow;

extern "C" {

// out (canonical Fp12) = item `item` of m pairs over n_tables device-form tables (Montgomery limbs), n_pairs G1 points
// (wire form) and optional flags / indices.  The inputs are copied to 16-byte aligned buffers (the body loads uint4).
void hs_miller_tables(int m, const uint8_t* tables, size_t n_tables, const uint32_t* idx, const uint8_t* g1,
                      const uint8_t* g1_inf, size_t n_pairs, size_t item, uint8_t* out) {
  std::vector<uint4> t(n_tables * SY_TABLE_BYTES / 16), p(n_pairs * 4), o(24);
  memcpy(t.data(), tables, n_tables * SY_TABLE_BYTES);
  memcpy(p.data(), g1, n_pairs * 64);
  const uint8_t* tb = reinterpret_cast<const uint8_t*>(t.data());
  const uint8_t* pb = reinterpret_cast<const uint8_t*>(p.data());
  Fp12 f;
  if (m == 4)
    f = miller_tables_item<4>(tb, n_tables, idx, pb, g1_inf, item);
  else if (m == 2)
    f = miller_tables_item<2>(tb, n_tables, idx, pb, g1_inf, item);
  else
    f = miller_tables_item<1>(tb, n_tables, idx, pb, g1_inf, item);
  fp12_store(reinterpret_cast<uint8_t*>(o.data()), f);
  memcpy(out, o.data(), 384);
}

}  // extern "C"

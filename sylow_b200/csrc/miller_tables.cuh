// Miller loops over per-pair precomputed G2 tables (G2PreComputed::miller_loop, pairing.rs:590-619, and
// glued_miller_loop(&[G2PreComputed], &[G1Affine]), :970-1022), one item of M pairs per thread.
// Kept apart from the kernel so that the host simulation (tests/hostsim/miller_tables.cu) runs the same body.
#pragma once
#include "wire.cuh"

// One table: 87 Ell triples (c0, c1, c2), Montgomery form, 192 bytes each (the device form of
// sylow_b200_tables_to_device and sylow_b200_g2_precompute_dev).
#define SY_TABLE_BYTES (87 * 192)

namespace sylow {

// Item `item` multiplies the Miller values of pairs [item * M, item * M + M): pair k is g1[k] against table
// table_idx[k] (table k if table_idx is null), a flagged-infinite G1 point contributes 1 (MillerG1::skip).  A table
// index >= n_tables reads table 0 instead (never out of bounds) and makes the item's value the Fp12 zero, so a product
// over it is zero and its final exponentiation is zero, never the identity.  Montgomery form out.  n_tables >= 1.
template <int M>
SY_HD Fp12 miller_tables_item(const uint8_t* tables, size_t n_tables, const uint32_t* table_idx, const uint8_t* g1,
                              const uint8_t* g1_inf, size_t item, Fp12* acc = nullptr) {
  MillerG1 p[M];
  const Ell* tabs[M];
  bool bad = false;
  for (int j = 0; j < M; j++) {
    const size_t k = item * M + j;
    const size_t t = table_idx ? (size_t)table_idx[k] : k;
    const bool oob = t >= n_tables;
    bad |= oob;
    tabs[j] = reinterpret_cast<const Ell*>(tables + (oob ? 0 : t) * SY_TABLE_BYTES);
    p[j].x = fp_load(g1 + k * 64);
    p[j].y = fp_load(g1 + k * 64 + 32);
    p[j].skip = g1_inf && g1_inf[k];
  }
  Fp12 f = glued_miller_loop<0, M, 1>(p, nullptr, nullptr, tabs, acc);
  if (bad) f = Fp12{fp6_zero(), fp6_zero()};
  return f;
}

}  // namespace sylow

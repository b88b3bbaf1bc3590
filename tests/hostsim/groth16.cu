// TEST-ONLY host simulation of the per-thread bodies of the Groth16 kernels (csrc/groth16.cuh): k_groth16_assemble
// (groth16_public_term, put_point's negated affine -L, groth16_record) and the weighted Fr sums of
// k_groth16_fr_partial / k_groth16_fr_final (fr_words_canonical, fr_weighted, fr_add, fr_unscale).  Used by
// tests/test_groth16_hostsim.py.
#include "../../sylow_b200/csrc/groth16.cuh"

#include <cstring>
#include <vector>

using namespace sylow;

extern "C" {

void hs_g16_layout(size_t* neg_alpha, size_t* ic0, size_t* tables, size_t* table_bytes) {
  *neg_alpha = kG16NegAlpha;
  *ic0 = kG16Ic0;
  *tables = kG16Tables;
  *table_bytes = kG16IcTable;
}

// The record of one proof against the device-form key vk (l inputs x, proof A || B || C, flags inf[3] or null):
// rec = [A, -alpha, -L, -C] (256 B), rec_inf[4], b (128 B), *b_inf, *in_range.
void hs_g16_assemble(const uint8_t* vk, size_t vk_bytes, size_t l, const uint8_t* x, const uint8_t* proof,
                     const uint8_t* inf, uint8_t* rec, uint8_t* rec_inf, uint8_t* b, uint8_t* b_inf, int* in_range) {
  std::vector<uint4> k(vk_bytes / 16), xs(2 * l + 1), p(16), r(16), q(8);
  memcpy(k.data(), vk, vk_bytes);
  memcpy(xs.data(), x, 32 * l);
  memcpy(p.data(), proof, 256);
  const uint8_t* kv = reinterpret_cast<const uint8_t*>(k.data());
  uint8_t* rv = reinterpret_cast<uint8_t*>(r.data());
  bool ok;
  Affine<Fp> L = proj_to_affine(groth16_public_term(kv, l, reinterpret_cast<const uint8_t*>(xs.data()), ok));
  if (!L.inf) L.y = fp_neg(L.y);  // put_point with negate
  fp_store(rv + 128, L.x);
  fp_store(rv + 160, L.y);
  rec_inf[2] = L.inf;
  groth16_record(kv, reinterpret_cast<const uint8_t*>(p.data()), inf, rv, rec_inf, reinterpret_cast<uint8_t*>(q.data()),
                 b_inf);
  memcpy(rec, rv, 256);
  memcpy(b, q.data(), 128);
  *in_range = ok;
}

// out = sum_j r_j x_j mod r (canonical), summed as the kernels do: per-"thread" partials over a stride of `threads`
// proofs, then the partials added up, then one fr_unscale.  x null: every x_j = 1 (s_0 = sum r_j).  *in_range: all x_j < r.
void hs_g16_weighted_sum(const uint8_t* x, const uint64_t* r, size_t n, size_t threads, uint8_t* out, int* in_range) {
  const uint32_t one[8] = {1, 0, 0, 0, 0, 0, 0, 0};
  std::vector<Fr> part(threads, Fr{});
  bool ok = true;
  for (size_t j = 0; j < n; j++) {
    uint32_t w[8];
    if (x) {
      memcpy(w, x + 32 * j, 32);
      ok &= fr_words_canonical(w);
    } else {
      memcpy(w, one, 32);
    }
    part[j % threads] = fr_add(part[j % threads], fr_weighted(w, r[j]));
  }
  Fr acc{};
  for (const Fr& v : part) acc = fr_add(acc, v);
  acc = fr_unscale(acc);
  memcpy(out, acc.l, 32);
  *in_range = ok;
}

}  // extern "C"

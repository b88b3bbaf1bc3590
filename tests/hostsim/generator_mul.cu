// TEST-ONLY host simulation of the per-thread body of k_g1_mul_gen / k_g2_mul_gen (csrc/curve.cuh: scalar_reduce_r,
// scalar_digit, proj_add_mixed, gen_scalar_mul).  Used by tests/test_generator_mul_hostsim.py.
#include "../../sylow_b200/csrc/wire.cuh"

#include <cstring>
#include <vector>

using namespace sylow;

namespace {
// canonical wire values -> Montgomery form; the inputs are copied to 16-byte aligned storage (the loads are uint4)
Fp ld(const uint8_t* p, Fp*) {
  alignas(16) uint8_t b[32];
  memcpy(b, p, 32);
  return fp_load(b);
}
Fp2 ld(const uint8_t* p, Fp2*) { return Fp2{ld(p, (Fp*)nullptr), ld(p + 32, (Fp*)nullptr)}; }
void st(uint8_t* p, const Fp& v) {
  alignas(16) uint8_t b[32];
  fp_store(b, v);
  memcpy(p, b, 32);
}
void st(uint8_t* p, const Fp2& v) {
  st(p, v.c0);
  st(p + 32, v.c1);
}
template <class F>
void store_affine(const Proj<F>& q, uint8_t* out, uint8_t* out_inf) {
  Affine<F> r = proj_to_affine(q);
  st(out, r.x);
  st(out + sizeof(F), r.y);
  *out_inf = r.inf;
}
template <class F>
void add_mixed(const uint8_t* acc, const uint8_t* e, uint8_t* out, uint8_t* out_inf) {
  constexpr size_t W = sizeof(F);
  Proj<F> a{ld(acc, (F*)nullptr), ld(acc + W, (F*)nullptr), ld(acc + 2 * W, (F*)nullptr)};
  Affine<F> b{ld(e, (F*)nullptr), ld(e + W, (F*)nullptr), false};
  store_affine(proj_add_mixed(a, b), out, out_inf);
}
template <class F>
void gen_mul(const uint8_t* table, size_t table_bytes, const uint8_t* k, uint8_t* out, uint8_t* out_inf) {
  std::vector<uint4> t(table_bytes / 16);
  memcpy(t.data(), table, table_bytes);
  uint32_t kw[8];
  memcpy(kw, k, 32);
  store_affine(gen_scalar_mul<F>(reinterpret_cast<const uint8_t*>(t.data()), kw), out, out_inf);
}
}  // namespace

extern "C" {

void hs_gen_params(int* c, int* w, int* e) {
  *c = SY_GEN_C;
  *w = SY_GEN_W;
  *e = SY_GEN_E;
}

// k mod r (32 bytes LE) and its SY_GEN_W signed digits, least significant first
void hs_gen_digits(const uint8_t* k, int* digits, uint8_t* k_mod_r) {
  uint32_t kw[8];
  memcpy(kw, k, 32);
  scalar_reduce_r(kw);
  memcpy(k_mod_r, kw, 32);
  int carry = 0;
  for (int w = 0; w < SY_GEN_W; w++) digits[w] = scalar_digit<SY_GEN_C>(kw, w, carry);
}

// affine(acc + e) for a canonical projective acc (x, y, z) and a canonical affine e (x, y); g2 selects the group
void hs_add_mixed(int g2, const uint8_t* acc, const uint8_t* e, uint8_t* out, uint8_t* out_inf) {
  if (g2)
    add_mixed<Fp2>(acc, e, out, out_inf);
  else
    add_mixed<Fp>(acc, e, out, out_inf);
}

// affine(k G) over the device-form table of G (SY_GEN_W x SY_GEN_E affine entries, Montgomery form)
void hs_gen_mul(int g2, const uint8_t* table, size_t table_bytes, const uint8_t* k, uint8_t* out, uint8_t* out_inf) {
  if (g2)
    gen_mul<Fp2>(table, table_bytes, k, out, out_inf);
  else
    gen_mul<Fp>(table, table_bytes, k, out, out_inf);
}

}  // extern "C"

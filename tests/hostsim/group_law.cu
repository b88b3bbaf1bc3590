// TEST-ONLY host simulation of the per-item bodies of k_g1_add / k_g2_add and of the EIP-196 steps (csrc/group_law.cuh:
// add_pair, decode_be_item, g1_validate_item, eip196_scalar_item, eip196_finish_item).  Used by
// tests/test_group_law_hostsim.py.
#include "../../sylow_b200/csrc/group_law.cuh"

#include <cstring>

using namespace sylow;

namespace {
void st(uint8_t* p, const Fp& v) {
  alignas(16) uint8_t b[32];
  fp_store(b, v);
  memcpy(p, b, 32);
}
void st(uint8_t* p, const Fp2& v) {
  st(p, v.c0);
  st(p + 32, v.c1);
}
// the kernels' small-batch path: add_pair, then proj_to_affine in the same thread
template <class F>
void add(const uint8_t* a, int a_inf, const uint8_t* b, int b_inf, int subtract, uint8_t* out, uint8_t* out_inf) {
  constexpr size_t W = sizeof(F);
  alignas(16) uint8_t ab[2 * W], bb[2 * W];  // the loads are uint4
  memcpy(ab, a, 2 * W);
  memcpy(bb, b, 2 * W);
  const uint8_t ai = (uint8_t)a_inf, bi = (uint8_t)b_inf;
  Affine<F> r = proj_to_affine(add_pair<F>(ab, &ai, bb, &bi, 0, subtract));
  st(out, r.x);
  st(out + W, r.y);
  *out_inf = r.inf;
}
}  // namespace

extern "C" {

// affine(a +- b) for canonical affine points with infinity flags; g2 selects the group
void hs_add_pair(int g2, const uint8_t* a, int a_inf, const uint8_t* b, int b_inf, int subtract, uint8_t* out,
                 uint8_t* out_inf) {
  if (g2)
    add<Fp2>(a, a_inf, b, b_inf, subtract, out, out_inf);
  else
    add<Fp>(a, a_inf, b, b_inf, subtract, out, out_inf);
}

// The steps of sylow_b200_eip196_add_batch / _mul_batch before the group operation, for one input (mul = 0: ecAdd,
// 128 bytes; mul = 1: ecMul, 96 bytes): decode (mode 1) and validate each point; for ecMul also the scalar
void hs_eip196_decode(const uint8_t* in, int mul, uint8_t* pts /* 2 x 64 */, uint8_t* infs /* 2 */, int8_t* sts /* 2 */,
                      uint8_t* scalar_le) {
  alignas(16) uint8_t p[128];
  for (int j = 0; j < (mul ? 1 : 2); j++) {
    decode_be_item<2>(in + 64 * j, 1, p + 64 * j, infs + j, sts + j);
    sts[j] = g1_validate_item(p, infs, sts, j, 1);
  }
  memcpy(pts, p, 128);
  if (mul) eip196_scalar_item(in + 64, scalar_le);
}
// the whole ecAdd body of one input
void hs_eip196_add(const uint8_t* in, uint8_t* out, int8_t* status) {
  alignas(16) uint8_t p[128], r[64];
  uint8_t inf[2];
  int8_t sts[2];
  hs_eip196_decode(in, 0, p, inf, sts, nullptr);
  Affine<Fp> a = proj_to_affine(add_pair<Fp>(p, inf, p + 64, inf + 1, 0, 0));
  fp_store(r, a.x);
  fp_store(r + 32, a.y);
  eip196_finish_item(r, a.inf, sts[0], sts[1], out, status);
}
// the epilogue of one input: status fold and big-endian encoding of a wire-form result
void hs_eip196_finish(const uint8_t* pt, int inf, int st_a, int st_b, uint8_t* out, int8_t* status) {
  alignas(16) uint8_t p[64];
  memcpy(p, pt, 64);
  eip196_finish_item(p, inf != 0, (int8_t)st_a, (int8_t)st_b, out, status);
}

}  // extern "C"

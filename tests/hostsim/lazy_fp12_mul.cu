// TEST-ONLY host simulation of the lazily reduced Fp12 product (tower.cuh: fp4_mul_redc, fp12_mul_assign) on RAW
// Montgomery limbs, so that the tests can place operands exactly at the stated bounds.  The host build aborts when an
// fp4_mul_redc output reaches 2^256 or a lin9_reduce input reaches 2^262.  Used by tests/test_lazy_fp12_mul.py.
#include "../../sylow_b200/csrc/tower.cuh"

#include <cstring>

using namespace sylow;

extern "C" {

// one Fp4 product: in = x0, x1, y0, y1 (4 Fp2, 64 words), out = the four unreduced outputs V (32 words)
void hs_fp4_mul_redc(const uint32_t* in, uint32_t* out) {
  Fp2 v[4];
  Fp V[4];
  memcpy(v, in, sizeof(v));
  fp4_mul_redc(V, v[0], v[1], v[2], v[3]);
  memcpy(out, V, sizeof(V));
}

// a <- a b or a conj(b) on 12 raw coefficients each (96 words)
void hs_fp12_mul_assign(const uint32_t* a, const uint32_t* b, int conj_b, uint32_t* out) {
  Fp12 f, g;
  memcpy(&f, a, sizeof(f));
  memcpy(&g, b, sizeof(g));
  fp12_mul_assign(f, g, conj_b != 0);
  memcpy(out, &f, sizeof(f));
}

}  // extern "C"

// TEST-ONLY host simulation of the wide-accumulator reduction (fp.cuh: fp_redc_acc, lin9_reduce) and of the
// Granger-Scott squaring built on it (pairing.cuh: gs_fp4_square, cyclotomic_square_assign), on RAW Montgomery limbs so
// that the tests can place values exactly at the stated bounds.  Used by tests/test_lazy_fp4_square.py.
#include "../../sylow_b200/csrc/pairing.cuh"

#include <cstring>

using namespace sylow;

extern "C" {

// V (9 limbs) = fp_redc_acc(A) for a 17-limb accumulator A
void hs_redc_acc(const uint32_t* A, uint32_t* V) { fp_redc_acc(V, A); }

// lin9_reduce of a 9-limb T < 2^262
void hs_lin9_reduce(const uint32_t* T, uint32_t* r) {
  Fp x = lin9_reduce(T);
  memcpy(r, x.l, 32);
}

// one Fp4 squaring: in = a, b, x, y (4 Fp2, 64 words), out = new x, y (32 words)
void hs_gs_fp4_square(const uint32_t* in, int xi, uint32_t* out) {
  Fp2 v[4];
  memcpy(v, in, sizeof(v));
  gs_fp4_square(v[0], v[1], v[2], v[3], xi != 0);
  memcpy(out, &v[2], 2 * sizeof(Fp2));
}

// the in-place Granger-Scott squaring on 12 raw coefficients (96 words)
void hs_cyclotomic_square(const uint32_t* in, uint32_t* out) {
  Fp12 f;
  memcpy(&f, in, sizeof(f));
  cyclotomic_square_assign(f);
  memcpy(out, &f, sizeof(f));
}

}  // extern "C"

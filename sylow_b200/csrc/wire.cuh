// Wire formats of the C ABI (include/sylow_b200.h) <-> Montgomery-form device values.
//   Fp      : 32 bytes, little-endian canonical integer in [0, p)  (== U256::to_words(), fp.rs:232-234)
//   G1 affine: x || y (64 B);  G2 affine: x.c0 || x.c1 || y.c0 || y.c1 (128 B)
//   Fp12/Gt : 12 Fp in tower order c0.c0.c0, c0.c0.c1, ..., c1.c2.c1 (384 B)  (fp12.rs:561-574)
// Buffers handed to the library must be 16-byte aligned for the vector loads (cudaMalloc/pinned
// allocations are); the host entry points stage through the library's own buffers.
#pragma once
#include "pairing.cuh"

namespace sylow {

SY_HD Fp fp_load_raw(const uint8_t* p) {
  Fp r;
  const uint4* q = reinterpret_cast<const uint4*>(p);
  uint4 a = q[0], b = q[1];
  r.l[0] = a.x; r.l[1] = a.y; r.l[2] = a.z; r.l[3] = a.w;
  r.l[4] = b.x; r.l[5] = b.y; r.l[6] = b.z; r.l[7] = b.w;
  return r;
}
SY_HD void fp_store_raw(uint8_t* p, const Fp& v) {
  uint4* q = reinterpret_cast<uint4*>(p);
  q[0] = make_uint4(v.l[0], v.l[1], v.l[2], v.l[3]);
  q[1] = make_uint4(v.l[4], v.l[5], v.l[6], v.l[7]);
}
// canonical -> Montgomery.  Values >= p are reduced (fp_mul accepts any a < 2^256 here).
SY_HD Fp fp_load(const uint8_t* p) { return fp_to_mont(fp_load_raw(p)); }
SY_HD void fp_store(uint8_t* p, const Fp& v) { fp_store_raw(p, fp_from_mont(v)); }
// true iff the 32-byte value is a canonical residue (< p)
SY_HD bool fp_raw_is_canonical(const Fp& a) {
  int64_t bw = 0;  // borrow of a - p
  for (int i = 0; i < 8; i++) bw = ((int64_t)a.l[i] - (int64_t)SY_TAB(kP)[i] + bw) >> 32;
  return bw != 0;
}

SY_HD Fp2 fp2_load(const uint8_t* p) { return Fp2{fp_load(p), fp_load(p + 32)}; }
SY_HD void fp2_store(uint8_t* p, const Fp2& v) {
  fp_store(p, v.c0);
  fp_store(p + 32, v.c1);
}
SY_HD Fp2 fp2_load_raw(const uint8_t* p) { return Fp2{fp_load_raw(p), fp_load_raw(p + 32)}; }
SY_HD void fp2_store_raw(uint8_t* p, const Fp2& v) {
  fp_store_raw(p, v.c0);
  fp_store_raw(p + 32, v.c1);
}

// ---- G1 (F = Fp) and G2 (F = Fp2) point records ----------------------------------------------------------------
// A coordinate of either group, canonical (f_load / f_store) or Montgomery form (f_load_raw / f_store_raw).
template <class F>
SY_HD F f_load(const uint8_t* p);
template <>
SY_HD Fp f_load<Fp>(const uint8_t* p) { return fp_load(p); }
template <>
SY_HD Fp2 f_load<Fp2>(const uint8_t* p) { return fp2_load(p); }
template <class F>
SY_HD F f_load_raw(const uint8_t* p);
template <>
SY_HD Fp f_load_raw<Fp>(const uint8_t* p) { return fp_load_raw(p); }
template <>
SY_HD Fp2 f_load_raw<Fp2>(const uint8_t* p) { return fp2_load_raw(p); }
SY_HD void f_store(uint8_t* p, const Fp& v) { fp_store(p, v); }
SY_HD void f_store(uint8_t* p, const Fp2& v) { fp2_store(p, v); }
SY_HD void f_store_raw(uint8_t* p, const Fp& v) { fp_store_raw(p, v); }
SY_HD void f_store_raw(uint8_t* p, const Fp2& v) { fp2_store_raw(p, v); }

// Point i of an affine wire array (x || y, 2 sizeof(F) bytes per point) with its flag from the optional array inf.
template <class F>
SY_HD Affine<F> affine_load(const uint8_t* pts, const uint8_t* inf, size_t i) {
  constexpr size_t W = sizeof(F);
  return Affine<F>{f_load<F>(pts + i * 2 * W), f_load<F>(pts + i * 2 * W + W), inf && inf[i]};
}
// The device-internal projective record: x || y || z in Montgomery form, 96 bytes for G1 and 192 for G2.
template <class F>
SY_HD Proj<F> proj_load_raw(const uint8_t* p) {
  constexpr size_t W = sizeof(F);
  return Proj<F>{f_load_raw<F>(p), f_load_raw<F>(p + W), f_load_raw<F>(p + 2 * W)};
}
template <class F>
SY_HD void proj_store_raw(uint8_t* p, const Proj<F>& q) {
  constexpr size_t W = sizeof(F);
  f_store_raw(p, q.x);
  f_store_raw(p + W, q.y);
  f_store_raw(p + 2 * W, q.z);
}

// Fp12 in tower order.  *_raw keeps Montgomery form (device-internal intermediates).
SY_HD Fp12 fp12_load(const uint8_t* p) {
  Fp12 r;
  r.c0.c0 = fp2_load(p);
  r.c0.c1 = fp2_load(p + 64);
  r.c0.c2 = fp2_load(p + 128);
  r.c1.c0 = fp2_load(p + 192);
  r.c1.c1 = fp2_load(p + 256);
  r.c1.c2 = fp2_load(p + 320);
  return r;
}
SY_HD void fp12_store(uint8_t* p, const Fp12& v) {
  fp2_store(p, v.c0.c0);
  fp2_store(p + 64, v.c0.c1);
  fp2_store(p + 128, v.c0.c2);
  fp2_store(p + 192, v.c1.c0);
  fp2_store(p + 256, v.c1.c1);
  fp2_store(p + 320, v.c1.c2);
}
SY_HD Fp12 fp12_load_raw(const uint8_t* p) {
  Fp12 r;
  r.c0.c0 = fp2_load_raw(p);
  r.c0.c1 = fp2_load_raw(p + 64);
  r.c0.c2 = fp2_load_raw(p + 128);
  r.c1.c0 = fp2_load_raw(p + 192);
  r.c1.c1 = fp2_load_raw(p + 256);
  r.c1.c2 = fp2_load_raw(p + 320);
  return r;
}
SY_HD void fp12_store_raw(uint8_t* p, const Fp12& v) {
  fp2_store_raw(p, v.c0.c0);
  fp2_store_raw(p + 64, v.c0.c1);
  fp2_store_raw(p + 128, v.c0.c2);
  fp2_store_raw(p + 192, v.c1.c0);
  fp2_store_raw(p + 256, v.c1.c1);
  fp2_store_raw(p + 320, v.c1.c2);
}

}  // namespace sylow

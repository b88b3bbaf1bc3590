// Tower Fp2 -> Fp6 -> Fp12 for BN254 (u^2 = -1, v^3 = xi = 9+u, w^2 = v), Montgomery-form limbs.
//
// Value-level replacement of /root/reference/src/fields/{extensions,fp2,fp6,fp12}.rs.  The reference
// uses schoolbook Fp2/Fp6 products "for constant time"; field arithmetic is exact, so Karatsuba forms
// give bit-identical values with fewer limb products (SURVEY.md 8a rows a3-a5).
#pragma once
#include "fp.cuh"

// The Fp2 product and square stay out of line (one copy per kernel: the hot instruction footprint is what the
// instruction caches see); the Fp2 additions are inlined into their callers.
#define SY_HD_MUL2 SY_HD_NOINLINE
#define SY_HD_ADD SY_HD

namespace sylow {

struct Fp2 {
  Fp c0, c1;
};
struct Fp6 {
  Fp2 c0, c1, c2;
};
struct Fp12 {
  Fp6 c0, c1;
};

// ------------------------------------------------------------------------------------------ Fp2
SY_HD Fp2 fp2_zero() { return Fp2{fp_zero(), fp_zero()}; }
SY_HD Fp2 fp2_one() { return Fp2{fp_one(), fp_zero()}; }
SY_HD bool fp2_is_zero(const Fp2& a) { return fp_is_zero(a.c0) & fp_is_zero(a.c1); }
SY_HD bool fp2_eq(const Fp2& a, const Fp2& b) { return fp_eq(a.c0, b.c0) & fp_eq(a.c1, b.c1); }
SY_HD_ADD Fp2 fp2_add(const Fp2& a, const Fp2& b) { return Fp2{fp_add(a.c0, b.c0), fp_add(a.c1, b.c1)}; }
SY_HD_ADD Fp2 fp2_sub(const Fp2& a, const Fp2& b) { return Fp2{fp_sub(a.c0, b.c0), fp_sub(a.c1, b.c1)}; }
SY_HD_ADD Fp2 fp2_dbl(const Fp2& a) { return Fp2{fp_dbl(a.c0), fp_dbl(a.c1)}; }
SY_HD_ADD Fp2 fp2_neg(const Fp2& a) { return Fp2{fp_neg(a.c0), fp_neg(a.c1)}; }
SY_HD_ADD Fp2 fp2_mul3(const Fp2& a) { return fp2_add(fp2_dbl(a), a); }
// frobenius(1): the Fp non-residue is -1, so this is conjugation (fp2.rs:119-133)
SY_HD Fp2 fp2_conj(const Fp2& a) { return Fp2{a.c0, fp_neg(a.c1)}; }
SY_HD Fp2 fp2_select(bool c, const Fp2& a, const Fp2& b) {
  return Fp2{fp_select(c, a.c0, b.c0), fp_select(c, a.c1, b.c1)};
}
// scale(1/2) (pairing.rs:799,805): halving the Montgomery representative halves the value
SY_HD_ADD Fp2 fp2_halve(const Fp2& a) { return Fp2{fp_halve(a.c0), fp_halve(a.c1)}; }

// (a0 + a1 u)(9 + u) = (9 a0 - a1) + (a0 + 9 a1) u    (fp2.rs:99-107)
SY_HD_ADD Fp2 fp2_mul_xi(const Fp2& a) {
  return Fp2{fp_lin9(a.c0, fp_neg_nr(a.c1)), fp_lin9(a.c1, a.c0)};
}
// t + xi a and t - xi a: the addition rides in the same reduction
SY_HD_ADD Fp2 fp2_mul_xi_add(const Fp2& a, const Fp2& t) {
  return Fp2{fp_lin9(a.c0, fp_neg_nr(a.c1), t.c0), fp_lin9(a.c1, a.c0, t.c1)};
}
SY_HD_ADD Fp2 fp2_sub_mul_xi(const Fp2& t, const Fp2& a) {
  // (t0 - 9 a0 + a1, t1 - 9 a1 - a0) = (9 (p - a0) + a1 + t0, 9 (p - a1) + (p - a0) + t1)
  Fp n0 = fp_neg_nr(a.c0), n1 = fp_neg_nr(a.c1);
  return Fp2{fp_lin9(n0, a.c1, t.c0), fp_lin9(n1, n0, t.c1)};
}

// Karatsuba with lazy reduction: 3 full 512-bit products, the linear combinations on the unreduced
// values, and only 2 Montgomery reductions (value-equal to the schoolbook of fp2.rs:302-305).
//   c0 = a0 b0 - a1 b1            in (-p^2, p^2): add p*R when negative, then < p*R
//   c1 = (a0+a1)(b0+b1) - a0 b0 - a1 b1 = a0 b1 + a1 b0   in [0, 2 p^2) subset [0, p*R)
// The sums a0+a1, b0+b1 are NOT reduced (< 2p < 2^255, product < 4 p^2 < 2^510).
// ptxas interleaves every independent carry chain it can find; with three products and two reductions in one
// function it runs out of the seven predicate registers that hold the carries and spills them into a bit mask
// (about 50 LOP3 set/test instructions per Fp2 product).  Two chains per warp already saturate the multiplier
// pipe, so the products and the reductions are ordered by empty asm statements that make the next one's first
// operand depend on the previous one's last limb.
#if defined(__CUDA_ARCH__)
#define SY_AFTER(x, y) asm volatile("" : "+r"(x) : "r"(y))
// every limb of v waits for y: nothing of the next product can be hoisted above the previous one
#define SY_AFTER8(v, y)                            \
  do {                                             \
    _Pragma("unroll") for (int i_ = 0; i_ < 8; i_++) SY_AFTER((v)[i_], y); \
  } while (0)
#else
#define SY_AFTER(x, y) ((void)0)
#define SY_AFTER8(v, y) ((void)0)
#endif
// An Fp2 operand arrives by reference (generic pointer into the caller's frame); ptxas loads it limb by limb unless
// told that the 64 bytes are four aligned 128-bit words (Fp is alignas(16)).
SY_HD Fp2 fp2_ldv(const Fp2& a) {
#if defined(__CUDA_ARCH__)
  const uint4* p = reinterpret_cast<const uint4*>(&a);
  uint4 w0 = p[0], w1 = p[1], w2 = p[2], w3 = p[3];
  Fp2 r;
  r.c0.l[0] = w0.x; r.c0.l[1] = w0.y; r.c0.l[2] = w0.z; r.c0.l[3] = w0.w;
  r.c0.l[4] = w1.x; r.c0.l[5] = w1.y; r.c0.l[6] = w1.z; r.c0.l[7] = w1.w;
  r.c1.l[0] = w2.x; r.c1.l[1] = w2.y; r.c1.l[2] = w2.z; r.c1.l[3] = w2.w;
  r.c1.l[4] = w3.x; r.c1.l[5] = w3.y; r.c1.l[6] = w3.z; r.c1.l[7] = w3.w;
  return r;
#else
  return a;
#endif
}
SY_HD_MUL2 Fp2 fp2_mul(const Fp2& a_, const Fp2& b_) {
  const Fp2 a = fp2_ldv(a_), b = fp2_ldv(b_);
  uint32_t t0[16], t1[16], t2[16], sa[8], sb[8], a1[8];
  fp_mul_wide(t0, a.c0.l, b.c0.l);
#pragma unroll
  for (int i = 0; i < 8; i++) a1[i] = a.c1.l[i];
  SY_AFTER8(a1, t0[15]);
  fp_mul_wide(t1, a1, b.c1.l);
  fp_add_nr(sa, a.c0.l, a1);
  fp_add_nr(sb, b.c0.l, b.c1.l);
  SY_AFTER8(sa, t1[15]);
  fp_mul_wide(t2, sa, sb);
  wide_sub(t2, t0);
  wide_sub(t2, t1);
  uint32_t neg = wide_sub(t0, t1);
  wide_add_pR(t0, neg);
  Fp2 r;
  r.c0 = fp_redc_wide(t0);
  SY_AFTER(t2[0], r.c0.l[7]);
  r.c1 = fp_redc_wide(t2);
  return r;
}

// fp2.rs:164-171: ((a0+a1)(a0-a1), 2 a0 a1).  The factors a0+a1 and a0-a1+p are left unreduced
// (< 2p each, product < 4p^2 < p*R, which is all fp_mul needs) and 2 a0 a1 is doubled before its single
// reduction (2 a0 a1 < 2p^2 < p*R).
SY_HD_MUL2 Fp2 fp2_sqr(const Fp2& a_) {
  const Fp2 a = fp2_ldv(a_);
  Fp s, d, pp;
#pragma unroll
  for (int i = 0; i < 8; i++) pp.l[i] = SY_TAB(kP)[i];
  fp_add_nr(s.l, a.c0.l, a.c1.l);          // a0 + a1        < 2p
  fp_add_nr(d.l, a.c0.l, pp.l);            // a0 + p         < 2p
  fp_sub_nr(d.l, d.l, a.c1.l);             // a0 + p - a1    in (0, 2p)
  uint32_t t[16];
  fp_mul_wide(t, a.c0.l, a.c1.l);
  wide_dbl(t);
  Fp2 r;
  r.c0 = fp_mul(s, d);
  r.c1 = fp_redc_wide(t);
  return r;
}

// FieldExtension::scale by a base-field element (extensions.rs:86-94)
SY_HD_NOINLINE Fp2 fp2_mul_fp(const Fp2& a_, const Fp& k_) {
  const Fp2 a = fp2_ldv(a_);
  const Fp k = k_;
  return Fp2{fp_mul(a.c0, k), fp_mul(a.c1, k)};
}

// fp2.rs:343-361
SY_HD_NOINLINE Fp2 fp2_inv(const Fp2& a) {
  Fp t = fp_inv(fp_add(fp_sqr(a.c0), fp_sqr(a.c1)));
  return Fp2{fp_mul(a.c0, t), fp_neg(fp_mul(a.c1, t))};
}

// ------------------------------------------------------------------------------------------ Fp6
SY_HD Fp6 fp6_zero() { return Fp6{fp2_zero(), fp2_zero(), fp2_zero()}; }
SY_HD Fp6 fp6_one() { return Fp6{fp2_one(), fp2_zero(), fp2_zero()}; }
SY_HD Fp6 fp6_add(const Fp6& a, const Fp6& b) {
  return Fp6{fp2_add(a.c0, b.c0), fp2_add(a.c1, b.c1), fp2_add(a.c2, b.c2)};
}
SY_HD Fp6 fp6_sub(const Fp6& a, const Fp6& b) {
  return Fp6{fp2_sub(a.c0, b.c0), fp2_sub(a.c1, b.c1), fp2_sub(a.c2, b.c2)};
}
SY_HD Fp6 fp6_neg(const Fp6& a) { return Fp6{fp2_neg(a.c0), fp2_neg(a.c1), fp2_neg(a.c2)}; }
SY_HD Fp6 fp6_dbl(const Fp6& a) { return Fp6{fp2_dbl(a.c0), fp2_dbl(a.c1), fp2_dbl(a.c2)}; }
// multiplication by v (fp6.rs:189-191)
SY_HD Fp6 fp6_mul_v(const Fp6& a) { return Fp6{fp2_mul_xi(a.c2), a.c0, a.c1}; }
SY_HD bool fp6_eq(const Fp6& a, const Fp6& b) { return fp2_eq(a.c0, b.c0) & fp2_eq(a.c1, b.c1) & fp2_eq(a.c2, b.c2); }

// Karatsuba, 6 Fp2 products (value-equal to the 36-product schoolbook of fp6.rs:267-368; this is
// the form the reference quotes in its own comment at fp6.rs:274-283)
SY_HD_NOINLINE Fp6 fp6_mul(const Fp6& a, const Fp6& b) {
  Fp2 t0 = fp2_mul(a.c0, b.c0);
  Fp2 t1 = fp2_mul(a.c1, b.c1);
  Fp2 t2 = fp2_mul(a.c2, b.c2);
  Fp2 r0 = fp2_mul(fp2_add(a.c1, a.c2), fp2_add(b.c1, b.c2));
  r0 = fp2_mul_xi_add(fp2_sub(fp2_sub(r0, t1), t2), t0);
  Fp2 r1 = fp2_mul(fp2_add(a.c0, a.c1), fp2_add(b.c0, b.c1));
  r1 = fp2_mul_xi_add(t2, fp2_sub(fp2_sub(r1, t0), t1));
  Fp2 r2 = fp2_mul(fp2_add(a.c0, a.c2), fp2_add(b.c0, b.c2));
  r2 = fp2_sub(fp2_add(fp2_sub(r2, t0), t1), t2);
  return Fp6{r0, r1, r2};
}

// CH-SQR (fp6.rs:219-236)
SY_HD_NOINLINE Fp6 fp6_sqr(const Fp6& a) {
  Fp2 t0 = fp2_sqr(a.c0);
  Fp2 t1 = fp2_dbl(fp2_mul(a.c0, a.c1));
  Fp2 t2 = fp2_sqr(fp2_add(fp2_sub(a.c0, a.c1), a.c2));
  Fp2 s3 = fp2_dbl(fp2_mul(a.c1, a.c2));
  Fp2 s4 = fp2_sqr(a.c2);
  Fp6 r;
  r.c0 = fp2_mul_xi_add(s3, t0);
  r.c1 = fp2_mul_xi_add(s4, t1);
  r.c2 = fp2_sub(fp2_sub(fp2_add(fp2_add(t1, t2), s3), t0), s4);
  return r;
}

// scale by an Fp2 factor (extensions.rs:86-94)
SY_HD_NOINLINE Fp6 fp6_scale(const Fp6& a, const Fp2& k) {
  return Fp6{fp2_mul(a.c0, k), fp2_mul(a.c1, k), fp2_mul(a.c2, k)};
}

// Alg. 17 of eprint 2010/354 (fp6.rs:400-424)
SY_HD_NOINLINE Fp6 fp6_inv(const Fp6& a) {
  Fp2 t0 = fp2_sub(fp2_sqr(a.c0), fp2_mul(a.c1, fp2_mul_xi(a.c2)));
  Fp2 t1 = fp2_sub(fp2_mul_xi(fp2_sqr(a.c2)), fp2_mul(a.c0, a.c1));
  Fp2 t2 = fp2_sub(fp2_sqr(a.c1), fp2_mul(a.c0, a.c2));
  Fp2 d = fp2_add(fp2_mul_xi(fp2_add(fp2_mul(a.c2, t1), fp2_mul(a.c1, t2))), fp2_mul(a.c0, t0));
  d = fp2_inv(d);
  return Fp6{fp2_mul(d, t0), fp2_mul(d, t1), fp2_mul(d, t2)};
}

// ------------------------------------------------------------------------------------------ Fp12
SY_HD Fp12 fp12_one() { return Fp12{fp6_one(), fp6_zero()}; }
SY_HD bool fp12_eq(const Fp12& a, const Fp12& b) { return fp6_eq(a.c0, b.c0) & fp6_eq(a.c1, b.c1); }
// unitary_inverse (fp12.rs:381-383)
SY_HD Fp12 fp12_conj(const Fp12& a) { return Fp12{a.c0, fp6_neg(a.c1)}; }

// Karatsuba (fp12.rs:210-239)
// The *_assign forms update their first operand in place.  A call like f = fp12_sqr(f) makes the callee write into a
// hidden temporary that the caller then copies over f (24 + 24 128-bit local loads and stores, each store waiting for
// its load: 8 % of the final exponentiation's stall samples); with one reference parameter there is no temporary.
// conj_b = true multiplies by the conjugate (b.c0, -b.c1) without materialising it (the flag is uniform across the
// block: exponent digits are compile-time tables):  a conj(b) = (a0 b0 - v a1 b1) + ((a0 + a1)(b0 - b1) - a0 b0 + a1 b1) w.
SY_HD_NOINLINE void fp12_mul_assign(Fp12& a, const Fp12& b, bool conj_b = false) {  // b must not alias a
  Fp6 t0 = fp6_mul(a.c0, b.c0);
  Fp6 t1 = fp6_mul(a.c1, b.c1);
  if (conj_b) t1 = fp6_neg(t1);
  Fp6 s = fp6_mul(fp6_add(a.c0, a.c1), conj_b ? fp6_sub(b.c0, b.c1) : fp6_add(b.c0, b.c1));
  a.c0 = Fp6{fp2_mul_xi_add(t1.c2, t0.c0), fp2_add(t1.c0, t0.c1), fp2_add(t1.c1, t0.c2)};  // v t1 + t0
  a.c1 = fp6_sub(fp6_sub(s, t0), t1);
}
SY_HD Fp12 fp12_mul(const Fp12& a, const Fp12& b) {
  Fp12 r = a;
  fp12_mul_assign(r, b);
  return r;
}
SY_HD void fp12_conj_assign(Fp12& a) { a.c1 = fp6_neg(a.c1); }

// complex squaring (fp12.rs:536-550)
SY_HD_NOINLINE void fp12_sqr_assign(Fp12& a) {
  Fp6 c0 = fp6_sub(a.c0, a.c1);
  Fp6 c3{fp2_sub_mul_xi(a.c0.c0, a.c1.c2), fp2_sub(a.c0.c1, a.c1.c0), fp2_sub(a.c0.c2, a.c1.c1)};  // a0 - v a1
  Fp6 c2 = fp6_mul(a.c0, a.c1);
  c0 = fp6_add(fp6_mul(c0, c3), c2);
  a.c1 = fp6_dbl(c2);
  a.c0 = Fp6{fp2_mul_xi_add(c2.c2, c0.c0), fp2_add(c2.c0, c0.c1), fp2_add(c2.c1, c0.c2)};  // c0 + v c2
}
SY_HD Fp12 fp12_sqr(const Fp12& a) {
  Fp12 r = a;
  fp12_sqr_assign(r);
  return r;
}

// Alg. 23 of eprint 2010/354 (fp12.rs:270-287)
SY_HD_NOINLINE Fp12 fp12_inv(const Fp12& a) {
  Fp6 t = fp6_inv(fp6_sub(fp6_sqr(a.c0), fp6_mul_v(fp6_sqr(a.c1))));
  return Fp12{fp6_mul(a.c0, t), fp6_neg(fp6_mul(a.c1, t))};
}

// Multiplication by the sparse element l0 + l_vv v^2 + l_vw v w, i.e. slots z0, z2, z4 of
// (c0.c0, c0.c1, c0.c2, c1.c0, c1.c1, c1.c2).  Same 13-product schedule as fp12.rs:426-503.
// In place (x0, x2, x4 must not alias f): the four products that need sums of z first, then every slot is overwritten
// as soon as its last reader is done (z0 after z1 x2, z2 after z3 x4, z1 after z5 x4, z3 after z3 x0, z4 and z5 after
// z5 x2) - no result record and
// no copy back (the one-record form stored the six outputs to the frame, re-loaded them and wrote f word by word:
// k_miller 166.1 -> 162.7 ms per 2^20 without it, profiles/r02s_kbench_inplace.jsonl).
SY_HD_NOINLINE void fp12_sparse_mul_assign(Fp12& f, const Fp2& x0, const Fp2& x4 /*ell_vw*/, const Fp2& x2 /*ell_vv*/) {
  Fp2 &z0 = f.c0.c0, &z1 = f.c0.c1, &z2 = f.c0.c2, &z3 = f.c1.c0, &z4 = f.c1.c1, &z5 = f.c1.c2;
  Fp2 x02 = fp2_add(x0, x2);
  Fp2 p4 = fp2_mul(fp2_add(z0, z2), x02);                                      // (z0 + z2)(x0 + x2)
  Fp2 p6 = fp2_mul(fp2_add(z2, z4), fp2_add(x2, x4));                          // (z2 + z4)(x2 + x4)
  Fp2 p9 = fp2_mul(fp2_add(z0, z4), fp2_add(x0, x4));                          // (z0 + z4)(x0 + x4)
  Fp2 p10 = fp2_mul(fp2_add(fp2_add(z1, z3), z5), fp2_add(x02, x4));           // (z1 + z3 + z5)(x0 + x2 + x4)
  Fp2 d0 = fp2_mul(z0, x0);
  Fp2 d2 = fp2_mul(z2, x2);
  Fp2 d4 = fp2_mul(z4, x4);
  Fp2 s1 = fp2_mul(z1, x2);
  z0 = fp2_mul_xi_add(fp2_add(s1, d4), d0);                                    // r00
  Fp2 t = fp2_mul(z3, x4);
  s1 = fp2_add(s1, t);
  z2 = fp2_add(fp2_sub(fp2_sub(p4, d0), d2), t);                               // r02
  t = fp2_mul(z1, x0);
  s1 = fp2_add(s1, t);
  Fp2 u = fp2_mul(z5, x4);
  s1 = fp2_add(s1, u);
  z1 = fp2_mul_xi_add(fp2_add(u, d2), t);                                      // r01
  t = fp2_mul(z3, x0);
  s1 = fp2_add(s1, t);
  z3 = fp2_mul_xi_add(fp2_sub(fp2_sub(p6, d2), d4), t);                        // r10
  t = fp2_mul(z5, x2);
  s1 = fp2_add(s1, t);
  z4 = fp2_mul_xi_add(t, fp2_sub(fp2_sub(p9, d0), d4));                        // r11
  z5 = fp2_sub(p10, s1);                                                       // r12
}
SY_HD Fp12 fp12_sparse_mul(const Fp12& f, const Fp2& x0, const Fp2& x4, const Fp2& x2) {
  Fp12 r = f;
  fp12_sparse_mul_assign(r, x0, x4, x2);
  return r;
}

}  // namespace sylow

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

SY_HD void fp12_conj_assign(Fp12& a) { a.c1 = fp6_neg(a.c1); }

// ---- Fp12 product over Fp4 = Fp2[y] / (y^2 - xi), Fp12 = Fp4[w] / (w^3 - y)  (y = w^3, the Granger-Scott view) --------
// With w^2 = v the coefficient pairs are A0 = (c0.c0, c1.c1), A1 = (c1.c0, c0.c2), A2 = (c0.c1, c1.c2).
// Lifts of the Fp4 product's accumulators (17 limbs) and of the combinations of its outputs (9 limbs).  They are
// immediates, not __constant__ tables, so the constant bank of every other kernel keeps its layout.
struct Acc17 {
  uint32_t l[17];
};
struct U9 {
  uint32_t l[9];
};
SY_HD Acc17 acc_p2() {  // p^2
  return Acc17{{0x275d69b1u, 0x3b5458a2u, 0x09eac101u, 0xa602072du, 0x6d96cadcu, 0x4a50189cu, 0x7a1242c8u, 0x04689e95u,
                0x34c6b38du, 0x26edfa5cu, 0x16375606u, 0xb00b8551u, 0x0348d21cu, 0x599a6f7cu, 0x763cbf9cu, 0x0925c4b8u,
                0x00000000u}};
}
SY_HD Acc17 acc_3p2() {  // 3 p^2
  return Acc17{{0x76183d13u, 0xb1fd09e6u, 0x1dc04303u, 0xf2061587u, 0x48c46095u, 0xdef049d5u, 0x6e36c858u, 0x0d39dbc0u,
                0x9e541aa7u, 0x74c9ef14u, 0x42a60212u, 0x10228ff3u, 0x09da7656u, 0x0ccf4e74u, 0x62b63ed5u, 0x1b714e29u,
                0x00000000u}};
}
SY_HD U9 u9_36p() {  // 36 p
  return U9{{0x71939dfcu, 0x7493b336u, 0xb0007bdcu, 0x4e32fc72u, 0x36306d29u, 0xeb49cdaau, 0xaafa85ddu, 0xce1b0827u,
             0x00000006u}};
}

// fp12_mul_assign's locals: the six Fp4 product outputs it keeps and the operand sums of the current product
struct Fp12MulFrame {
  Fp t0[4], t1[4], t2[4], m12[4], m[4];
  Fp2 x0, x1, y0, y1;
};
#if defined(__CUDA_ARCH__)
// the operands are read again from memory after this point instead of being kept in registers across the products
#define SY_RELOAD() asm volatile("" ::: "memory")
// references a, b, l to a_, b_, l_ whose member addresses are formed afresh here: otherwise the twelve coefficient
// addresses of a and b and those of the locals are kept live across every call of fp4_mul_redc, and the callee saves
// and restores them in local memory
#define SY_FRESH(a, b, l)                                        \
  Fp12* a##p_ = &a##_;                                           \
  const Fp12* b##p_ = &b##_;                                     \
  Fp12MulFrame* l##p_ = &l##_;                                   \
  asm volatile("" : "+l"(a##p_), "+l"(b##p_), "+l"(l##p_));      \
  Fp12& a = *a##p_;                                              \
  const Fp12& b = *b##p_;                                        \
  Fp12MulFrame& l = *l##p_
#else
#define SY_RELOAD() ((void)0)
#define SY_FRESH(a, b, l) \
  Fp12& a = a##_;         \
  const Fp12& b = b##_;   \
  Fp12MulFrame& l = l##_
#endif

// an fp4_mul_redc output as 8 limbs (its bound keeps W[8] = 0)
SY_HD Fp fp4_v8(const uint32_t* W) {
#if defined(SYLOW_HOSTSIM) && !defined(__CUDA_ARCH__)
  if (W[8] != 0) {
    fprintf(stderr, "fp4_mul_redc: output >= 2^256\n");
    abort();
  }
#endif
  return Fp{{W[0], W[1], W[2], W[3], W[4], W[5], W[6], W[7]}};
}

// An Fp operand by reference, as two 128-bit loads (fp2_ldv)
SY_HD Fp fp_ldv(const Fp& a) {
#if defined(__CUDA_ARCH__)
  const uint4* p = reinterpret_cast<const uint4*>(&a);
  uint4 w0 = p[0], w1 = p[1];
  return Fp{{w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w}};
#else
  return a;
#endif
}
// the Karatsuba sums x0 + x1 and y0 + y1 of two Fp2 operands, not reduced
SY_HD void fp4_sums(uint32_t* s, uint32_t* d, const Fp2& x_, const Fp2& y_) {
  const Fp2 x = fp2_ldv(x_), y = fp2_ldv(y_);
  fp_add_nr(s, x.c0.l, x.c1.l);
  fp_add_nr(d, y.c0.l, y.c1.l);
}

SY_HD void fp2_mul_acc(uint32_t* Re, uint32_t* Im, const Fp2& x_, const Fp2& y_, const uint32_t* L) {
  uint32_t T[16], s[8], d[8];
  fp4_sums(s, d, x_, y_);
  fp_mul_wide(T, s, d);
#pragma unroll
  for (int i = 0; i < 16; i++) Im[i] = T[i];
  Im[16] = 0;
  SY_RELOAD();
  {
    const Fp x = fp_ldv(x_.c0), y = fp_ldv(y_.c0);
    SY_AFTER8(x.l, T[15]);
    fp_mul_wide(T, x.l, y.l);
    acc_sub(Im, T);
    SY_AFTER(T[0], Im[16]);
    acc_const_add(Re, L, T);
  }
  SY_RELOAD();
  {
    const Fp x = fp_ldv(x_.c1), y = fp_ldv(y_.c1);
    SY_AFTER8(x.l, Re[16]);
    fp_mul_wide(T, x.l, y.l);
    acc_sub(Im, T);
    SY_AFTER(T[0], Im[16]);
    acc_sub(Re, T);
  }
}
// One Fp4 product (X0 + X1 y)(Y0 + Y1 y) = (X0 Y0 + xi X1 Y1) + (X0 Y1 + X1 Y0) y with lazy reduction.  Nine 512-bit
// products, Karatsuba over Fp2 and over Fp4: Q = X1 Y1, P = X0 Y0 and Z = (X0 + X1)(Y0 + Y1) (the coefficients of
// X0 + X1 are < 2p, their sum < 4p, so Z's largest product < 16 p^2).  With Re Q, Re P in (-p^2, p^2) and Im Q,
// Im P in [0, 2 p^2), four 17-limb accumulators:
//   A = 3 p^2 - Im Q + 9 (Re Q + p^2) + Re P    = Re X0Y0 + 9 Re X1Y1 - Im X1Y1 + 12 p^2    in (0, 22 p^2)
//   B = (Re Q + p^2) + 9 Im Q + Im P            = Im X0Y0 + Re X1Y1 + 9 Im X1Y1 + p^2      in (0, 22 p^2)
//   E = 3 p^2 - (Re Q + p^2) - Re P + Re Z      = Re (X0Y1 + X1Y0) + 2 p^2                  in (0, 4 p^2)
//   F = -Im Q - Im P + Im Z                     = Im (X0Y1 + X1Y0)                          in [0, 4 p^2)
// (xi = 9 + u, u^2 = -1; every input coefficient < p; the ranges are those of the exact integer values, since the
// Karatsuba identities hold over the integers, and the limbs are exact mod 2^544, so intermediate steps may wrap).
// Q is formed first as two accumulators (fp2_mul_acc) and spread into A, B, E, F; then the products of P and Z are
// added to those four directly, so at most four accumulators and one product are live while a product is formed.
// Each accumulator is reduced once (fp_redc_acc): V = W + floor(acc / R) with W <= p, so V < p + 22 p^2 / R = 5.16 p
// (A, B) and V < 1.76 p (E, F), below 2^256 = 5.29 p: V is stored as 8 limbs, not reduced mod p.
// Four Montgomery reductions instead of the six of three Fp2 products.  V may not alias an operand.
SY_HD_NOINLINE void fp4_mul_redc(Fp* V, const Fp2& x0_, const Fp2& x1_, const Fp2& y0_, const Fp2& y1_) {
  uint32_t T[16], s[8], d[8], W[9], A[17], B[17], E[17], F[17];
  {  // X1 Y1
    uint32_t C[17], D[17];
    fp2_mul_acc(C, D, x1_, y1_, acc_p2().l);  // C = Re Q + p^2, D = Im Q
    acc_const_sub(E, acc_3p2().l, C);
    SY_AFTER(D[0], E[16]);
    acc_neg(F, D);
    SY_AFTER(D[0], F[16]);
    acc_const_sub(A, acc_3p2().l, D);
    SY_AFTER(C[0], A[16]);
    acc_madd<9>(A, C);
#pragma unroll
    for (int i = 0; i < 17; i++) B[i] = C[i];
    SY_AFTER(B[0], A[16]);
    acc_madd<9>(B, D);
  }
  SY_RELOAD();
  {  // X0 Y0
    fp4_sums(s, d, x0_, y0_);
    SY_AFTER8(s, B[16]);
    fp_mul_wide(T, s, d);  // (x00 + x01)(y00 + y01)
    acc_add(B, T);
    SY_AFTER(T[0], B[16]);
    acc_sub(F, T);
  }
  SY_RELOAD();
  {
    const Fp x = fp_ldv(x0_.c0), y = fp_ldv(y0_.c0);
    SY_AFTER8(x.l, F[16]);
    fp_mul_wide(T, x.l, y.l);  // x00 y00
    acc_add(A, T);
    SY_AFTER(T[0], A[16]);
    acc_sub(B, T);
    SY_AFTER(T[0], B[16]);
    acc_sub(E, T);
    SY_AFTER(T[0], E[16]);
    acc_add(F, T);
  }
  SY_RELOAD();
  {
    const Fp x = fp_ldv(x0_.c1), y = fp_ldv(y0_.c1);
    SY_AFTER8(x.l, F[16]);
    fp_mul_wide(T, x.l, y.l);  // x01 y01
    acc_sub(A, T);
    SY_AFTER(T[0], A[16]);
    acc_sub(B, T);
    SY_AFTER(T[0], B[16]);
    acc_add(E, T);
    SY_AFTER(T[0], E[16]);
    acc_add(F, T);
  }
  SY_AFTER(A[0], F[16]);
  fp_redc_acc(W, A);
  V[0] = fp4_v8(W);
  SY_AFTER(B[0], W[7]);
  fp_redc_acc(W, B);
  V[1] = fp4_v8(W);
  SY_RELOAD();
  {  // (X0 + X1)(Y0 + Y1)
    Fp2 x, y;
    {
      const Fp2 xa = fp2_ldv(x0_), xb = fp2_ldv(x1_);
      fp_add_nr(x.c0.l, xa.c0.l, xb.c0.l);
      fp_add_nr(x.c1.l, xa.c1.l, xb.c1.l);
    }
    {
      const Fp2 ya = fp2_ldv(y0_), yb = fp2_ldv(y1_);
      fp_add_nr(y.c0.l, ya.c0.l, yb.c0.l);
      fp_add_nr(y.c1.l, ya.c1.l, yb.c1.l);
    }
    fp_add_nr(s, x.c0.l, x.c1.l);
    fp_add_nr(d, y.c0.l, y.c1.l);
    SY_AFTER8(x.c0.l, W[7]);
    fp_mul_wide(T, x.c0.l, y.c0.l);  // z0
    acc_add(E, T);
    SY_AFTER(T[0], E[16]);
    acc_sub(F, T);
    SY_AFTER8(x.c1.l, F[16]);
    fp_mul_wide(T, x.c1.l, y.c1.l);  // z1
    acc_sub(E, T);
    SY_AFTER(T[0], E[16]);
    acc_sub(F, T);
    SY_AFTER8(s, F[16]);
    fp_mul_wide(T, s, d);  // zS
    acc_add(F, T);
  }
  SY_AFTER(E[0], F[16]);
  fp_redc_acc(W, E);
  V[2] = fp4_v8(W);
  SY_AFTER(F[0], W[7]);
  fp_redc_acc(W, F);
  V[3] = fp4_v8(W);
}

// 9-limb copy of an fp4_mul_redc output
SY_HD void u9_of(uint32_t* r, const Fp& v) {
#pragma unroll
  for (int i = 0; i < 8; i++) r[i] = v.l[i];
  r[8] = 0;
}
// (B0 + 9 Dr - Di, B1 + Dr + 9 Di) + 36 p, reduced: B + xi D for 9-limb combinations B, D (fp12_mul_assign)
SY_HD Fp2 fp2_xi_glue(uint32_t* B0, uint32_t* B1, const uint32_t* Dr, const uint32_t* Di) {
  u9_add_shl(B0, B0, Dr, 3);
  u9_add_shl(B0, B0, Dr, 0);
  u9_sub(B0, B0, Di);
  u9_add_shl(B0, B0, u9_36p().l, 0);
  u9_add_shl(B1, B1, Di, 3);
  u9_add_shl(B1, B1, Di, 0);
  u9_add_shl(B1, B1, Dr, 0);
  u9_add_shl(B1, B1, u9_36p().l, 0);
  return Fp2{lin9_reduce(B0), lin9_reduce(B1)};
}
// u + v - w - t + 36 p, reduced
SY_HD Fp fp_glue(const Fp& u, const Fp& v, const Fp& w, const Fp& t) {
  uint32_t B[9], X[9];
  u9_of(B, u);
  u9_of(X, v);
  u9_add_shl(B, B, X, 0);
  u9_of(X, w);
  u9_sub(B, B, X);
  u9_of(X, t);
  u9_sub(B, B, X);
  u9_add_shl(B, B, u9_36p().l, 0);
  return lin9_reduce(B);
}
// B = u - v - w (9 limbs, mod 2^288)
SY_HD void u9_diff(uint32_t* B, const Fp& u, const Fp& v, const Fp& w) {
  uint32_t X[9];
  u9_of(B, u);
  u9_of(X, v);
  u9_sub(B, B, X);
  u9_of(X, w);
  u9_sub(B, B, X);
}

// Karatsuba over the three Fp4 coefficients (A0 + A1 w + A2 w^2)(B0 + B1 w + B2 w^2) with w^3 = y:
//   T0 = A0 B0, T1 = A1 B1, T2 = A2 B2, M01 = (A0 + A1)(B0 + B1), M02 = (A0 + A2)(B0 + B2), M12 = (A1 + A2)(B1 + B2)
//   R0 = T0 + y (M12 - T1 - T2),  R1 = M01 - T0 - T1 + y T2,  R2 = M02 - T0 - T2 + T1,   y (a + b y) = xi b + a y.
// 18 Fp2 products as six fp4_mul_redc (54 512-bit products, 24 Montgomery reductions instead of 36).  The operand sums
// are reduced (fp2_add), so every fp4_mul_redc input is < p.  The combinations act on its unreduced outputs
// (V < 5.16 p for the y^0 coefficient of an Fp4 value, < 1.76 p for the y^1 one) in 9 limbs, each lifted by 36 p and
// finished by one lin9_reduce.  The largest lin9_reduce inputs are those of R0's y^0 coefficient:
//   T0 + 9 (M12 - T1 - T2)_r - (M12 - T1 - T2)_i + 36 p < 5.16 p + 9 * 1.76 p + 2 * 1.76 p + 36 p < 61 p
// and its negative part is at most 9 * 2 * 1.76 p + 1.76 p < 36 p (the u coefficient: 2 * 1.76 p + 9 * 2 * 1.76 p
// < 36 p); every other combination has fewer and smaller negative terms (at most 2 * 5.16 p + 1.76 p).  All inputs
// are below lin9_reduce's 338 p.
// The output of one Fp4 coefficient is written once the last product that reads its input is done: M12 first (its
// value is kept for R0), then M01 -> R1, M02 -> R2, and R0 last.
// The *_assign forms update their first operand in place.  A call like f = fp12_sqr(f) makes the callee write into a
// hidden temporary that the caller then copies over f (24 + 24 128-bit local loads and stores, each store waiting for
// its load: 8 % of the final exponentiation's stall samples); with one reference parameter there is no temporary.
// conj_b = true multiplies by the conjugate (b.c0, -b.c1) without materialising it (the flag is uniform across the
// block: exponent digits are compile-time tables): a conj(b) = conj(conj(a) b), so a is conjugated before and after.
SY_HD_NOINLINE void fp12_mul_assign(Fp12& a_, const Fp12& b_, bool conj_b = false) {  // b must not alias a
  if (conj_b) fp12_conj_assign(a_);
  Fp12MulFrame l_;  // one frame object: one base address is live across the calls, not nine
  {
    SY_FRESH(a, b, l);
    fp4_mul_redc(l.t0, a.c0.c0, a.c1.c1, b.c0.c0, b.c1.c1);  // A0 B0
  }
  {
    SY_FRESH(a, b, l);
    fp4_mul_redc(l.t1, a.c1.c0, a.c0.c2, b.c1.c0, b.c0.c2);  // A1 B1
  }
  {
    SY_FRESH(a, b, l);
    fp4_mul_redc(l.t2, a.c0.c1, a.c1.c2, b.c0.c1, b.c1.c2);  // A2 B2
  }
  {
    SY_FRESH(a, b, l);
    l.x0 = fp2_add(a.c1.c0, a.c0.c1);
    l.x1 = fp2_add(a.c0.c2, a.c1.c2);
    l.y0 = fp2_add(b.c1.c0, b.c0.c1);
    l.y1 = fp2_add(b.c0.c2, b.c1.c2);
    fp4_mul_redc(l.m12, l.x0, l.x1, l.y0, l.y1);  // M12
  }
  uint32_t B0[9], B1[9], Dr[9], Di[9];
  {  // R1 = M01 - T0 - T1 + y T2
    SY_FRESH(a, b, l);
    l.x0 = fp2_add(a.c0.c0, a.c1.c0);
    l.x1 = fp2_add(a.c1.c1, a.c0.c2);
    l.y0 = fp2_add(b.c0.c0, b.c1.c0);
    l.y1 = fp2_add(b.c1.c1, b.c0.c2);
    fp4_mul_redc(l.m, l.x0, l.x1, l.y0, l.y1);
  }
  {
    SY_FRESH(a, b, l);
    u9_diff(B0, l.m[0], l.t0[0], l.t1[0]);
    u9_diff(B1, l.m[1], l.t0[1], l.t1[1]);
    u9_of(Dr, l.t2[2]);
    u9_of(Di, l.t2[3]);
    a.c1.c0 = fp2_xi_glue(B0, B1, Dr, Di);
    a.c0.c2 = Fp2{fp_glue(l.m[2], l.t2[0], l.t0[2], l.t1[2]), fp_glue(l.m[3], l.t2[1], l.t0[3], l.t1[3])};
  }
  {  // R2 = M02 - T0 - T2 + T1
    SY_FRESH(a, b, l);
    l.x0 = fp2_add(a.c0.c0, a.c0.c1);
    l.x1 = fp2_add(a.c1.c1, a.c1.c2);
    l.y0 = fp2_add(b.c0.c0, b.c0.c1);
    l.y1 = fp2_add(b.c1.c1, b.c1.c2);
    fp4_mul_redc(l.m, l.x0, l.x1, l.y0, l.y1);
  }
  {
    SY_FRESH(a, b, l);
    a.c0.c1 = Fp2{fp_glue(l.m[0], l.t1[0], l.t0[0], l.t2[0]), fp_glue(l.m[1], l.t1[1], l.t0[1], l.t2[1])};
    a.c1.c2 = Fp2{fp_glue(l.m[2], l.t1[2], l.t0[2], l.t2[2]), fp_glue(l.m[3], l.t1[3], l.t0[3], l.t2[3])};
    // R0 = T0 + y (M12 - T1 - T2)
    u9_of(B0, l.t0[0]);
    u9_of(B1, l.t0[1]);
    u9_diff(Dr, l.m12[2], l.t1[2], l.t2[2]);
    u9_diff(Di, l.m12[3], l.t1[3], l.t2[3]);
    a.c0.c0 = fp2_xi_glue(B0, B1, Dr, Di);
    a.c1.c1 = Fp2{fp_glue(l.t0[2], l.m12[0], l.t1[0], l.t2[0]), fp_glue(l.t0[3], l.m12[1], l.t1[1], l.t2[1])};
  }
  if (conj_b) fp12_conj_assign(a_);
}
SY_HD Fp12 fp12_mul(const Fp12& a, const Fp12& b) {
  Fp12 r = a;
  fp12_mul_assign(r, b);
  return r;
}

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

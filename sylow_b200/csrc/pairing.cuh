// Optimal-ate pairing on BN254: fused Miller loop and final exponentiation.
//
// Replaces /root/reference/src/pairing.rs: G2Affine::precompute (:676-708) composed with
// G2PreComputed::miller_loop (:590-619) as ONE pass (no 16.7 KB coefficient table round trip), the
// Costello-Lange-Naehrig doubling/addition steps (:756-818) with exactly the reference's line
// scalings so the MillerLoopResult itself is bit-identical (SURVEY Q15), and
// MillerLoopResult::final_exponentiation (:245-492).
#pragma once
#include "curve.cuh"

namespace sylow {

struct Ell {
  Fp2 c0, c1, c2;
};

// pairing.rs:798-818.  Mutates R, returns the line triple.
SY_HD_NOINLINE Ell g2_doubling_step(G2Proj& r) {
  Fp2 a = fp2_halve(fp2_mul(r.x, r.y));
  Fp2 b = fp2_sqr(r.y);
  Fp2 c = fp2_sqr(r.z);
  Fp2 d = fp2_mul3(c);
  Fp2 e = fp2_mul(SY_TAB(kTwistB)[0], d);
  Fp2 f = fp2_mul3(e);
  Fp2 g = fp2_halve(fp2_add(b, f));
  Fp2 h = fp2_sub(fp2_sqr(fp2_add(r.y, r.z)), fp2_add(b, c));
  Fp2 i = fp2_sub(e, b);
  Fp2 j = fp2_sqr(r.x);
  Fp2 e_sq = fp2_sqr(e);
  r.x = fp2_mul(a, fp2_sub(b, f));
  r.y = fp2_sub(fp2_sqr(g), fp2_mul3(e_sq));
  r.z = fp2_mul(b, h);
  return Ell{fp2_mul_xi(i), fp2_neg(h), fp2_mul3(j)};
}

// pairing.rs:756-772
SY_HD_NOINLINE Ell g2_addition_step(G2Proj& r, const Fp2& qx, const Fp2& qy) {
  Fp2 d = fp2_sub(r.x, fp2_mul(r.z, qx));
  Fp2 e = fp2_sub(r.y, fp2_mul(r.z, qy));
  Fp2 f = fp2_sqr(d);
  Fp2 g = fp2_sqr(e);
  Fp2 h = fp2_mul(d, f);
  Fp2 i = fp2_mul(r.x, f);
  Fp2 j = fp2_sub(fp2_add(fp2_mul(r.z, g), h), fp2_dbl(i));
  Fp2 ry = fp2_sub(fp2_mul(e, fp2_sub(i, j)), fp2_mul(h, r.y));
  r.x = fp2_mul(d, j);
  r.y = ry;
  r.z = fp2_mul(r.z, h);
  return Ell{fp2_mul_xi(fp2_sub(fp2_mul(e, qx), fp2_mul(d, qy))), d, fp2_neg(e)};
}

// f <- f * l(P),  l(P) = (c0, c1 * yP, c2 * xP)   (pairing.rs:597)
SY_HD void miller_mul_line(Fp12& f, const Ell& l, const Fp& xp, const Fp& yp) {
  Fp2 lvw = fp2_mul_fp(l.c1, yp);
  Fp2 lvv = fp2_mul_fp(l.c2, xp);
  fp12_sparse_mul_assign(f, l.c0, lvw, lvv);
}

// Fused precompute + miller_loop for one (P, Q) pair of finite affine points.
// `acc` (optional) is where the Fp12 accumulator lives during the loop - the kernels pass a shared-memory slot.
SY_HD_NOINLINE Fp12 miller_loop(const Fp& xp, const Fp& yp, const Fp2& qx, const Fp2& qy, Fp12* acc = nullptr) {
  G2Proj r{qx, qy, fp2_one()};
  Fp2 nqy = fp2_neg(qy);
  Fp12 f_local;
  Fp12& f = acc ? *acc : f_local;
  f = fp12_one();
  for (int i = 0; i < 64; i++) {
    SY_LOOP_SYNC();
    Ell l = g2_doubling_step(r);
    if (i != 0) fp12_sqr_assign(f);  // 1^2 = 1 (SURVEY Q6)
    miller_mul_line(f, l, xp, yp);
    int digit = SY_TAB(kAteNaf)[i];
    if (digit != 0) {
      l = g2_addition_step(r, qx, digit > 0 ? qy : nqy);
      miller_mul_line(f, l, xp, yp);
    }
  }
  // Q1 = psi(Q), Q2 = -psi(Q1)   (pairing.rs:701-706, g2.rs:140-152)
  Fp2 q1x = fp2_mul(SY_TAB(kEpsExp0)[0], fp2_conj(qx));
  Fp2 q1y = fp2_mul(SY_TAB(kEpsExp1)[0], fp2_conj(qy));
  Fp2 q2x = fp2_mul(SY_TAB(kEpsExp0)[0], fp2_conj(q1x));
  Fp2 q2y = fp2_neg(fp2_mul(SY_TAB(kEpsExp1)[0], fp2_conj(q1y)));
  Ell l = g2_addition_step(r, q1x, q1y);
  miller_mul_line(f, l, xp, yp);
  l = g2_addition_step(r, q2x, q2y);
  miller_mul_line(f, l, xp, yp);
  return f;
}

// G2Affine::precompute (pairing.rs:676-708): the 87 line-coefficient triples of a fixed G2 point, in
// the reference's order (64 doublings interleaved with 21 additions, then the two Frobenius additions).
SY_HD_NOINLINE void g2_precompute(const Fp2& qx, const Fp2& qy, Ell* out) {
  G2Proj r{qx, qy, fp2_one()};
  Fp2 nqy = fp2_neg(qy);
  int idx = 0;
  for (int i = 0; i < 64; i++) {
    SY_LOOP_SYNC();
    out[idx++] = g2_doubling_step(r);
    int digit = SY_TAB(kAteNaf)[i];
    if (digit != 0) out[idx++] = g2_addition_step(r, qx, digit > 0 ? qy : nqy);
  }
  Fp2 q1x = fp2_mul(SY_TAB(kEpsExp0)[0], fp2_conj(qx));
  Fp2 q1y = fp2_mul(SY_TAB(kEpsExp1)[0], fp2_conj(qy));
  Fp2 q2x = fp2_mul(SY_TAB(kEpsExp0)[0], fp2_conj(q1x));
  Fp2 q2y = fp2_neg(fp2_mul(SY_TAB(kEpsExp1)[0], fp2_conj(q1y)));
  out[idx++] = g2_addition_step(r, q1x, q1y);
  out[idx++] = g2_addition_step(r, q2x, q2y);
}

// One G1 point of a glued loop.  `skip` pairs contribute the identity line (1, 0, 0): f * 1 = f exactly.
struct MillerG1 {
  Fp x, y;
  bool skip;
};
SY_HD void glued_mul_line(Fp12& f, const Ell& l, const MillerG1& p) {
  Fp2 l0 = fp2_select(p.skip, fp2_one(), l.c0);
  Fp2 lvw = fp2_select(p.skip, fp2_zero(), fp2_mul_fp(l.c1, p.y));
  Fp2 lvv = fp2_select(p.skip, fp2_zero(), fp2_mul_fp(l.c2, p.x));
  fp12_sparse_mul_assign(f, l0, lvw, lvv);
}

// glued_miller_loop (pairing.rs:970-1022) for NV pairs whose G2 point is per-item (line coefficients
// computed on the fly, fused) followed by NF pairs against fixed, precomputed G2 tables (87 triples each,
// Montgomery form; on the device they sit in shared memory and every thread reads the same triple).
// One shared Fp12 squaring per digit for all NV + NF pairs.  The product equals the reference's
// (multiplication order differs; Fp12 multiplication is exact and commutative).
// COPY only names a separate compiled copy: ptxas builds one body of a noinline function for all its callers, so a new
// kernel calling an existing instantiation would change the register allocation of the kernels that already call it.
// The loops over per-pair tables in global memory (miller_tables.cuh) use COPY = 1.
template <int NV, int NF, int COPY = 0>
SY_HD_NOINLINE Fp12 glued_miller_loop(const MillerG1* p /* NV + NF */, const Fp2* qx, const Fp2* qy /* NV */,
                                      const Ell* const* tables /* NF */, Fp12* acc = nullptr) {
  G2Proj r[NV > 0 ? NV : 1];
  Fp2 nqy[NV > 0 ? NV : 1];
  for (int v = 0; v < NV; v++) {
    r[v] = G2Proj{qx[v], qy[v], fp2_one()};
    nqy[v] = fp2_neg(qy[v]);
  }
  Fp12 f_local;
  Fp12& f = acc ? *acc : f_local;  // the kernels pass a shared-memory slot (see miller_loop)
  f = fp12_one();
  int idx = 0;
  for (int i = 0; i < 64; i++) {
    SY_LOOP_SYNC();
    if (i != 0) fp12_sqr_assign(f);
    for (int v = 0; v < NV; v++) {
      Ell l = g2_doubling_step(r[v]);
      glued_mul_line(f, l, p[v]);
    }
    for (int t = 0; t < NF; t++) glued_mul_line(f, tables[t][idx], p[NV + t]);
    idx++;
    int digit = SY_TAB(kAteNaf)[i];
    if (digit != 0) {
      for (int v = 0; v < NV; v++) {
        Ell l = g2_addition_step(r[v], qx[v], digit > 0 ? qy[v] : nqy[v]);
        glued_mul_line(f, l, p[v]);
      }
      for (int t = 0; t < NF; t++) glued_mul_line(f, tables[t][idx], p[NV + t]);
      idx++;
    }
  }
  for (int k = 0; k < 2; k++) {
    for (int v = 0; v < NV; v++) {
      // Q1 = psi(Q), then Q2 = -psi(Q1)
      Fp2 q1x = fp2_mul(SY_TAB(kEpsExp0)[0], fp2_conj(qx[v]));
      Fp2 q1y = fp2_mul(SY_TAB(kEpsExp1)[0], fp2_conj(qy[v]));
      if (k == 1) {
        Fp2 tx = fp2_mul(SY_TAB(kEpsExp0)[0], fp2_conj(q1x));
        Fp2 ty = fp2_neg(fp2_mul(SY_TAB(kEpsExp1)[0], fp2_conj(q1y)));
        q1x = tx;
        q1y = ty;
      }
      Ell l = g2_addition_step(r[v], q1x, q1y);
      glued_mul_line(f, l, p[v]);
    }
    for (int t = 0; t < NF; t++) glued_mul_line(f, tables[t][idx], p[NV + t]);
    idx++;
  }
  return f;
}

// ---------------------------------------------------------------------------- final exponentiation
// fp6.rs:203-209 / fp12.rs:515-522 for e in {1, 2, 3}; r must not alias a
SY_HD_NOINLINE void fp12_frobenius_to(Fp12& r, const Fp12& a, int e) {
  bool odd = e & 1;
  const Fp2 c61 = SY_TAB(kFrob6C1)[e], c62 = SY_TAB(kFrob6C2)[e], c12 = SY_TAB(kFrob12C1)[e];
  r.c0.c0 = odd ? fp2_conj(a.c0.c0) : a.c0.c0;
  r.c0.c1 = fp2_mul(odd ? fp2_conj(a.c0.c1) : a.c0.c1, c61);
  r.c0.c2 = fp2_mul(odd ? fp2_conj(a.c0.c2) : a.c0.c2, c62);
  r.c1.c0 = fp2_mul(odd ? fp2_conj(a.c1.c0) : a.c1.c0, c12);
  r.c1.c1 = fp2_mul(fp2_mul(odd ? fp2_conj(a.c1.c1) : a.c1.c1, c61), c12);
  r.c1.c2 = fp2_mul(fp2_mul(odd ? fp2_conj(a.c1.c2) : a.c1.c2, c62), c12);
}
SY_HD Fp12 fp12_frobenius(const Fp12& a, int e) {
  Fp12 r;
  fp12_frobenius_to(r, a, e);
  return r;
}

// One Fp4 squaring of Granger-Scott (pairing.rs:274-289 and the update of its two outputs, :309-346) with lazy reduction:
//   A = a^2 + xi b^2,  B = 2 a b = (a + b)^2 - a^2 - b^2,  x <- 3 A - 2 x,  y <- 3 B + 2 y  (3 xi B + 2 y when xi is set)
// Every coefficient of A and B is ONE signed combination of 512-bit products in a 17-limb accumulator (fp.cuh: acc_*),
// reduced once; the factor 3, the +-2 x / y term and the multiplication by xi = 9 + u act on the 9-limb values after
// that reduction (fp_lin3).  With u^2 = -1, and all inputs canonical (< p):
//   S_a = (a0 + a1)(a0 + p - a1) = a0^2 - a1^2 (mod p)  < 4 p^2      Q_a = 2 a0 a1 < 2 p^2     (S_b, Q_b alike)
//   S_c, Q_c the same for c = a + b (c0, c1 < 2p, not reduced):  S_c < 16 p^2,  Q_c < 8 p^2
//   A0 = S_a + 9 S_b - Q_b + p R        < 45.3 p^2       A1 = Q_a + S_b + 9 Q_b         < 24 p^2
//   B0 = S_c - S_a - S_b + 2 p R        < 26.6 p^2       B1 = Q_c - Q_a - Q_b + p R     < 13.3 p^2
// (p R = 5.29 p^2; every lift exceeds what it covers, so each value is non-negative, and all are below 2^513).  After
// fp_redc_acc, V = W + floor(acc / R) with W <= p: V_A0 < 9.57 p, V_A1 < 5.54 p, V_B0 < 6.03 p, V_B1 < 3.52 p, and
// the reduced inputs of lin9_reduce are at most 3 * 9.57 p + 2 p (x), 3 * 6.03 p + 2 p (y) or, with xi,
// 3 (9 V_B0 + 4 p - V_B1) + 2 p < 177 p and 3 (V_B0 + 9 V_B1) + 2 p < 116 p: all below its 338 p.
// Six 512-bit products and four Montgomery reductions instead of three Fp2 squarings (nine reductions) and about thirty
// modular additions.  a and x, b and y may alias (the outputs are written after the last read of the inputs).
SY_HD_NOINLINE void gs_fp4_square(const Fp2& a_, const Fp2& b_, Fp2& x, Fp2& y, bool xi) {
  const Fp2 a = fp2_ldv(a_), b = fp2_ldv(b_);
  uint32_t pp[8], T[16], s[8], d[8], A0[17], A1[17], B0[17], B1[17];
#pragma unroll
  for (int i = 0; i < 8; i++) pp[i] = SY_TAB(kP)[i];
  // Q_b: B1 = p R - Q_b, A0 = p R - Q_b, A1 = 9 Q_b
  fp_add_nr(s, b.c0.l, b.c0.l);
  fp_mul_wide(T, s, b.c1.l);
  acc_lift_sub(B1, pp, T);
  SY_AFTER(T[0], B1[15]);
  acc_lift_sub(A0, pp, T);
#pragma unroll
  for (int i = 0; i < 17; i++) A1[i] = 0;
  SY_AFTER(A1[0], A0[15]);
  acc_madd<9>(A1, T);
  // Q_a
  fp_add_nr(s, a.c0.l, a.c0.l);
  SY_AFTER8(s, A1[16]);
  fp_mul_wide(T, s, a.c1.l);
  acc_add(A1, T);
  SY_AFTER(B1[0], A1[16]);
  acc_sub(B1, T);
  // S_b: B0 = 2 p R - S_b
  fp_add_nr(s, b.c0.l, b.c1.l);
  fp_add_nr(d, b.c0.l, pp);
  fp_sub_nr(d, d, b.c1.l);
  SY_AFTER8(s, B1[16]);
  SY_AFTER8(d, B1[16]);
  fp_mul_wide(T, s, d);
  acc_madd<9>(A0, T);
  SY_AFTER(A1[0], A0[16]);
  acc_add(A1, T);
  SY_AFTER(T[0], A1[16]);
  acc_lift_sub(B0, SY_TAB(kP2), T);
  // S_a
  fp_add_nr(s, a.c0.l, a.c1.l);
  fp_add_nr(d, a.c0.l, pp);
  fp_sub_nr(d, d, a.c1.l);
  SY_AFTER8(s, B0[15]);
  SY_AFTER8(d, B0[15]);
  fp_mul_wide(T, s, d);
  acc_add(A0, T);
  SY_AFTER(B0[0], A0[16]);
  acc_sub(B0, T);
  // c = a + b; from here on only c and the accumulators are live
  Fp2 c;
  fp_add_nr(c.c0.l, a.c0.l, b.c0.l);
  fp_add_nr(c.c1.l, a.c1.l, b.c1.l);
  // x <- 3 A - 2 x
  uint32_t V[9];
  Fp2 r;
  const Fp2 xo = fp2_ldv(x);
  SY_AFTER(A0[0], B0[16]);
  fp_redc_acc(V, A0);
  fp_sub_nr(s, pp, xo.c0.l);  // 2 (p - x0) <= 2p
  fp_add_nr(s, s, s);
  r.c0 = fp_lin3(V, Fp{{s[0], s[1], s[2], s[3], s[4], s[5], s[6], s[7]}});
  SY_AFTER(A1[0], r.c0.l[7]);
  fp_redc_acc(V, A1);
  fp_sub_nr(s, pp, xo.c1.l);
  fp_add_nr(s, s, s);
  r.c1 = fp_lin3(V, Fp{{s[0], s[1], s[2], s[3], s[4], s[5], s[6], s[7]}});
  x = r;
  // S_c, Q_c
  fp_add_nr(s, c.c0.l, c.c1.l);  // < 4p
#pragma unroll
  for (int i = 0; i < 8; i++) d[i] = SY_TAB(kP2)[i];
  fp_add_nr(d, c.c0.l, d);
  fp_sub_nr(d, d, c.c1.l);       // c0 + 2p - c1 in (0, 4p)
  SY_AFTER8(s, r.c1.l[7]);
  SY_AFTER8(d, r.c1.l[7]);
  fp_mul_wide(T, s, d);
  acc_add(B0, T);
  uint32_t VB0[9], VB1[9];
  SY_AFTER(B0[0], T[15]);
  fp_redc_acc(VB0, B0);
  fp_add_nr(s, c.c0.l, c.c0.l);  // 2 c0 < 4p
  SY_AFTER8(s, VB0[8]);
  fp_mul_wide(T, s, c.c1.l);
  acc_add(B1, T);
  SY_AFTER(B1[0], T[15]);
  fp_redc_acc(VB1, B1);
  // y <- 3 B + 2 y, or 3 xi B + 2 y with xi B = (9 B0 - B1) + (B0 + 9 B1) u
  const Fp2 yo = fp2_ldv(y);
  if (xi) {
#pragma unroll
    for (int i = 0; i < 8; i++) d[i] = SY_TAB(kP4)[i];
    fp_sub_nr(V, d, VB1);  // V_B1 < 3.52 p < 2^256: 4p - V_B1 > 0 in 8 limbs
    V[8] = 0;
    u9_add_shl(V, V, VB0, 3);
    u9_add_shl(V, V, VB0, 0);     // 9 V_B0 + 4p - V_B1
    u9_add_shl(VB1, VB1, VB1, 3);
    u9_add_shl(VB1, VB1, VB0, 0);  // V_B0 + 9 V_B1
#pragma unroll
    for (int i = 0; i < 9; i++) VB0[i] = V[i];
  }
  fp_add_nr(s, yo.c0.l, yo.c0.l);
  r.c0 = fp_lin3(VB0, Fp{{s[0], s[1], s[2], s[3], s[4], s[5], s[6], s[7]}});
  fp_add_nr(s, yo.c1.l, yo.c1.l);
  r.c1 = fp_lin3(VB1, Fp{{s[0], s[1], s[2], s[3], s[4], s[5], s[6], s[7]}});
  y = r;
}

// Granger-Scott (pairing.rs:309-346), in place: (z0, z1) -> (z0, z1), (z2, z3) -> (z4, z5), (z4, z5) -> (z3, z2).
// The second pair's outputs overwrite the third pair's inputs, so those two coefficients are copied first.
SY_HD_NOINLINE void cyclotomic_square_assign(Fp12& f) {
  Fp2 &z0 = f.c0.c0, &z4 = f.c0.c1, &z3 = f.c0.c2, &z2 = f.c1.c0, &z1 = f.c1.c1, &z5 = f.c1.c2;
  gs_fp4_square(z0, z1, z0, z1, false);
  const Fp2 t4 = z4, t5 = z5;
  gs_fp4_square(z2, z3, z4, z5, false);
  gs_fp4_square(t4, t5, z3, z2, true);
}
SY_HD Fp12 cyclotomic_squared(const Fp12& f) {
  Fp12 r = f;
  cyclotomic_square_assign(r);
  return r;
}

// f <- conj(f^x) with x = BLS_X (pairing.rs:366-392), in place.  The reference walks 256 exponent bits one at a time;
// the value f^x is the same for any addition chain, so this uses the width-4 NAF of x (63 digits, 14 of them non-zero,
// digits +-1 .. +-7): 62 + 1 cyclotomic squarings and 13 + 3 multiplications instead of 62 + 27.  A negative digit
// multiplies by the conjugate (the inverse on the cyclotomic subgroup f lives in) through fp12_mul_assign's flag, so
// the table holds only f^3, f^5, f^7 (f itself stays in the caller's slot): 4 Fp12 of frame instead of 10.
SY_HD_NOINLINE void exp_by_neg_z_assign(Fp12& f, Fp12* acc = nullptr) {
  Fp12 tab[3], res_local;
  Fp12& res = acc ? *acc : res_local;  // the running value: the kernels pass a shared-memory slot
  res = f;
  cyclotomic_square_assign(res);  // f^2
  tab[0] = f;
  fp12_mul_assign(tab[0], res);
  tab[1] = tab[0];
  fp12_mul_assign(tab[1], res);
  tab[2] = tab[1];
  fp12_mul_assign(tab[2], res);
  {
    int i0 = (SY_TAB(kXWnaf4)[0] - 1) >> 1;  // the leading digit is positive
    res = i0 ? tab[i0 - 1] : f;
  }
  for (int i = 1; i < SY_XWNAF4_LEN; i++) {
    // the block re-converges every SECOND digit: 177.0 -> 174.4 ms per 2^20 against a barrier per digit (every third or
    // fourth digit, or only after the digits that multiply, are slower again: profiles/r02p_kbench_sync.jsonl)
    if (i % 2 == 0) SY_LOOP_SYNC();
    cyclotomic_square_assign(res);
    int d = SY_TAB(kXWnaf4)[i];
    if (d != 0) {
      int idx = ((d > 0 ? d : -d) - 1) >> 1;
      fp12_mul_assign(res, idx ? tab[idx - 1] : f, d < 0);
    }
  }
  fp12_conj_assign(res);
  f = res;
}
SY_HD Fp12 exp_by_neg_z(const Fp12& f) {
  Fp12 r = f;
  exp_by_neg_z_assign(r);
  return r;
}

// pairing.rs:245-492, in place.  Five Fp12 slots in all (f and four locals): every product updates one of its factors,
// Frobenius images go through one scratch slot, and conjugated factors use fp12_mul_assign's flag.
SY_HD_NOINLINE void final_exponentiation_assign(Fp12& f, Fp12* acc = nullptr) {
  Fp12 A, C, E, G;
  // easy part (:410-415)
  SY_LOOP_SYNC();
  A = fp12_inv(f);
  fp12_conj_assign(f);
  fp12_mul_assign(f, A);
  SY_LOOP_SYNC();
  fp12_frobenius_to(A, f, 2);
  fp12_mul_assign(f, A);  // f = inp
  // hard part (:437-489); the comments give the reference's names
  A = f;
  exp_by_neg_z_assign(A, acc);    // a
  cyclotomic_square_assign(A);    // b
  C = A;
  cyclotomic_square_assign(C);    // c
  fp12_mul_assign(C, A);          // d = c b
  E = C;
  exp_by_neg_z_assign(E, acc);    // e
  G = E;
  cyclotomic_square_assign(G);    // f
  exp_by_neg_z_assign(G, acc);    // g
  SY_LOOP_SYNC();
  fp12_conj_assign(G);
  fp12_mul_assign(G, E);          // h = conj(g) e    (:463-465)
  fp12_mul_assign(G, C, true);    // k = h conj(d)
  fp12_mul_assign(A, G);          // l = k b
  SY_LOOP_SYNC();
  fp12_mul_assign(E, G);          // m = k e
  fp12_mul_assign(E, f);          // n = inp m
  fp12_frobenius_to(C, A, 1);
  fp12_mul_assign(E, C);          // p = frobenius(l, 1) n
  SY_LOOP_SYNC();
  fp12_frobenius_to(C, G, 2);
  fp12_mul_assign(E, C);          // r = frobenius(k, 2) p
  fp12_mul_assign(A, f, true);    // t = conj(inp) l
  fp12_frobenius_to(C, A, 3);
  fp12_mul_assign(E, C);          // frobenius(t, 3) r
  f = E;
}
SY_HD Fp12 final_exponentiation(const Fp12& f0) {
  Fp12 r = f0;
  final_exponentiation_assign(r);
  return r;
}


// `&Gt * &Fr` (gt.rs:188-215): g^k for g in the cyclotomic subgroup (every Gt value is a final
// exponentiation output).  The reference runs a 256-digit NAF ladder with Fp12 squarings; the value g^k does
// not depend on the chain, so this uses fixed 4-bit windows with cyclotomic squarings and no data-dependent
// control flow.
SY_HD_NOINLINE Fp12 gt_pow(const Fp12& g, const uint32_t* k) {
  Fp12 tab[16];
  tab[0] = fp12_one();
  tab[1] = g;
  for (int i = 2; i < 16; i++) tab[i] = (i & 1) ? fp12_mul(tab[i - 1], g) : cyclotomic_squared(tab[i >> 1]);
  // g^p is the Frobenius map and p = mu (mod r), the order of Gt: the G2 decomposition k = sum k_j mu^j (curve.cuh)
  // turns the exponentiation into 17 windows of 4 cyclotomic squarings and 4 multiplications by frobenius^j(tab[d_j]);
  // a negative k_j multiplies by the conjugate (the inverse on the cyclotomic subgroup).
  uint32_t mag[4][3];
  bool neg[4];
  gls_decompose(k, mag, neg);
  Fp12 acc = fp12_one();
  for (int w = 16; w >= 0; w--) {
    SY_LOOP_SYNC();
    if (w != 16) {
      cyclotomic_square_assign(acc);
      cyclotomic_square_assign(acc);
      cyclotomic_square_assign(acc);
      cyclotomic_square_assign(acc);
    }
    for (int e = 0; e < 4; e++) {
      Fp12 t = tab[(mag[e][w >> 3] >> ((w & 7) * 4)) & 15u];
      if (e) t = fp12_frobenius(t, e);
      if (neg[e]) t = fp12_conj(t);
      fp12_mul_assign(acc, t);
    }
  }
  return acc;
}

}  // namespace sylow

// G1 = E(Fp): y^2 = x^3 + 3 and G2 in E'(Fp2): y^2 = x^3 + 3/(9+u), homogeneous projective
// coordinates with the complete a = 0 formulas of Renes-Costello-Batina (eprint 2015/1060 Algs 7, 9).
//
// Value-level replacement of /root/reference/src/groups/group.rs:339-386 (double), :528-599 (add),
// :639-667 (scalar multiplication by an Fp-range scalar) and :475-495 (projective -> affine).  Parity
// is defined on AFFINE coordinates (SURVEY.md Q14), so the scalar multiplication is free to use a
// GLV split with fixed 4-bit windows and no data-dependent branches instead of the reference's NAF loop.
#pragma once
#include "constants.cuh"

namespace sylow {

// field dispatch by overload
SY_HD Fp f_add(const Fp& a, const Fp& b) { return fp_add(a, b); }
SY_HD Fp f_sub(const Fp& a, const Fp& b) { return fp_sub(a, b); }
SY_HD Fp f_mul(const Fp& a, const Fp& b) { return fp_mul(a, b); }
SY_HD Fp f_sqr(const Fp& a) { return fp_sqr(a); }
SY_HD Fp f_mul_b3(const Fp& a) { return fp_mul9(a); }  // 3b = 9
SY_HD Fp f_neg(const Fp& a) { return fp_neg(a); }
SY_HD bool f_is_zero(const Fp& a) { return fp_is_zero(a); }
SY_HD void f_set_zero(Fp& a) { a = fp_zero(); }
SY_HD void f_set_one(Fp& a) { a = fp_one(); }
SY_HD Fp f_inv(const Fp& a) { return fp_inv(a); }

SY_HD Fp2 f_add(const Fp2& a, const Fp2& b) { return fp2_add(a, b); }
SY_HD Fp2 f_sub(const Fp2& a, const Fp2& b) { return fp2_sub(a, b); }
SY_HD Fp2 f_mul(const Fp2& a, const Fp2& b) { return fp2_mul(a, b); }
SY_HD Fp2 f_sqr(const Fp2& a) { return fp2_sqr(a); }
SY_HD Fp2 f_mul_b3(const Fp2& a) { return fp2_mul(a, SY_TAB(kTwistB3)[0]); }
SY_HD Fp2 f_neg(const Fp2& a) { return fp2_neg(a); }
SY_HD bool f_is_zero(const Fp2& a) { return fp2_is_zero(a); }
SY_HD void f_set_zero(Fp2& a) { a = fp2_zero(); }
SY_HD void f_set_one(Fp2& a) { a = fp2_one(); }
SY_HD Fp2 f_inv(const Fp2& a) { return fp2_inv(a); }

template <class F>
struct Proj {
  F x, y, z;
};
template <class F>
struct Affine {
  F x, y;
  bool inf;
};
typedef Proj<Fp> G1Proj;
typedef Proj<Fp2> G2Proj;
typedef Affine<Fp> G1Aff;
typedef Affine<Fp2> G2Aff;

// (0 : 1 : 0), group.rs:320-331
template <class F>
SY_HD Proj<F> proj_zero() {
  Proj<F> r;
  f_set_zero(r.x);
  f_set_one(r.y);
  f_set_zero(r.z);
  return r;
}

// Alg. 9 (group.rs:339-386).  The formula maps (0:1:0) to (0:Y:0), so no select is needed for the
// value of the affine result; the reference's select only normalises the representative.
template <class F>
SY_HD_NOINLINE Proj<F> proj_double(const Proj<F>& p) {
  F t0 = f_sqr(p.y);
  F z3 = f_add(t0, t0);
  z3 = f_add(z3, z3);
  z3 = f_add(z3, z3);
  F t1 = f_mul(p.y, p.z);
  F t2 = f_sqr(p.z);
  t2 = f_mul_b3(t2);
  F x3 = f_mul(t2, z3);
  F y3 = f_add(t0, t2);
  z3 = f_mul(t1, z3);
  t1 = f_add(t2, t2);
  t2 = f_add(t1, t2);
  t0 = f_sub(t0, t2);
  y3 = f_mul(t0, y3);
  y3 = f_add(x3, y3);
  t1 = f_mul(p.x, p.y);
  x3 = f_mul(t0, t1);
  x3 = f_add(x3, x3);
  return Proj<F>{x3, y3, z3};
}

// Alg. 7 (group.rs:528-599)
template <class F>
SY_HD_NOINLINE Proj<F> proj_add(const Proj<F>& a, const Proj<F>& b) {
  F t0 = f_mul(a.x, b.x);
  F t1 = f_mul(a.y, b.y);
  F t2 = f_mul(a.z, b.z);
  F t3 = f_mul(f_add(a.x, a.y), f_add(b.x, b.y));
  t3 = f_sub(t3, f_add(t0, t1));
  F t4 = f_mul(f_add(a.y, a.z), f_add(b.y, b.z));
  t4 = f_sub(t4, f_add(t1, t2));
  F y3 = f_mul(f_add(a.x, a.z), f_add(b.x, b.z));
  y3 = f_sub(y3, f_add(t0, t2));
  F x3 = f_add(t0, t0);
  t0 = f_add(x3, t0);
  t2 = f_mul_b3(t2);
  F z3 = f_add(t1, t2);
  t1 = f_sub(t1, t2);
  y3 = f_mul_b3(y3);
  x3 = f_mul(t4, y3);
  t2 = f_mul(t3, t1);
  x3 = f_sub(t2, x3);
  y3 = f_mul(y3, t0);
  t1 = f_mul(t1, z3);
  y3 = f_add(t1, y3);
  t0 = f_mul(t0, t3);
  z3 = f_mul(z3, t4);
  z3 = f_add(z3, t0);
  return Proj<F>{x3, y3, z3};
}

template <class F>
SY_HD Proj<F> affine_to_proj(const Affine<F>& a) {
  // a flagged point is (0 : 1 : 0) whatever its coordinate bytes hold (GroupAffine::zero(), group.rs:236-244)
  Proj<F> r = proj_zero<F>();
  if (!a.inf) {
    r.x = a.x;
    r.y = a.y;
    f_set_one(r.z);
  }
  return r;
}

// group.rs:475-495: x/z, y/z; z == 0 gives (0, 1, infinity)
template <class F>
SY_HD_NOINLINE Affine<F> proj_to_affine(const Proj<F>& p) {
  Affine<F> r;
  F zi = f_inv(p.z);
  r.inf = f_is_zero(zi);
  r.x = f_mul(p.x, zi);
  r.y = f_mul(p.y, zi);
  if (r.inf) {
    f_set_zero(r.x);
    f_set_one(r.y);
  }
  return r;
}

// k * P for a 256-bit scalar k (8 LE words; the reference takes an Fp-range scalar and does not reduce
// it mod r, group.rs:639-667 / SURVEY Q8 - the group has order r so the affine result is the same).
// Fixed 4-bit windows, table of 0..15 multiples, complete additions: no data-dependent control flow.
template <class F>
SY_HD_NOINLINE Proj<F> proj_scalar_mul(const Proj<F>& p, const uint32_t* k) {
  Proj<F> tab[16];
  tab[0] = proj_zero<F>();
  tab[1] = p;
  for (int i = 2; i < 16; i++) tab[i] = (i & 1) ? proj_add(tab[i - 1], p) : proj_double(tab[i >> 1]);
  Proj<F> acc = tab[k[7] >> 28];
  for (int w = 62; w >= 0; w--) {
    SY_LOOP_SYNC();
    acc = proj_double(acc);
    acc = proj_double(acc);
    acc = proj_double(acc);
    acc = proj_double(acc);
    uint32_t d = (k[w >> 3] >> ((w & 7) * 4)) & 15u;
    acc = proj_add(acc, tab[d]);
  }
  return acc;
}

// k * P for a 64-bit k (the random weights of batch verification): 16 windows of 4 bits.
template <class F>
SY_HD_NOINLINE Proj<F> proj_scalar_mul_u64(const Proj<F>& p, uint64_t k) {
  Proj<F> tab[16];
  tab[0] = proj_zero<F>();
  tab[1] = p;
  for (int i = 2; i < 16; i++) tab[i] = (i & 1) ? proj_add(tab[i - 1], p) : proj_double(tab[i >> 1]);
  Proj<F> acc = tab[(uint32_t)(k >> 60)];
  for (int w = 14; w >= 0; w--) {
    SY_LOOP_SYNC();
    acc = proj_double(acc);
    acc = proj_double(acc);
    acc = proj_double(acc);
    acc = proj_double(acc);
    acc = proj_add(acc, tab[(uint32_t)(k >> (4 * w)) & 15u]);
  }
  return acc;
}

// Signed 4-bit windows of a magnitude of NW * 4 bits whose top window is at most 7: digits in [-8, 8], least significant
// first.  A table of the multiples 0..8 then serves every window (half the table of unsigned windows, half the
// additions to build it); a negative digit negates the selected point's y.
template <int NW>
SY_HD void signed_windows4(const uint32_t* mag, int8_t* digit) {
  int carry = 0;
  for (int w = 0; w < NW; w++) {
    int d = (int)((mag[w >> 3] >> ((w & 7) * 4)) & 15u) + carry;
    carry = d > 8;
    digit[w] = (int8_t)(d - (carry << 4));
  }
}
// multiples 0..8 of p
template <class F>
SY_HD void small_multiples(Proj<F>* tab, const Proj<F>& p) {
  tab[0] = proj_zero<F>();
  tab[1] = p;
  tab[2] = proj_double(p);
  tab[3] = proj_add(tab[2], p);
  tab[4] = proj_double(tab[2]);
  tab[5] = proj_add(tab[4], p);
  tab[6] = proj_double(tab[3]);
  tab[7] = proj_add(tab[6], p);
  tab[8] = proj_double(tab[4]);
}

// ---- GLV scalar multiplication --------------------------------------------------------------------
// phi(x, y) = (beta x, y) is an endomorphism of both curves (j = 0) and acts on the r-torsion as
// multiplication by lambda, lambda^2 + lambda + 1 = 0 mod r.  k = k1 + k2 lambda (mod r) with
// |k1|, |k2| < 2^127 halves the number of doublings.  The result equals k * P as a group element for
// every P of order r, i.e. the same affine point as the reference's loop (group.rs:639-667).
SY_HD Fp f_mul_beta(const Fp& x) { return fp_mul(x, SY_TAB(kBetaG1)[0]); }
SY_HD Fp2 f_mul_beta(const Fp2& x) { return fp2_mul_fp(x, SY_TAB(kBetaG2)[0]); }

// t[0..NA+NB) = a * b, schoolbook on 32-bit limbs
template <int NA, int NB>
SY_HD void mp_mul(uint32_t* t, const uint32_t* a, const uint32_t* b) {
  for (int i = 0; i < NA + NB; i++) t[i] = 0;
  for (int i = 0; i < NA; i++) {
    uint64_t carry = 0;
    for (int j = 0; j < NB; j++) {
      uint64_t v = (uint64_t)a[i] * b[j] + t[i + j] + carry;
      t[i + j] = (uint32_t)v;
      carry = v >> 32;
    }
    t[i + NB] = (uint32_t)carry;
  }
}
// r[0..8) -= a[0..n) mod 2^256
SY_HD void mp_sub256(uint32_t* r, const uint32_t* a, int n) {
  uint32_t borrow = 0;
  for (int i = 0; i < 8; i++) {
    uint64_t v = (uint64_t)r[i] - (i < n ? a[i] : 0u) - borrow;
    r[i] = (uint32_t)v;
    borrow = (uint32_t)(v >> 63);
  }
}
// two's complement 256-bit value -> magnitude (4 limbs, the bound above) and sign
SY_HD bool mp_abs128(uint32_t* mag, const uint32_t* v) {
  bool neg = (v[7] >> 31) != 0;
  uint32_t carry = neg ? 1u : 0u, m = neg ? 0xFFFFFFFFu : 0u;
  for (int i = 0; i < 4; i++) {
    uint64_t s = (uint64_t)(v[i] ^ m) + carry;
    mag[i] = (uint32_t)s;
    carry = (uint32_t)(s >> 32);
  }
  return neg;
}
// Babai rounding with precomputed g_i = round(2^320 b_i / r): c_i = (k g_i) >> 320 is within one of
// k b_i / r, so the remainders are bounded by |a1| + |a2| and |b1| + |b2| < 2^127.
SY_HD void glv_decompose(const uint32_t* k, uint32_t* k1, bool& neg1, uint32_t* k2, bool& neg2) {
  uint32_t t[16], c1[3], c2[5], u[9], s1[8], s2[8];
  mp_mul<8, 5>(t, k, SY_TAB(kGlvG1));
  for (int i = 0; i < 3; i++) c1[i] = t[10 + i];
  mp_mul<8, 7>(t, k, SY_TAB(kGlvG2));
  for (int i = 0; i < 5; i++) c2[i] = t[10 + i];
  for (int i = 0; i < 8; i++) s1[i] = k[i];
  mp_mul<3, 2>(u, c1, SY_TAB(kGlvA1));
  mp_sub256(s1, u, 5);
  mp_mul<5, 4>(u, c2, SY_TAB(kGlvA2));
  mp_sub256(s1, u, 8);
  mp_mul<3, 4>(u, c1, SY_TAB(kGlvNB1));
  for (int i = 0; i < 8; i++) s2[i] = i < 7 ? u[i] : 0u;
  mp_mul<5, 2>(u, c2, SY_TAB(kGlvB2));
  mp_sub256(s2, u, 7);
  neg1 = mp_abs128(k1, s1);
  neg2 = mp_abs128(k2, s2);
}

// k * P = k1 * P + k2 * phi(P): one table of 0..15 multiples of P serves both halves (phi is applied to
// the selected entry), 32 windows of 4 bits, complete additions, no data-dependent control flow.
template <class F>
SY_HD_NOINLINE Proj<F> proj_scalar_mul_glv(const Proj<F>& p, const uint32_t* k) {
  uint32_t k1[4], k2[4];
  bool neg1, neg2;
  glv_decompose(k, k1, neg1, k2, neg2);
  int8_t d1[32], d2[32];
  signed_windows4<32>(k1, d1);  // |k1|, |k2| < 2^127: the top window is at most 7
  signed_windows4<32>(k2, d2);
  Proj<F> tab[9];
  small_multiples(tab, p);
  Proj<F> acc = proj_zero<F>();
  for (int w = 31; w >= 0; w--) {
    SY_LOOP_SYNC();
    if (w != 31) {
      acc = proj_double(acc);
      acc = proj_double(acc);
      acc = proj_double(acc);
      acc = proj_double(acc);
    }
    int a = d1[w], b = d2[w];
    Proj<F> t = tab[a < 0 ? -a : a];
    if (neg1 != (a < 0)) t.y = f_neg(t.y);
    acc = proj_add(acc, t);
    t = tab[b < 0 ? -b : b];
    t.x = f_mul_beta(t.x);
    if (neg2 != (b < 0)) t.y = f_neg(t.y);
    acc = proj_add(acc, t);
  }
  return acc;
}

// psi on a projective point (also used by the subgroup check below)
SY_HD G2Proj g2_psi_1(const G2Proj& q) {
  return G2Proj{fp2_mul(SY_TAB(kEpsExp0)[0], fp2_conj(q.x)), fp2_mul(SY_TAB(kEpsExp1)[0], fp2_conj(q.y)), fp2_conj(q.z)};
}
// ---- 4-dimensional GLS scalar multiplication on G2 ----------------------------------------------------
// psi (g2.rs:140-152) acts on the r-torsion of the twist as multiplication by mu = p mod r = 6 x^2, so
// k = k0 + k1 mu + k2 mu^2 + k3 mu^3 with |k_j| < 2^67 (Galbraith-Scott basis, Babai rounding with precomputed
// 320-bit-scaled cofactors; constants.cuh) needs 64 doublings instead of GLV's 128.
SY_HD void mp_add256(uint32_t* r, const uint32_t* a, int n) {
  uint64_t c = 0;
  for (int i = 0; i < 8; i++) {
    c += (uint64_t)r[i] + (i < n ? a[i] : 0u);
    r[i] = (uint32_t)c;
    c >>= 32;
  }
}
// two's complement 256-bit value -> magnitude (3 limbs: < 2^67 here) and sign
SY_HD bool mp_abs96(uint32_t* mag, const uint32_t* v) {
  bool neg = (v[7] >> 31) != 0;
  uint32_t carry = neg ? 1u : 0u, m = neg ? 0xFFFFFFFFu : 0u;
  for (int i = 0; i < 3; i++) {
    uint64_t s = (uint64_t)(v[i] ^ m) + carry;
    mag[i] = (uint32_t)s;
    carry = (uint32_t)(s >> 32);
  }
  return neg;
}
template <int NC>
SY_HD void gls_apply_row(uint32_t acc[4][8], const uint32_t* c, int i) {
  for (int j = 0; j < 4; j++) {
    uint32_t t[NC + 3];
    mp_mul<NC, 3>(t, c, SY_TAB(kGlsB) + 3 * (4 * i + j));
    if ((SY_GLS_SUBMASK >> (4 * i + j)) & 1u)
      mp_sub256(acc[j], t, NC + 3);
    else
      mp_add256(acc[j], t, NC + 3);
  }
}
SY_HD void gls_decompose(const uint32_t* k, uint32_t mag[4][3], bool neg[4]) {
  uint32_t acc[4][8], t[17];
  for (int j = 0; j < 4; j++)
    for (int i = 0; i < 8; i++) acc[j][i] = j == 0 ? k[i] : 0u;
  mp_mul<8, 6>(t, k, SY_TAB(kGlsG0));
  gls_apply_row<4>(acc, t + 10, 0);
  mp_mul<8, 9>(t, k, SY_TAB(kGlsG1));
  gls_apply_row<7>(acc, t + 10, 1);
  mp_mul<8, 8>(t, k, SY_TAB(kGlsG2));
  gls_apply_row<6>(acc, t + 10, 2);
  mp_mul<8, 6>(t, k, SY_TAB(kGlsG3));
  gls_apply_row<4>(acc, t + 10, 3);
  for (int j = 0; j < 4; j++) neg[j] = mp_abs96(mag[j], acc[j]);
}
// psi^e of a projective point, e = 0..3 (conjugation is the p-power Frobenius of Fp2; the constants are
// xi^((p-1)/3), xi^((p-1)/2) and their products with their own norms)
SY_HD G2Proj g2_psi_pow(const G2Proj& q, int e) {
  switch (e) {
    case 1: return g2_psi_1(q);
    case 2: return G2Proj{fp2_mul_fp(q.x, SY_TAB(kPsi2X)[0]), fp2_mul_fp(q.y, SY_TAB(kPsi2Y)[0]), q.z};
    case 3: return G2Proj{fp2_mul(SY_TAB(kPsi3X)[0], fp2_conj(q.x)), fp2_mul(SY_TAB(kPsi3Y)[0], fp2_conj(q.y)), fp2_conj(q.z)};
    default: return q;
  }
}
SY_HD_NOINLINE G2Proj g2_scalar_mul_gls(const G2Proj& p, const uint32_t* k) {
  uint32_t mag[4][3];
  bool neg[4];
  gls_decompose(k, mag, neg);
  int8_t dg[4][17];
  for (int e = 0; e < 4; e++) signed_windows4<17>(mag[e], dg[e]);  // |k_j| < 2^67: the top window is at most 7
  G2Proj tab[9];
  small_multiples(tab, p);
  G2Proj acc = proj_zero<Fp2>();
  for (int w = 16; w >= 0; w--) {
    SY_LOOP_SYNC();
    if (w != 16) {
      acc = proj_double(acc);
      acc = proj_double(acc);
      acc = proj_double(acc);
      acc = proj_double(acc);
    }
    for (int e = 0; e < 4; e++) {
      int d = dg[e][w];
      G2Proj t = g2_psi_pow(tab[d < 0 ? -d : d], e);
      if (neg[e] != (d < 0)) t.y = fp2_neg(t.y);
      acc = proj_add(acc, t);
    }
  }
  return acc;
}

// ---- fixed-base multiplication by a generator -------------------------------------------------------------
// k G with a table of affine multiples of G: T[w][j] = (j + 1) 2^(C w) G, j < 2^(C-1), Montgomery form, x || y.
// k mod r is recoded into W = ceil(254 / C) signed C-bit digits, least significant first, and the selected entries are
// added up: W mixed additions and no doublings.  The table is built on the device from the variable-base ladder
// (sylow_b200.cu: build_mul_tables), so its entries are the ladder's own affine points.
#define SY_GEN_C 8
#define SY_GEN_W ((254 + SY_GEN_C - 1) / SY_GEN_C)
#define SY_GEN_E (1 << (SY_GEN_C - 1))  // entries per window
static_assert(SY_GEN_C >= 6 && SY_GEN_C <= 8, "the top digit bound below is shown for C = 6, 7, 8");

SY_HD Fp f_select(bool c, const Fp& a, const Fp& b) { return fp_select(c, a, b); }
SY_HD Fp2 f_select(bool c, const Fp2& a, const Fp2& b) { return fp2_select(c, a, b); }

// Renes-Costello-Batina Alg. 8 (a = 0): a + (b.x : b.y : 1), 11M + 2 m_3b.  Complete for every projective a, b.inf
// ignored (the caller never adds the point at infinity): a = O gives b, a = -b gives O, a = b doubles.
template <class F>
SY_HD_NOINLINE Proj<F> proj_add_mixed(const Proj<F>& a, const Affine<F>& b) {
  F t0 = f_mul(a.x, b.x);
  F t1 = f_mul(a.y, b.y);
  F t3 = f_mul(f_add(b.x, b.y), f_add(a.x, a.y));
  t3 = f_sub(t3, f_add(t0, t1));
  F t4 = f_add(f_mul(b.y, a.z), a.y);
  F y3 = f_add(f_mul(b.x, a.z), a.x);
  F x3 = f_add(t0, t0);
  t0 = f_add(x3, t0);
  F t2 = f_mul_b3(a.z);
  F z3 = f_add(t1, t2);
  t1 = f_sub(t1, t2);
  y3 = f_mul_b3(y3);
  x3 = f_mul(t4, y3);
  t2 = f_mul(t3, t1);
  x3 = f_sub(t2, x3);
  y3 = f_mul(y3, t0);
  t1 = f_mul(t1, z3);
  y3 = f_add(t1, y3);
  t0 = f_mul(t0, t3);
  z3 = f_mul(z3, t4);
  z3 = f_add(z3, t0);
  return Proj<F>{x3, y3, z3};
}

// k mod r in place for any 256-bit k: 2^256 < 6 r, so five conditional subtractions leave k < r < 2^254
SY_HD void scalar_reduce_r(uint32_t* k) {
  for (int s = 0; s < 5; s++) {
    uint32_t d[8], borrow = 0;
    for (int i = 0; i < 8; i++) {
      uint64_t v = (uint64_t)k[i] - SY_TAB(kFrMod)[i] - borrow;
      d[i] = (uint32_t)v;
      borrow = (uint32_t)(v >> 63);
    }
    for (int i = 0; i < 8; i++) k[i] = borrow ? k[i] : d[i];
  }
}
// bits [pos, pos + C) of the 256-bit k (pos + C may pass bit 255: those bits read as 0)
template <int C>
SY_HD uint32_t scalar_window(const uint32_t* k, int pos) {
  const int i = pos >> 5, s = pos & 31;
  uint64_t v = k[i];
  if (i < 7) v |= (uint64_t)k[i + 1] << 32;
  return (uint32_t)(v >> s) & ((1u << C) - 1);
}
// Signed digit of window w of k < 2^254, and the carry into window w + 1: d in [-2^(C-1) + 1, 2^(C-1)].  The top
// window holds at most 254 - C (W - 1) <= C - 2 bits, so its digit plus carry stays below 2^(C-1) and never carries.
template <int C>
SY_HD int scalar_digit(const uint32_t* k, int w, int& carry) {
  int d = (int)scalar_window<C>(k, C * w) + carry;
  carry = d > (1 << (C - 1));
  return d - (carry << C);
}

SY_HD uint4 ld_nc(const uint8_t* p) {
#if defined(__CUDA_ARCH__)
  return __ldg(reinterpret_cast<const uint4*>(p));  // ld.global.nc: the table is read-only while a kernel reads it
#else
  return *reinterpret_cast<const uint4*>(p);
#endif
}
SY_HD void gen_entry_load(const uint8_t* p, Affine<Fp>& e) {
  uint4 v[4] = {ld_nc(p), ld_nc(p + 16), ld_nc(p + 32), ld_nc(p + 48)};
  e.x = Fp{{v[0].x, v[0].y, v[0].z, v[0].w, v[1].x, v[1].y, v[1].z, v[1].w}};
  e.y = Fp{{v[2].x, v[2].y, v[2].z, v[2].w, v[3].x, v[3].y, v[3].z, v[3].w}};
}
SY_HD void gen_entry_load(const uint8_t* p, Affine<Fp2>& e) {
  Affine<Fp> a, b;
  gen_entry_load(p, a);
  gen_entry_load(p + 64, b);
  e.x = Fp2{a.x, a.y};
  e.y = Fp2{b.x, b.y};
}

// acc + k G over the table `tab` of G (SY_GEN_W x SY_GEN_E entries of 2 sizeof(F) bytes): the digit only selects an entry
// and the sign of its y, a zero digit keeps the accumulator; no data-dependent branches.  A non-zero start lets one
// accumulator walk the tables of several bases (groth16.cuh: groth16_public_term).
template <class F>
SY_HD Proj<F> gen_scalar_mul_add(const uint8_t* __restrict__ tab, const uint32_t* k_in, Proj<F> acc) {
  uint32_t k[8];
  for (int i = 0; i < 8; i++) k[i] = k_in[i];
  scalar_reduce_r(k);
  int carry = 0;
#pragma unroll
  for (int w = 0; w < SY_GEN_W; w++) {
    const int d = scalar_digit<SY_GEN_C>(k, w, carry);
    const int m = d < 0 ? -d : d;
    Affine<F> e;
    gen_entry_load(tab + ((size_t)w * SY_GEN_E + (m ? m - 1 : 0)) * 2 * sizeof(F), e);
    e.y = f_select(d < 0, f_neg(e.y), e.y);
    Proj<F> s = proj_add_mixed(acc, e);
    acc.x = f_select(m != 0, s.x, acc.x);
    acc.y = f_select(m != 0, s.y, acc.y);
    acc.z = f_select(m != 0, s.z, acc.z);
  }
  return acc;
}
// k G (gen_scalar_mul_add from O)
template <class F>
SY_HD_NOINLINE Proj<F> gen_scalar_mul(const uint8_t* __restrict__ tab, const uint32_t* k_in) {
  return gen_scalar_mul_add<F>(tab, k_in, proj_zero<F>());
}

// y^2 == x^3 + b
SY_HD bool g1_on_curve(const Fp& x, const Fp& y) {
  Fp rhs = fp_add(fp_mul(fp_sqr(x), x), SY_TAB(kFpThree)[0]);
  return fp_eq(fp_sqr(y), rhs);
}
SY_HD bool g2_on_curve(const Fp2& x, const Fp2& y) {
  Fp2 rhs = fp2_add(fp2_mul(fp2_sqr(x), x), SY_TAB(kTwistB)[0]);
  return fp2_eq(fp2_sqr(y), rhs);
}


// ---- input validation (SURVEY.md 8f-1) ------------------------------------------------------------
// psi on a projective point: (eps0 * conj(x), eps1 * conj(y), conj(z)) - the same point the reference
// reaches through affine coordinates (g2.rs:140-152, :207-210).
SY_HD G2Proj g2_psi(const G2Proj& q) { return g2_psi_1(q); }
// cross-multiplied projective equality (group.rs:426-447)
SY_HD bool g2_proj_eq(const G2Proj& a, const G2Proj& b) {
  bool az = fp2_is_zero(a.z), bz = fp2_is_zero(b.z);
  bool same = fp2_eq(fp2_mul(a.x, b.z), fp2_mul(b.x, a.z)) & fp2_eq(fp2_mul(a.y, b.z), fp2_mul(b.y, a.z));
  return (az & bz) | (!az & !bz & same);
}
// [x]Q for the BN parameter x (63 bits, compile-time constant: uniform control flow), width-4 NAF: the odd
// multiples Q, 3Q, 5Q, 7Q and 13 additions instead of the 27 of the binary expansion
SY_HD_NOINLINE G2Proj g2_mul_by_x(const G2Proj& q) {
  G2Proj tab[4];
  {
    G2Proj q2 = proj_double(q);
    tab[0] = q;
    for (int i = 1; i < 4; i++) tab[i] = proj_add(tab[i - 1], q2);
  }
  G2Proj acc = tab[(SY_TAB(kXWnaf4)[0] - 1) >> 1];
  for (int i = 1; i < SY_XWNAF4_LEN; i++) {
    SY_LOOP_SYNC();
    acc = proj_double(acc);
    int d = SY_TAB(kXWnaf4)[i];
    if (d != 0) {
      G2Proj t = tab[((d > 0 ? d : -d) - 1) >> 1];
      if (d < 0) t.y = fp2_neg(t.y);
      acc = proj_add(acc, t);
    }
  }
  return acc;
}
// G2Projective::new's subgroup relation (g2.rs:460-525): (x+1)Q + psi(xQ) + psi^2(xQ) == psi^3(2xQ)
SY_HD_NOINLINE bool g2_in_subgroup(const Fp2& x, const Fp2& y) {
  G2Proj q{x, y, fp2_one()};
  G2Proj a = g2_mul_by_x(q);
  G2Proj b = g2_psi(a);
  a = proj_add(a, q);
  G2Proj c = g2_psi(b);
  G2Proj lhs = proj_add(proj_add(c, b), a);
  G2Proj rhs = proj_double(g2_psi(c));
  return g2_proj_eq(lhs, rhs);
}

}  // namespace sylow

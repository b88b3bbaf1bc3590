// Fp arithmetic for BN254 on sm_100a: 8 x 32-bit limbs, Montgomery form (R = 2^256).
//
// Replaces (value-level) sylow's `Fp` operators, /root/reference/src/fields/fp.rs:304-457, which
// delegate to crypto-bigint ConstMontyForm<U256>.  Every value that leaves the device is converted
// back to the canonical residue in [0, p), so results are bit-identical to the reference.
//
// Multiplication is a CIOS Montgomery product written as PTX mad.lo.cc / madc.hi.cc carry chains
// over two interleaved accumulators ("even" holds 64-bit columns aligned at limb 0,2,4,6 and "odd"
// the columns aligned at limb 1,3,5,7).  ptxas fuses every mad.lo.cc/madc.hi.cc pair into ONE
// IMAD.WIDE.U32(.X) with a predicate carry, so one Fp multiplication is 136 IMAD-pipe instructions
// (64 for a*b, 64 for m*p, 8 for m) - the 136 "limb products" SURVEY.md 8(d) counts.
#pragma once
#if defined(SYLOW_HOSTSIM)
#include <cstdio>
#include <cstdlib>
#endif
#include <cstdint>

#if defined(__CUDACC__)
#define SY_HD __host__ __device__ __forceinline__
#define SY_HD_NOINLINE __host__ __device__ __noinline__
#else
#define SY_HD inline
#define SY_HD_NOINLINE
#endif
// Tables live in __constant__ memory on the device.  The host copy exists only so that the
// test-only host simulation (tests/hostsim, -DSYLOW_HOSTSIM) can run the same tower/pairing source
// on a CPU; the product library never executes it.
#if defined(__CUDA_ARCH__)
#define SY_TAB(name) name##_d
#else
#define SY_TAB(name) name##_h
#endif
#define SY_DEFINE_TABLE(type, name, n, ...)                       \
  __device__ __constant__ const type name##_d[n] = {__VA_ARGS__}; \
  static const type name##_h[n] = {__VA_ARGS__};

// Block-wide re-convergence inside the long loops: keeps the warps of a block in the same region of
// the (large) instruction stream so instruction-cache lines fetched by one warp are hit by the others.
// Only legal when every thread of the block runs the loop (the kernels guarantee it).
#if defined(__CUDA_ARCH__)
#define SY_LOOP_SYNC() __syncthreads()
#else
#define SY_LOOP_SYNC() ((void)0)
#endif

namespace sylow {

// 16-byte alignment lets every load/store of a field element (including the local-memory frame traffic of
// the out-of-line Fp2 routines) be a 128-bit access.
struct alignas(16) Fp {
  uint32_t l[8];
};

// p = 0x30644e72e131a029b85045b68181585d97816a916871ca8d3c208c16d87cfd47 (fp.rs:51-56)
#define SY_P0 0xd87cfd47
#define SY_P1 0x3c208c16
#define SY_P2 0x6871ca8d
#define SY_P3 0x97816a91
#define SY_P4 0x8181585d
#define SY_P5 0xb85045b6
#define SY_P6 0xe131a029
#define SY_P7 0x30644e72
#define SY_STR2(x) #x
#define SY_STR(x) SY_STR2(x)
#define SY_INV 0xe4866389u  // -p^{-1} mod 2^32
#define SY_INV_ASM 0xe4866389

SY_DEFINE_TABLE(uint32_t, kP, 8, SY_P0, SY_P1, SY_P2, SY_P3, SY_P4, SY_P5, SY_P6, SY_P7)

SY_HD Fp fp_zero() {
  Fp r;
#pragma unroll
  for (int i = 0; i < 8; i++) r.l[i] = 0;
  return r;
}
// R mod p  (Montgomery form of 1)
SY_HD Fp fp_one() {
  return Fp{{0xc58f0d9du, 0xd35d438du, 0xf5c70b3du, 0x0a78eb28u, 0x7879462cu, 0x666ea36fu, 0x9a07df2fu, 0x0e0a77c1u}};
}
// R^2 mod p (to-Montgomery multiplier) and R^3 mod p (for 2^256 * hi in hash_to_field)
SY_HD Fp fp_R2() {
  return Fp{{0x538afa89u, 0xf32cfc5bu, 0xd44501fbu, 0xb5e71911u, 0x0a417ff6u, 0x47ab1effu, 0xcab8351fu, 0x06d89f71u}};
}
SY_HD Fp fp_R3() {
  return Fp{{0xda1530dfu, 0xb1cd6dafu, 0xa7283db6u, 0x62f210e6u, 0x0ada0afbu, 0xef7f0b0cu, 0x2d592544u, 0x20fd6e90u}};
}

SY_HD bool fp_is_zero(const Fp& a) {
  uint32_t o = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) o |= a.l[i];
  return o == 0;
}
SY_HD bool fp_eq(const Fp& a, const Fp& b) {
  uint32_t o = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) o |= a.l[i] ^ b.l[i];
  return o == 0;
}
SY_HD Fp fp_select(bool c, const Fp& a, const Fp& b) {  // c ? a : b
  Fp r;
#pragma unroll
  for (int i = 0; i < 8; i++) r.l[i] = c ? a.l[i] : b.l[i];
  return r;
}

// r = a - p if a >= p else a      (a < 2p)
SY_HD void fp_final_sub(uint32_t* a) {
  uint32_t t[8], borrow;
#if !defined(__CUDA_ARCH__)
  int64_t bw = 0;
  for (int i = 0; i < 8; i++) {
    int64_t d = (int64_t)a[i] - (int64_t)SY_TAB(kP)[i] + bw;
    t[i] = (uint32_t)d;
    bw = d >> 32;
  }
  borrow = (uint32_t)bw;
#else
  asm("sub.cc.u32 %0, %9, " SY_STR(SY_P0) ";\n\t"
      "subc.cc.u32 %1, %10, " SY_STR(SY_P1) ";\n\t"
      "subc.cc.u32 %2, %11, " SY_STR(SY_P2) ";\n\t"
      "subc.cc.u32 %3, %12, " SY_STR(SY_P3) ";\n\t"
      "subc.cc.u32 %4, %13, " SY_STR(SY_P4) ";\n\t"
      "subc.cc.u32 %5, %14, " SY_STR(SY_P5) ";\n\t"
      "subc.cc.u32 %6, %15, " SY_STR(SY_P6) ";\n\t"
      "subc.cc.u32 %7, %16, " SY_STR(SY_P7) ";\n\t"
      "subc.u32 %8, 0, 0;"
      : "=r"(t[0]), "=r"(t[1]), "=r"(t[2]), "=r"(t[3]), "=r"(t[4]), "=r"(t[5]), "=r"(t[6]), "=r"(t[7]), "=r"(borrow)
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]));
#endif
#pragma unroll
  for (int i = 0; i < 8; i++) a[i] = borrow ? a[i] : t[i];
}

SY_HD Fp fp_add(const Fp& a, const Fp& b) {
  Fp r;
#if !defined(__CUDA_ARCH__)
  uint64_t c = 0;
  for (int i = 0; i < 8; i++) {
    c += (uint64_t)a.l[i] + b.l[i];
    r.l[i] = (uint32_t)c;
    c >>= 32;
  }
#else
  asm("add.cc.u32 %0, %8, %16;\n\t"
      "addc.cc.u32 %1, %9, %17;\n\t"
      "addc.cc.u32 %2, %10, %18;\n\t"
      "addc.cc.u32 %3, %11, %19;\n\t"
      "addc.cc.u32 %4, %12, %20;\n\t"
      "addc.cc.u32 %5, %13, %21;\n\t"
      "addc.cc.u32 %6, %14, %22;\n\t"
      "addc.u32 %7, %15, %23;"
      : "=r"(r.l[0]), "=r"(r.l[1]), "=r"(r.l[2]), "=r"(r.l[3]), "=r"(r.l[4]), "=r"(r.l[5]), "=r"(r.l[6]), "=r"(r.l[7])
      : "r"(a.l[0]), "r"(a.l[1]), "r"(a.l[2]), "r"(a.l[3]), "r"(a.l[4]), "r"(a.l[5]), "r"(a.l[6]), "r"(a.l[7]),
        "r"(b.l[0]), "r"(b.l[1]), "r"(b.l[2]), "r"(b.l[3]), "r"(b.l[4]), "r"(b.l[5]), "r"(b.l[6]), "r"(b.l[7]));
#endif
  fp_final_sub(r.l);  // a + b < 2p < 2^255: no carry out of limb 7
  return r;
}

SY_HD Fp fp_sub(const Fp& a, const Fp& b) {
  Fp r;
  uint32_t borrow;
#if !defined(__CUDA_ARCH__)
  int64_t bw = 0;
  for (int i = 0; i < 8; i++) {
    int64_t d = (int64_t)a.l[i] - (int64_t)b.l[i] + bw;
    r.l[i] = (uint32_t)d;
    bw = d >> 32;
  }
  borrow = (uint32_t)bw;
  uint64_t c = 0;
  for (int i = 0; i < 8; i++) {
    c += (uint64_t)r.l[i] + (borrow & SY_TAB(kP)[i]);
    r.l[i] = (uint32_t)c;
    c >>= 32;
  }
#else
  asm("sub.cc.u32 %0, %9, %17;\n\t"
      "subc.cc.u32 %1, %10, %18;\n\t"
      "subc.cc.u32 %2, %11, %19;\n\t"
      "subc.cc.u32 %3, %12, %20;\n\t"
      "subc.cc.u32 %4, %13, %21;\n\t"
      "subc.cc.u32 %5, %14, %22;\n\t"
      "subc.cc.u32 %6, %15, %23;\n\t"
      "subc.cc.u32 %7, %16, %24;\n\t"
      "subc.u32 %8, 0, 0;"
      : "=r"(r.l[0]), "=r"(r.l[1]), "=r"(r.l[2]), "=r"(r.l[3]), "=r"(r.l[4]), "=r"(r.l[5]), "=r"(r.l[6]), "=r"(r.l[7]),
        "=r"(borrow)
      : "r"(a.l[0]), "r"(a.l[1]), "r"(a.l[2]), "r"(a.l[3]), "r"(a.l[4]), "r"(a.l[5]), "r"(a.l[6]), "r"(a.l[7]),
        "r"(b.l[0]), "r"(b.l[1]), "r"(b.l[2]), "r"(b.l[3]), "r"(b.l[4]), "r"(b.l[5]), "r"(b.l[6]), "r"(b.l[7]));
  // borrow is 0 or 0xffffffff: add back p & borrow
  asm("add.cc.u32 %0, %0, %8;\n\t"
      "addc.cc.u32 %1, %1, %9;\n\t"
      "addc.cc.u32 %2, %2, %10;\n\t"
      "addc.cc.u32 %3, %3, %11;\n\t"
      "addc.cc.u32 %4, %4, %12;\n\t"
      "addc.cc.u32 %5, %5, %13;\n\t"
      "addc.cc.u32 %6, %6, %14;\n\t"
      "addc.u32 %7, %7, %15;"
      : "+r"(r.l[0]), "+r"(r.l[1]), "+r"(r.l[2]), "+r"(r.l[3]), "+r"(r.l[4]), "+r"(r.l[5]), "+r"(r.l[6]), "+r"(r.l[7])
      : "r"(borrow & SY_P0), "r"(borrow & SY_P1), "r"(borrow & SY_P2), "r"(borrow & SY_P3), "r"(borrow & SY_P4),
        "r"(borrow & SY_P5), "r"(borrow & SY_P6), "r"(borrow & SY_P7));
#endif
  return r;
}

// a / 2 mod p: (a + (a odd ? p : 0)) >> 1.  Works on the Montgomery representative directly.
SY_HD Fp fp_halve(const Fp& a) {
  uint32_t m = 0u - (a.l[0] & 1u);
  Fp t;
#if !defined(__CUDA_ARCH__)
  uint64_t c = 0;
  for (int i = 0; i < 8; i++) {
    c += (uint64_t)a.l[i] + (m & SY_TAB(kP)[i]);
    t.l[i] = (uint32_t)c;
    c >>= 32;
  }
#else
  asm("add.cc.u32 %0, %8, %16;\n\t"
      "addc.cc.u32 %1, %9, %17;\n\t"
      "addc.cc.u32 %2, %10, %18;\n\t"
      "addc.cc.u32 %3, %11, %19;\n\t"
      "addc.cc.u32 %4, %12, %20;\n\t"
      "addc.cc.u32 %5, %13, %21;\n\t"
      "addc.cc.u32 %6, %14, %22;\n\t"
      "addc.u32 %7, %15, %23;"
      : "=r"(t.l[0]), "=r"(t.l[1]), "=r"(t.l[2]), "=r"(t.l[3]), "=r"(t.l[4]), "=r"(t.l[5]), "=r"(t.l[6]), "=r"(t.l[7])
      : "r"(a.l[0]), "r"(a.l[1]), "r"(a.l[2]), "r"(a.l[3]), "r"(a.l[4]), "r"(a.l[5]), "r"(a.l[6]), "r"(a.l[7]),
        "r"(m & SY_P0), "r"(m & SY_P1), "r"(m & SY_P2), "r"(m & SY_P3), "r"(m & SY_P4), "r"(m & SY_P5), "r"(m & SY_P6), "r"(m & SY_P7));
#endif
  Fp r;  // a + p < 2^255: the sum fits in 8 limbs
#pragma unroll
  for (int i = 0; i < 7; i++) r.l[i] = (t.l[i] >> 1) | (t.l[i + 1] << 31);
  r.l[7] = t.l[7] >> 1;
  return r;
}

SY_HD Fp fp_neg(const Fp& a) { return fp_sub(fp_zero(), a); }
SY_HD Fp fp_dbl(const Fp& a) { return fp_add(a, a); }

// Four 32x32->64 products with no addend, one IMAD.WIDE each: (X[2k], X[2k+1]) = a_k * b.  Written as mul.wide.u32
// because ptxas does not fuse a mul.lo / mul.hi pair (it emits IMAD + IMAD.HI, two multiplier-pipe instructions).
#if defined(__CUDA_ARCH__)
__device__ __forceinline__ void mul_row4(uint32_t* X, uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b) {
  asm("{\n\t"
      ".reg .u64 t0, t1, t2, t3;\n\t"
      "mul.wide.u32 t0, %8, %12;\n\t"
      "mul.wide.u32 t1, %9, %12;\n\t"
      "mul.wide.u32 t2, %10, %12;\n\t"
      "mul.wide.u32 t3, %11, %12;\n\t"
      "mov.b64 {%0, %1}, t0;\n\t"
      "mov.b64 {%2, %3}, t1;\n\t"
      "mov.b64 {%4, %5}, t2;\n\t"
      "mov.b64 {%6, %7}, t3;\n\t"
      "}"
      : "=r"(X[0]), "=r"(X[1]), "=r"(X[2]), "=r"(X[3]), "=r"(X[4]), "=r"(X[5]), "=r"(X[6]), "=r"(X[7])
      : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b));
}
#endif

// ---- Montgomery multiplication ------------------------------------------------------------------
// One CIOS round for multiplier limb bi.  T = X + Y * 2^32 (X: columns at limbs 0,2,4,6; Y: columns at
// limbs 1,3,5,7).  After the round X[0] == 0 and the caller swaps the roles of X and Y, which divides
// T by 2^32.  Bounds: T < 2p on entry, T + a*bi + m*p < 2^287, so neither accumulator overflows.
#if defined(__CUDA_ARCH__)
template <bool FIRST>
__device__ __forceinline__ void mont_round(uint32_t* X, uint32_t* Y, const uint32_t* a, uint32_t bi) {
  if (FIRST) {
    mul_row4(X, a[0], a[2], a[4], a[6], bi);
    mul_row4(Y, a[1], a[3], a[5], a[7], bi);
  } else {
    // X[0] += Y[1]; Y = (Y >> 64) + a_odd * bi   (carry of the first add feeds the chain)
    asm("add.cc.u32 %0, %0, %2;\n\t"
        "madc.lo.cc.u32 %1, %9, %13, %3;\n\t"
        "madc.hi.cc.u32 %2, %9, %13, %4;\n\t"
        "madc.lo.cc.u32 %3, %10, %13, %5;\n\t"
        "madc.hi.cc.u32 %4, %10, %13, %6;\n\t"
        "madc.lo.cc.u32 %5, %11, %13, %7;\n\t"
        "madc.hi.cc.u32 %6, %11, %13, %8;\n\t"
        "madc.lo.cc.u32 %7, %12, %13, 0;\n\t"
        "madc.hi.u32 %8, %12, %13, 0;"
        : "+r"(X[0]), "+r"(Y[0]), "+r"(Y[1]), "+r"(Y[2]), "+r"(Y[3]), "+r"(Y[4]), "+r"(Y[5]), "+r"(Y[6]), "+r"(Y[7])
        : "r"(a[1]), "r"(a[3]), "r"(a[5]), "r"(a[7]), "r"(bi));
    // X += a_even * bi; carry out (weight 2^256) lands in Y[7]
    asm("mad.lo.cc.u32 %0, %9, %13, %0;\n\t"
        "madc.hi.cc.u32 %1, %9, %13, %1;\n\t"
        "madc.lo.cc.u32 %2, %10, %13, %2;\n\t"
        "madc.hi.cc.u32 %3, %10, %13, %3;\n\t"
        "madc.lo.cc.u32 %4, %11, %13, %4;\n\t"
        "madc.hi.cc.u32 %5, %11, %13, %5;\n\t"
        "madc.lo.cc.u32 %6, %12, %13, %6;\n\t"
        "madc.hi.cc.u32 %7, %12, %13, %7;\n\t"
        "addc.u32 %8, %8, 0;"
        : "+r"(X[0]), "+r"(X[1]), "+r"(X[2]), "+r"(X[3]), "+r"(X[4]), "+r"(X[5]), "+r"(X[6]), "+r"(X[7]), "+r"(Y[7])
        : "r"(a[0]), "r"(a[2]), "r"(a[4]), "r"(a[6]), "r"(bi));
  }
  uint32_t m = X[0] * SY_INV;
  // Y += m * p_odd   (no carry out: Y * 2^32 <= T < 2^287)
  asm("mad.lo.cc.u32 %0, %8, " SY_STR(SY_P1) ", %0;\n\t"
      "madc.hi.cc.u32 %1, %8, " SY_STR(SY_P1) ", %1;\n\t"
      "madc.lo.cc.u32 %2, %8, " SY_STR(SY_P3) ", %2;\n\t"
      "madc.hi.cc.u32 %3, %8, " SY_STR(SY_P3) ", %3;\n\t"
      "madc.lo.cc.u32 %4, %8, " SY_STR(SY_P5) ", %4;\n\t"
      "madc.hi.cc.u32 %5, %8, " SY_STR(SY_P5) ", %5;\n\t"
      "madc.lo.cc.u32 %6, %8, " SY_STR(SY_P7) ", %6;\n\t"
      "madc.hi.u32 %7, %8, " SY_STR(SY_P7) ", %7;"
      : "+r"(Y[0]), "+r"(Y[1]), "+r"(Y[2]), "+r"(Y[3]), "+r"(Y[4]), "+r"(Y[5]), "+r"(Y[6]), "+r"(Y[7])
      : "r"(m));
  // X += m * p_even; carry out lands in Y[7]; X[0] becomes 0
  asm("mad.lo.cc.u32 %0, %9, " SY_STR(SY_P0) ", %0;\n\t"
      "madc.hi.cc.u32 %1, %9, " SY_STR(SY_P0) ", %1;\n\t"
      "madc.lo.cc.u32 %2, %9, " SY_STR(SY_P2) ", %2;\n\t"
      "madc.hi.cc.u32 %3, %9, " SY_STR(SY_P2) ", %3;\n\t"
      "madc.lo.cc.u32 %4, %9, " SY_STR(SY_P4) ", %4;\n\t"
      "madc.hi.cc.u32 %5, %9, " SY_STR(SY_P4) ", %5;\n\t"
      "madc.lo.cc.u32 %6, %9, " SY_STR(SY_P6) ", %6;\n\t"
      "madc.hi.cc.u32 %7, %9, " SY_STR(SY_P6) ", %7;\n\t"
      "addc.u32 %8, %8, 0;"
      : "+r"(X[0]), "+r"(X[1]), "+r"(X[2]), "+r"(X[3]), "+r"(X[4]), "+r"(X[5]), "+r"(X[6]), "+r"(X[7]), "+r"(Y[7])
      : "r"(m));
}

// r = a * b / R mod p, fully reduced.  Requires a < 2p (a is the multiplicand of every round: the
// running value stays below a + p, which must fit the 8-limb accumulators) and a * b < p * R; b may be
// ANY 256-bit value as long as the product bound holds - so conversions of unreduced inputs put the
// constant first: fp_mul(R^2, x) is valid for every x < 2^256.
__device__ __forceinline__ Fp fp_mul(const Fp& a, const Fp& b) {
  uint32_t ev[8], od[8];
  mont_round<true>(ev, od, a.l, b.l[0]);
  mont_round<false>(od, ev, a.l, b.l[1]);
  mont_round<false>(ev, od, a.l, b.l[2]);
  mont_round<false>(od, ev, a.l, b.l[3]);
  mont_round<false>(ev, od, a.l, b.l[4]);
  mont_round<false>(od, ev, a.l, b.l[5]);
  mont_round<false>(ev, od, a.l, b.l[6]);
  mont_round<false>(od, ev, a.l, b.l[7]);
  // last round used X = od, Y = ev: result = ev + (od >> 32)
  Fp r;
  asm("add.cc.u32 %0, %8, %16;\n\t"
      "addc.cc.u32 %1, %9, %17;\n\t"
      "addc.cc.u32 %2, %10, %18;\n\t"
      "addc.cc.u32 %3, %11, %19;\n\t"
      "addc.cc.u32 %4, %12, %20;\n\t"
      "addc.cc.u32 %5, %13, %21;\n\t"
      "addc.cc.u32 %6, %14, %22;\n\t"
      "addc.u32 %7, %15, 0;"
      : "=r"(r.l[0]), "=r"(r.l[1]), "=r"(r.l[2]), "=r"(r.l[3]), "=r"(r.l[4]), "=r"(r.l[5]), "=r"(r.l[6]), "=r"(r.l[7])
      : "r"(ev[0]), "r"(ev[1]), "r"(ev[2]), "r"(ev[3]), "r"(ev[4]), "r"(ev[5]), "r"(ev[6]), "r"(ev[7]),
        "r"(od[1]), "r"(od[2]), "r"(od[3]), "r"(od[4]), "r"(od[5]), "r"(od[6]), "r"(od[7]));
  fp_final_sub(r.l);
  return r;
}
#else
// host simulation only (tests/hostsim): textbook CIOS with 64-bit temporaries
inline Fp fp_mul(const Fp& a, const Fp& b) {
  uint32_t t[10] = {0};
  for (int i = 0; i < 8; i++) {
    uint64_t c = 0;
    for (int j = 0; j < 8; j++) {
      c += (uint64_t)a.l[j] * b.l[i] + t[j];
      t[j] = (uint32_t)c;
      c >>= 32;
    }
    c += t[8];
    t[8] = (uint32_t)c;
    t[9] = (uint32_t)(c >> 32);
    uint32_t m = t[0] * SY_INV;
    c = (uint64_t)m * kP_h[0] + t[0];
    c >>= 32;
    for (int j = 1; j < 8; j++) {
      c += (uint64_t)m * kP_h[j] + t[j];
      t[j - 1] = (uint32_t)c;
      c >>= 32;
    }
    c += t[8];
    t[7] = (uint32_t)c;
    t[8] = t[9] + (uint32_t)(c >> 32);
  }
  Fp r;
  for (int i = 0; i < 8; i++) r.l[i] = t[i];
  fp_final_sub(r.l);
  return r;
}
#endif

// ---- lazy reduction: full 512-bit products and a separate Montgomery reduction ----------------------
// fp_mul_wide: T = a * b as 16 plain limbs (64 IMAD.WIDE).  fp_redc_wide: T * R^-1 mod p for T < p * R
// (72 IMAD).  An Fp2 product needs 3 wide products and only 2 reductions (tower.cuh), 336 IMAD-pipe
// instructions instead of 3 * 136.  Inputs of fp_mul_wide may be unreduced sums (< 2^256).
#if defined(__CUDA_ARCH__)
// X[0..7] += (a0,a1,a2,a3) * b at limb pairs (0,1),(2,3),(4,5),(6,7); the carry out (weight 2^256 relative to X[0]) is
// added into `fold`, the limb of the OTHER accumulator that sits at that weight.  `fold` is always the top limb of a
// pair that wide_row_top has just written: hi(a7 * b) + carry <= a7, so the addition cannot overflow as long as the
// multiplicand's top limb is not 0xffffffff (every first operand of fp_mul_wide is below 4p < 2^256 - 2^224).
__device__ __forceinline__ void wide_row_fold(uint32_t* X, uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b,
                                              uint32_t& fold) {
  asm("mad.lo.cc.u32 %0, %9, %13, %0;\n\t"
      "madc.hi.cc.u32 %1, %9, %13, %1;\n\t"
      "madc.lo.cc.u32 %2, %10, %13, %2;\n\t"
      "madc.hi.cc.u32 %3, %10, %13, %3;\n\t"
      "madc.lo.cc.u32 %4, %11, %13, %4;\n\t"
      "madc.hi.cc.u32 %5, %11, %13, %5;\n\t"
      "madc.lo.cc.u32 %6, %12, %13, %6;\n\t"
      "madc.hi.cc.u32 %7, %12, %13, %7;\n\t"
      "addc.u32 %8, %8, 0;"
      : "+r"(X[0]), "+r"(X[1]), "+r"(X[2]), "+r"(X[3]), "+r"(X[4]), "+r"(X[5]), "+r"(X[6]), "+r"(X[7]), "+r"(fold)
      : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b));
}
// X[0..5] += ..., the top pair (X[6], X[7]) is fresh (written): the product a3 * b plus the chain's carry
__device__ __forceinline__ void wide_row_top(uint32_t* X, uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b) {
  asm("mad.lo.cc.u32 %0, %8, %12, %0;\n\t"
      "madc.hi.cc.u32 %1, %8, %12, %1;\n\t"
      "madc.lo.cc.u32 %2, %9, %12, %2;\n\t"
      "madc.hi.cc.u32 %3, %9, %12, %3;\n\t"
      "madc.lo.cc.u32 %4, %10, %12, %4;\n\t"
      "madc.hi.cc.u32 %5, %10, %12, %5;\n\t"
      "madc.lo.cc.u32 %6, %11, %12, 0;\n\t"
      "madc.hi.u32 %7, %11, %12, 0;"
      : "+r"(X[0]), "+r"(X[1]), "+r"(X[2]), "+r"(X[3]), "+r"(X[4]), "+r"(X[5]), "=r"(X[6]), "=r"(X[7])
      : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b));
}
__device__ __forceinline__ void wide_row_first(uint32_t* X, uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b) {
  mul_row4(X, a0, a1, a2, a3, b);
}

// T = a * b.  E collects the products whose position i+j is even, O (offset by one limb) the others.  For every
// multiplier limb the row of the odd multiplicand limbs goes first and WRITES its top pair, then the row of the even
// limbs accumulates below it and folds its carry into that pair's top limb - no carry is ever materialised in a
// register of its own.  Requires a[7] != 0xffffffff (see wide_row_fold); b is any 256-bit value.
__device__ __forceinline__ void fp_mul_wide(uint32_t* T, const uint32_t* a, const uint32_t* b) {
  uint32_t E[16], O[16];
  wide_row_first(E, a[0], a[2], a[4], a[6], b[0]);
  wide_row_first(O, a[1], a[3], a[5], a[7], b[0]);
  // b1: odd limbs -> E[2..9] (E[8], E[9] fresh); even limbs -> O[0..7], carry into E[9]
  wide_row_top(E + 2, a[1], a[3], a[5], a[7], b[1]);
  wide_row_fold(O + 0, a[0], a[2], a[4], a[6], b[1], E[9]);
#pragma unroll
  for (int i = 2; i < 8; i += 2) {
    // b_i: odd limbs -> O[i..i+7] (top pair fresh); even limbs -> E[i..i+7], carry into O[i+7]
    wide_row_top(O + i, a[1], a[3], a[5], a[7], b[i]);
    wide_row_fold(E + i, a[0], a[2], a[4], a[6], b[i], O[i + 7]);
    // b_(i+1): odd limbs -> E[i+2..i+9] (top pair fresh); even limbs -> O[i..i+7], carry into E[i+9]
    wide_row_top(E + i + 2, a[1], a[3], a[5], a[7], b[i + 1]);
    wide_row_fold(O + i, a[0], a[2], a[4], a[6], b[i + 1], E[i + 9]);
  }
  // T = E + (O << 32); O[0..13] are defined, the sum is < 2^512
  T[0] = E[0];
  asm("add.cc.u32 %0, %15, %30;\n\t"
      "addc.cc.u32 %1, %16, %31;\n\t"
      "addc.cc.u32 %2, %17, %32;\n\t"
      "addc.cc.u32 %3, %18, %33;\n\t"
      "addc.cc.u32 %4, %19, %34;\n\t"
      "addc.cc.u32 %5, %20, %35;\n\t"
      "addc.cc.u32 %6, %21, %36;\n\t"
      "addc.cc.u32 %7, %22, %37;\n\t"
      "addc.cc.u32 %8, %23, %38;\n\t"
      "addc.cc.u32 %9, %24, %39;\n\t"
      "addc.cc.u32 %10, %25, %40;\n\t"
      "addc.cc.u32 %11, %26, %41;\n\t"
      "addc.cc.u32 %12, %27, %42;\n\t"
      "addc.cc.u32 %13, %28, %43;\n\t"
      "addc.u32 %14, %29, 0;"
      : "=r"(T[1]), "=r"(T[2]), "=r"(T[3]), "=r"(T[4]), "=r"(T[5]), "=r"(T[6]), "=r"(T[7]), "=r"(T[8]), "=r"(T[9]),
        "=r"(T[10]), "=r"(T[11]), "=r"(T[12]), "=r"(T[13]), "=r"(T[14]), "=r"(T[15])
      : "r"(E[1]), "r"(E[2]), "r"(E[3]), "r"(E[4]), "r"(E[5]), "r"(E[6]), "r"(E[7]), "r"(E[8]), "r"(E[9]), "r"(E[10]),
        "r"(E[11]), "r"(E[12]), "r"(E[13]), "r"(E[14]), "r"(E[15]), "r"(O[0]), "r"(O[1]), "r"(O[2]), "r"(O[3]),
        "r"(O[4]), "r"(O[5]), "r"(O[6]), "r"(O[7]), "r"(O[8]), "r"(O[9]), "r"(O[10]), "r"(O[11]), "r"(O[12]),
        "r"(O[13]));
}

// One reduce-only CIOS round (mont_round without the a * b_i terms): T = X + Y * 2^32, X[0] -> 0, roles swap.
template <bool FIRST>
__device__ __forceinline__ void redc_round(uint32_t* X, uint32_t* Y) {
  uint32_t m;
  if (FIRST) {
    m = X[0] * SY_INV;
    mul_row4(Y, SY_P1, SY_P3, SY_P5, SY_P7, m);
  } else {
    // X[0] += Y[1]; m = X[0] * inv; Y = (Y >> 64) + m * p_odd   (the fold carry feeds the chain)
    asm("add.cc.u32 %0, %0, %2;\n\t"
        "mul.lo.u32 %9, %0, " SY_STR(SY_INV_ASM) ";\n\t"
        "madc.lo.cc.u32 %1, %9, " SY_STR(SY_P1) ", %3;\n\t"
        "madc.hi.cc.u32 %2, %9, " SY_STR(SY_P1) ", %4;\n\t"
        "madc.lo.cc.u32 %3, %9, " SY_STR(SY_P3) ", %5;\n\t"
        "madc.hi.cc.u32 %4, %9, " SY_STR(SY_P3) ", %6;\n\t"
        "madc.lo.cc.u32 %5, %9, " SY_STR(SY_P5) ", %7;\n\t"
        "madc.hi.cc.u32 %6, %9, " SY_STR(SY_P5) ", %8;\n\t"
        "madc.lo.cc.u32 %7, %9, " SY_STR(SY_P7) ", 0;\n\t"
        "madc.hi.u32 %8, %9, " SY_STR(SY_P7) ", 0;"
        : "+r"(X[0]), "+r"(Y[0]), "+r"(Y[1]), "+r"(Y[2]), "+r"(Y[3]), "+r"(Y[4]), "+r"(Y[5]), "+r"(Y[6]), "+r"(Y[7]),
          "=&r"(m));
  }
  asm("mad.lo.cc.u32 %0, %9, " SY_STR(SY_P0) ", %0;\n\t"
      "madc.hi.cc.u32 %1, %9, " SY_STR(SY_P0) ", %1;\n\t"
      "madc.lo.cc.u32 %2, %9, " SY_STR(SY_P2) ", %2;\n\t"
      "madc.hi.cc.u32 %3, %9, " SY_STR(SY_P2) ", %3;\n\t"
      "madc.lo.cc.u32 %4, %9, " SY_STR(SY_P4) ", %4;\n\t"
      "madc.hi.cc.u32 %5, %9, " SY_STR(SY_P4) ", %5;\n\t"
      "madc.lo.cc.u32 %6, %9, " SY_STR(SY_P6) ", %6;\n\t"
      "madc.hi.cc.u32 %7, %9, " SY_STR(SY_P6) ", %7;\n\t"
      "addc.u32 %8, %8, 0;"
      : "+r"(X[0]), "+r"(X[1]), "+r"(X[2]), "+r"(X[3]), "+r"(X[4]), "+r"(X[5]), "+r"(X[6]), "+r"(X[7]), "+r"(Y[7])
      : "r"(m));
}

// W = (T_lo + M p) / R <= p for the low half T_lo = T[0..7] (8 reduce-only CIOS rounds): W = T_lo * R^-1 mod p.
__device__ __forceinline__ Fp redc_low(const uint32_t* T) {
  uint32_t ev[8], od[8];
#pragma unroll
  for (int i = 0; i < 8; i++) ev[i] = T[i];
  redc_round<true>(ev, od);
  redc_round<false>(od, ev);
  redc_round<false>(ev, od);
  redc_round<false>(od, ev);
  redc_round<false>(ev, od);
  redc_round<false>(od, ev);
  redc_round<false>(ev, od);
  redc_round<false>(od, ev);
  // last round: X = od, Y = ev  ->  W = ev + (od >> 32)
  Fp w;
  asm("add.cc.u32 %0, %8, %16;\n\t"
      "addc.cc.u32 %1, %9, %17;\n\t"
      "addc.cc.u32 %2, %10, %18;\n\t"
      "addc.cc.u32 %3, %11, %19;\n\t"
      "addc.cc.u32 %4, %12, %20;\n\t"
      "addc.cc.u32 %5, %13, %21;\n\t"
      "addc.cc.u32 %6, %14, %22;\n\t"
      "addc.u32 %7, %15, 0;"
      : "=r"(w.l[0]), "=r"(w.l[1]), "=r"(w.l[2]), "=r"(w.l[3]), "=r"(w.l[4]), "=r"(w.l[5]), "=r"(w.l[6]), "=r"(w.l[7])
      : "r"(ev[0]), "r"(ev[1]), "r"(ev[2]), "r"(ev[3]), "r"(ev[4]), "r"(ev[5]), "r"(ev[6]), "r"(ev[7]),
        "r"(od[1]), "r"(od[2]), "r"(od[3]), "r"(od[4]), "r"(od[5]), "r"(od[6]), "r"(od[7]));
  return w;
}

// r = T * R^-1 mod p, fully reduced, for T < p * R: W + T_hi with W <= p, T_hi < p.
__device__ __forceinline__ Fp fp_redc_wide(const uint32_t* T) {
  Fp w = redc_low(T), r;
  asm("add.cc.u32 %0, %8, %16;\n\t"
      "addc.cc.u32 %1, %9, %17;\n\t"
      "addc.cc.u32 %2, %10, %18;\n\t"
      "addc.cc.u32 %3, %11, %19;\n\t"
      "addc.cc.u32 %4, %12, %20;\n\t"
      "addc.cc.u32 %5, %13, %21;\n\t"
      "addc.cc.u32 %6, %14, %22;\n\t"
      "addc.u32 %7, %15, %23;"
      : "=r"(r.l[0]), "=r"(r.l[1]), "=r"(r.l[2]), "=r"(r.l[3]), "=r"(r.l[4]), "=r"(r.l[5]), "=r"(r.l[6]), "=r"(r.l[7])
      : "r"(w.l[0]), "r"(w.l[1]), "r"(w.l[2]), "r"(w.l[3]), "r"(w.l[4]), "r"(w.l[5]), "r"(w.l[6]), "r"(w.l[7]),
        "r"(T[8]), "r"(T[9]), "r"(T[10]), "r"(T[11]), "r"(T[12]), "r"(T[13]), "r"(T[14]), "r"(T[15]));
  fp_final_sub(r.l);  // W <= p, T_hi < p  ->  r < 2p
  return r;
}

// 16-limb a -= b; returns 0xffffffff if the subtraction borrowed (a < b), else 0
__device__ __forceinline__ uint32_t wide_sub(uint32_t* a, const uint32_t* b) {
  uint32_t borrow;
  asm("sub.cc.u32 %0, %0, %17;\n\t"
      "subc.cc.u32 %1, %1, %18;\n\t"
      "subc.cc.u32 %2, %2, %19;\n\t"
      "subc.cc.u32 %3, %3, %20;\n\t"
      "subc.cc.u32 %4, %4, %21;\n\t"
      "subc.cc.u32 %5, %5, %22;\n\t"
      "subc.cc.u32 %6, %6, %23;\n\t"
      "subc.cc.u32 %7, %7, %24;\n\t"
      "subc.cc.u32 %8, %8, %25;\n\t"
      "subc.cc.u32 %9, %9, %26;\n\t"
      "subc.cc.u32 %10, %10, %27;\n\t"
      "subc.cc.u32 %11, %11, %28;\n\t"
      "subc.cc.u32 %12, %12, %29;\n\t"
      "subc.cc.u32 %13, %13, %30;\n\t"
      "subc.cc.u32 %14, %14, %31;\n\t"
      "subc.cc.u32 %15, %15, %32;\n\t"
      "subc.u32 %16, 0, 0;"
      : "+r"(a[0]), "+r"(a[1]), "+r"(a[2]), "+r"(a[3]), "+r"(a[4]), "+r"(a[5]), "+r"(a[6]), "+r"(a[7]), "+r"(a[8]),
        "+r"(a[9]), "+r"(a[10]), "+r"(a[11]), "+r"(a[12]), "+r"(a[13]), "+r"(a[14]), "+r"(a[15]), "=r"(borrow)
      : "r"(b[0]), "r"(b[1]), "r"(b[2]), "r"(b[3]), "r"(b[4]), "r"(b[5]), "r"(b[6]), "r"(b[7]), "r"(b[8]), "r"(b[9]),
        "r"(b[10]), "r"(b[11]), "r"(b[12]), "r"(b[13]), "r"(b[14]), "r"(b[15]));
  return borrow;
}
// a[8..15] += p & mask   (adds p * R to the 512-bit value when mask = 0xffffffff)
__device__ __forceinline__ void wide_add_pR(uint32_t* a, uint32_t mask) {
  asm("add.cc.u32 %0, %0, %8;\n\t"
      "addc.cc.u32 %1, %1, %9;\n\t"
      "addc.cc.u32 %2, %2, %10;\n\t"
      "addc.cc.u32 %3, %3, %11;\n\t"
      "addc.cc.u32 %4, %4, %12;\n\t"
      "addc.cc.u32 %5, %5, %13;\n\t"
      "addc.cc.u32 %6, %6, %14;\n\t"
      "addc.u32 %7, %7, %15;"
      : "+r"(a[8]), "+r"(a[9]), "+r"(a[10]), "+r"(a[11]), "+r"(a[12]), "+r"(a[13]), "+r"(a[14]), "+r"(a[15])
      : "r"(mask & SY_P0), "r"(mask & SY_P1), "r"(mask & SY_P2), "r"(mask & SY_P3), "r"(mask & SY_P4),
        "r"(mask & SY_P5), "r"(mask & SY_P6), "r"(mask & SY_P7));
}
// r = a + b without reduction (caller guarantees a + b < 2^256)
__device__ __forceinline__ void fp_add_nr(uint32_t* r, const uint32_t* a, const uint32_t* b) {
  asm("add.cc.u32 %0, %8, %16;\n\t"
      "addc.cc.u32 %1, %9, %17;\n\t"
      "addc.cc.u32 %2, %10, %18;\n\t"
      "addc.cc.u32 %3, %11, %19;\n\t"
      "addc.cc.u32 %4, %12, %20;\n\t"
      "addc.cc.u32 %5, %13, %21;\n\t"
      "addc.cc.u32 %6, %14, %22;\n\t"
      "addc.u32 %7, %15, %23;"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]),
        "r"(b[0]), "r"(b[1]), "r"(b[2]), "r"(b[3]), "r"(b[4]), "r"(b[5]), "r"(b[6]), "r"(b[7]));
}
// r = a - b without correction (caller guarantees a >= b)
__device__ __forceinline__ void fp_sub_nr(uint32_t* r, const uint32_t* a, const uint32_t* b) {
  asm("sub.cc.u32 %0, %8, %16;\n\t"
      "subc.cc.u32 %1, %9, %17;\n\t"
      "subc.cc.u32 %2, %10, %18;\n\t"
      "subc.cc.u32 %3, %11, %19;\n\t"
      "subc.cc.u32 %4, %12, %20;\n\t"
      "subc.cc.u32 %5, %13, %21;\n\t"
      "subc.cc.u32 %6, %14, %22;\n\t"
      "subc.u32 %7, %15, %23;"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]),
        "r"(b[0]), "r"(b[1]), "r"(b[2]), "r"(b[3]), "r"(b[4]), "r"(b[5]), "r"(b[6]), "r"(b[7]));
}
// 16-limb a <<= 1 (caller guarantees no overflow)
__device__ __forceinline__ void wide_dbl(uint32_t* a) {
#pragma unroll
  for (int i = 15; i > 0; i--) a[i] = __funnelshift_l(a[i - 1], a[i], 1);
  a[0] <<= 1;
}

// ---- 17-limb accumulators: a signed combination of 512-bit products, reduced once ---------------------------------
// A = sum k_i T_i + L p R with small integers k_i and a lift L p R (a multiple of p, so the residue is unchanged) that
// makes the sum non-negative.  The limbs are exact mod 2^544, so only the FINAL value has to lie in [0, 2^544); the
// callers state their bounds.  Each helper is one carry chain (acc_madd: two chains of 8 IMAD.WIDE).
// The top limb is materialised at the end of every helper: ptxas otherwise defers its final carry addition to the
// reduction, keeps that carry in a predicate register across the next products and spills predicates into a bit mask.
#define SY_ACC_TOP(A) asm volatile("" : "+r"((A)[16]))
// A = L p R - T for T < L p R; the 8 limbs of L p (< 2^256) are Lp.  A[16] = 0.
__device__ __forceinline__ void acc_lift_sub(uint32_t* A, const uint32_t* Lp, const uint32_t* T) {
  asm("sub.cc.u32 %0, 0, %17;\n\t"
      "subc.cc.u32 %1, 0, %18;\n\t"
      "subc.cc.u32 %2, 0, %19;\n\t"
      "subc.cc.u32 %3, 0, %20;\n\t"
      "subc.cc.u32 %4, 0, %21;\n\t"
      "subc.cc.u32 %5, 0, %22;\n\t"
      "subc.cc.u32 %6, 0, %23;\n\t"
      "subc.cc.u32 %7, 0, %24;\n\t"
      "subc.cc.u32 %8, %33, %25;\n\t"
      "subc.cc.u32 %9, %34, %26;\n\t"
      "subc.cc.u32 %10, %35, %27;\n\t"
      "subc.cc.u32 %11, %36, %28;\n\t"
      "subc.cc.u32 %12, %37, %29;\n\t"
      "subc.cc.u32 %13, %38, %30;\n\t"
      "subc.cc.u32 %14, %39, %31;\n\t"
      "subc.u32 %15, %40, %32;\n\t"
      "mov.u32 %16, 0;"
      : "=r"(A[0]), "=r"(A[1]), "=r"(A[2]), "=r"(A[3]), "=r"(A[4]), "=r"(A[5]), "=r"(A[6]), "=r"(A[7]), "=r"(A[8]),
        "=r"(A[9]), "=r"(A[10]), "=r"(A[11]), "=r"(A[12]), "=r"(A[13]), "=r"(A[14]), "=r"(A[15]), "=r"(A[16])
      : "r"(T[0]), "r"(T[1]), "r"(T[2]), "r"(T[3]), "r"(T[4]), "r"(T[5]), "r"(T[6]), "r"(T[7]), "r"(T[8]), "r"(T[9]),
        "r"(T[10]), "r"(T[11]), "r"(T[12]), "r"(T[13]), "r"(T[14]), "r"(T[15]), "r"(Lp[0]), "r"(Lp[1]), "r"(Lp[2]),
        "r"(Lp[3]), "r"(Lp[4]), "r"(Lp[5]), "r"(Lp[6]), "r"(Lp[7]));
}
// A = C + T and A = C - T (mod 2^544) for a 17-limb constant C: the first term of an accumulator together with its
// whole lift (a table of fp.cuh or tower.cuh)
__device__ __forceinline__ void acc_const_add(uint32_t* A, const uint32_t* C, const uint32_t* T) {
  asm("add.cc.u32 %0, %17, %34;\n\t"
      "addc.cc.u32 %1, %18, %35;\n\t"
      "addc.cc.u32 %2, %19, %36;\n\t"
      "addc.cc.u32 %3, %20, %37;\n\t"
      "addc.cc.u32 %4, %21, %38;\n\t"
      "addc.cc.u32 %5, %22, %39;\n\t"
      "addc.cc.u32 %6, %23, %40;\n\t"
      "addc.cc.u32 %7, %24, %41;\n\t"
      "addc.cc.u32 %8, %25, %42;\n\t"
      "addc.cc.u32 %9, %26, %43;\n\t"
      "addc.cc.u32 %10, %27, %44;\n\t"
      "addc.cc.u32 %11, %28, %45;\n\t"
      "addc.cc.u32 %12, %29, %46;\n\t"
      "addc.cc.u32 %13, %30, %47;\n\t"
      "addc.cc.u32 %14, %31, %48;\n\t"
      "addc.cc.u32 %15, %32, %49;\n\t"
      "addc.u32 %16, %33, 0;"
      : "=r"(A[0]), "=r"(A[1]), "=r"(A[2]), "=r"(A[3]), "=r"(A[4]), "=r"(A[5]), "=r"(A[6]), "=r"(A[7]), "=r"(A[8]),
        "=r"(A[9]), "=r"(A[10]), "=r"(A[11]), "=r"(A[12]), "=r"(A[13]), "=r"(A[14]), "=r"(A[15]), "=r"(A[16])
      : "r"(C[0]), "r"(C[1]), "r"(C[2]), "r"(C[3]), "r"(C[4]), "r"(C[5]), "r"(C[6]), "r"(C[7]), "r"(C[8]), "r"(C[9]),
        "r"(C[10]), "r"(C[11]), "r"(C[12]), "r"(C[13]), "r"(C[14]), "r"(C[15]), "r"(C[16]), "r"(T[0]), "r"(T[1]),
        "r"(T[2]), "r"(T[3]), "r"(T[4]), "r"(T[5]), "r"(T[6]), "r"(T[7]), "r"(T[8]), "r"(T[9]), "r"(T[10]), "r"(T[11]),
        "r"(T[12]), "r"(T[13]), "r"(T[14]), "r"(T[15]));
  SY_ACC_TOP(A);
}
__device__ __forceinline__ void acc_const_sub(uint32_t* A, const uint32_t* C, const uint32_t* T) {
  asm("sub.cc.u32 %0, %17, %34;\n\t"
      "subc.cc.u32 %1, %18, %35;\n\t"
      "subc.cc.u32 %2, %19, %36;\n\t"
      "subc.cc.u32 %3, %20, %37;\n\t"
      "subc.cc.u32 %4, %21, %38;\n\t"
      "subc.cc.u32 %5, %22, %39;\n\t"
      "subc.cc.u32 %6, %23, %40;\n\t"
      "subc.cc.u32 %7, %24, %41;\n\t"
      "subc.cc.u32 %8, %25, %42;\n\t"
      "subc.cc.u32 %9, %26, %43;\n\t"
      "subc.cc.u32 %10, %27, %44;\n\t"
      "subc.cc.u32 %11, %28, %45;\n\t"
      "subc.cc.u32 %12, %29, %46;\n\t"
      "subc.cc.u32 %13, %30, %47;\n\t"
      "subc.cc.u32 %14, %31, %48;\n\t"
      "subc.cc.u32 %15, %32, %49;\n\t"
      "subc.u32 %16, %33, 0;"
      : "=r"(A[0]), "=r"(A[1]), "=r"(A[2]), "=r"(A[3]), "=r"(A[4]), "=r"(A[5]), "=r"(A[6]), "=r"(A[7]), "=r"(A[8]),
        "=r"(A[9]), "=r"(A[10]), "=r"(A[11]), "=r"(A[12]), "=r"(A[13]), "=r"(A[14]), "=r"(A[15]), "=r"(A[16])
      : "r"(C[0]), "r"(C[1]), "r"(C[2]), "r"(C[3]), "r"(C[4]), "r"(C[5]), "r"(C[6]), "r"(C[7]), "r"(C[8]), "r"(C[9]),
        "r"(C[10]), "r"(C[11]), "r"(C[12]), "r"(C[13]), "r"(C[14]), "r"(C[15]), "r"(C[16]), "r"(T[0]), "r"(T[1]),
        "r"(T[2]), "r"(T[3]), "r"(T[4]), "r"(T[5]), "r"(T[6]), "r"(T[7]), "r"(T[8]), "r"(T[9]), "r"(T[10]), "r"(T[11]),
        "r"(T[12]), "r"(T[13]), "r"(T[14]), "r"(T[15]));
  SY_ACC_TOP(A);
}
// A = -T mod 2^544 (17 limbs)
__device__ __forceinline__ void acc_neg(uint32_t* A, const uint32_t* T) {
  asm("sub.cc.u32 %0, 0, %17;\n\t"
      "subc.cc.u32 %1, 0, %18;\n\t"
      "subc.cc.u32 %2, 0, %19;\n\t"
      "subc.cc.u32 %3, 0, %20;\n\t"
      "subc.cc.u32 %4, 0, %21;\n\t"
      "subc.cc.u32 %5, 0, %22;\n\t"
      "subc.cc.u32 %6, 0, %23;\n\t"
      "subc.cc.u32 %7, 0, %24;\n\t"
      "subc.cc.u32 %8, 0, %25;\n\t"
      "subc.cc.u32 %9, 0, %26;\n\t"
      "subc.cc.u32 %10, 0, %27;\n\t"
      "subc.cc.u32 %11, 0, %28;\n\t"
      "subc.cc.u32 %12, 0, %29;\n\t"
      "subc.cc.u32 %13, 0, %30;\n\t"
      "subc.cc.u32 %14, 0, %31;\n\t"
      "subc.cc.u32 %15, 0, %32;\n\t"
      "subc.u32 %16, 0, %33;"
      : "=r"(A[0]), "=r"(A[1]), "=r"(A[2]), "=r"(A[3]), "=r"(A[4]), "=r"(A[5]), "=r"(A[6]), "=r"(A[7]), "=r"(A[8]),
        "=r"(A[9]), "=r"(A[10]), "=r"(A[11]), "=r"(A[12]), "=r"(A[13]), "=r"(A[14]), "=r"(A[15]), "=r"(A[16])
      : "r"(T[0]), "r"(T[1]), "r"(T[2]), "r"(T[3]), "r"(T[4]), "r"(T[5]), "r"(T[6]), "r"(T[7]), "r"(T[8]), "r"(T[9]),
        "r"(T[10]), "r"(T[11]), "r"(T[12]), "r"(T[13]), "r"(T[14]), "r"(T[15]), "r"(T[16]));
  SY_ACC_TOP(A);
}
// A += T
__device__ __forceinline__ void acc_add(uint32_t* A, const uint32_t* T) {
  asm("add.cc.u32 %0, %0, %17;\n\t"
      "addc.cc.u32 %1, %1, %18;\n\t"
      "addc.cc.u32 %2, %2, %19;\n\t"
      "addc.cc.u32 %3, %3, %20;\n\t"
      "addc.cc.u32 %4, %4, %21;\n\t"
      "addc.cc.u32 %5, %5, %22;\n\t"
      "addc.cc.u32 %6, %6, %23;\n\t"
      "addc.cc.u32 %7, %7, %24;\n\t"
      "addc.cc.u32 %8, %8, %25;\n\t"
      "addc.cc.u32 %9, %9, %26;\n\t"
      "addc.cc.u32 %10, %10, %27;\n\t"
      "addc.cc.u32 %11, %11, %28;\n\t"
      "addc.cc.u32 %12, %12, %29;\n\t"
      "addc.cc.u32 %13, %13, %30;\n\t"
      "addc.cc.u32 %14, %14, %31;\n\t"
      "addc.cc.u32 %15, %15, %32;\n\t"
      "addc.u32 %16, %16, 0;"
      : "+r"(A[0]), "+r"(A[1]), "+r"(A[2]), "+r"(A[3]), "+r"(A[4]), "+r"(A[5]), "+r"(A[6]), "+r"(A[7]), "+r"(A[8]),
        "+r"(A[9]), "+r"(A[10]), "+r"(A[11]), "+r"(A[12]), "+r"(A[13]), "+r"(A[14]), "+r"(A[15]), "+r"(A[16])
      : "r"(T[0]), "r"(T[1]), "r"(T[2]), "r"(T[3]), "r"(T[4]), "r"(T[5]), "r"(T[6]), "r"(T[7]), "r"(T[8]), "r"(T[9]),
        "r"(T[10]), "r"(T[11]), "r"(T[12]), "r"(T[13]), "r"(T[14]), "r"(T[15]));
  SY_ACC_TOP(A);
}
// A -= T
__device__ __forceinline__ void acc_sub(uint32_t* A, const uint32_t* T) {
  asm("sub.cc.u32 %0, %0, %17;\n\t"
      "subc.cc.u32 %1, %1, %18;\n\t"
      "subc.cc.u32 %2, %2, %19;\n\t"
      "subc.cc.u32 %3, %3, %20;\n\t"
      "subc.cc.u32 %4, %4, %21;\n\t"
      "subc.cc.u32 %5, %5, %22;\n\t"
      "subc.cc.u32 %6, %6, %23;\n\t"
      "subc.cc.u32 %7, %7, %24;\n\t"
      "subc.cc.u32 %8, %8, %25;\n\t"
      "subc.cc.u32 %9, %9, %26;\n\t"
      "subc.cc.u32 %10, %10, %27;\n\t"
      "subc.cc.u32 %11, %11, %28;\n\t"
      "subc.cc.u32 %12, %12, %29;\n\t"
      "subc.cc.u32 %13, %13, %30;\n\t"
      "subc.cc.u32 %14, %14, %31;\n\t"
      "subc.cc.u32 %15, %15, %32;\n\t"
      "subc.u32 %16, %16, 0;"
      : "+r"(A[0]), "+r"(A[1]), "+r"(A[2]), "+r"(A[3]), "+r"(A[4]), "+r"(A[5]), "+r"(A[6]), "+r"(A[7]), "+r"(A[8]),
        "+r"(A[9]), "+r"(A[10]), "+r"(A[11]), "+r"(A[12]), "+r"(A[13]), "+r"(A[14]), "+r"(A[15]), "+r"(A[16])
      : "r"(T[0]), "r"(T[1]), "r"(T[2]), "r"(T[3]), "r"(T[4]), "r"(T[5]), "r"(T[6]), "r"(T[7]), "r"(T[8]), "r"(T[9]),
        "r"(T[10]), "r"(T[11]), "r"(T[12]), "r"(T[13]), "r"(T[14]), "r"(T[15]));
  SY_ACC_TOP(A);
}
// A += K T: the even limbs of T in one chain over A[0..16], the odd limbs in a second one over A[1..16]
template <uint32_t K>
__device__ __forceinline__ void acc_madd(uint32_t* A, const uint32_t* T) {
  asm("mad.lo.cc.u32 %0, %17, %25, %0;\n\t"
      "madc.hi.cc.u32 %1, %17, %25, %1;\n\t"
      "madc.lo.cc.u32 %2, %18, %25, %2;\n\t"
      "madc.hi.cc.u32 %3, %18, %25, %3;\n\t"
      "madc.lo.cc.u32 %4, %19, %25, %4;\n\t"
      "madc.hi.cc.u32 %5, %19, %25, %5;\n\t"
      "madc.lo.cc.u32 %6, %20, %25, %6;\n\t"
      "madc.hi.cc.u32 %7, %20, %25, %7;\n\t"
      "madc.lo.cc.u32 %8, %21, %25, %8;\n\t"
      "madc.hi.cc.u32 %9, %21, %25, %9;\n\t"
      "madc.lo.cc.u32 %10, %22, %25, %10;\n\t"
      "madc.hi.cc.u32 %11, %22, %25, %11;\n\t"
      "madc.lo.cc.u32 %12, %23, %25, %12;\n\t"
      "madc.hi.cc.u32 %13, %23, %25, %13;\n\t"
      "madc.lo.cc.u32 %14, %24, %25, %14;\n\t"
      "madc.hi.cc.u32 %15, %24, %25, %15;\n\t"
      "addc.u32 %16, %16, 0;"
      : "+r"(A[0]), "+r"(A[1]), "+r"(A[2]), "+r"(A[3]), "+r"(A[4]), "+r"(A[5]), "+r"(A[6]), "+r"(A[7]), "+r"(A[8]),
        "+r"(A[9]), "+r"(A[10]), "+r"(A[11]), "+r"(A[12]), "+r"(A[13]), "+r"(A[14]), "+r"(A[15]), "+r"(A[16])
      : "r"(T[0]), "r"(T[2]), "r"(T[4]), "r"(T[6]), "r"(T[8]), "r"(T[10]), "r"(T[12]), "r"(T[14]), "n"(K));
  asm("mad.lo.cc.u32 %0, %16, %24, %0;\n\t"
      "madc.hi.cc.u32 %1, %16, %24, %1;\n\t"
      "madc.lo.cc.u32 %2, %17, %24, %2;\n\t"
      "madc.hi.cc.u32 %3, %17, %24, %3;\n\t"
      "madc.lo.cc.u32 %4, %18, %24, %4;\n\t"
      "madc.hi.cc.u32 %5, %18, %24, %5;\n\t"
      "madc.lo.cc.u32 %6, %19, %24, %6;\n\t"
      "madc.hi.cc.u32 %7, %19, %24, %7;\n\t"
      "madc.lo.cc.u32 %8, %20, %24, %8;\n\t"
      "madc.hi.cc.u32 %9, %20, %24, %9;\n\t"
      "madc.lo.cc.u32 %10, %21, %24, %10;\n\t"
      "madc.hi.cc.u32 %11, %21, %24, %11;\n\t"
      "madc.lo.cc.u32 %12, %22, %24, %12;\n\t"
      "madc.hi.cc.u32 %13, %22, %24, %13;\n\t"
      "madc.lo.cc.u32 %14, %23, %24, %14;\n\t"
      "madc.hi.u32 %15, %23, %24, %15;"
      : "+r"(A[1]), "+r"(A[2]), "+r"(A[3]), "+r"(A[4]), "+r"(A[5]), "+r"(A[6]), "+r"(A[7]), "+r"(A[8]), "+r"(A[9]),
        "+r"(A[10]), "+r"(A[11]), "+r"(A[12]), "+r"(A[13]), "+r"(A[14]), "+r"(A[15]), "+r"(A[16])
      : "r"(T[1]), "r"(T[3]), "r"(T[5]), "r"(T[7]), "r"(T[9]), "r"(T[11]), "r"(T[13]), "r"(T[15]), "n"(K));
  SY_ACC_TOP(A);
}
// V = A * R^-1 mod p, not reduced: V = W + A_hi with W <= p (redc_low) and A_hi = floor(A / R).  9 limbs, the caller
// keeps A small enough for lin9_reduce (V < 2^262).
__device__ __forceinline__ void fp_redc_acc(uint32_t* V, const uint32_t* A) {
  Fp w = redc_low(A);
  asm("add.cc.u32 %0, %9, %17;\n\t"
      "addc.cc.u32 %1, %10, %18;\n\t"
      "addc.cc.u32 %2, %11, %19;\n\t"
      "addc.cc.u32 %3, %12, %20;\n\t"
      "addc.cc.u32 %4, %13, %21;\n\t"
      "addc.cc.u32 %5, %14, %22;\n\t"
      "addc.cc.u32 %6, %15, %23;\n\t"
      "addc.cc.u32 %7, %16, %24;\n\t"
      "addc.u32 %8, %25, 0;"
      : "=r"(V[0]), "=r"(V[1]), "=r"(V[2]), "=r"(V[3]), "=r"(V[4]), "=r"(V[5]), "=r"(V[6]), "=r"(V[7]), "=r"(V[8])
      : "r"(w.l[0]), "r"(w.l[1]), "r"(w.l[2]), "r"(w.l[3]), "r"(w.l[4]), "r"(w.l[5]), "r"(w.l[6]), "r"(w.l[7]),
        "r"(A[8]), "r"(A[9]), "r"(A[10]), "r"(A[11]), "r"(A[12]), "r"(A[13]), "r"(A[14]), "r"(A[15]), "r"(A[16]));
}
#else
// host simulation only: same contracts with 64-bit temporaries
inline void fp_sub_nr(uint32_t* r, const uint32_t* a, const uint32_t* b) {
  int64_t bw = 0;
  for (int i = 0; i < 8; i++) {
    int64_t d = (int64_t)a[i] - (int64_t)b[i] + bw;
    r[i] = (uint32_t)d;
    bw = d >> 32;
  }
}
inline void wide_dbl(uint32_t* a) {
  for (int i = 15; i > 0; i--) a[i] = (a[i] << 1) | (a[i - 1] >> 31);
  a[0] <<= 1;
}
inline void fp_mul_wide(uint32_t* T, const uint32_t* a, const uint32_t* b) {
  for (int i = 0; i < 16; i++) T[i] = 0;
  for (int i = 0; i < 8; i++) {
    uint64_t c = 0;
    for (int j = 0; j < 8; j++) {
      c += (uint64_t)a[j] * b[i] + T[i + j];
      T[i + j] = (uint32_t)c;
      c >>= 32;
    }
    T[i + 8] = (uint32_t)c;
  }
}
inline Fp fp_redc_wide(const uint32_t* T0) {
  uint32_t T[17];
  for (int i = 0; i < 16; i++) T[i] = T0[i];
  T[16] = 0;
  for (int i = 0; i < 8; i++) {
    uint32_t m = T[i] * SY_INV;
    uint64_t c = 0;
    for (int j = 0; j < 8; j++) {
      c += (uint64_t)m * kP_h[j] + T[i + j];
      T[i + j] = (uint32_t)c;
      c >>= 32;
    }
    for (int j = i + 8; j < 17 && c; j++) {
      c += T[j];
      T[j] = (uint32_t)c;
      c >>= 32;
    }
  }
  Fp r;
  for (int i = 0; i < 8; i++) r.l[i] = T[8 + i];
  fp_final_sub(r.l);
  return r;
}
inline uint32_t wide_sub(uint32_t* a, const uint32_t* b) {
  int64_t bw = 0;
  for (int i = 0; i < 16; i++) {
    int64_t d = (int64_t)a[i] - (int64_t)b[i] + bw;
    a[i] = (uint32_t)d;
    bw = d >> 32;
  }
  return (uint32_t)bw;
}
inline void wide_add_pR(uint32_t* a, uint32_t mask) {
  uint64_t c = 0;
  for (int i = 0; i < 8; i++) {
    c += (uint64_t)a[8 + i] + (mask & kP_h[i]);
    a[8 + i] = (uint32_t)c;
    c >>= 32;
  }
}
inline void fp_add_nr(uint32_t* r, const uint32_t* a, const uint32_t* b) {
  uint64_t c = 0;
  for (int i = 0; i < 8; i++) {
    c += (uint64_t)a[i] + b[i];
    r[i] = (uint32_t)c;
    c >>= 32;
  }
}
inline void acc_lift_sub(uint32_t* A, const uint32_t* Lp, const uint32_t* T) {
  int64_t bw = 0;
  for (int i = 0; i < 16; i++) {
    int64_t d = (int64_t)(i < 8 ? 0u : Lp[i - 8]) - (int64_t)T[i] + bw;
    A[i] = (uint32_t)d;
    bw = d >> 32;
  }
  A[16] = 0;
}
inline void acc_const_add(uint32_t* A, const uint32_t* C, const uint32_t* T) {
  uint64_t c = 0;
  for (int i = 0; i < 17; i++) {
    c += (uint64_t)C[i] + (i < 16 ? T[i] : 0u);
    A[i] = (uint32_t)c;
    c >>= 32;
  }
}
inline void acc_const_sub(uint32_t* A, const uint32_t* C, const uint32_t* T) {
  int64_t bw = 0;
  for (int i = 0; i < 17; i++) {
    int64_t d = (int64_t)C[i] - (int64_t)(i < 16 ? T[i] : 0u) + bw;
    A[i] = (uint32_t)d;
    bw = d >> 32;
  }
}
inline void acc_neg(uint32_t* A, const uint32_t* T) {
  int64_t bw = 0;
  for (int i = 0; i < 17; i++) {
    int64_t d = -(int64_t)T[i] + bw;
    A[i] = (uint32_t)d;
    bw = d >> 32;
  }
}
inline void acc_add(uint32_t* A, const uint32_t* T) {
  uint64_t c = 0;
  for (int i = 0; i < 17; i++) {
    c += (uint64_t)A[i] + (i < 16 ? T[i] : 0u);
    A[i] = (uint32_t)c;
    c >>= 32;
  }
}
inline void acc_sub(uint32_t* A, const uint32_t* T) {
  int64_t bw = 0;
  for (int i = 0; i < 17; i++) {
    int64_t d = (int64_t)A[i] - (int64_t)(i < 16 ? T[i] : 0u) + bw;
    A[i] = (uint32_t)d;
    bw = d >> 32;
  }
}
template <uint32_t K>
inline void acc_madd(uint32_t* A, const uint32_t* T) {
  uint64_t c = 0;
  for (int i = 0; i < 17; i++) {
    c += (uint64_t)A[i] + (i < 16 ? (uint64_t)K * T[i] : 0u);
    A[i] = (uint32_t)c;
    c >>= 32;
  }
}
inline void fp_redc_acc(uint32_t* V, const uint32_t* A) {
  uint32_t t[17] = {0};
  for (int i = 0; i < 8; i++) t[i] = A[i];
  for (int i = 0; i < 8; i++) {  // W = (A_lo + M p) / R, as the device's redc_low
    uint32_t m = t[i] * SY_INV;
    uint64_t c = 0;
    for (int j = 0; j < 8; j++) {
      c += (uint64_t)m * kP_h[j] + t[i + j];
      t[i + j] = (uint32_t)c;
      c >>= 32;
    }
    for (int j = i + 8; j < 17 && c; j++) {
      c += t[j];
      t[j] = (uint32_t)c;
      c >>= 32;
    }
  }
  uint64_t c = 0;
  for (int i = 0; i < 9; i++) {
    c += (uint64_t)(i < 8 ? t[8 + i] : 0u) + A[8 + i];
    V[i] = (uint32_t)c;
    c >>= 32;
  }
#if defined(SYLOW_HOSTSIM)
  if (t[16] != 0 || c != 0) {
    fprintf(stderr, "fp_redc_acc: W > p or V >= 2^288\n");
    abort();
  }
#endif
}
#endif

SY_DEFINE_TABLE(uint32_t, kP2, 8, 0xb0f9fa8eu, 0x7841182du, 0xd0e3951au, 0x2f02d522u, 0x0302b0bbu, 0x70a08b6du, 0xc2634053u, 0x60c89ce5u)  // 2p
SY_DEFINE_TABLE(uint32_t, kP4, 8, 0x61f3f51cu, 0xf082305bu, 0xa1c72a34u, 0x5e05aa45u, 0x06056176u, 0xe14116dau, 0x84c680a6u, 0xc19139cbu)  // 4p

// ---- 9 x + y + t mod p in one pass (the multiplications by xi = 9 + u, tower.cuh) --------------------------------
// x, y, t < p, so T = 9x + y + t < 11p needs 9 limbs.  lin9_reduce takes any 9-limb T < 2^262 (338 p; the wide
// accumulators of the cyclotomic squaring end there, fp_redc_acc).  The quotient is estimated from the top 32 bits,
// q = floor(floor(T / 2^230) * 338 / 2^32): 338 / 2^262 is below 1 / p (2^262 / p = 338.57), so q never exceeds T / p,
// and it falls short by less than 338.57 * (1 - 338 / 338.57) + 1 < 2.  T - q p in [0, 2p) is formed mod 2^256 as
// T + q (2^256 - p) with one multiplier row, then one conditional subtraction.
// 8 IMAD.WIDE + about 60 ALU instructions instead of the 120 of three doublings, two additions and their reductions.
#define SY_NP0 0x278302b9
#define SY_NP1 0xc3df73e9
#define SY_NP2 0x978e3572
#define SY_NP3 0x687e956e
#define SY_NP4 0x7e7ea7a2
#define SY_NP5 0x47afba49
#define SY_NP6 0x1ece5fd6
#define SY_NP7 0xcf9bb18d
SY_DEFINE_TABLE(uint32_t, kNegP, 8, SY_NP0, SY_NP1, SY_NP2, SY_NP3, SY_NP4, SY_NP5, SY_NP6, SY_NP7)

// T[0..8] += a[0..7]
SY_HD void lin9_acc(uint32_t* T, const uint32_t* a) {
#if defined(__CUDA_ARCH__)
  asm("add.cc.u32 %0, %0, %9;\n\t"
      "addc.cc.u32 %1, %1, %10;\n\t"
      "addc.cc.u32 %2, %2, %11;\n\t"
      "addc.cc.u32 %3, %3, %12;\n\t"
      "addc.cc.u32 %4, %4, %13;\n\t"
      "addc.cc.u32 %5, %5, %14;\n\t"
      "addc.cc.u32 %6, %6, %15;\n\t"
      "addc.cc.u32 %7, %7, %16;\n\t"
      "addc.u32 %8, %8, 0;"
      : "+r"(T[0]), "+r"(T[1]), "+r"(T[2]), "+r"(T[3]), "+r"(T[4]), "+r"(T[5]), "+r"(T[6]), "+r"(T[7]), "+r"(T[8])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]));
#else
  uint64_t c = 0;
  for (int i = 0; i < 8; i++) {
    c += (uint64_t)T[i] + a[i];
    T[i] = (uint32_t)c;
    c >>= 32;
  }
  T[8] += (uint32_t)c;
#endif
}
// T (9 limbs, < 2^262) -> canonical residue
SY_HD Fp lin9_reduce(const uint32_t* T) {
  uint32_t h = (T[8] << 26) | (T[7] >> 6);
  Fp r;
#if defined(__CUDA_ARCH__)
  uint32_t q = __umulhi(h, 338u);
  uint32_t e[8], o[8];
  asm("mad.lo.cc.u32 %0, %8, " SY_STR(SY_NP0) ", %9;\n\t"
      "madc.hi.cc.u32 %1, %8, " SY_STR(SY_NP0) ", %10;\n\t"
      "madc.lo.cc.u32 %2, %8, " SY_STR(SY_NP2) ", %11;\n\t"
      "madc.hi.cc.u32 %3, %8, " SY_STR(SY_NP2) ", %12;\n\t"
      "madc.lo.cc.u32 %4, %8, " SY_STR(SY_NP4) ", %13;\n\t"
      "madc.hi.cc.u32 %5, %8, " SY_STR(SY_NP4) ", %14;\n\t"
      "madc.lo.cc.u32 %6, %8, " SY_STR(SY_NP6) ", %15;\n\t"
      "madc.hi.u32 %7, %8, " SY_STR(SY_NP6) ", %16;"
      : "=r"(e[0]), "=r"(e[1]), "=r"(e[2]), "=r"(e[3]), "=r"(e[4]), "=r"(e[5]), "=r"(e[6]), "=r"(e[7])
      : "r"(q), "r"(T[0]), "r"(T[1]), "r"(T[2]), "r"(T[3]), "r"(T[4]), "r"(T[5]), "r"(T[6]), "r"(T[7]));
  asm("mul.lo.u32 %0, %7, " SY_STR(SY_NP1) "; mul.hi.u32 %1, %7, " SY_STR(SY_NP1) ";\n\t"
      "mul.lo.u32 %2, %7, " SY_STR(SY_NP3) "; mul.hi.u32 %3, %7, " SY_STR(SY_NP3) ";\n\t"
      "mul.lo.u32 %4, %7, " SY_STR(SY_NP5) "; mul.hi.u32 %5, %7, " SY_STR(SY_NP5) ";\n\t"
      "mul.lo.u32 %6, %7, " SY_STR(SY_NP7) ";"
      : "=r"(o[1]), "=r"(o[2]), "=r"(o[3]), "=r"(o[4]), "=r"(o[5]), "=r"(o[6]), "=r"(o[7])
      : "r"(q));
  r.l[0] = e[0];
  asm("add.cc.u32 %0, %7, %14;\n\t"
      "addc.cc.u32 %1, %8, %15;\n\t"
      "addc.cc.u32 %2, %9, %16;\n\t"
      "addc.cc.u32 %3, %10, %17;\n\t"
      "addc.cc.u32 %4, %11, %18;\n\t"
      "addc.cc.u32 %5, %12, %19;\n\t"
      "addc.u32 %6, %13, %20;"
      : "=r"(r.l[1]), "=r"(r.l[2]), "=r"(r.l[3]), "=r"(r.l[4]), "=r"(r.l[5]), "=r"(r.l[6]), "=r"(r.l[7])
      : "r"(e[1]), "r"(e[2]), "r"(e[3]), "r"(e[4]), "r"(e[5]), "r"(e[6]), "r"(e[7]), "r"(o[1]), "r"(o[2]), "r"(o[3]),
        "r"(o[4]), "r"(o[5]), "r"(o[6]), "r"(o[7]));
#else
#if defined(SYLOW_HOSTSIM)
  if (T[8] >> 6) {
    fprintf(stderr, "lin9_reduce: input >= 2^262\n");
    abort();
  }
#endif
  uint32_t q = (uint32_t)(((uint64_t)h * 338u) >> 32);
  uint64_t c = 0;
  for (int i = 0; i < 8; i++) {  // T + q (2^256 - p) mod 2^256
    c += (uint64_t)T[i] + (uint64_t)q * SY_TAB(kNegP)[i];
    r.l[i] = (uint32_t)c;
    c >>= 32;
  }
#if defined(SYLOW_HOSTSIM)
  {  // the estimate may be one short, never more: T - q p < 2p
    uint32_t chk[8];
    for (int i = 0; i < 8; i++) chk[i] = r.l[i];
    int64_t bw = 0;
    for (int i = 0; i < 8; i++) bw = ((int64_t)chk[i] - (int64_t)SY_TAB(kP2)[i] + bw) >> 32;
    if (bw == 0) {
      fprintf(stderr, "lin9_reduce: remainder >= 2p\n");
      abort();
    }
  }
#endif
#endif
  fp_final_sub(r.l);
  return r;
}
// 9 x + y  and  9 x + y + t   (all operands < p)
SY_HD void lin9_start(uint32_t* T, const Fp& x) {
#pragma unroll
  for (int i = 7; i > 0; i--) T[i] = (x.l[i] << 3) | (x.l[i - 1] >> 29);
  T[0] = x.l[0] << 3;
  T[8] = x.l[7] >> 29;
  lin9_acc(T, x.l);
}
SY_HD Fp fp_lin9(const Fp& x, const Fp& y) {
  uint32_t T[9];
  lin9_start(T, x);
  lin9_acc(T, y.l);
  return lin9_reduce(T);
}
SY_HD Fp fp_lin9(const Fp& x, const Fp& y, const Fp& t) {
  uint32_t T[9];
  lin9_start(T, x);
  lin9_acc(T, y.l);
  lin9_acc(T, t.l);
  return lin9_reduce(T);
}
SY_HD Fp fp_mul9(const Fp& x) {  // 3b = 9 of G1's complete formulas (curve.cuh)
  uint32_t T[9];
  lin9_start(T, x);
  return lin9_reduce(T);
}
// p - z without reduction: in (0, p] for z < p (p itself stands for 0 and is a valid fp_lin9 operand)
SY_HD Fp fp_neg_nr(const Fp& z) {
  Fp r, pp;
#pragma unroll
  for (int i = 0; i < 8; i++) pp.l[i] = SY_TAB(kP)[i];
  fp_sub_nr(r.l, pp.l, z.l);
  return r;
}

// ---- 9-limb combinations of fp_redc_acc outputs, finished by lin9_reduce ---------------------------------------------
// r = a + (b << s)   (9 limbs, s < 32 a compile-time constant; the caller guarantees no overflow)
SY_HD void u9_add_shl(uint32_t* r, const uint32_t* a, const uint32_t* b, int s) {
  uint32_t t[9];
#if defined(__CUDA_ARCH__)
#pragma unroll
  for (int i = 8; i > 0; i--) t[i] = s ? __funnelshift_l(b[i - 1], b[i], s) : b[i];
  t[0] = b[0] << s;
  asm("add.cc.u32 %0, %9, %18;\n\t"
      "addc.cc.u32 %1, %10, %19;\n\t"
      "addc.cc.u32 %2, %11, %20;\n\t"
      "addc.cc.u32 %3, %12, %21;\n\t"
      "addc.cc.u32 %4, %13, %22;\n\t"
      "addc.cc.u32 %5, %14, %23;\n\t"
      "addc.cc.u32 %6, %15, %24;\n\t"
      "addc.cc.u32 %7, %16, %25;\n\t"
      "addc.u32 %8, %17, %26;"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]), "r"(a[8]),
        "r"(t[0]), "r"(t[1]), "r"(t[2]), "r"(t[3]), "r"(t[4]), "r"(t[5]), "r"(t[6]), "r"(t[7]), "r"(t[8]));
#else
  for (int i = 8; i > 0; i--) t[i] = s ? (b[i] << s) | (b[i - 1] >> (32 - s)) : b[i];
  t[0] = b[0] << s;
  uint64_t c = 0;
  for (int i = 0; i < 9; i++) {
    c += (uint64_t)a[i] + t[i];
    r[i] = (uint32_t)c;
    c >>= 32;
  }
#endif
}
// r = a - b mod 2^288 (9 limbs; the caller's final sum, not each step, lies in [0, 2^262))
SY_HD void u9_sub(uint32_t* r, const uint32_t* a, const uint32_t* b) {
#if defined(__CUDA_ARCH__)
  asm("sub.cc.u32 %0, %9, %18;\n\t"
      "subc.cc.u32 %1, %10, %19;\n\t"
      "subc.cc.u32 %2, %11, %20;\n\t"
      "subc.cc.u32 %3, %12, %21;\n\t"
      "subc.cc.u32 %4, %13, %22;\n\t"
      "subc.cc.u32 %5, %14, %23;\n\t"
      "subc.cc.u32 %6, %15, %24;\n\t"
      "subc.cc.u32 %7, %16, %25;\n\t"
      "subc.u32 %8, %17, %26;"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]), "r"(a[8]),
        "r"(b[0]), "r"(b[1]), "r"(b[2]), "r"(b[3]), "r"(b[4]), "r"(b[5]), "r"(b[6]), "r"(b[7]), "r"(b[8]));
#else
  int64_t bw = 0;
  for (int i = 0; i < 9; i++) {
    int64_t d = (int64_t)a[i] - (int64_t)b[i] + bw;
    r[i] = (uint32_t)d;
    bw = d >> 32;
  }
#endif
}
// 3 V + y mod p for a 9-limb V and y < 2^256 (3 V + y < 2^262)
SY_HD Fp fp_lin3(const uint32_t* V, const Fp& y) {
  uint32_t T[9];
  u9_add_shl(T, V, V, 1);
  lin9_acc(T, y.l);
  return lin9_reduce(T);
}

SY_HD Fp fp_sqr(const Fp& a) { return fp_mul(a, a); }

SY_HD Fp fp_to_mont(const Fp& a) { return fp_mul(fp_R2(), a); }  // any a < 2^256 (reduces mod p)
SY_HD Fp fp_from_mont(const Fp& a) {
  Fp one = fp_zero();
  one.l[0] = 1;
  return fp_mul(a, one);
}

// small-constant helpers (additions only)
SY_HD Fp fp_mul3(const Fp& a) { return fp_add(fp_dbl(a), a); }

// a^e for a fixed 256-bit exponent given as 8 LE words (uniform across the warp); top_bit = index of its
// highest set bit.  Fixed 4-bit windows: 14 multiplications for the table, then 4 squarings and at most one
// multiplication per window (the digit is uniform, so skipping a zero digit does not diverge).
SY_HD_NOINLINE Fp fp_pow(const Fp& a, const uint32_t* e, int top_bit) {
  Fp tab[16];
  tab[1] = a;
  tab[2] = fp_sqr(a);
  for (int i = 3; i < 16; i++) tab[i] = fp_mul(tab[i - 1], a);
  int w = top_bit >> 2;
  Fp r = tab[(e[w >> 3] >> ((w & 7) * 4)) & 15u];
  for (w--; w >= 0; w--) {
    if ((w & 3) == 3) SY_LOOP_SYNC();
    r = fp_sqr(fp_sqr(fp_sqr(fp_sqr(r))));
    uint32_t d = (e[w >> 3] >> ((w & 7) * 4)) & 15u;
    if (d) r = fp_mul(r, tab[d]);
  }
  return r;
}

// p-2, (p-1)/2, (p+1)/4 as LE words
SY_DEFINE_TABLE(uint32_t, kPm2, 8, 0xd87cfd45, 0x3c208c16, 0x6871ca8d, 0x97816a91, 0x8181585d, 0xb85045b6, 0xe131a029, 0x30644e72)
SY_DEFINE_TABLE(uint32_t, kPm1h, 8, 0x6c3e7ea3, 0x9e10460b, 0xb438e546, 0xcbc0b548, 0x40c0ac2e, 0xdc2822db, 0x7098d014, 0x18322739)
SY_DEFINE_TABLE(uint32_t, kPp1q, 8, 0xb61f3f52, 0x4f082305, 0x5a1c72a3, 0x65e05aa4, 0xa0605617, 0x6e14116d, 0xb84c680a, 0x0c19139c)

// ---- inversion and the quadratic character by a branch-free binary GCD ----------------------------------------------
// Replaces the Fermat ladders x^(p-2) and x^((p-1)/2) (253 squarings + 75 products each, about 45 k IMAD.WIDE) by
// 510 add/shift steps on 256-bit integers (about 60 ALU instructions each, no multiplier work).  Every lane runs the
// same 510 steps; the data only feeds masks and selects.
// One step on (a, n), n odd:   a even: a <- a / 2;   a odd: (a, n) <- (|a - n| / 2, min(a, n)).
// bits(a) + bits(n) falls by at least one per step while a != 0, so 2 * 254 + 2 steps reach a = 0, n = gcd.
// r = a - b mod 2^256; returns 0xffffffff when the subtraction borrowed (a < b), else 0
SY_HD uint32_t u256_sub_b(uint32_t* r, const uint32_t* a, const uint32_t* b) {
  uint32_t borrow;
#if defined(__CUDA_ARCH__)
  asm("sub.cc.u32 %0, %9, %17;\n\t"
      "subc.cc.u32 %1, %10, %18;\n\t"
      "subc.cc.u32 %2, %11, %19;\n\t"
      "subc.cc.u32 %3, %12, %20;\n\t"
      "subc.cc.u32 %4, %13, %21;\n\t"
      "subc.cc.u32 %5, %14, %22;\n\t"
      "subc.cc.u32 %6, %15, %23;\n\t"
      "subc.cc.u32 %7, %16, %24;\n\t"
      "subc.u32 %8, 0, 0;"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(borrow)
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]), "r"(b[0]), "r"(b[1]),
        "r"(b[2]), "r"(b[3]), "r"(b[4]), "r"(b[5]), "r"(b[6]), "r"(b[7]));
#else
  int64_t bw = 0;
  for (int i = 0; i < 8; i++) {
    int64_t d = (int64_t)a[i] - (int64_t)b[i] + bw;
    r[i] = (uint32_t)d;
    bw = d >> 32;
  }
  borrow = (uint32_t)bw;
#endif
  return borrow;
}
// odd / sw are returned as masks: odd = a was odd, sw = a was odd and smaller than n (the pair was swapped)
SY_HD void bingcd_step(uint32_t* a, uint32_t* n, uint32_t& odd, uint32_t& sw) {
  uint32_t d[8], e[8];
  odd = 0u - (a[0] & 1u);
  uint32_t lt = u256_sub_b(d, a, n);  // d = a - n
  fp_sub_nr(e, n, a);                 // e = n - a
  sw = odd & lt;
#pragma unroll
  for (int i = 0; i < 8; i++) {
    uint32_t y = lt ? e[i] : d[i];
    d[i] = odd ? y : a[i];
    n[i] = sw ? a[i] : n[i];
  }
#pragma unroll
  for (int i = 0; i < 7; i++) a[i] = (d[i] >> 1) | (d[i + 1] << 31);
  a[7] = d[7] >> 1;
}
#define SY_GCD_STEPS 510  // 17 rounds of 30

// Jacobi symbol (v / p) in {1, 0, -1} for v < p.  Montgomery form may be passed as is: R = 2^256 is a square.
// Reciprocity when an odd pair is swapped (flip iff both are 3 mod 4) and (2 / n) for every halving (flip iff n is
// 3 or 5 mod 8).  Once a = 0 the halving rule keeps running on n = gcd, which is 1 (no flip) - or p = 7 mod 8 for v = 0.
SY_HD_NOINLINE int fp_jacobi(const Fp& v) {
  uint32_t a[8], n[8], t = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) {
    a[i] = v.l[i];
    n[i] = SY_TAB(kP)[i];
  }
#pragma unroll 1
  for (int it = 0; it < SY_GCD_STEPS; it++) {
    uint32_t a0 = a[0], n0 = n[0], odd, sw;
    bingcd_step(a, n, odd, sw);
    t ^= ((a0 & n0) >> 1) & sw;
    t ^= (n[0] >> 1) ^ (n[0] >> 2);
  }
  uint32_t rest = n[0] ^ 1u;
#pragma unroll
  for (int i = 1; i < 8; i++) rest |= n[i];
  return rest ? 0 : ((t & 1u) ? -1 : 1);
}

// Two Jacobi symbols in one loop: the 510 steps are a serial dependency chain (subtract, select, shift, repeat), so two
// independent inputs interleaved in the same iterations give the scheduler twice the work per stall.  SvdW tests g(x1)
// and g(x2) for squareness (svdw.rs:211-222), which do not depend on each other.
SY_HD_NOINLINE void fp_jacobi2(const Fp& v0, const Fp& v1, int& j0, int& j1) {
  uint32_t a[8], n[8], b[8], m[8], t = 0, u = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) {
    a[i] = v0.l[i];
    b[i] = v1.l[i];
    n[i] = m[i] = SY_TAB(kP)[i];
  }
#pragma unroll 1
  for (int it = 0; it < SY_GCD_STEPS; it++) {
    uint32_t a0 = a[0], n0 = n[0], b0 = b[0], m0 = m[0], odd, sw, odd2, sw2;
    bingcd_step(a, n, odd, sw);
    bingcd_step(b, m, odd2, sw2);
    t ^= ((a0 & n0) >> 1) & sw;
    t ^= (n[0] >> 1) ^ (n[0] >> 2);
    u ^= ((b0 & m0) >> 1) & sw2;
    u ^= (m[0] >> 1) ^ (m[0] >> 2);
  }
  uint32_t rest = n[0] ^ 1u, rest2 = m[0] ^ 1u;
#pragma unroll
  for (int i = 1; i < 8; i++) {
    rest |= n[i];
    rest2 |= m[i];
  }
  j0 = rest ? 0 : ((t & 1u) ? -1 : 1);
  j1 = rest2 ? 0 : ((u & 1u) ? -1 : 1);
}

// (f u + g v) / 2^32 mod p for u, v < p and signed f, g with |f| + |g| <= 2^30: negative factors act on p - u, the sum
// (< 2^30 p) takes one Montgomery step (< 1.25 p) and one conditional subtraction.
SY_HD void bingcd_lincomb(uint32_t* r, int32_t f, const uint32_t* u, int32_t g, const uint32_t* v) {
  uint32_t uu[8], vv[8], pp[8], T[9];
#pragma unroll
  for (int i = 0; i < 8; i++) pp[i] = SY_TAB(kP)[i];
  fp_sub_nr(uu, pp, u);
  fp_sub_nr(vv, pp, v);
  bool fn = f < 0, gn = g < 0;
  uint32_t fa = (uint32_t)(fn ? -f : f), ga = (uint32_t)(gn ? -g : g);
  uint64_t c = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) {
    c += (uint64_t)fa * (fn ? uu[i] : u[i]);
    uint64_t c2 = (uint64_t)ga * (gn ? vv[i] : v[i]);
    uint64_t s = (c & 0xffffffffu) + (c2 & 0xffffffffu);
    T[i] = (uint32_t)s;
    c = (c >> 32) + (c2 >> 32) + (s >> 32);
  }
  T[8] = (uint32_t)c;
  uint32_t m = T[0] * SY_INV;
  c = ((uint64_t)m * pp[0] + T[0]) >> 32;
#pragma unroll
  for (int i = 1; i < 8; i++) {
    c += (uint64_t)m * pp[i] + T[i];
    r[i - 1] = (uint32_t)c;
    c >>= 32;
  }
  r[7] = (uint32_t)(c + T[8]);
  fp_final_sub(r);
}

// 2^34 R^3 mod p: the 17 rounds leave v = y^-1 / 2^(17 (32 - 30)); the input is the Montgomery representative Y R, the
// output must be Y^-1 R = (Y R)^-1 R^2, so the last step is one Montgomery product of v with 2^34 R^3.
SY_HD Fp fp_gcd_fix() {
  return Fp{{0x13bd45e1u, 0x31d6a0d9u, 0x382c59a2u, 0x45fbf2bcu, 0x1ab31dfbu, 0x5b5fa369u, 0xb36fd339u, 0x24811383u}};
}
// Invariant: a = u y c, n = v y c (mod p) with y the input integer.  30 steps are tracked as a 2 x 2 integer matrix
// (entries below 2^30 in absolute value: row0 <- row0 - row1 when a is odd, row1 doubles every step, rows swap with
// the pair), then applied to (u, v) at once.  inv(0) = 0 like the reference (fp.rs:418-424): a starts at 0 and v stays 0.
SY_HD_NOINLINE Fp fp_inv(const Fp& y) {
  uint32_t a[8], n[8], u[8], v[8];
#pragma unroll
  for (int i = 0; i < 8; i++) {
    a[i] = y.l[i];
    n[i] = SY_TAB(kP)[i];
    u[i] = i == 0;
    v[i] = 0;
  }
#pragma unroll 1
  for (int round = 0; round < SY_GCD_STEPS / 30; round++) {
    int32_t f0 = 1, g0 = 0, f1 = 0, g1 = 1;
#pragma unroll 1
    for (int j = 0; j < 30; j++) {
      uint32_t odd, sw;
      bingcd_step(a, n, odd, sw);
      int32_t tf = (f0 ^ f1) & (int32_t)sw, tg = (g0 ^ g1) & (int32_t)sw;
      f0 ^= tf;
      f1 ^= tf;
      g0 ^= tg;
      g1 ^= tg;
      f0 -= f1 & (int32_t)odd;
      g0 -= g1 & (int32_t)odd;
      f1 <<= 1;
      g1 <<= 1;
    }
    uint32_t nu[8], nv[8];
    bingcd_lincomb(nu, f0, u, g0, v);
    bingcd_lincomb(nv, f1, u, g1, v);
#pragma unroll
    for (int i = 0; i < 8; i++) {
      u[i] = nu[i];
      v[i] = nv[i];
    }
  }
  Fp r;
#pragma unroll
  for (int i = 0; i < 8; i++) r.l[i] = v[i];
  return fp_mul(r, fp_gcd_fix());
}
// the Fermat ladder, kept as the cross-check of the tests (fp_op 7)
SY_HD Fp fp_inv_fermat(const Fp& a) { return fp_pow(a, SY_TAB(kPm2), 253); }

}  // namespace sylow

// Groth16 verification (sylow_b200.cu: sylow_b200_groth16_*): the per-thread bodies, shared by the device build and the
// host simulation (tests/hostsim/groth16.cu).
//   check:  e(A, B) e(-alpha, beta) e(-L, gamma) e(-C, delta) == 1,  L = IC_0 + sum_i x_i IC_i
//   batch:  prod_j check_j^{r_j} with 64-bit weights r_j: per proof one fused pair (r_j A_j, B_j); for the whole batch
//           (-s_0 alpha, beta), (-(s_0 IC_0 + sum_i s_i IC_i), gamma), (-sum_j r_j C_j, delta) with s_0 = sum_j r_j and
//           s_i = sum_j r_j x_ji in Fr.
#pragma once
#include "fr.cuh"
#include "wire.cuh"

namespace sylow {

// Device form of a prepared verifying key (SYLOW_B200_GROTH16_VK_DEV_BYTES, include/sylow_b200.h), all offsets 16-byte
// aligned:
//   [0, 3 T)                the beta, gamma, delta line tables in k_glued's device form (T = 87 x 192 bytes each)
//   [kG16NegAlpha, +64)     -alpha, canonical affine
//   [kG16Ic0, +64)          IC_0, canonical affine (directly behind -alpha: the batch's one-point ladders read both)
//   [kG16Tables, ...)       the fixed-base table of IC_i for i = 1 .. l, kG16IcTable bytes each (gen_scalar_mul's
//                           layout: SY_GEN_W x SY_GEN_E affine multiples in Montgomery form)
constexpr size_t kG16NegAlpha = 3 * (87 * 192), kG16Ic0 = kG16NegAlpha + 64, kG16Tables = kG16Ic0 + 64;
constexpr size_t kG16IcTable = (size_t)SY_GEN_W * SY_GEN_E * 64;
SY_HD constexpr size_t g16_vk_bytes(size_t l) { return kG16Tables + l * kG16IcTable; }

// x < r for a 32-byte little-endian integer (8 words).  Public inputs are NOT reduced: an input >= r fails the proof,
// as the snarkjs / Solidity verifiers reject it (a reduced alias would make the public input malleable).
SY_HD bool fr_words_canonical(const uint32_t* x) {
  int64_t bw = 0;  // borrow of x - r
  for (int i = 0; i < 8; i++) bw = ((int64_t)x[i] - (int64_t)SY_TAB(kFrMod)[i] + bw) >> 32;
  return bw != 0;
}

// L = IC_0 + sum_{i < l} x_i IC_{i+1} over the prepared key `vk`, x = the proof's l inputs (32 bytes each): ONE projective
// accumulator, started at IC_0, walks the l tables with gen_scalar_mul_add's signed digits - no per-input affine
// conversion.
// in_range = every x_i < r.  An input >= r is walked like any other (reduced), so a thread's work does not depend on it.
SY_HD_NOINLINE G1Proj groth16_public_term(const uint8_t* __restrict__ vk, size_t l, const uint8_t* __restrict__ x,
                                          bool& in_range) {
  G1Proj acc{fp_load(vk + kG16Ic0), fp_load(vk + kG16Ic0 + 32), fp_one()};
  bool ok = true;
  for (size_t i = 0; i < l; i++) {
    const Fp k = fp_load_raw(x + i * 32);
    ok &= fr_words_canonical(k.l);
    acc = gen_scalar_mul_add<Fp>(vk + kG16Tables + i * kG16IcTable, k.l, acc);
  }
  in_range = ok;
  return acc;
}

// The rest of proof j's check record [A, -alpha, -L, -C] (k_groth16_assemble; -L and its flag come from put_point):
// A, -alpha from the key and -C (p - y unless C is flagged) to rec, the flags [A, 0, -, C] to rec_inf, and the proof's
// B with its flag to b / b_inf.  proof_inf: the proof's three flags (A, B, C) or null.  16-byte aligned buffers.
SY_HD void groth16_record(const uint8_t* __restrict__ vk, const uint8_t* __restrict__ proof,
                          const uint8_t* __restrict__ proof_inf, uint8_t* __restrict__ rec, uint8_t* __restrict__ rec_inf,
                          uint8_t* __restrict__ b, uint8_t* __restrict__ b_inf) {
  const uint4* p = reinterpret_cast<const uint4*>(proof);
  const uint4* na = reinterpret_cast<const uint4*>(vk + kG16NegAlpha);
  uint4* r = reinterpret_cast<uint4*>(rec);
  uint4* q = reinterpret_cast<uint4*>(b);
  for (int k = 0; k < 4; k++) {
    r[k] = p[k];       // A
    r[4 + k] = na[k];  // -alpha
  }
  for (int k = 0; k < 8; k++) q[k] = p[4 + k];  // B
  const bool c_inf = proof_inf && proof_inf[2];
  Fp cy = fp_load_raw(proof + 224);
  if (!c_inf) cy = fp_neg(cy);  // p - y: negation is the same on canonical and Montgomery values
  r[12] = p[12];
  r[13] = p[13];
  fp_store_raw(rec + 224, cy);
  rec_inf[0] = proof_inf ? proof_inf[0] : 0;
  rec_inf[1] = 0;
  rec_inf[3] = c_inf;
  *b_inf = proof_inf ? proof_inf[1] : 0;
}

// One term of a weighted Fr sum: x r / R mod r (fr_mul of the plain integers x < r and r < 2^64, canonical).  Sums of such
// terms are sum x r / R; fr_unscale multiplies by R once at the end.
SY_HD Fr fr_weighted(const uint32_t* x, uint64_t r) {
  Fr a, b;
  for (int i = 0; i < 8; i++) {
    a.l[i] = x[i];
    b.l[i] = i == 0 ? (uint32_t)r : i == 1 ? (uint32_t)(r >> 32) : 0u;
  }
  return fr_mul(a, b);
}
// (sum x r / R) -> sum x r mod r, canonical words: a R^2 / R
SY_HD Fr fr_unscale(const Fr& a) {
  Fr r2;
  for (int i = 0; i < 8; i++) r2.l[i] = SY_TAB(kFrR2)[i];
  return fr_mul(a, r2);
}

}  // namespace sylow

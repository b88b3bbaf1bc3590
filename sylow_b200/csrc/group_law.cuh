// Pointwise group law (`&GroupProjective + / - &GroupProjective`, group.rs:528-624, then GroupAffine::from, :475-495)
// and the per-item steps of the EIP-196 ecAdd / ecMul precompile bodies (examples/reth_bn128.rs) with the big-endian
// codec they share with the ecPairing body.  Kept apart from the kernels so that the host simulation
// (tests/hostsim/group_law.cu) runs the same bodies.
#pragma once
#include "../../include/sylow_b200.h"
#include "wire.cuh"

namespace sylow {

// a[i] + b[i], or a[i] - b[i] when subtract != 0, for canonical affine points (x || y, 2 sizeof(F) bytes each) with
// optional infinity flags; projective, Montgomery form.  proj_add_mixed is complete for a = O, a = b and a = -b but
// ignores b.inf, so an infinite b selects a.  No data-dependent branches.
template <class F>
SY_HD Proj<F> add_pair(const uint8_t* a, const uint8_t* a_inf, const uint8_t* b, const uint8_t* b_inf, size_t i,
                       int subtract) {
  // the loads of affine_load written out: through the call, k_g1_add spills 16 more bytes (CUDA 12.9, sm_100a)
  constexpr size_t W = sizeof(F);
  Affine<F> pa{f_load<F>(a + i * 2 * W), f_load<F>(a + i * 2 * W + W), a_inf && a_inf[i]};
  Affine<F> pb{f_load<F>(b + i * 2 * W), f_load<F>(b + i * 2 * W + W), b_inf && b_inf[i]};
  pb.y = f_select(subtract && !pb.inf, f_neg(pb.y), pb.y);
  Proj<F> p = affine_to_proj(pa);
  Proj<F> s = proj_add_mixed(p, pb);
  s.x = f_select(pb.inf, p.x, s.x);
  s.y = f_select(pb.inf, p.y, s.y);
  s.z = f_select(pb.inf, p.z, s.z);
  return s;
}

// ---- big-endian codecs (SURVEY.md 8f-2) -------------------------------------------------------------
// 32 big-endian bytes -> Fp limbs (little-endian words), no reduction
SY_HD Fp fp_from_be32(const uint8_t* b, uint32_t top_mask) {
  Fp r;
#pragma unroll
  for (int i = 0; i < 8; i++) {
    const uint8_t* q = b + 28 - 4 * i;
    r.l[i] = ((uint32_t)q[0] << 24) | ((uint32_t)q[1] << 16) | ((uint32_t)q[2] << 8) | q[3];
  }
  r.l[7] &= top_mask;
  return r;
}
SY_HD void fp_to_be32(uint8_t* b, const Fp& v) {
#pragma unroll
  for (int i = 0; i < 8; i++) {
    uint8_t* q = b + 28 - 4 * i;
    q[0] = (uint8_t)(v.l[i] >> 24);
    q[1] = (uint8_t)(v.l[i] >> 16);
    q[2] = (uint8_t)(v.l[i] >> 8);
    q[3] = (uint8_t)v.l[i];
  }
}
SY_HD bool fp_raw_is_u32(const Fp& a, uint32_t v) {
  uint32_t o = a.l[0] ^ v;
#pragma unroll
  for (int i = 1; i < 8; i++) o |= a.l[i];
  return o == 0;
}
// One point of NF big-endian field elements (2 for G1, 4 for G2 with the imaginary parts first, g2.rs:325-328) at b
// -> little-endian wire form at out + infinity flag + decode status.
//   mode 0: sylow's codec (g1.rs:151-280, g2.rs:319-433): bit 7 of byte 0 flags infinity and must come
//           with x = 0, y = 1;   mode 1: EIP-196/197: the all-zero encoding is the point at infinity
//           (examples/reth_bn128.rs:118-126,187-194) and there is no flag bit.
// A point that fails to decode is written as (0, 1), off the curve, with no infinity flag.
template <int NF>
SY_HD void decode_be_item(const uint8_t* b, int mode, uint8_t* out, uint8_t* out_inf, int8_t* status) {
  bool flag = mode == 0 && (b[0] >> 7);
  Fp f[NF];
  bool canon = true, all_zero = true;
  for (int j = 0; j < NF; j++) {
    f[j] = fp_from_be32(b + 32 * j, (mode == 0 && j == 0) ? 0x7fffffffu : 0xffffffffu);
    canon &= fp_raw_is_canonical(f[j]);
    all_zero &= fp_raw_is_u32(f[j], 0);
  }
  // wire order: G1 (x, y); G2 (x.c0, x.c1, y.c0, y.c1) from (x.c1, x.c0, y.c1, y.c0)
  Fp w[NF];
  if (NF == 2) {
    w[0] = f[0];
    w[1] = f[1];
  } else {
    w[0] = f[1];
    w[1] = f[0];
    w[2] = f[3];
    w[3] = f[2];
  }
  bool x_zero = true, y_one = true;
  for (int j = 0; j < NF / 2; j++) x_zero &= fp_raw_is_u32(w[j], 0);
  for (int j = 0; j < NF / 2; j++) y_one &= fp_raw_is_u32(w[NF / 2 + j], j == 0 ? 1u : 0u);
  int8_t st = canon ? 0 : SYLOW_B200_ERR_DECODE;
  bool inf = false;
  if (mode == 0) {
    if (flag) {
      inf = true;
      if (st == 0 && !(x_zero && y_one)) st = SYLOW_B200_ERR_DECODE;
    }
  } else {
    inf = all_zero;
  }
  if (inf || st != 0) {  // GroupAffine::zero(): (0, 1, infinity)
    for (int j = 0; j < NF; j++) w[j] = fp_zero();
    w[NF / 2].l[0] = 1;
  }
  for (int j = 0; j < NF; j++) fp_store_raw(out + 32 * j, w[j]);
  *out_inf = inf ? 1 : 0;
  *status = st;
}

// The status of wire-form G1 point i (g1.rs:111-132): with keep_errors, a non-zero status[i] stays; an infinite point
// keeps its status; otherwise 0, SYLOW_B200_ERR_DECODE (a coordinate >= p) or SYLOW_B200_ERR_NOT_ON_CURVE.
SY_HD int8_t g1_validate_item(const uint8_t* g1, const uint8_t* inf, const int8_t* status, size_t i, int keep_errors) {
  Fp xr = fp_load_raw(g1 + i * 64), yr = fp_load_raw(g1 + i * 64 + 32);
  int8_t st = keep_errors ? status[i] : 0;
  if (st == 0 && !(inf && inf[i])) {
    if (!fp_raw_is_canonical(xr) || !fp_raw_is_canonical(yr))
      st = SYLOW_B200_ERR_DECODE;
    else if (!g1_on_curve(fp_to_mont(xr), fp_to_mont(yr)))
      st = SYLOW_B200_ERR_NOT_ON_CURVE;
  }
  return st;
}

// ecMul's scalar: 32 big-endian bytes -> the 32-byte little-endian integer g1_mul_batch reads (any 256-bit value)
SY_HD void eip196_scalar_item(const uint8_t* be, uint8_t* le) {
  for (int j = 0; j < 32; j++) le[j] = be[31 - j];
}

// The EIP-196 result of one input: status = st_a, or st_b when st_a is 0; out = the 64-byte big-endian affine point,
// all zero for the point at infinity and for a failed input (whose point is meaningless).
SY_HD void eip196_finish_item(const uint8_t* pt, bool inf, int8_t st_a, int8_t st_b, uint8_t* out, int8_t* status) {
  const int8_t st = st_a ? st_a : st_b;
  Fp x = fp_load_raw(pt), y = fp_load_raw(pt + 32);
  if (inf || st) {
    x = fp_zero();
    y = fp_zero();
  }
  fp_to_be32(out, x);
  fp_to_be32(out + 32, y);
  *status = st;
}

}  // namespace sylow

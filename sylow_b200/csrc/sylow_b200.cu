// libsylow_b200.so: kernels + C ABI (include/sylow_b200.h).  sm_100a only, no CPU fallback.
#include "../../include/sylow_b200.h"

#include <cuda_runtime.h>

#include <cstdio>
#include <cstdlib>
#include <thread>
#include <cstring>
#include <new>
#include <vector>

#include "hash.cuh"
#include "fr.cuh"
#include "wire.cuh"
#include "kernels_pairing.cuh"
#include "miller_tables.cuh"
#include "group_law.cuh"
#include "launch_plan.h"

using namespace sylow;

// ------------------------------------------------------------------------------------------------
// kernels.  One item (pair / point / message / check) per thread; control flow is uniform across
// a warp except for the infinity early-outs and the message-length loops of the hash.
// ------------------------------------------------------------------------------------------------
#define SY_MUL_THREADS 256
#define SY_G2_THREADS 256
#define SY_G2_MINB 2
#define SY_HASH_THREADS 256
#define SY_G1_MINB 2  // resident 256-thread blocks per SM for the Fp-only kernels (G1 ladder, hash-to-curve)
#define SY_SMALL_THREADS 128

struct DstPrime {
  uint8_t b[256];
  uint32_t len;
  int hash_id;  // 0 XMD Keccak-256, 1 XMD SHA-256, 2 XOF SHAKE128
};

// coeffs[i] = G2Affine::precompute(g2[i]): 87 triples (c0, c1, c2), 16704 B per point, Montgomery (raw) or canonical
__global__ void __launch_bounds__(SY_GLUED_THREADS, SY_GLUED_MINB)
k_g2_precompute(const uint8_t* __restrict__ g2, size_t n, uint8_t* __restrict__ coeffs, int raw_out) {
  size_t i0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t i = i0 < n ? i0 : n - 1;
  Ell c[87];
  g2_precompute(fp2_load(g2 + i * 128), fp2_load(g2 + i * 128 + 64), c);
  if (i0 >= n) return;
  uint8_t* o = coeffs + i * (87 * 192);
  for (int j = 0; j < 87; j++) {
    if (raw_out) {
      fp2_store_raw(o + 192 * j, c[j].c0);
      fp2_store_raw(o + 192 * j + 64, c[j].c1);
      fp2_store_raw(o + 192 * j + 128, c[j].c2);
    } else {
      fp2_store(o + 192 * j, c[j].c0);
      fp2_store(o + 192 * j + 64, c[j].c1);
      fp2_store(o + 192 * j + 128, c[j].c2);
    }
  }
}

// canonical <-> Montgomery for n Fp values (line-coefficient tables)
__global__ void k_fp_convert(const uint8_t* in, size_t n, uint8_t* out, int to_mont) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  if (to_mont)
    fp_store_raw(out + i * 32, fp_load(in + i * 32));
  else
    fp_store(out + i * 32, fp_load_raw(in + i * 32));
}

// Item i multiplies NV fused pairs (g1v[i*sv + v], g2v[i*NV + v]) and NF pairs against the fixed tables
// (g1f[i*sf + t], table t): f_out[i] = glued_miller_loop of those NV + NF pairs, Montgomery form.
// The NF tables (87 * 192 B each, Montgomery form) are staged once per block in shared memory; every
// thread of a warp then reads the same triple (broadcast, conflict-free).
template <int NV, int NF>
__global__ void __launch_bounds__(SY_GLUED_THREADS, SY_GLUED_MINB)
k_glued(const uint8_t* __restrict__ g1v, size_t sv, const uint8_t* __restrict__ g1v_inf, const uint8_t* __restrict__ g2v,
        const uint8_t* __restrict__ g2v_inf, const uint8_t* __restrict__ g1f, size_t sf,
        const uint8_t* __restrict__ g1f_inf, const uint8_t* __restrict__ tables, size_t n,
        uint8_t* __restrict__ f_out) {
  extern __shared__ uint4 sy_smem[];
  {
    const uint4* src = reinterpret_cast<const uint4*>(tables);
    for (int w = threadIdx.x; w < NF * 87 * 12; w += blockDim.x) sy_smem[w] = src[w];
    __syncthreads();
  }
  const Ell* tabs[NF > 0 ? NF : 1];
  for (int t = 0; t < NF; t++) tabs[t] = reinterpret_cast<const Ell*>(sy_smem) + 87 * t;
  size_t i0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t i = i0 < n ? i0 : n - 1;
  MillerG1 p[NV + NF];
  Fp2 qx[NV > 0 ? NV : 1], qy[NV > 0 ? NV : 1];
  for (int v = 0; v < NV; v++) {
    const uint8_t* a = g1v + (i * sv + v) * 64;
    const uint8_t* q = g2v + (i * NV + v) * 128;
    p[v].x = fp_load(a);
    p[v].y = fp_load(a + 32);
    p[v].skip = (g1v_inf && g1v_inf[i * sv + v]) || (g2v_inf && g2v_inf[i * NV + v]);
    qx[v] = fp2_load(q);
    qy[v] = fp2_load(q + 64);
  }
  for (int t = 0; t < NF; t++) {
    const uint8_t* a = g1f + (i * sf + t) * 64;
    p[NV + t].x = fp_load(a);
    p[NV + t].y = fp_load(a + 32);
    p[NV + t].skip = g1f_inf && g1f_inf[i * sf + t];
  }
  // the accumulator's shared-memory slot sits behind the NF tables (16-byte aligned: 87 * 192 is a multiple of 16)
  Fp12* acc = reinterpret_cast<Fp12*>(reinterpret_cast<char*>(sy_smem) + (size_t)NF * 87 * 192 +
                                      (size_t)threadIdx.x * SY_ACC_STRIDE);
  Fp12 f = glued_miller_loop<NV, NF>(p, qx, qy, tabs, acc);
  if (i0 >= n) return;
  fp12_store_raw(f_out + i * 384, f);
}

// f_out[i] = the glued Miller loop of pairs [i M, i M + M), each against its own table in global memory
// (miller_tables_item), Montgomery form if raw_out, else canonical.  The accumulator lives in the thread's shared-memory
// slot like k_miller's; every thread runs the loop (SY_LOOP_SYNC) and surplus threads redo the last item.
template <int M>
__global__ void __launch_bounds__(SY_GLUED_THREADS, SY_GLUED_MINB)
k_miller_tables(const uint8_t* __restrict__ tables, size_t n_tables, const uint32_t* __restrict__ table_idx,
                const uint8_t* __restrict__ g1, const uint8_t* __restrict__ g1_inf, size_t n_items,
                uint8_t* __restrict__ f_out, int raw_out) {
  size_t i0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t i = i0 < n_items ? i0 : n_items - 1;
  Fp12 f = miller_tables_item<M>(tables, n_tables, table_idx, g1, g1_inf, i, acc_slot());
  if (i0 >= n_items) return;
  if (raw_out)
    fp12_store_raw(f_out + i * 384, f);
  else
    fp12_store(f_out + i * 384, f);
}

// out[t] = in[t] * in[t + T] * in[t + 2T] * ...   (Montgomery form in and out)
__global__ void __launch_bounds__(SY_SMALL_THREADS)
k_fp12_product_strided(const uint8_t* in, size_t n, uint8_t* out, size_t T) {
  size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= T) return;
  Fp12 acc = fp12_one();
  bool first = true;
  for (size_t i = t; i < n; i += T) {
    Fp12 v = fp12_load_raw(in + i * 384);
    acc = first ? v : fp12_mul(acc, v);
    first = false;
  }
  fp12_store_raw(out + t * 384, acc);
}

// canonical <-> Montgomery for n Fp12 values
__global__ void k_fp12_convert(const uint8_t* in, size_t n, uint8_t* out, int to_mont) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  if (to_mont)
    fp12_store_raw(out + i * 384, fp12_load(in + i * 384));
  else
    fp12_store(out + i * 384, fp12_load_raw(in + i * 384));
}

// ok[c] = final_exp(prod_{j<k} f[c*k + j]) == 1
__global__ void __launch_bounds__(SY_FEXP_THREADS, SY_FEXP_MINB)
k_check_products(const uint8_t* f_raw, size_t k, size_t n_checks, uint8_t* ok) {
  size_t c0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t c = c0 < n_checks ? c0 : n_checks - 1;
  Fp12 acc = fp12_one();
  for (size_t j = 0; j < k; j++) {
    Fp12 v = fp12_load_raw(f_raw + (c * k + j) * 384);
    acc = j == 0 ? v : fp12_mul(acc, v);
  }
  final_exponentiation_assign(acc, acc_slot());
  bool one = fp12_eq(acc, fp12_one());
  if (c0 >= n_checks) return;
  ok[c] = one ? 1 : 0;
}

// The two halves of k_check_products as kernels of their own, around k_final_exp_lanes for small batches:
// out[c] = prod_{j<k} f[c*k + j] (Montgomery form), and ok[c] = (gt[c] == 1) on canonical values.
__global__ void k_group_products(const uint8_t* f_raw, size_t k, size_t n_checks, uint8_t* out_raw) {
  size_t c = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= n_checks) return;
  Fp12 acc = fp12_load_raw(f_raw + c * k * 384);
  for (size_t j = 1; j < k; j++) acc = fp12_mul(acc, fp12_load_raw(f_raw + (c * k + j) * 384));
  fp12_store_raw(out_raw + c * 384, acc);
}
__global__ void k_gt_is_one(const uint8_t* gt, size_t n, uint8_t* ok) {
  size_t c = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= n) return;
  const uint4* p = reinterpret_cast<const uint4*>(gt + c * 384);
  uint32_t d = 0;
  for (int i = 0; i < 24; i++) {
    uint4 v = p[i];
    d |= (i == 0 ? v.x ^ 1u : v.x) | v.y | v.z | v.w;
  }
  ok[c] = d == 0 ? 1 : 0;
}

// Projective (Montgomery form) -> affine wire format for a whole batch with Montgomery's trick: thread t owns the
// SY_AFF_K points t, t + T, t + 2T, ... (coalesced), multiplies their Z together, inverts ONCE and unwinds.  A point at
// infinity (Z = 0) enters the product as 1 and is written as (0, 1) + flag, like GroupAffine::from (group.rs:475-495).
// F = Fp: G1, 96-byte projective / 64-byte affine points; F = Fp2: G2, 192 / 128 bytes.
#define SY_AFF_K 8
template <class F>
__device__ __forceinline__ void batch_affine(const uint8_t* __restrict__ proj, size_t n, int negate,
                                             uint8_t* __restrict__ out, uint8_t* __restrict__ out_inf) {
  constexpr size_t W = sizeof(F);  // bytes per coordinate in both encodings
  F one;
  f_set_one(one);
  const size_t T = (n + SY_AFF_K - 1) / SY_AFF_K;
  size_t t0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t t = t0 < T ? t0 : T - 1;  // the inversion ladder is block-synchronised: every thread runs it
  F pre[SY_AFF_K];
  F acc = one;
  for (int j = 0; j < SY_AFF_K; j++) {
    size_t i = t + (size_t)j * T;
    F z = i < n ? f_load_raw<F>(proj + i * 3 * W + 2 * W) : one;
    z = f_select(f_is_zero(z), one, z);
    acc = f_mul(acc, z);
    pre[j] = acc;
  }
  F inv = f_inv(acc);
  for (int j = SY_AFF_K - 1; j >= 0; j--) {
    size_t i = t + (size_t)j * T;
    if (i >= n) continue;  // only the last stride can be short; its z entered the product as 1
    F z = f_load_raw<F>(proj + i * 3 * W + 2 * W);
    bool inf = f_is_zero(z);
    z = f_select(inf, one, z);
    F zi = j ? f_mul(inv, pre[j - 1]) : inv;
    inv = f_mul(inv, z);
    if (t0 >= T) continue;
    F x = f_mul(f_load_raw<F>(proj + i * 3 * W), zi), y = f_mul(f_load_raw<F>(proj + i * 3 * W + W), zi);
    if (inf) {
      f_set_zero(x);
      y = one;
    } else if (negate) {
      y = f_neg(y);
    }
    f_store(out + i * 2 * W, x);
    f_store(out + i * 2 * W + W, y);
    if (out_inf) out_inf[i] = inf;
  }
}
__global__ void __launch_bounds__(SY_MUL_THREADS, SY_G1_MINB)
k_g1_batch_affine(const uint8_t* __restrict__ proj, size_t n, int negate, uint8_t* __restrict__ out,
                  uint8_t* __restrict__ out_inf) {
  batch_affine<Fp>(proj, n, negate, out, out_inf);
}
__global__ void __launch_bounds__(SY_MUL_THREADS, 1)
k_g2_batch_affine(const uint8_t* __restrict__ proj, size_t n, uint8_t* __restrict__ out, uint8_t* __restrict__ out_inf) {
  batch_affine<Fp2>(proj, n, 0, out, out_inf);
}

// The result q of item i = min(i0, n - 1) of a point-batch kernel, from thread i0, to its output:
//  - every thread of the block calls it, surplus threads (i0 >= n) included: proj_to_affine's inversion ladder is
//    block-synchronised; surplus threads store nothing;
//  - with proj_out (large batches) the raw projective record for batch_affine, which shares one inversion between
//    SY_AFF_K points and applies the negation;
//  - otherwise the affine wire form and flag, y negated when negate is set and the point is finite.
template <class F>
__device__ __forceinline__ void put_point(const Proj<F>& q, size_t i0, size_t i, size_t n, int negate,
                                          uint8_t* __restrict__ out, uint8_t* __restrict__ out_inf,
                                          uint8_t* __restrict__ proj_out) {
  constexpr size_t W = sizeof(F);
  if (proj_out) {
    if (i0 < n) proj_store_raw(proj_out + i * 3 * W, q);
    return;
  }
  Affine<F> r = proj_to_affine(q);
  if (i0 >= n) return;
  if (negate && !r.inf) r.y = f_neg(r.y);
  f_store(out + i * 2 * W, r.x);
  f_store(out + i * 2 * W + W, r.y);
  if (out_inf) out_inf[i] = r.inf;
}

// the variable-base ladders: GLV on G1, GLS on G2
SY_HD G1Proj scalar_mul(const G1Proj& p, const uint32_t* k) { return proj_scalar_mul_glv(p, k); }
SY_HD G2Proj scalar_mul(const G2Proj& p, const uint32_t* k) { return g2_scalar_mul_gls(p, k); }

// out[i] = affine(scalars[i] * pts[i]) for any 256-bit scalar
template <class F>
__device__ __forceinline__ void mul_batch(const uint8_t* __restrict__ pts, const uint8_t* __restrict__ pts_inf,
                                          const uint8_t* __restrict__ scalars, size_t n, uint8_t* __restrict__ out,
                                          uint8_t* __restrict__ out_inf, uint8_t* __restrict__ proj_out) {
  size_t i0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t i = i0 < n ? i0 : n - 1;  // every thread runs the block-synchronised ladder
  Affine<F> a = affine_load<F>(pts, pts_inf, i);
  Fp k = fp_load_raw(scalars + i * 32);
  put_point(scalar_mul(affine_to_proj(a), k.l), i0, i, n, 0, out, out_inf, proj_out);
}
__global__ void __launch_bounds__(SY_MUL_THREADS, SY_G1_MINB)
k_g1_mul(const uint8_t* __restrict__ pts, const uint8_t* __restrict__ pts_inf, const uint8_t* __restrict__ scalars,
         size_t n, uint8_t* __restrict__ out, uint8_t* __restrict__ out_inf, uint8_t* __restrict__ proj_out) {
  mul_batch<Fp>(pts, pts_inf, scalars, n, out, out_inf, proj_out);
}
__global__ void __launch_bounds__(SY_G2_THREADS, SY_G2_MINB)
k_g2_mul(const uint8_t* __restrict__ pts, const uint8_t* __restrict__ pts_inf, const uint8_t* __restrict__ scalars,
         size_t n, uint8_t* __restrict__ out, uint8_t* __restrict__ out_inf, uint8_t* __restrict__ proj_out) {
  mul_batch<Fp2>(pts, pts_inf, scalars, n, out, out_inf, proj_out);
}

// proj_out[i] = r_i * pts[i] (projective, Montgomery form), r_i the weight of item first_index + i
__global__ void __launch_bounds__(SY_MUL_THREADS, SY_G1_MINB)
k_g1_mul_weight(const uint8_t* __restrict__ pts, const uint8_t* __restrict__ pts_inf, const __grid_constant__ WeightSeed seed,
                uint64_t first_index, size_t n, uint8_t* __restrict__ proj_out) {
  size_t i0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t i = i0 < n ? i0 : n - 1;
  G1Aff a = affine_load<Fp>(pts, pts_inf, i);
  G1Proj q = proj_scalar_mul_u64(affine_to_proj(a), batch_weight(seed, first_index + i));
  if (i0 < n) proj_store_raw(proj_out + i * 96, q);
}
// out[i] = the 64-bit weight of item first_index + i (tests)
__global__ void k_batch_weights(const __grid_constant__ WeightSeed seed, uint64_t first_index, size_t n, uint64_t* out) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = batch_weight(seed, first_index + i);
}

// out[i] = affine(scalars[i] * G) for the generator G of `table` (gen_scalar_mul; ensure_mul_table), any 256-bit scalar
template <class F>
__device__ __forceinline__ void mul_gen(const uint8_t* __restrict__ table, const uint8_t* __restrict__ scalars, size_t n,
                                        uint8_t* __restrict__ out, uint8_t* __restrict__ out_inf,
                                        uint8_t* __restrict__ proj_out) {
  size_t i0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t i = i0 < n ? i0 : n - 1;
  Fp k = fp_load_raw(scalars + i * 32);
  put_point(gen_scalar_mul<F>(table, k.l), i0, i, n, 0, out, out_inf, proj_out);
}
__global__ void __launch_bounds__(SY_MUL_THREADS, SY_G1_MINB)
k_g1_mul_gen(const uint8_t* __restrict__ table, const uint8_t* __restrict__ scalars, size_t n, uint8_t* __restrict__ out,
             uint8_t* __restrict__ out_inf, uint8_t* __restrict__ proj_out) {
  mul_gen<Fp>(table, scalars, n, out, out_inf, proj_out);
}
__global__ void __launch_bounds__(SY_G2_THREADS, SY_G2_MINB)
k_g2_mul_gen(const uint8_t* __restrict__ table, const uint8_t* __restrict__ scalars, size_t n, uint8_t* __restrict__ out,
             uint8_t* __restrict__ out_inf, uint8_t* __restrict__ proj_out) {
  mul_gen<Fp2>(table, scalars, n, out, out_inf, proj_out);
}

// out[i] = affine(a[i] + b[i]), or affine(a[i] - b[i]) when subtract != 0 (add_pair, group_law.cuh)
template <class F>
__device__ __forceinline__ void add_batch(const uint8_t* __restrict__ a, const uint8_t* __restrict__ a_inf,
                                          const uint8_t* __restrict__ b, const uint8_t* __restrict__ b_inf, size_t n,
                                          int subtract, uint8_t* __restrict__ out, uint8_t* __restrict__ out_inf,
                                          uint8_t* __restrict__ proj_out) {
  size_t i0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t i = i0 < n ? i0 : n - 1;
  put_point(add_pair<F>(a, a_inf, b, b_inf, i, subtract), i0, i, n, 0, out, out_inf, proj_out);
}
__global__ void __launch_bounds__(SY_MUL_THREADS, SY_G1_MINB)
k_g1_add(const uint8_t* __restrict__ a, const uint8_t* __restrict__ a_inf, const uint8_t* __restrict__ b,
         const uint8_t* __restrict__ b_inf, size_t n, int subtract, uint8_t* __restrict__ out,
         uint8_t* __restrict__ out_inf, uint8_t* __restrict__ proj_out) {
  add_batch<Fp>(a, a_inf, b, b_inf, n, subtract, out, out_inf, proj_out);
}
__global__ void __launch_bounds__(SY_G2_THREADS, SY_G2_MINB)
k_g2_add(const uint8_t* __restrict__ a, const uint8_t* __restrict__ a_inf, const uint8_t* __restrict__ b,
         const uint8_t* __restrict__ b_inf, size_t n, int subtract, uint8_t* __restrict__ out,
         uint8_t* __restrict__ out_inf, uint8_t* __restrict__ proj_out) {
  add_batch<Fp2>(a, a_inf, b, b_inf, n, subtract, out, out_inf, proj_out);
}

// out[i] = affine(+-hash_to_curve(msg_i)); *fail_flag = 1 if the SvdW sqrt check failed for any message
__global__ void __launch_bounds__(SY_HASH_THREADS, SY_G1_MINB)
k_hash_to_g1(const uint8_t* __restrict__ msgs, const uint64_t* __restrict__ offsets, size_t n,
             const __grid_constant__ DstPrime dst, int negate, uint8_t* __restrict__ out,
             uint8_t* __restrict__ out_inf, int* __restrict__ fail_flag, uint8_t* __restrict__ proj_out) {
  size_t i0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t i = i0 < n ? i0 : n - 1;
  uint64_t o0 = offsets[i], o1 = offsets[i + 1];
  G1Proj p;
  bool ok = hash_to_g1(msgs + o0, (size_t)(o1 - o0), dst.b, dst.len, p, dst.hash_id);
  put_point(p, i0, i, n, negate, out, out_inf, proj_out);
  if (i0 < n && !ok) atomicExch(fail_flag, 1);
}

// status[i]: 0 ok, SYLOW_B200_ERR_DECODE (a coordinate >= p), SYLOW_B200_ERR_NOT_ON_CURVE   (g1.rs:111-132)
__global__ void k_g1_validate(const uint8_t* __restrict__ g1, const uint8_t* __restrict__ inf, size_t n,
                              int8_t* __restrict__ status, int keep_errors) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  status[i] = g1_validate_item(g1, inf, status, i, keep_errors);
}

// + SYLOW_B200_ERR_NOT_IN_SUBGROUP: (x+1)Q + psi(xQ) + psi^2(xQ) != psi^3(2xQ)   (g2.rs:279-297, :460-525)
__global__ void __launch_bounds__(SY_MUL_THREADS, 1)
k_g2_validate(const uint8_t* __restrict__ g2, const uint8_t* __restrict__ inf, size_t n, int8_t* __restrict__ status,
              int keep_errors) {
  size_t i0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t i = i0 < n ? i0 : n - 1;
  Fp2 xr = fp2_load_raw(g2 + i * 128), yr = fp2_load_raw(g2 + i * 128 + 64);
  bool canon = fp_raw_is_canonical(xr.c0) & fp_raw_is_canonical(xr.c1) & fp_raw_is_canonical(yr.c0) &
               fp_raw_is_canonical(yr.c1);
  Fp2 x{fp_to_mont(xr.c0), fp_to_mont(xr.c1)}, y{fp_to_mont(yr.c0), fp_to_mont(yr.c1)};
  bool on = g2_on_curve(x, y);
  bool sub = g2_in_subgroup(x, y);  // every thread runs the (block-synchronised) ladder
  if (i0 >= n) return;
  int8_t st = keep_errors ? status[i] : 0;
  if (st == 0 && !(inf && inf[i])) {
    if (!canon)
      st = SYLOW_B200_ERR_DECODE;
    else if (!on)
      st = SYLOW_B200_ERR_NOT_ON_CURVE;
    else if (!sub)
      st = SYLOW_B200_ERR_NOT_IN_SUBGROUP;
  }
  status[i] = st;
}


// ---- big-endian codecs (group_law.cuh) --------------------------------------------------------------
template <int NF>
__global__ void k_decode_be(const uint8_t* __restrict__ be, size_t stride, size_t n, int mode, uint8_t* __restrict__ out,
                            uint8_t* __restrict__ out_inf, int8_t* __restrict__ status) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  decode_be_item<NF>(be + i * stride, mode, out + i * (32 * NF), out_inf + i, status + i);
}

// wire form -> big-endian (to_be_bytes / to_be_bytes_scrubbed, g1.rs:136-160, g2.rs:319-333)
template <int NF>
__global__ void k_encode_be(const uint8_t* __restrict__ pts, const uint8_t* __restrict__ inf, size_t n, int scrub,
                            uint8_t* __restrict__ be) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  bool is_inf = inf && inf[i];
  Fp w[NF];
  for (int j = 0; j < NF; j++) w[j] = fp_load_raw(pts + i * (32 * NF) + 32 * j);
  if (is_inf) {
    for (int j = 0; j < NF; j++) w[j] = fp_zero();
    if (!scrub) w[NF / 2].l[0] = 1;
  }
  uint8_t* b = be + i * (32 * NF);
  if (NF == 2) {
    fp_to_be32(b, w[0]);
    fp_to_be32(b + 32, w[1]);
  } else {
    fp_to_be32(b, w[1]);
    fp_to_be32(b + 32, w[0]);
    fp_to_be32(b + 64, w[3]);
    fp_to_be32(b + 96, w[2]);
  }
  if (is_inf && !scrub) b[0] |= 0x80;
}

// ecMul scalars: the 32 big-endian bytes at in + i * stride -> out[i], 32 bytes little-endian (k_g1_mul's form)
__global__ void k_eip196_scalars(const uint8_t* __restrict__ in, size_t stride, size_t n, uint8_t* __restrict__ out) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) eip196_scalar_item(in + i * stride, out + i * 32);
}
// EIP-196 results: the statuses of each input's one (st_b null) or two points folded, and the 64-byte big-endian
// point, all zero for infinity and for a failed input
__global__ void k_eip196_finish(const uint8_t* __restrict__ pts, const uint8_t* __restrict__ inf,
                                const int8_t* __restrict__ st_a, const int8_t* __restrict__ st_b, size_t n,
                                uint8_t* __restrict__ out, int8_t* __restrict__ status) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) eip196_finish_item(pts + i * 64, inf[i], st_a[i], st_b ? st_b[i] : 0, out + i * 64, status + i);
}

// per check: the first non-zero pair status wins and forces ok = 0
__global__ void k_fold_status(const int8_t* __restrict__ st_g1, const int8_t* __restrict__ st_g2, size_t k, size_t n_checks,
                              uint8_t* __restrict__ ok, int8_t* __restrict__ status) {
  size_t c = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= n_checks) return;
  int8_t st = 0;
  for (size_t j = 0; j < k && st == 0; j++) {
    st = st_g1[c * k + j];
    if (st == 0) st = st_g2[c * k + j];
  }
  if (st != 0) ok[c] = 0;
  status[c] = st;
}


// out[i] = gt[i]^scalars[i]   (`Gt * Fr`, gt.rs:188-215)
__global__ void __launch_bounds__(SY_FEXP_THREADS, SY_FEXP_MINB)
k_gt_pow(const uint8_t* __restrict__ gt, const uint8_t* __restrict__ scalars, size_t n, uint8_t* __restrict__ out) {
  size_t i0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t i = i0 < n ? i0 : n - 1;
  Fp12 g = fp12_load(gt + i * 384);
  Fp k = fp_load_raw(scalars + i * 32);
  Fp12 r = gt_pow(g, k.l);
  if (i0 >= n) return;
  fp12_store(out + i * 384, r);
}


// out[i] = expand_message_xmd(msg_i, DST, len_in_bytes)   (Expander::expand_message, hasher.rs:70,201-250)
__global__ void k_expand_message(const uint8_t* __restrict__ msgs, const uint64_t* __restrict__ offsets, size_t n,
                                 const __grid_constant__ DstPrime dst, uint32_t len_in_bytes, uint8_t* __restrict__ out) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint64_t o0 = offsets[i], o1 = offsets[i + 1];
  expand_message(dst.hash_id, msgs + o0, (size_t)(o1 - o0), dst.b, dst.len, len_in_bytes, out + i * len_in_bytes);
}
// out[i] = hash_to_field(msg_i, 2, 48): two canonical Fp (Expander::hash_to_field, hasher.rs:84-128)
__global__ void k_hash_to_field(const uint8_t* __restrict__ msgs, const uint64_t* __restrict__ offsets, size_t n,
                                const __grid_constant__ DstPrime dst, uint8_t* __restrict__ out) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint64_t o0 = offsets[i], o1 = offsets[i + 1];
  Fp u0, u1;
  hash_to_field_xmd(dst.hash_id, msgs + o0, (size_t)(o1 - o0), dst.b, dst.len, u0, u1);
  fp_store(out + i * 64, u0);
  fp_store(out + i * 64 + 32, u1);
}
// DST longer than 255 bytes: DST' = H("H2C-OVERSIZE-DST-" || DST)   (XMDExpander::new, hasher.rs:157-172)
__global__ void k_oversize_dst(const uint8_t* __restrict__ dst, size_t dst_len, int hash_id, uint8_t* __restrict__ out32) {
  if (blockIdx.x || threadIdx.x) return;
  const char prefix[] = "H2C-OVERSIZE-DST-";
  if (hash_id == 2) {  // XOFExpander::new (hasher.rs:274-281): ceil(2k / 8) = 32 output bytes for k = 128
    Shake128 h;
    shake_init(h);
    for (int i = 0; i < 17; i++) shake_absorb_byte(h, (uint8_t)prefix[i]);
    for (size_t i = 0; i < dst_len; i++) shake_absorb_byte(h, dst[i]);
    shake_squeeze(h, out32, 32);
  } else if (hash_id == 1) {
    Sha256 h;
    hash_init(h);
    for (int i = 0; i < 17; i++) hash_absorb_byte(h, (uint8_t)prefix[i]);
    for (size_t i = 0; i < dst_len; i++) hash_absorb_byte(h, dst[i]);
    hash_final(h, out32);
  } else {
    Keccak256H h;
    hash_init(h);
    for (int i = 0; i < 17; i++) hash_absorb_byte(h, (uint8_t)prefix[i]);
    for (size_t i = 0; i < dst_len; i++) hash_absorb_byte(h, dst[i]);
    hash_final(h, out32);
  }
}


// out[t] = sum of in[t], in[t + T], ...  as projective points in Montgomery form (96 B each).  affine_in = 1: the
// input is the affine wire format (64 B) with an optional infinity flag array.  Complete additions, so
// infinities and repeated points need no special cases.
__global__ void __launch_bounds__(SY_MUL_THREADS, SY_G1_MINB)
k_g1_sum_strided(const uint8_t* __restrict__ in, const uint8_t* __restrict__ in_inf, int affine_in, size_t n,
                 uint8_t* __restrict__ out, size_t T) {
  size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= T) return;
  G1Proj acc = proj_zero<Fp>();
  for (size_t i = t; i < n; i += T) {
    G1Proj v;
    if (affine_in)
      v = affine_to_proj(affine_load<Fp>(in, in_inf, i));
    else
      v = proj_load_raw<Fp>(in + i * 96);
    acc = proj_add(acc, v);
  }
  proj_store_raw(out + t * 96, acc);
}
// one projective point (Montgomery form) -> affine wire format + infinity flag, optionally negated
__global__ void k_g1_finish_sum(const uint8_t* __restrict__ in, int negate, uint8_t* __restrict__ out,
                                uint8_t* __restrict__ out_inf) {
  if (blockIdx.x || threadIdx.x) return;
  G1Aff r = proj_to_affine(proj_load_raw<Fp>(in));
  if (negate && !r.inf) r.y = fp_neg(r.y);
  fp_store(out, r.x);
  fp_store(out + 32, r.y);
  out_inf[0] = r.inf ? 1 : 0;
}

// ---- threshold-signature aggregation (SURVEY 8f-4; examples/dkg.rs:190-226, threshold_signing.rs:124-155) ----
// lambda[s][i] = prod_{j != i} x_j / (x_j - x_i) in Fr for the participant ids of set s, canonical 32-byte LE.
__global__ void k_lagrange(const uint64_t* __restrict__ ids, size_t n_sets, size_t t, uint8_t* __restrict__ out) {
  size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= n_sets * t) return;
  size_t s = g / t, i = g % t;
  Fr lam = fr_lagrange_at_zero(ids + s * t, t, i);
  uint32_t w[8];
  fr_to_words(w, lam);
  for (int k = 0; k < 8; k++) reinterpret_cast<uint32_t*>(out + g * 32)[k] = w[k];
}
// lambda[s][i] * sig[s][i] as a projective point in Montgomery form (96 B): no per-share inversion
__global__ void __launch_bounds__(SY_MUL_THREADS, SY_G1_MINB)
k_lagrange_mul(const uint64_t* __restrict__ ids, const uint8_t* __restrict__ sigs, const uint8_t* __restrict__ sigs_inf,
               size_t n_sets, size_t t, uint8_t* __restrict__ out) {
  size_t g0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t g = g0 < n_sets * t ? g0 : n_sets * t - 1;  // all threads run the block-synchronised ladder
  size_t s = g / t, i = g % t;
  Fr lam = fr_lagrange_at_zero(ids + s * t, t, i);
  uint32_t w[8];
  fr_to_words(w, lam);
  G1Aff a = affine_load<Fp>(sigs, sigs_inf, g);
  G1Proj r = proj_scalar_mul_glv(affine_to_proj(a), w);
  if (g0 != g) return;
  proj_store_raw(out + g * 96, r);
}
// One warp per set: sum of the set's t projective points, then affine wire format + infinity flag.
__global__ void __launch_bounds__(128) k_g1_segment_sum(const uint8_t* __restrict__ in, size_t n_sets, size_t t,
                                                         uint8_t* __restrict__ out, uint8_t* __restrict__ out_inf) {
  __shared__ G1Proj sh[128];
  size_t s0 = (size_t)blockIdx.x * 4 + (threadIdx.x >> 5);
  size_t s = s0 < n_sets ? s0 : n_sets - 1;
  unsigned lane = threadIdx.x & 31;
  G1Proj acc = proj_zero<Fp>();
  for (size_t i = lane; i < t; i += 32) acc = proj_add(acc, proj_load_raw<Fp>(in + (s * t + i) * 96));
  sh[threadIdx.x] = acc;
  __syncthreads();
  for (unsigned off = 16; off > 0; off >>= 1) {
    if (lane < off) acc = proj_add(sh[threadIdx.x], sh[threadIdx.x + off]);
    __syncthreads();
    if (lane < off) sh[threadIdx.x] = acc;
    __syncthreads();
  }
  G1Aff r = proj_to_affine(sh[threadIdx.x & ~31u]);  // every thread: the inversion ladder is block-synchronised
  if (lane == 0 && s0 < n_sets) {
    fp_store(out + s * 64, r.x);
    fp_store(out + s * 64 + 32, r.y);
    out_inf[s] = r.inf ? 1 : 0;
  }
}

SY_HD Fp fp_final_sub_copy(Fp a) {  // p -> 0, anything below p unchanged
  fp_final_sub(a.l);
  return a;
}
// ---- bucket (Pippenger) multi-scalar multiplication on G1 (SURVEY 8f-4) -----------------------------------------
// sum_i k_i P_i = sum_w 2^(c w) sum_d d * B[w][d], B[w][d] = sum of the points whose c-bit digit in window w is d.
//   k_msm_count / k_msm_offsets / k_msm_scatter : counting sort of the point indices by (window, digit)
//   k_msm_bucket_sum   : one thread per bucket adds its points (complete additions: repeated points and infinities
//                        need no special case)
//   k_msm_chunk_reduce : per window, 64 chunks of digits: local running sums S_j = sum (d - d0_j) B_d, T_j = sum B_d
//   k_msm_window_final : R_w = sum_j S_j + d0_j T_j (small double-and-add), then Horner over the windows
SY_HD uint32_t msm_digit(const uint8_t* scalar, int w, int c) {
  // c <= 16 bits starting at bit w * c of a 32-byte little-endian scalar
  int bit = w * c;
  uint64_t v = 0;
  for (int b = 0; b < 5; b++) {
    int byte = (bit >> 3) + b;
    if (byte < 32) v |= (uint64_t)scalar[byte] << (8 * b);
  }
  return (uint32_t)((v >> (bit & 7)) & ((1u << c) - 1u));
}
__global__ void k_msm_count(const uint8_t* __restrict__ scalars, const uint8_t* __restrict__ inf, size_t n, int c, int nw,
                            uint32_t* __restrict__ count) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n || (inf && inf[i])) return;
  for (int w = 0; w < nw; w++) {
    uint32_t d = msm_digit(scalars + i * 32, w, c);
    if (d) atomicAdd(&count[((size_t)w << c) + d], 1u);
  }
}
// Per window (one thread each): exclusive prefix sums of the bucket counts, and the work items of the bucket sums -
// a bucket of `count` points is cut into ceil(count / SY_MSM_ITEM) items so that no thread adds more than SY_MSM_ITEM
// points however skewed the digits are (the top window of 254-bit scalars has a handful of digits; equal scalars put
// everything into one bucket).  Items of window w live at [w * max_items, ...).
#define SY_MSM_ITEM 256
__global__ void k_msm_offsets(const uint32_t* __restrict__ count, int c, int nw, size_t max_items,
                              uint32_t* __restrict__ offset, uint32_t* __restrict__ cursor,
                              uint32_t* __restrict__ item_first, uint32_t* __restrict__ item_start,
                              uint32_t* __restrict__ item_len, uint32_t* __restrict__ items_in_window) {
  int w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= nw) return;
  uint32_t run = 0, items = 0;
  for (uint32_t d = 0; d < (1u << c); d++) {
    size_t k = ((size_t)w << c) + d;
    uint32_t cnt = count[k];
    offset[k] = run;
    cursor[k] = run;
    item_first[k] = items;
    for (uint32_t j = 0; j < cnt; j += SY_MSM_ITEM) {
      item_start[(size_t)w * max_items + items] = run + j;
      item_len[(size_t)w * max_items + items] = cnt - j < SY_MSM_ITEM ? cnt - j : SY_MSM_ITEM;
      items++;
    }
    run += cnt;
  }
  items_in_window[w] = items;
}
__global__ void k_msm_scatter(const uint8_t* __restrict__ scalars, const uint8_t* __restrict__ inf, size_t n, int c, int nw,
                              uint32_t* __restrict__ cursor, uint32_t* __restrict__ idx) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n || (inf && inf[i])) return;
  for (int w = 0; w < nw; w++) {
    uint32_t d = msm_digit(scalars + i * 32, w, c);
    if (d) {
      uint32_t pos = atomicAdd(&cursor[((size_t)w << c) + d], 1u);
      idx[(size_t)w * n + pos] = (uint32_t)i;
    }
  }
}
__global__ void __launch_bounds__(SY_MUL_THREADS, SY_G1_MINB)
k_msm_item_sum(const uint8_t* __restrict__ pts, size_t n, int nw, size_t max_items,
               const uint32_t* __restrict__ item_start, const uint32_t* __restrict__ item_len,
               const uint32_t* __restrict__ items_in_window, const uint32_t* __restrict__ idx,
               uint8_t* __restrict__ item_sum) {
  size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (size_t)nw * max_items) return;
  size_t w = t / max_items;
  if (t - w * max_items >= items_in_window[w]) return;
  G1Proj acc = proj_zero<Fp>();
  const uint32_t* list = idx + w * n + item_start[t];
  for (uint32_t j = 0; j < item_len[t]; j++) {
    const uint8_t* p = pts + (size_t)list[j] * 64;  // Montgomery form (converted once by k_fp_convert)
    acc = proj_add(acc, G1Proj{fp_load_raw(p), fp_load_raw(p + 32), fp_one()});
  }
  proj_store_raw(item_sum + t * 96, acc);
}
__global__ void __launch_bounds__(SY_MUL_THREADS, SY_G1_MINB)
k_msm_bucket_sum(int c, int nw, size_t max_items, const uint32_t* __restrict__ count,
                 const uint32_t* __restrict__ item_first, const uint8_t* __restrict__ item_sum,
                 uint8_t* __restrict__ buckets) {
  size_t b = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= ((size_t)nw << c)) return;
  size_t w = b >> c;
  uint32_t items = (count[b] + SY_MSM_ITEM - 1) / SY_MSM_ITEM;
  G1Proj acc = proj_zero<Fp>();
  for (uint32_t j = 0; j < items; j++)
    acc = proj_add(acc, proj_load_raw<Fp>(item_sum + (w * max_items + item_first[b] + j) * 96));
  proj_store_raw(buckets + b * 96, acc);
}
// small multiple m * P, m < 2^16, double-and-add from the top bit
SY_HD G1Proj g1_mul_small(const G1Proj& p, uint32_t m) {
  G1Proj acc = proj_zero<Fp>();
  for (int b = 15; b >= 0; b--) {
    acc = proj_double(acc);
    if ((m >> b) & 1u) acc = proj_add(acc, p);
  }
  return acc;
}
#define SY_MSM_CHUNKS 64
__global__ void __launch_bounds__(64) k_msm_chunk_reduce(const uint8_t* __restrict__ buckets, int c, int nw,
                                                          uint8_t* __restrict__ partial) {
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nw * SY_MSM_CHUNKS) return;
  int w = t / SY_MSM_CHUNKS, j = t % SY_MSM_CHUNKS;
  uint32_t per = ((1u << c) + SY_MSM_CHUNKS - 1) / SY_MSM_CHUNKS;
  uint32_t d0 = (uint32_t)j * per, d1 = d0 + per < (1u << c) ? d0 + per : (1u << c);
  // digits d0 + 1 .. d1 - 1 and d1 itself belong to the next chunk's base: use the half-open range (d0, d1] mapped
  // to local weights 1 .. d1 - d0; digit 0 never holds points, the top digit 2^c - 1 is < 2^c = last d1
  G1Proj run = proj_zero<Fp>(), sum = proj_zero<Fp>();
  for (uint32_t d = d1; d > d0; d--) {
    if (d < (1u << c)) run = proj_add(run, proj_load_raw<Fp>(buckets + (((size_t)w << c) + d) * 96));
    sum = proj_add(sum, run);
  }
  // sum = sum_{d in (d0, d1]} (d - d0) B_d, run = sum B_d; the window value needs d B_d = (d - d0) B_d + d0 B_d
  G1Proj r = proj_add(sum, g1_mul_small(run, d0));
  proj_store_raw(partial + (size_t)t * 96, r);
}
// R_w = sum of the 64 chunk values of window w (one thread per window), written over the window's first partial
__global__ void k_msm_window_sum(uint8_t* __restrict__ partial, int nw) {
  int w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= nw) return;
  G1Proj r = proj_zero<Fp>();
  for (int j = 0; j < SY_MSM_CHUNKS; j++)
    r = proj_add(r, proj_load_raw<Fp>(partial + ((size_t)w * SY_MSM_CHUNKS + j) * 96));
  proj_store_raw(partial + (size_t)w * SY_MSM_CHUNKS * 96, r);
}
// Horner over the windows: ((R_{nw-1} 2^c + R_{nw-2}) 2^c + ...) - 256 doublings, the only serial part
__global__ void k_msm_window_final(const uint8_t* __restrict__ partial, int c, int nw, uint8_t* __restrict__ out_proj) {
  if (blockIdx.x || threadIdx.x) return;
  G1Proj acc = proj_zero<Fp>();
  for (int w = nw - 1; w >= 0; w--) {
    for (int b = 0; b < c; b++) acc = proj_double(acc);
    acc = proj_add(acc, proj_load_raw<Fp>(partial + (size_t)w * SY_MSM_CHUNKS * 96));
  }
  proj_store_raw(out_proj, acc);
}

__global__ void k_fp_op(int op, const uint8_t* a, const uint8_t* b, size_t n, uint8_t* out) {
  size_t i0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t i = i0 < n ? i0 : n - 1;
  Fp x = fp_load(a + i * 32), y = fp_load(b + i * 32), r;
  switch (op) {
    case 0: r = fp_mul(x, y); break;
    case 1: r = fp_add(x, y); break;
    case 2: r = fp_sub(x, y); break;
    case 3: r = fp_inv(x); break;
    case 4: r = fp_halve(x); break;
    case 6: r = fp_inv_fermat(x); break;  // the Fermat ladder the binary-GCD inversion replaced (cross-check)
    case 7: {  // quadratic character: (x / p) + 1 in {0, 1, 2} from the Jacobi iteration, +4 if the Fermat form disagrees
      int j = fp_jacobi(x);
      Fp l = fp_pow(x, SY_TAB(kPm1h), 252);
      int e = fp_is_zero(l) ? 0 : fp_eq(l, fp_one()) ? 1 : -1;
      r = fp_zero();
      r.l[0] = (uint32_t)(j + 1) + (j != e ? 4u : 0u);
      if (i0 < n) fp_store_raw(out + i * 32, r);
      return;
    }
    case 8:  // raw limbs in and out: 9 a + b and 9 a + b + b mod p for operands <= p (fp_lin9)
    case 9: {
      Fp xr = fp_load_raw(a + i * 32), yr = fp_load_raw(b + i * 32);
      r = op == 8 ? fp_lin9(xr, yr) : fp_lin9(xr, yr, fp_final_sub_copy(yr));
      if (i0 < n) fp_store_raw(out + i * 32, r);
      return;
    }
    default: r = fp_neg(x);
  }
  if (i0 >= n) return;
  fp_store(out + i * 32, r);
}

__global__ void __launch_bounds__(SY_SMALL_THREADS)
k_fp12_op(int op, const uint8_t* a, const uint8_t* b, size_t n, uint8_t* out) {
  size_t i0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t i = i0 < n ? i0 : n - 1;
  Fp12 x = fp12_load(a + i * 384), y = fp12_load(b + i * 384), r;
  switch (op) {
    case 0: r = fp12_mul(x, y); break;
    case 1: r = fp12_sqr(x); break;
    case 2: r = fp12_inv(x); break;
    case 3: r = fp12_frobenius(x, 1); break;
    case 4: r = fp12_frobenius(x, 2); break;
    case 5: r = fp12_frobenius(x, 3); break;
    case 6: r = cyclotomic_squared(x); break;
    case 7: r = fp12_sparse_mul(x, y.c0.c0, y.c0.c1, y.c0.c2); break;
    // the tower's lower levels on their own (operands in the leading coefficients, the rest of the output is 0)
    case 8: r = Fp12{Fp6{fp2_mul(x.c0.c0, y.c0.c0), fp2_zero(), fp2_zero()}, fp6_zero()}; break;
    case 9: r = Fp12{Fp6{fp2_sqr(x.c0.c0), fp2_zero(), fp2_zero()}, fp6_zero()}; break;
    case 10: r = Fp12{fp6_mul(x.c0, y.c0), fp6_zero()}; break;
    case 11: r = Fp12{fp6_sqr(x.c0), fp6_zero()}; break;
    case 12: r = Fp12{Fp6{fp2_inv(x.c0.c0), fp2_zero(), fp2_zero()}, fp6_zero()}; break;
    case 13: r = Fp12{Fp6{fp2_mul_xi(x.c0.c0), fp2_mul_xi_add(x.c0.c0, y.c0.c0), fp2_sub_mul_xi(y.c0.c0, x.c0.c0)}, fp6_zero()}; break;
    case 14: r = Fp12{fp6_inv(x.c0), fp6_zero()}; break;
    case 15: r = Fp12{Fp6{fp2_mul_fp(x.c0.c0, y.c0.c0.c0), fp2_halve(x.c0.c0), fp2_conj(x.c0.c0)}, fp6_zero()}; break;
    default: r = fp12_one();
  }
  if (i0 >= n) return;
  fp12_store(out + i * 384, r);
}


// Register-resident Montgomery-multiplication throughput probe (the roofline denominator).
template <int CHAINS>
__global__ void k_imad_probe(int iters, const uint32_t* src, uint32_t* sink) {
  Fp x[CHAINS], y;
  for (int i = 0; i < 8; i++) y.l[i] = src[i];  // run-time multiplier: no constant folding
  for (int c = 0; c < CHAINS; c++) {
    x[c] = fp_one();
    x[c].l[0] += threadIdx.x + c;
  }
  for (int it = 0; it < iters; it++) {
#pragma unroll
    for (int c = 0; c < CHAINS; c++) x[c] = fp_mul(x[c], y);
  }
  uint32_t acc = 0;
  for (int c = 0; c < CHAINS; c++)
    for (int i = 0; i < 8; i++) acc ^= x[c].l[i];
  if (acc == 0x12345678u) sink[0] = acc;  // practically never true; keeps the loop alive
}

// Raw pipe probes.  MODE 0: independent mad.wide.u32 (IMAD.WIDE.U32); MODE 1: independent 32-bit
// mad.lo.u32 (IMAD); MODE 2: mad.lo.cc/madc.hi.cc carry chains of 4 pairs (IMAD.WIDE.U32.X with
// predicate carries, the exact instruction form fp_mul uses).  64 multiply-adds per loop iteration.
template <int MODE>
__global__ void k_pipe_probe(int iters, const uint32_t* src, uint32_t* sink) {
  uint32_t a = src[0] | 1u, b = src[1] | 3u;
  uint32_t r[16];
#pragma unroll
  for (int i = 0; i < 16; i++) r[i] = threadIdx.x + i;
  for (int it = 0; it < iters; it++) {
#pragma unroll
    for (int rep = 0; rep < (MODE == 1 ? 4 : 8); rep++) {
      if (MODE == 0) {
#pragma unroll
        for (int c = 0; c < 8; c++) {
          uint64_t acc = ((uint64_t)r[2 * c + 1] << 32) | r[2 * c];
          asm volatile("mad.wide.u32 %0, %1, %2, %0;" : "+l"(acc) : "r"(a), "r"(r[2 * c]));
          r[2 * c] = (uint32_t)acc;
          r[2 * c + 1] = (uint32_t)(acc >> 32);
        }
      } else if (MODE == 1) {
#pragma unroll
        for (int c = 0; c < 16; c++) asm volatile("mad.lo.u32 %0, %1, %2, %0;" : "+r"(r[c]) : "r"(a), "r"(b));
      } else {
#pragma unroll
        for (int c = 0; c < 2; c++) {
          uint32_t* q = r + 8 * c;
          asm volatile(
              "mad.lo.cc.u32 %0, %8, %9, %0;\n\t"
              "madc.hi.cc.u32 %1, %8, %9, %1;\n\t"
              "madc.lo.cc.u32 %2, %8, %9, %2;\n\t"
              "madc.hi.cc.u32 %3, %8, %9, %3;\n\t"
              "madc.lo.cc.u32 %4, %8, %9, %4;\n\t"
              "madc.hi.cc.u32 %5, %8, %9, %5;\n\t"
              "madc.lo.cc.u32 %6, %8, %9, %6;\n\t"
              "madc.hi.u32 %7, %8, %9, %7;"
              : "+r"(q[0]), "+r"(q[1]), "+r"(q[2]), "+r"(q[3]), "+r"(q[4]), "+r"(q[5]), "+r"(q[6]), "+r"(q[7])
              : "r"(a), "r"(b));
        }
      }
    }
  }
  uint32_t acc = 0;
#pragma unroll
  for (int i = 0; i < 16; i++) acc ^= r[i];
  if (acc == 0x12345678u) sink[0] = acc;
}

// FP64 FMA probe (16 independent chains, 64 DFMA per loop iteration): how fast the OTHER multiplier on the SM
// is.  Recorded for DESIGN.md section 7 (double-precision limb products as a possible second pipe).
__global__ void k_dfma_probe(int iters, const uint32_t* src, uint32_t* sink) {
  double a = 1.0 + (double)(src[0] & 1023) * 1e-9, b = 1e-7 + (double)(src[1] & 1023) * 1e-12;
  double r[16];
#pragma unroll
  for (int i = 0; i < 16; i++) r[i] = (double)(threadIdx.x + i);
  for (int it = 0; it < iters; it++) {
#pragma unroll
    for (int rep = 0; rep < 4; rep++) {
#pragma unroll
      for (int c = 0; c < 16; c++) asm volatile("fma.rn.f64 %0, %0, %1, %2;" : "+d"(r[c]) : "d"(a), "d"(b));
    }
  }
  double acc = 0;
#pragma unroll
  for (int i = 0; i < 16; i++) acc += r[i];
  if (acc == 0.12345) sink[0] = 1;
}

// ------------------------------------------------------------------------------------------------
// context
// ------------------------------------------------------------------------------------------------
// device memory of one context, freed with it (the context's device is current when its destructor runs)
struct DevBuf {
  uint8_t* p = nullptr;
  size_t cap = 0;
  DevBuf() = default;
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  ~DevBuf() {
    if (p) cudaFree(p);
  }
};

struct sylow_b200_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  cudaStream_t copy_in = nullptr, copy_out = nullptr;  // host<->device copies of the chunked host-pointer calls
  cudaStream_t stream2 = nullptr;                      // second compute stream: odd chunks (their tails overlap)
  cudaEvent_t ev_fork = nullptr;                       // copy_in -> compute stream hand-off of verify_batch_partial
  int sms = 148;
  int last_cuda = 0;
  uint64_t launches = 0;
  DevBuf stage[7];  // staging slots of the host-pointer calls (Staging); seven is the most one call takes
  DevBuf scratch0, scratch1, scratch2;
  int* d_fail = nullptr;
  uint8_t* d_gen_table = nullptr;  // G2PreComputed of the G2 generator, Montgomery form (16704 B)
  uint8_t* d_mul_table[2] = {};    // fixed-base tables of the G1 and G2 generators (ensure_mul_table)
  DevBuf tables, sum0, sum1, proj, msm;
  DevBuf check_stage[2];  // group products / Gt values of launch_check_products' two-lane path, per compute stream
  DevBuf fexp_lanes[2];  // FexpCold records of k_final_exp_lanes, one buffer per compute stream (stream, stream2)
  // multi-device parent (sylow_b200_create_multi): owns one single-device context per GPU and nothing else
  std::vector<sylow_b200_ctx*> children;

  // releases whatever was created, so it also undoes a partly finished sylow_b200_create (hidden: the library exports
  // its C ABI, not C++ members)
  __attribute__((visibility("hidden"))) ~sylow_b200_ctx() {
    for (sylow_b200_ctx* c : children) delete c;
    if (!children.empty()) return;
    cudaSetDevice(device);  // the DevBuf members are freed after this body, on the same device
    if (d_fail) cudaFree(d_fail);
    if (d_gen_table) cudaFree(d_gen_table);
    for (uint8_t* t : d_mul_table)
      if (t) cudaFree(t);
    for (cudaStream_t s : {stream, copy_in, copy_out, stream2})
      if (s) cudaStreamDestroy(s);
    if (ev_fork) cudaEventDestroy(ev_fork);
  }
};

static int fail_cuda(sylow_b200_ctx* ctx, cudaError_t e) {
  if (ctx) ctx->last_cuda = (int)e;
  return SYLOW_B200_ERR_CUDA;
}
#define CK(call)                                   \
  do {                                             \
    cudaError_t e__ = (call);                      \
    if (e__ != cudaSuccess) return fail_cuda(ctx, e__); \
  } while (0)
#define CKS(call)                  \
  do {                             \
    int s__ = (call);              \
    if (s__ != 0) return s__;      \
  } while (0)

#define ENTER(ctx)                                          \
  if (!(ctx)) return SYLOW_B200_ERR_ARG;                    \
  if (!(ctx)->children.empty()) (ctx) = (ctx)->children[0]; \
  CK(cudaSetDevice((ctx)->device));
// `_dev` entry points work on one device's memory: they need a single-device context (sylow_b200_device_ctx), and run
// on its device whatever device the calling thread has current
#define ENTER_DEV(ctx)                                                   \
  if (!(ctx) || !(ctx)->children.empty()) return SYLOW_B200_ERR_ARG; \
  CK(cudaSetDevice((ctx)->device));

static int reserve(sylow_b200_ctx* ctx, DevBuf& b, size_t bytes) {
  if (bytes <= b.cap) return 0;
  if (b.p) CK(cudaFree(b.p));
  b.p = nullptr;
  b.cap = 0;
  size_t cap = bytes + (bytes >> 3) + 256;
  cudaError_t e = cudaMalloc(&b.p, cap);
  if (e != cudaSuccess) {
    ctx->last_cuda = (int)e;
    return e == cudaErrorMemoryAllocation ? SYLOW_B200_ERR_NOMEM : SYLOW_B200_ERR_CUDA;
  }
  b.cap = cap;
  return 0;
}

// Staging of one host-pointer call: the context's staging slots, handed out in the order they are asked for, so two
// areas of one call never overlap (and no host form calls another while its staging is live).  `_dev` forms and the
// static helpers they call never touch the staging slots: that is what lets a host form's staged inputs survive the
// device form it calls.  A slot keeps the largest area ever asked of it, so calls ask for their large areas first.
// The first error sticks (later requests give null and queue nothing) and finish() returns it.  A call that returns
// without finishing waits for ctx->stream and ctx->copy_in in the destructor: whatever the status, no copy from or into
// caller memory runs on after a host entry point returns.
namespace {
struct Staging {
  sylow_b200_ctx* const ctx;
  int err = 0, used = 0;
  bool finished = false;
  explicit Staging(sylow_b200_ctx* c) : ctx(c) {}
  ~Staging() {
    if (finished) return;
    cudaStreamSynchronize(ctx->stream);
    cudaStreamSynchronize(ctx->copy_in);
  }
  // a device-only area for outputs and intermediates; null, and no slot, for 0 bytes; ERR_NOMEM past the last slot
  uint8_t* area(size_t bytes) {
    if (err || !bytes) return nullptr;
    err = used < (int)std::size(ctx->stage) ? reserve(ctx, ctx->stage[used], bytes) : SYLOW_B200_ERR_NOMEM;
    return err ? nullptr : ctx->stage[used++].p;
  }
  // a device copy of `bytes` of host memory at h, queued on ctx->stream; null for a null h or 0 bytes
  const uint8_t* up(const void* h, size_t bytes) {
    uint8_t* d = area(h ? bytes : 0);
    if (d) check(cudaMemcpyAsync(d, h, bytes, cudaMemcpyHostToDevice, ctx->stream));
    return err ? nullptr : d;
  }
  // queues the copy of `bytes` at device address d back to host memory at h
  void down(void* h, const void* d, size_t bytes) {
    if (!err) check(cudaMemcpyAsync(h, d, bytes, cudaMemcpyDeviceToHost, ctx->stream));
  }
  // waits for ctx->stream; the first error of the call, or 0
  int finish() {
    if (!err) check(cudaStreamSynchronize(ctx->stream));
    finished = !err;
    return err;
  }
  void check(cudaError_t e) {
    if (e != cudaSuccess) err = fail_cuda(ctx, e);
  }
};
}  // namespace

static constexpr size_t sy_gcd(size_t a, size_t b) { return b ? sy_gcd(b, a % b) : a; }
static constexpr size_t sy_lcm(size_t a, size_t b) { return a / sy_gcd(a, b) * b; }
static inline cudaStream_t pick(sylow_b200_ctx* ctx, void* stream) {
  return stream ? (cudaStream_t)stream : ctx->stream;
}
#define LAUNCHED(ctx)        \
  do {                       \
    (ctx)->launches++;       \
    CK(cudaGetLastError());  \
  } while (0)

static inline const uint8_t* adv(const uint8_t* p, size_t bytes) { return p ? p + bytes : nullptr; }
static inline uint8_t* adv(uint8_t* p, size_t bytes) { return p ? p + bytes : nullptr; }

// block shapes of the batch kernels (kernels_pairing.cuh), for the launch policy of launch_plan.h
static constexpr BlockShape kMillerShape{SY_MILLER_THREADS, SY_MILLER_MINB}, kFexpShape{SY_FEXP_THREADS, SY_FEXP_MINB},
    kLanesShape{SY_LANES_THREADS, SY_LANES_MINB}, kGluedShape{SY_GLUED_THREADS, SY_GLUED_MINB};

// SYLOW_B200_LANES: 0 never, 1 automatic (default), 2 always (measurement and the parity tests); see batch_plan.
static int lanes_mode() {  // read on every call (the tests flip it inside one process)
  const char* v = getenv("SYLOW_B200_LANES");
  return v ? atoi(v) : 1;
}
static int launch_miller(sylow_b200_ctx* ctx, const uint8_t* g1, const uint8_t* g1_inf, const uint8_t* g2,
                         const uint8_t* g2_inf, size_t n, uint8_t* f_out, int raw_out, cudaStream_t s) {
  for (const Segment& g : batch_plan(ctx->sms, n, kMillerShape, kLanesShape, lanes_mode())) {
    const size_t o = g.first;
    if (g.lanes)
      k_miller_lanes<<<g.blocks, g.threads, SY_LANES_SMEM_BYTES(g.threads), s>>>(
          g1 + o * 64, adv(g1_inf, o), g2 + o * 128, adv(g2_inf, o), g.count, f_out + o * 384, raw_out);
    else
      k_miller<<<g.blocks, g.threads, SY_MILLER_SMEM_BYTES(g.threads), s>>>(
          g1 + o * 64, adv(g1_inf, o), g2 + o * 128, adv(g2_inf, o), 1, g.count, f_out + o * 384, raw_out);
    LAUNCHED(ctx);
  }
  return 0;
}
// k_final_exp_lanes over the items of g; its FexpCold scratch is kept per compute stream
static int launch_final_exp_lanes(sylow_b200_ctx* ctx, const Segment& g, const uint8_t* f, int raw_in, uint8_t* gt_out,
                                  cudaStream_t s) {
  DevBuf& scratch = ctx->fexp_lanes[s == ctx->stream2 ? 1 : 0];
  CKS(reserve(ctx, scratch, SY_FLANES_SCRATCH_BYTES((size_t)g.blocks * (g.threads / 2))));
  k_final_exp_lanes<<<g.blocks, g.threads, SY_FLANES_SMEM_BYTES(g.threads), s>>>(f + g.first * 384, raw_in, g.count,
                                                                                 gt_out + g.first * 384, scratch.p);
  LAUNCHED(ctx);
  return 0;
}
static int launch_final_exp(sylow_b200_ctx* ctx, const uint8_t* f, int raw_in, size_t n, uint8_t* gt_out, cudaStream_t s) {
  for (const Segment& g : batch_plan(ctx->sms, n, kFexpShape, kLanesShape, lanes_mode())) {
    if (g.lanes) {
      CKS(launch_final_exp_lanes(ctx, g, f, raw_in, gt_out, s));
      continue;
    }
    k_final_exp<<<g.blocks, g.threads, SY_FEXP_SMEM_BYTES(g.threads), s>>>(f + g.first * 384, raw_in, g.count,
                                                                           gt_out + g.first * 384);
    LAUNCHED(ctx);
  }
  return 0;
}

// ok[c] = final_exp(prod_{j<k} f[c*k + j]) == 1 for the Montgomery-form Miller values at f (check_products_segment)
static int launch_check_products(sylow_b200_ctx* ctx, const uint8_t* f, size_t k, size_t n_checks, uint8_t* ok,
                                 cudaStream_t s) {
  const Segment g = check_products_segment(ctx->sms, n_checks, kFexpShape, kLanesShape, lanes_mode());
  if (g.lanes) {
    DevBuf& stage = ctx->check_stage[s == ctx->stream2 ? 1 : 0];
    CKS(reserve(ctx, stage, n_checks * 384));
    if (k > 1) {
      k_group_products<<<nblocks(n_checks, 32), 32, 0, s>>>(f, k, n_checks, stage.p);
      LAUNCHED(ctx);
    }
    CKS(launch_final_exp_lanes(ctx, g, k > 1 ? stage.p : f, 1, stage.p, s));
    k_gt_is_one<<<nblocks(n_checks, SY_SMALL_THREADS), SY_SMALL_THREADS, 0, s>>>(stage.p, n_checks, ok);
    LAUNCHED(ctx);
    return 0;
  }
  k_check_products<<<g.blocks, g.threads, SY_FEXP_SMEM_BYTES(g.threads), s>>>(f, k, n_checks, ok);
  LAUNCHED(ctx);
  return 0;
}

// The compiled glued-loop shapes k_glued<NV, NF>: NV fused pairs and NF pairs against fixed tables per item.
static const struct {
  size_t nv, nf;
  decltype(&k_glued<0, 1>) kernel;
} kGlued[] = {{2, 0, k_glued<2, 0>}, {4, 0, k_glued<4, 0>}, {1, 1, k_glued<1, 1>}, {0, 1, k_glued<0, 1>}, {1, 3, k_glued<1, 3>}};
// the NF tables, then the accumulators
static size_t glued_smem(size_t nf) { return nf * SY_TABLE_BYTES + SY_MILLER_SMEM_BYTES(SY_GLUED_THREADS); }
static bool glued_shape_ok(size_t nv, size_t nf) {
  for (const auto& v : kGlued)
    if (v.nv == nv && v.nf == nf) return true;
  return false;
}
// one glued loop of nv fused + nf table pairs per item; SYLOW_B200_ERR_ARG for a shape that is not compiled
static int launch_glued(sylow_b200_ctx* ctx, size_t nv, size_t nf, const uint8_t* g1v, size_t sv, const uint8_t* g1v_inf,
                        const uint8_t* g2v, const uint8_t* g2v_inf, const uint8_t* g1f, size_t sf, const uint8_t* g1f_inf,
                        const uint8_t* tables, size_t n, uint8_t* f_out, cudaStream_t s) {
  for (const auto& v : kGlued) {
    if (v.nv != nv || v.nf != nf) continue;
    v.kernel<<<nblocks(n, SY_GLUED_THREADS), SY_GLUED_THREADS, glued_smem(nf), s>>>(g1v, sv, g1v_inf, g2v, g2v_inf, g1f, sf,
                                                                                   g1f_inf, tables, n, f_out);
    LAUNCHED(ctx);
    return 0;
  }
  return SYLOW_B200_ERR_ARG;
}

// The compiled k_miller_tables<M>: M pairs per item, each against its own table.
static const struct {
  int m;
  decltype(&k_miller_tables<1>) kernel;
} kMillerTables[] = {{1, k_miller_tables<1>}, {2, k_miller_tables<2>}, {4, k_miller_tables<4>}};
// n_items items of m pairs each -> f_out, one Fp12 per item; SYLOW_B200_ERR_ARG for an m that is not compiled
static int launch_miller_tables(sylow_b200_ctx* ctx, int m, const uint8_t* tables, size_t n_tables, const uint32_t* idx,
                                const uint8_t* g1, const uint8_t* g1_inf, size_t n_items, uint8_t* f_out, int raw_out,
                                cudaStream_t s) {
  for (const auto& v : kMillerTables) {
    if (v.m != m) continue;
    v.kernel<<<nblocks(n_items, SY_GLUED_THREADS), SY_GLUED_THREADS, SY_MILLER_SMEM_BYTES(SY_GLUED_THREADS), s>>>(
        tables, n_tables, idx, g1, g1_inf, n_items, f_out, raw_out);
    LAUNCHED(ctx);
    return 0;
  }
  return SYLOW_B200_ERR_ARG;
}

// Batches from SY_AFF_MIN_BATCH points on leave their results in projective form (Montgomery form) in ctx->proj and
// convert them to affine coordinates afterwards, with one inversion per SY_AFF_K points (k_g1/g2_batch_affine); smaller
// ones convert each point in the kernel.
#define SY_AFF_MIN_BATCH 32768
// The pointwise additions (k_g1_add, k_g2_add) are short enough that below these sizes the launch of
// k_g*_batch_affine and its serial walk over SY_AFF_K points per thread cost more than an inversion in every
// thread; measured crossovers on a B200 (DESIGN.md section 4, item 26): G1 between 2^15 and 2^16 points, G2
// between 2^16 and 2^17.  The definitions can be overridden only to build the variants tools/group_law_time.py
// times on both sides of them.
#ifndef SY_G1_ADD_AFF_MIN_BATCH
#define SY_G1_ADD_AFF_MIN_BATCH 65536
#endif
#ifndef SY_G2_ADD_AFF_MIN_BATCH
#define SY_G2_ADD_AFF_MIN_BATCH 131072
#endif
// n points of G1 or G2 (g2) -> affine wire format + infinity flags at out / out_inf, G1 points negated when negate is
// set: launch(proj) enqueues the point kernel on s with proj_out = proj, which is ctx->proj from min_batch points on
// (followed by the batched conversion) and null below.
template <class Launch>
static int point_batch(sylow_b200_ctx* ctx, bool g2, size_t n, size_t min_batch, int negate, uint8_t* out,
                       uint8_t* out_inf, cudaStream_t s, Launch launch) {
  uint8_t* proj = nullptr;
  if (n >= min_batch) {
    CKS(reserve(ctx, ctx->proj, n * (g2 ? 192 : 96)));
    proj = ctx->proj.p;
  }
  launch(proj);
  LAUNCHED(ctx);
  if (!proj) return 0;
  const unsigned blocks = nblocks((n + SY_AFF_K - 1) / SY_AFF_K, SY_MUL_THREADS);
  if (g2)
    k_g2_batch_affine<<<blocks, SY_MUL_THREADS, 0, s>>>(proj, n, out, out_inf);
  else
    k_g1_batch_affine<<<blocks, SY_MUL_THREADS, 0, s>>>(proj, n, negate, out, out_inf);
  LAUNCHED(ctx);
  return 0;
}

extern "C" {

int sylow_b200_create(sylow_b200_ctx** out, int device_id) {
  if (!out) return SYLOW_B200_ERR_ARG;
  *out = nullptr;
  sylow_b200_ctx* ctx = new (std::nothrow) sylow_b200_ctx();
  if (!ctx) return SYLOW_B200_ERR_NOMEM;
  ctx->device = device_id;
  cudaError_t e = cudaSetDevice(device_id);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ctx->copy_in, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ctx->copy_out, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ctx->stream2, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaDeviceGetAttribute(&ctx->sms, cudaDevAttrMultiProcessorCount, device_id);
  // opt-ins for more than 48 KB of dynamic shared memory (the accumulators, the glued loops' tables); per device
  const struct {
    const void* kernel;
    size_t bytes;
  } smem[] = {{(const void*)k_miller, SY_MILLER_SMEM_BYTES(SY_MILLER_THREADS)},
              {(const void*)k_miller_lanes, SY_LANES_SMEM_BYTES(SY_LANES_THREADS)},
              {(const void*)k_final_exp_lanes, SY_FLANES_SMEM_BYTES(SY_LANES_THREADS)},
              {(const void*)k_final_exp, SY_FEXP_SMEM_BYTES(SY_FEXP_THREADS)},
              {(const void*)k_check_products, SY_FEXP_SMEM_BYTES(SY_FEXP_THREADS)}};
  const cudaFuncAttribute max_smem = cudaFuncAttributeMaxDynamicSharedMemorySize;
  for (const auto& k : smem)
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k.kernel, max_smem, (int)k.bytes);
  for (const auto& v : kMillerTables)
    if (e == cudaSuccess) e = cudaFuncSetAttribute(v.kernel, max_smem, (int)SY_MILLER_SMEM_BYTES(SY_GLUED_THREADS));
  for (const auto& v : kGlued)
    if (e == cudaSuccess) e = cudaFuncSetAttribute(v.kernel, max_smem, (int)glued_smem(v.nf));
  if (e == cudaSuccess) e = cudaMalloc(&ctx->d_fail, sizeof(int));
  if (e == cudaSuccess) e = cudaMemset(ctx->d_fail, 0, sizeof(int));
  if (e != cudaSuccess) {
    delete ctx;
    return SYLOW_B200_ERR_CUDA;
  }
  *out = ctx;
  return 0;
}

int sylow_b200_destroy(sylow_b200_ctx* ctx) {
  if (!ctx) return SYLOW_B200_ERR_ARG;
  delete ctx;
  return 0;
}

int sylow_b200_create_multi(sylow_b200_ctx** out, const int* device_ids, int n_devices) {
  if (!out) return SYLOW_B200_ERR_ARG;
  *out = nullptr;
  if (!device_ids || n_devices < 1) return SYLOW_B200_ERR_ARG;
  sylow_b200_ctx* parent = new (std::nothrow) sylow_b200_ctx();
  if (!parent) return SYLOW_B200_ERR_NOMEM;
  parent->device = device_ids[0];
  for (int i = 0; i < n_devices; i++) {
    sylow_b200_ctx* c = nullptr;
    int st = sylow_b200_create(&c, device_ids[i]);
    if (st == 0) {
      try {
        parent->children.push_back(c);
      } catch (...) {
        delete c;
        st = SYLOW_B200_ERR_NOMEM;
      }
    }
    if (st != 0) {
      delete parent;
      return st;
    }
  }
  *out = parent;
  return 0;
}
int sylow_b200_device_count(const sylow_b200_ctx* ctx) {
  if (!ctx) return 0;
  return ctx->children.empty() ? 1 : (int)ctx->children.size();
}
sylow_b200_ctx* sylow_b200_device_ctx(sylow_b200_ctx* ctx, int i) {
  if (!ctx || i < 0) return nullptr;
  if (ctx->children.empty()) return i == 0 ? ctx : nullptr;
  return i < (int)ctx->children.size() ? ctx->children[i] : nullptr;
}

const char* sylow_b200_strerror(int status) {
  switch (status) {
    case SYLOW_B200_OK: return "ok";
    case SYLOW_B200_ERR_ARG: return "invalid argument";
    case SYLOW_B200_ERR_CUDA: return "CUDA error";
    case SYLOW_B200_ERR_NOT_ON_CURVE: return "point not on curve";
    case SYLOW_B200_ERR_NOT_IN_SUBGROUP: return "point not in the r-torsion subgroup";
    case SYLOW_B200_ERR_CANNOT_HASH: return "cannot hash to group";
    case SYLOW_B200_ERR_DECODE: return "coordinate is not a canonical field element";
    case SYLOW_B200_ERR_NOMEM: return "out of memory";
    default: return "unknown status";
  }
}
int sylow_b200_last_cuda_error(const sylow_b200_ctx* ctx) {
  if (!ctx) return 0;
  for (const sylow_b200_ctx* c : ctx->children)
    if (c->last_cuda) return c->last_cuda;
  return ctx->last_cuda;
}
uint64_t sylow_b200_launch_count(const sylow_b200_ctx* ctx) {
  if (!ctx) return 0;
  uint64_t t = ctx->launches;
  for (const sylow_b200_ctx* c : ctx->children) t += c->launches;
  return t;
}

// ------------------------------------------------------------------------------- device variants
int sylow_b200_miller_loop_batch_dev(sylow_b200_ctx* ctx, const uint8_t* g1, const uint8_t* g1_inf, const uint8_t* g2,
                                     const uint8_t* g2_inf, size_t n, uint8_t* f_out, void* stream) {
  ENTER_DEV(ctx);
  if (n && (!g1 || !g2 || !f_out)) return SYLOW_B200_ERR_ARG;
  if (!n) return 0;
  return launch_miller(ctx, g1, g1_inf, g2, g2_inf, n, f_out, 0, pick(ctx, stream));
}

int sylow_b200_final_exp_batch_dev(sylow_b200_ctx* ctx, const uint8_t* f, size_t n, uint8_t* gt_out, void* stream) {
  ENTER_DEV(ctx);
  if (n && (!f || !gt_out)) return SYLOW_B200_ERR_ARG;
  if (!n) return 0;
  return launch_final_exp(ctx, f, 0, n, gt_out, pick(ctx, stream));
}

// Miller loops then final exponentiations of one batch on one stream.  The Miller values (Montgomery form) are staged
// in gt_out itself; the final exponentiation is in place.  (Slicing the batch over two streams was measured and only
// adds wave tails: a k_final_exp block needs a whole SM's registers and a k_miller block half of them, so the partly
// filled last wave of one kernel never usefully overlaps the other stream's kernels, profiles/r02_pair_chunk_sweep.jsonl.
// The low-occupancy tail launches of launch_miller / launch_final_exp handle the tails instead.)
static int pairing_dev_single(sylow_b200_ctx* ctx, const uint8_t* g1, const uint8_t* g1_inf, const uint8_t* g2,
                              const uint8_t* g2_inf, size_t n, uint8_t* gt_out, cudaStream_t s) {
  CKS(launch_miller(ctx, g1, g1_inf, g2, g2_inf, n, gt_out, 1, s));
  return launch_final_exp(ctx, gt_out, 1, n, gt_out, s);
}

int sylow_b200_pairing_batch_dev(sylow_b200_ctx* ctx, const uint8_t* g1, const uint8_t* g1_inf, const uint8_t* g2,
                                 const uint8_t* g2_inf, size_t n, uint8_t* gt_out, void* stream) {
  ENTER_DEV(ctx);
  if (n && (!g1 || !g2 || !gt_out)) return SYLOW_B200_ERR_ARG;
  if (!n) return 0;
  return pairing_dev_single(ctx, g1, g1_inf, g2, g2_inf, n, gt_out, pick(ctx, stream));
}

// reduce n Montgomery-form Fp12 values at `buf` (clobbered, with `tmp` as ping-pong space of at least
// ceil(n/4) values) to one value written to d_out in canonical (raw_out = 0) or Montgomery form.
static int product_reduce(sylow_b200_ctx* ctx, uint8_t* buf, uint8_t* tmp, size_t n, uint8_t* d_out, int raw_out,
                          cudaStream_t s) {
  uint8_t* cur = buf;
  uint8_t* nxt = tmp;
  while (n > 1) {
    size_t T = n / 4;
    if (T < 1) T = 1;
    if (T > 148 * 256) T = 148 * 256;
    k_fp12_product_strided<<<nblocks(T, SY_SMALL_THREADS), SY_SMALL_THREADS, 0, s>>>(cur, n, nxt, T);
    LAUNCHED(ctx);
    uint8_t* t = cur;
    cur = nxt;
    nxt = t;
    n = T;
  }
  if (raw_out) {
    CK(cudaMemcpyAsync(d_out, cur, 384, cudaMemcpyDeviceToDevice, s));
  } else {
    k_fp12_convert<<<1, 32, 0, s>>>(cur, 1, d_out, 0);
    LAUNCHED(ctx);
  }
  return 0;
}

static const uint8_t kOneCanonical[384] = {1};

int sylow_b200_miller_product_dev(sylow_b200_ctx* ctx, const uint8_t* g1, const uint8_t* g1_inf, const uint8_t* g2,
                                  const uint8_t* g2_inf, size_t n, uint8_t* f_out, void* stream) {
  ENTER_DEV(ctx);
  if (!f_out || (n && (!g1 || !g2))) return SYLOW_B200_ERR_ARG;
  cudaStream_t s = pick(ctx, stream);
  if (!n) {
    CK(cudaMemcpyAsync(f_out, kOneCanonical, 384, cudaMemcpyHostToDevice, s));
    return 0;
  }
  CKS(reserve(ctx, ctx->scratch0, n * 384));
  CKS(reserve(ctx, ctx->scratch1, (n / 4 + 1) * 384));
  CKS(launch_miller(ctx, g1, g1_inf, g2, g2_inf, n, ctx->scratch0.p, 1, s));
  return product_reduce(ctx, ctx->scratch0.p, ctx->scratch1.p, n, f_out, 0, s);
}

int sylow_b200_pairing_check_batch_dev(sylow_b200_ctx* ctx, const uint8_t* g1, const uint8_t* g1_inf,
                                       const uint8_t* g2, const uint8_t* g2_inf, size_t k, size_t n_checks,
                                       uint8_t* ok_out, void* stream) {
  ENTER_DEV(ctx);
  if (n_checks && !ok_out) return SYLOW_B200_ERR_ARG;
  if (!n_checks) return 0;
  size_t n = k * n_checks;
  if (n && (!g1 || !g2)) return SYLOW_B200_ERR_ARG;
  cudaStream_t s = pick(ctx, stream);
  if (!k) {  // the product of no pairs is the identity: every check holds, and there is nothing to compute
    CK(cudaMemsetAsync(ok_out, 1, n_checks, s));
    return 0;
  }
  CKS(reserve(ctx, ctx->scratch0, n * 384));
  size_t k_prod = k;  // Miller values per check left for k_check_products to multiply
  // 2- and 4-pair checks as ONE glued loop per check: one Fp12 squaring per digit for all pairs of the check, like
  // glued_miller_loop (pairing.rs:970-1022)
  if (glued_checks(ctx->sms, k, n_checks, kGluedShape)) {
    CKS(launch_glued(ctx, k, 0, g1, k, g1_inf, g2, g2_inf, nullptr, 0, nullptr, nullptr, n_checks, ctx->scratch0.p, s));
    k_prod = 1;
  } else {
    CKS(launch_miller(ctx, g1, g1_inf, g2, g2_inf, n, ctx->scratch0.p, 1, s));
  }
  return launch_check_products(ctx, ctx->scratch0.p, k_prod, n_checks, ok_out, s);
}

// out[i] = affine(scalars[i] * pts[i]) in G1 (g2 = 0) or G2
static int mul_dev(sylow_b200_ctx* ctx, int g2, const uint8_t* pts, const uint8_t* pts_inf, const uint8_t* scalars,
                   size_t n, uint8_t* out, uint8_t* out_inf, void* stream) {
  ENTER_DEV(ctx);
  if (n && (!pts || !scalars || !out)) return SYLOW_B200_ERR_ARG;
  if (!n) return 0;
  cudaStream_t s = pick(ctx, stream);
  return point_batch(ctx, g2, n, SY_AFF_MIN_BATCH, 0, out, out_inf, s, [&](uint8_t* proj) {
    if (g2)
      k_g2_mul<<<nblocks(n, SY_G2_THREADS), SY_G2_THREADS, 0, s>>>(pts, pts_inf, scalars, n, out, out_inf, proj);
    else
      k_g1_mul<<<nblocks(n, SY_MUL_THREADS), SY_MUL_THREADS, 0, s>>>(pts, pts_inf, scalars, n, out, out_inf, proj);
  });
}
int sylow_b200_g1_mul_batch_dev(sylow_b200_ctx* ctx, const uint8_t* pts, const uint8_t* pts_inf,
                                const uint8_t* scalars, size_t n, uint8_t* out, uint8_t* out_inf, void* stream) {
  return mul_dev(ctx, 0, pts, pts_inf, scalars, n, out, out_inf, stream);
}
int sylow_b200_g2_mul_batch_dev(sylow_b200_ctx* ctx, const uint8_t* pts, const uint8_t* pts_inf,
                                const uint8_t* scalars, size_t n, uint8_t* out, uint8_t* out_inf, void* stream) {
  return mul_dev(ctx, 1, pts, pts_inf, scalars, n, out, out_inf, stream);
}

static int make_dst_prime(sylow_b200_ctx* ctx, const uint8_t* dst, size_t dst_len, int hash_id, DstPrime& dp) {
  if (hash_id != SYLOW_B200_HASH_KECCAK256 && hash_id != SYLOW_B200_HASH_SHA256 && hash_id != SYLOW_B200_HASH_SHAKE128)
    return SYLOW_B200_ERR_ARG;
  if (dst_len && !dst) return SYLOW_B200_ERR_ARG;
  memset(dp.b, 0, sizeof(dp.b));
  dp.hash_id = hash_id;
  if (dst_len > 255) {
    // oversize DST (hasher.rs:158-163): hashed on the device, like every other digest of this library
    if (!ctx) return SYLOW_B200_ERR_ARG;
    uint8_t* d_tmp = nullptr;
    CK(cudaMalloc(&d_tmp, dst_len + 32));
    cudaError_t e = cudaMemcpyAsync(d_tmp + 32, dst, dst_len, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) {
      k_oversize_dst<<<1, 32, 0, ctx->stream>>>(d_tmp + 32, dst_len, hash_id, d_tmp);
      ctx->launches++;
      e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(dp.b, d_tmp, 32, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    cudaFree(d_tmp);
    if (e != cudaSuccess) return fail_cuda(ctx, e);
    dst_len = 32;
  } else if (dst_len) {
    memcpy(dp.b, dst, dst_len);
  }
  dp.b[dst_len] = (uint8_t)dst_len;  // DST' || I2OSP(len(DST'), 1)   (hasher.rs:205-209)
  dp.len = (uint32_t)dst_len + 1;
  return 0;
}

static int hash_launch(sylow_b200_ctx* ctx, const uint8_t* d_msgs, const uint64_t* d_offsets, size_t n,
                       const DstPrime& dp, int negate, uint8_t* d_out, uint8_t* d_out_inf, cudaStream_t s) {
  CK(cudaMemsetAsync(ctx->d_fail, 0, sizeof(int), s));  // the flag reports THIS call's hashes only
  return point_batch(ctx, false, n, SY_AFF_MIN_BATCH, negate, d_out, d_out_inf, s, [&](uint8_t* proj) {
    k_hash_to_g1<<<nblocks(n, SY_HASH_THREADS), SY_HASH_THREADS, 0, s>>>(d_msgs, d_offsets, n, dp, negate, d_out,
                                                                       d_out_inf, ctx->d_fail, proj);
  });
}

int sylow_b200_hash_to_g1_batch_dev(sylow_b200_ctx* ctx, const uint8_t* d_msgs, const uint64_t* d_offsets, size_t n,
                                    const uint8_t* dst, size_t dst_len, int hash_id, uint8_t* d_out,
                                    uint8_t* d_out_inf, void* stream) {
  ENTER_DEV(ctx);
  if (n && (!d_offsets || !d_out)) return SYLOW_B200_ERR_ARG;
  DstPrime dp;
  CKS(make_dst_prime(ctx, dst, dst_len, hash_id, dp));
  if (!n) return 0;
  return hash_launch(ctx, d_msgs, d_offsets, n, dp, 0, d_out, d_out_inf, pick(ctx, stream));
}

// G2 generator in wire form, uploaded once per context on first use
static const uint64_t kG2GenWords[16] = {
    // x.c0, x.c1, y.c0, y.c1 as 4 LE u64 words each (g2.rs:47-77)
    5106727233969649389ull,  7440829307424791261ull,  4785637993704342649ull,  1729627375292849782ull,
    10945020018377822914ull, 17413811393473931026ull, 8241798111626485029ull,  1841571559660931130ull,
    5541340697920699818ull,  16416156555105522555ull, 5380518976772849807ull,  1353435754470862315ull,
    6173549831154472795ull,  13567992399387660019ull, 17050234209342075797ull, 650358724130500725ull};

// G2PreComputed of the generator, computed on the device once per context
static int ensure_gen_table(sylow_b200_ctx* ctx, cudaStream_t s) {
  if (ctx->d_gen_table) return 0;
  // the field is set only after the table has been computed: a failure on the way leaves it null (and frees both
  // buffers), so the next call builds it again instead of using an uninitialised table
  uint8_t *d_gen = nullptr, *d_tab = nullptr;
  cudaError_t e = cudaMalloc(&d_gen, 128);
  if (e == cudaSuccess) e = cudaMalloc(&d_tab, SY_TABLE_BYTES);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_gen, kG2GenWords, 128, cudaMemcpyHostToDevice, s);
  if (e == cudaSuccess) {
    k_g2_precompute<<<1, 32, 0, s>>>(d_gen, 1, d_tab, 1);
    ctx->launches++;
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) e = cudaStreamSynchronize(s);
  if (d_gen) cudaFree(d_gen);
  if (e != cudaSuccess) {
    if (d_tab) cudaFree(d_tab);
    return fail_cuda(ctx, e);
  }
  ctx->d_gen_table = d_tab;
  return 0;
}

// Fixed-base table of the G1 (g2 = 0) or G2 generator for gen_scalar_mul (curve.cuh), built on the device once per
// context: the ladder of mul_dev multiplies the generator by (j + 1) 2^(C w) mod r, and k_fp_convert takes
// the affine results to Montgomery form, so every entry is the ladder's own point.  The field is set only after the
// build has finished, like ensure_gen_table's.
static int ensure_mul_table(sylow_b200_ctx* ctx, int g2, cudaStream_t s) {
  if (ctx->d_mul_table[g2]) return 0;
  const size_t n = (size_t)SY_GEN_W * SY_GEN_E, pb = g2 ? 128 : 64, in_bytes = n * (32 + pb);
  std::vector<uint8_t> in(in_bytes);  // n scalars, then the generator n times
  Fr step{{1}};                       // 2^(C w) mod r
  for (int w = 0; w < SY_GEN_W; w++) {
    Fr m = step;
    for (int j = 0; j < SY_GEN_E; j++, m = fr_add(m, step)) memcpy(&in[((size_t)w * SY_GEN_E + j) * 32], m.l, 32);
    for (int b = 0; b < SY_GEN_C; b++) step = fr_add(step, step);
  }
  static const uint64_t kG1GenWords[8] = {1, 0, 0, 0, 2, 0, 0, 0};  // (1, 2)
  for (size_t i = 0; i < n; i++) memcpy(&in[n * 32 + i * pb], g2 ? (const void*)kG2GenWords : kG1GenWords, pb);
  uint8_t *d_in = nullptr, *d_tab = nullptr;
  cudaError_t e = cudaMalloc(&d_in, in_bytes + n * pb);  // inputs, then the canonical affine points
  if (e == cudaSuccess) e = cudaMalloc(&d_tab, n * pb);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_in, in.data(), in_bytes, cudaMemcpyHostToDevice, s);
  int st = e == cudaSuccess ? 0 : fail_cuda(ctx, e);
  uint8_t* d_aff = d_in + in_bytes;
  if (!st)
    st = mul_dev(ctx, g2, d_in + n * 32, nullptr, d_in, n, d_aff, nullptr, s);
  if (!st) {
    k_fp_convert<<<nblocks(n * pb / 32, 128), 128, 0, s>>>(d_aff, n * pb / 32, d_tab, 1);
    ctx->launches++;
    e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    if (e != cudaSuccess) st = fail_cuda(ctx, e);
  }
  if (d_in) cudaFree(d_in);
  if (st) {
    if (d_tab) cudaFree(d_tab);
    return st;
  }
  ctx->d_mul_table[g2] = d_tab;
  return 0;
}

// out[i] = affine(scalars[i] * G) for the G1 (g2 = 0) or G2 generator: the form of mul_dev with the
// fixed-base table in place of the ladder
static int mul_gen_dev(sylow_b200_ctx* ctx, int g2, const uint8_t* scalars, size_t n, uint8_t* out, uint8_t* out_inf,
                       void* stream) {
  ENTER_DEV(ctx);
  if (n && (!scalars || !out)) return SYLOW_B200_ERR_ARG;
  if (!n) return 0;
  cudaStream_t s = pick(ctx, stream);
  CKS(ensure_mul_table(ctx, g2, s));
  return point_batch(ctx, g2, n, SY_AFF_MIN_BATCH, 0, out, out_inf, s, [&](uint8_t* proj) {
    if (g2)
      k_g2_mul_gen<<<nblocks(n, SY_G2_THREADS), SY_G2_THREADS, 0, s>>>(ctx->d_mul_table[1], scalars, n, out, out_inf,
                                                                       proj);
    else
      k_g1_mul_gen<<<nblocks(n, SY_MUL_THREADS), SY_MUL_THREADS, 0, s>>>(ctx->d_mul_table[0], scalars, n, out, out_inf,
                                                                          proj);
  });
}
int sylow_b200_g1_mul_generator_batch_dev(sylow_b200_ctx* ctx, const uint8_t* d_scalars, size_t n, uint8_t* d_out,
                                          uint8_t* d_out_inf, void* stream) {
  return mul_gen_dev(ctx, 0, d_scalars, n, d_out, d_out_inf, stream);
}
int sylow_b200_g2_mul_generator_batch_dev(sylow_b200_ctx* ctx, const uint8_t* d_scalars, size_t n, uint8_t* d_out,
                                          uint8_t* d_out_inf, void* stream) {
  return mul_gen_dev(ctx, 1, d_scalars, n, d_out, d_out_inf, stream);
}

// out[i] = affine(a[i] +- b[i]) in G1 (g2 = 0) or G2 (add_pair, group_law.cuh)
static int add_dev(sylow_b200_ctx* ctx, int g2, const uint8_t* a, const uint8_t* a_inf, const uint8_t* b,
                   const uint8_t* b_inf, size_t n, int subtract, uint8_t* out, uint8_t* out_inf, void* stream) {
  ENTER_DEV(ctx);
  if (n && (!a || !b || !out)) return SYLOW_B200_ERR_ARG;
  if (!n) return 0;
  cudaStream_t s = pick(ctx, stream);
  const size_t min_batch = g2 ? SY_G2_ADD_AFF_MIN_BATCH : SY_G1_ADD_AFF_MIN_BATCH;
  return point_batch(ctx, g2, n, min_batch, 0, out, out_inf, s, [&](uint8_t* proj) {
    if (g2)
      k_g2_add<<<nblocks(n, SY_G2_THREADS), SY_G2_THREADS, 0, s>>>(a, a_inf, b, b_inf, n, subtract, out, out_inf, proj);
    else
      k_g1_add<<<nblocks(n, SY_MUL_THREADS), SY_MUL_THREADS, 0, s>>>(a, a_inf, b, b_inf, n, subtract, out, out_inf,
                                                                      proj);
  });
}
int sylow_b200_g1_add_batch_dev(sylow_b200_ctx* ctx, const uint8_t* d_a, const uint8_t* d_a_inf, const uint8_t* d_b,
                                const uint8_t* d_b_inf, size_t n, int subtract, uint8_t* d_out, uint8_t* d_out_inf,
                                void* stream) {
  return add_dev(ctx, 0, d_a, d_a_inf, d_b, d_b_inf, n, subtract, d_out, d_out_inf, stream);
}
int sylow_b200_g2_add_batch_dev(sylow_b200_ctx* ctx, const uint8_t* d_a, const uint8_t* d_a_inf, const uint8_t* d_b,
                                const uint8_t* d_b_inf, size_t n, int subtract, uint8_t* d_out, uint8_t* d_out_inf,
                                void* stream) {
  return add_dev(ctx, 1, d_a, d_a_inf, d_b, d_b_inf, n, subtract, d_out, d_out_inf, stream);
}

// f[i] = miller(sig_i, G2gen) * miller(-H(m_i), pk_i) for every signature, Montgomery form, in scratch0:
// one 2-pair glued loop per thread (shared squaring; the generator's lines come from shared memory).  An infinite
// signature or key makes its pair contribute 1, like pairing() does (pairing.rs:876-886).
static int verify_miller_values(sylow_b200_ctx* ctx, const uint8_t* d_pks, const uint8_t* d_pks_inf, const uint8_t* d_msgs,
                                const uint64_t* d_offsets, const uint8_t* d_sigs, const uint8_t* d_sigs_inf, size_t n,
                                const DstPrime& dp, cudaStream_t s) {
  CKS(ensure_gen_table(ctx, s));
  CKS(reserve(ctx, ctx->scratch0, n * 384));
  CKS(reserve(ctx, ctx->scratch2, n * 65 + 64));
  uint8_t* d_hm = ctx->scratch2.p;
  uint8_t* d_hm_inf = d_hm + n * 64;
  CKS(hash_launch(ctx, d_msgs, d_offsets, n, dp, 1, d_hm, d_hm_inf, s));
  return launch_glued(ctx, 1, 1, d_hm, 1, d_hm_inf, d_pks, d_pks_inf, d_sigs, 1, d_sigs_inf, ctx->d_gen_table, n,
                      ctx->scratch0.p, s);
}

// sum of n affine G1 points (wire format, optional infinity flags) -> one affine point + flag at d_out / d_out_inf
// (device).  Tree of strided partial sums in projective coordinates, then one inversion.  Launched <<<1, 1>>>
// at the end because fp_pow re-converges with __syncthreads().
static int g1_sum_reduce(sylow_b200_ctx* ctx, const uint8_t* d_pts, const uint8_t* d_inf, size_t n, int negate,
                         uint8_t* d_out, uint8_t* d_out_inf, cudaStream_t s, int affine_in = 1) {
  size_t T = n / 8;
  if (T < 1) T = 1;
  if (T > 148 * 512) T = 148 * 512;
  CKS(reserve(ctx, ctx->sum0, T * 96));
  CKS(reserve(ctx, ctx->sum1, (T / 4 + 1) * 96));
  k_g1_sum_strided<<<nblocks(T, SY_MUL_THREADS), SY_MUL_THREADS, 0, s>>>(d_pts, d_inf, affine_in, n, ctx->sum0.p, T);
  LAUNCHED(ctx);
  uint8_t* cur = ctx->sum0.p;
  uint8_t* nxt = ctx->sum1.p;
  size_t m = T;
  while (m > 1) {
    size_t T2 = m / 4;
    if (T2 < 1) T2 = 1;
    k_g1_sum_strided<<<nblocks(T2, SY_MUL_THREADS), SY_MUL_THREADS, 0, s>>>(cur, nullptr, 0, m, nxt, T2);
    LAUNCHED(ctx);
    uint8_t* t = cur;
    cur = nxt;
    nxt = t;
    m = T2;
  }
  k_g1_finish_sum<<<1, 1, 0, s>>>(cur, negate, d_out, d_out_inf);
  LAUNCHED(ctx);
  return 0;
}

static bool load_seed(const uint8_t* weight_seed, WeightSeed& ws) {
  if (!weight_seed) return false;
  memcpy(ws.w, weight_seed, 32);
  return true;
}

// `pairs_ready` (may be null): an event after which the keys and signatures are in device memory - the host entry point
// copies them on its copy stream while the hash-to-curve kernel, which only needs the messages, already runs
static int verify_partial_core(sylow_b200_ctx* ctx, const uint8_t* d_pks, const uint8_t* d_pks_inf, const uint8_t* d_msgs,
                               const uint64_t* d_offsets, const uint8_t* d_sigs, const uint8_t* d_sigs_inf, size_t n,
                               const uint8_t* dst, size_t dst_len, int hash_id, const uint8_t* weight_seed,
                               uint64_t first_index, uint8_t* d_f_out, void* stream, cudaEvent_t pairs_ready) {
  if (!ctx || !d_f_out || (n && (!d_pks || !d_offsets || !d_sigs))) return SYLOW_B200_ERR_ARG;
  DstPrime dp;
  CKS(make_dst_prime(ctx, dst, dst_len, hash_id, dp));
  cudaStream_t s = pick(ctx, stream);
  if (!n) {
    CK(cudaMemcpyAsync(d_f_out, kOneCanonical, 384, cudaMemcpyHostToDevice, s));
    return 0;
  }
  // prod_i e(sig_i, G2gen) = e(sum_i sig_i, G2gen): the n signature pairs collapse into ONE Miller loop against
  // the generator (bilinearity; the Gt value after the final exponentiation is the same), so the slice costs
  // n fused Miller loops (-H(m_i), pk_i), n point additions and one extra loop.  With weights the same identity
  // holds for r_i sig_i and r_i H(m_i): two 64-bit ladders per signature on top.
  WeightSeed ws;
  const bool weighted = load_seed(weight_seed, ws);
  CKS(ensure_gen_table(ctx, s));
  CKS(reserve(ctx, ctx->scratch0, (n + 1) * 384));
  CKS(reserve(ctx, ctx->scratch1, ((n + 1) / 4 + 1) * 384));
  CKS(reserve(ctx, ctx->scratch2, n * 65 + 256));
  uint8_t* d_hm = ctx->scratch2.p;
  uint8_t* d_hm_inf = d_hm + n * 64;
  uint8_t* d_sum = d_hm + ((n * 65 + 63) / 64) * 64;  // 64 B point + flag
  uint8_t* d_sum_inf = d_sum + 64;
  CKS(hash_launch(ctx, d_msgs, d_offsets, n, dp, 1, d_hm, d_hm_inf, s));
  if (pairs_ready) CK(cudaStreamWaitEvent(s, pairs_ready, 0));
  if (weighted) {  // r_i H(m_i) in place; k_g1_mul_weight writes projective points only (min_batch 0)
    CKS(point_batch(ctx, false, n, 0, 0, d_hm, d_hm_inf, s, [&](uint8_t* proj) {
      k_g1_mul_weight<<<nblocks(n, SY_MUL_THREADS), SY_MUL_THREADS, 0, s>>>(d_hm, d_hm_inf, ws, first_index, n, proj);
    }));
  }
  // The n Miller loops (-r_i H(m_i), pk_i) only ever meet as a product, so 1, 2 or 4 signatures share one thread
  // and ONE Fp12 squaring per loop digit - what glued_miller_loop does for the whole batch in the reference
  // (pairing.rs:970-1022).  A thread's 2 / 4 pairs save 63 x 36 of the 8 444 multiplications of every pair after its
  // first.  The n % GLUE leftover pairs go through k_miller.
  // The glue is the one of fewest wave-times (glue_pairs).  Measured at 2^20 signatures
  // (profiles/r02_verify_glue.jsonl): 192.4 / 171.2 / 163.3 ms for 1 / 2 / 4; at 2^13 the order reverses (9.3 / 12.4 /
  // 18.4 ms: a quarter of the threads, each four times as long).
  const int glue = glue_pairs(ctx->sms, n, 8444, kGluedShape);
  size_t n_f = n;  // Miller values in scratch0 before the signature pair's value is appended
  if (glue > 1 && n >= (size_t)glue) {
    const size_t items = n / glue, done = items * glue;
    CKS(launch_glued(ctx, glue, 0, d_hm, glue, d_hm_inf, d_pks, d_pks_inf, nullptr, 0, nullptr, nullptr, items,
                     ctx->scratch0.p, s));
    if (done < n)
      CKS(launch_miller(ctx, d_hm + done * 64, d_hm_inf + done, d_pks + done * 128, d_pks_inf ? d_pks_inf + done : nullptr,
                        n - done, ctx->scratch0.p + items * 384, 1, s));
    n_f = items + (n - done);
  } else {
    CKS(launch_miller(ctx, d_hm, d_hm_inf, d_pks, d_pks_inf, n, ctx->scratch0.p, 1, s));
  }
  if (weighted) {
    k_g1_mul_weight<<<nblocks(n, SY_MUL_THREADS), SY_MUL_THREADS, 0, s>>>(d_sigs, d_sigs_inf, ws, first_index, n,
                                                                       ctx->proj.p);
    LAUNCHED(ctx);
    CKS(g1_sum_reduce(ctx, ctx->proj.p, nullptr, n, 0, d_sum, d_sum_inf, s, 0));
  } else {
    CKS(g1_sum_reduce(ctx, d_sigs, d_sigs_inf, n, 0, d_sum, d_sum_inf, s));
  }
  CKS(launch_glued(ctx, 0, 1, nullptr, 0, nullptr, nullptr, nullptr, d_sum, 1, d_sum_inf, ctx->d_gen_table, 1,
                   ctx->scratch0.p + n_f * 384, s));
  return product_reduce(ctx, ctx->scratch0.p, ctx->scratch1.p, n_f + 1, d_f_out, 0, s);
}

int sylow_b200_verify_batch_partial_dev(sylow_b200_ctx* ctx, const uint8_t* d_pks, const uint8_t* d_pks_inf,
                                        const uint8_t* d_msgs, const uint64_t* d_offsets, const uint8_t* d_sigs,
                                        const uint8_t* d_sigs_inf, size_t n, const uint8_t* dst, size_t dst_len,
                                        int hash_id, const uint8_t* weight_seed, uint64_t first_index, uint8_t* d_f_out,
                                        void* stream) {
  ENTER_DEV(ctx);
  return verify_partial_core(ctx, d_pks, d_pks_inf, d_msgs, d_offsets, d_sigs, d_sigs_inf, n, dst, dst_len, hash_id,
                             weight_seed, first_index, d_f_out, stream, nullptr);
}

// *failed = 1 if a hash-to-curve of the last hashing `_dev` call enqueued on `stream` hit SvdW's failing square-root
// check (GroupError::CannotHashToGroup); synchronises the stream and clears the flag.
int sylow_b200_hash_failed_dev(sylow_b200_ctx* ctx, void* stream, int* failed) {
  ENTER_DEV(ctx);
  if (!failed) return SYLOW_B200_ERR_ARG;
  cudaStream_t s = pick(ctx, stream);
  int f = 0;
  CK(cudaMemcpyAsync(&f, ctx->d_fail, sizeof(int), cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  if (f) CK(cudaMemsetAsync(ctx->d_fail, 0, sizeof(int), s));
  *failed = f;
  return 0;
}

// ------------------------------------------------------------------------------- host variants
// Host-pointer pairing / Miller-loop batch.  Large batches are cut into chunks of whole waves of both kernels (SMs x
// 1536 pairs: six Miller-loop waves, four final-exponentiation waves) and pipelined over three streams: the
// host->device copy of chunk c+1 and the device->host copy of chunk c-1 run under the kernels of chunk c, so the
// PCIe time of the 576 bytes per pairing disappears from the call.
static int pairing_host(sylow_b200_ctx* ctx, const uint8_t* g1, const uint8_t* g1_inf, const uint8_t* g2,
                        const uint8_t* g2_inf, size_t n, uint8_t* out, bool final_exp) {
  Staging io(ctx);
  uint8_t *d_out = io.area(n * 384), *d2 = io.area(n * 128), *d1 = io.area(n * 64);
  const uint8_t *d1i = io.up(g1_inf, n), *d2i = io.up(g2_inf, n);
  CKS(io.err);
  if (d1i || d2i) CK(cudaStreamSynchronize(ctx->stream));  // the flags are read from both compute streams
  // whole waves of both kernels: a multiple of the threads each of them keeps resident per SM
  const size_t chunk =
      (size_t)ctx->sms * sy_lcm(sy_lcm(SY_MILLER_THREADS * SY_MILLER_MINB, SY_FEXP_THREADS * SY_FEXP_MINB), 768) * 2;
  const size_t n_chunks = n <= 2 * chunk ? 1 : (n + chunk - 1) / chunk;
  const size_t step = n_chunks == 1 ? n : chunk;
  std::vector<cudaEvent_t> ev(2 * n_chunks, nullptr);
  int rc = 0;
  cudaError_t e = cudaSuccess;
  for (size_t i = 0; i < ev.size() && e == cudaSuccess; i++) e = cudaEventCreateWithFlags(&ev[i], cudaEventDisableTiming);
  auto d2h = [&](size_t c) {
    size_t off = c * step, m = off + step < n ? step : n - off;
    cudaError_t r = cudaStreamWaitEvent(ctx->copy_out, ev[2 * c + 1], 0);
    if (r == cudaSuccess)
      r = cudaMemcpyAsync(out + off * 384, d_out + off * 384, m * 384, cudaMemcpyDeviceToHost, ctx->copy_out);
    return r;
  };
  for (size_t c = 0; c < n_chunks && e == cudaSuccess && rc == 0; c++) {
    size_t off = c * step, m = off + step < n ? step : n - off;
    e = cudaMemcpyAsync(d1 + off * 64, g1 + off * 64, m * 64, cudaMemcpyHostToDevice, ctx->copy_in);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d2 + off * 128, g2 + off * 128, m * 128, cudaMemcpyHostToDevice, ctx->copy_in);
    if (e == cudaSuccess) e = cudaEventRecord(ev[2 * c], ctx->copy_in);
    cudaStream_t cs = (c & 1) ? ctx->stream2 : ctx->stream;
    if (e == cudaSuccess) e = cudaStreamWaitEvent(cs, ev[2 * c], 0);
    if (e != cudaSuccess) break;
    uint8_t* o = d_out + off * 384;
    if (final_exp)
      rc = pairing_dev_single(ctx, d1 + off * 64, adv(d1i, off), d2 + off * 128, adv(d2i, off), m, o, cs);
    else
      rc = sylow_b200_miller_loop_batch_dev(ctx, d1 + off * 64, adv(d1i, off), d2 + off * 128, adv(d2i, off), m, o, cs);
    if (rc) break;
    e = cudaEventRecord(ev[2 * c + 1], cs);
    // the device->host copy of the PREVIOUS chunk is issued after this chunk's kernels are queued: with pageable
    // host memory that copy blocks the calling thread, and the GPU then still has a chunk of work in front of it
    if (e == cudaSuccess && c > 0) e = d2h(c - 1);
  }
  if (e == cudaSuccess && rc == 0) e = d2h(n_chunks - 1);
  cudaError_t e2 = cudaStreamSynchronize(ctx->copy_out);
  cudaError_t e3 = cudaStreamSynchronize(ctx->stream);
  cudaError_t e4 = cudaStreamSynchronize(ctx->copy_in);
  cudaError_t e5 = cudaStreamSynchronize(ctx->stream2);
  for (cudaEvent_t v : ev)
    if (v) cudaEventDestroy(v);
  if (rc) return rc;
  if (e == cudaSuccess) e = e2;
  if (e == cudaSuccess) e = e3;
  if (e == cudaSuccess) e = e4;
  if (e == cudaSuccess) e = e5;
  if (e != cudaSuccess) return fail_cuda(ctx, e);
  return io.finish();
}

}  // extern "C" (templates need C++ linkage)

// ------------------------------------------------------------------------------- multi-device dispatch
// A context made by sylow_b200_create_multi shards the batch as contiguous slices [g n / G, (g + 1) n / G), one
// host thread per GPU driving that GPU's own single-device context (SURVEY.md 8e).  Per-item outputs land in the
// caller's buffers directly; product forms combine the G 384-byte partials on the first device.  Nothing throws
// across the ABI: thread creation failures come back as SYLOW_B200_ERR_NOMEM.
template <class Fn>
static int multi_slices(sylow_b200_ctx* ctx, size_t n, Fn fn) {
  const size_t G = ctx->children.size();
  std::vector<int> rc(G, 0);
  try {
    std::vector<std::thread> th;
    th.reserve(G);
    for (size_t g = 0; g < G; g++) {
      size_t off = g * n / G, m = (g + 1) * n / G - off;
      if (!m) continue;
      sylow_b200_ctx* c = ctx->children[g];
      th.emplace_back([&rc, &fn, c, g, off, m] { rc[g] = fn(c, g, off, m); });
    }
    for (std::thread& t : th) t.join();
  } catch (...) {
    return SYLOW_B200_ERR_NOMEM;
  }
  for (int r : rc)
    if (r) return r;
  return 0;
}
// Product forms: fn(child, off, m, partial) writes the canonical product of its slice to `partial` (an empty slice
// contributes 1), and the first device multiplies the G partials into f_out.
template <class Fn>
static int multi_product(sylow_b200_ctx* ctx, size_t n, Fn fn, uint8_t* f_out) {
  const size_t G = ctx->children.size();
  std::vector<uint8_t> part(G * 384, 0);
  for (size_t g = 0; g < G; g++) part[g * 384] = 1;
  uint8_t* pp = part.data();
  CKS(multi_slices(ctx, n, [=](sylow_b200_ctx* c, size_t g, size_t off, size_t m) { return fn(c, off, m, pp + g * 384); }));
  return sylow_b200_fp12_product(ctx->children[0], pp, G, f_out);
}
static inline bool is_multi(const sylow_b200_ctx* ctx) { return ctx && ctx->children.size() > 1; }
// messages of the slice [off, off + m): the byte range and offsets rebased to 0
struct MsgSlice {
  const uint8_t* msgs;
  std::vector<uint64_t> offs;
  MsgSlice(const uint8_t* all, const uint64_t* offsets, size_t off, size_t m) : msgs(all ? all + offsets[off] : nullptr), offs(m + 1) {
    for (size_t i = 0; i <= m; i++) offs[i] = offsets[off + i] - offsets[off];
  }
};

extern "C" {

int sylow_b200_pairing_batch(sylow_b200_ctx* ctx, const uint8_t* g1, const uint8_t* g1_inf, const uint8_t* g2,
                             const uint8_t* g2_inf, size_t n, uint8_t* gt_out) {
  if (is_multi(ctx) && g1 && g2 && gt_out)
    return multi_slices(ctx, n, [=](sylow_b200_ctx* c, size_t, size_t off, size_t m) {
      return sylow_b200_pairing_batch(c, g1 + off * 64, adv(g1_inf, off), g2 + off * 128, adv(g2_inf, off), m,
                                      gt_out + off * 384);
    });
  ENTER(ctx);
  if (n && (!g1 || !g2 || !gt_out)) return SYLOW_B200_ERR_ARG;
  if (!n) return 0;
  return pairing_host(ctx, g1, g1_inf, g2, g2_inf, n, gt_out, true);
}

int sylow_b200_miller_loop_batch(sylow_b200_ctx* ctx, const uint8_t* g1, const uint8_t* g1_inf, const uint8_t* g2,
                                 const uint8_t* g2_inf, size_t n, uint8_t* f_out) {
  if (is_multi(ctx) && g1 && g2 && f_out)
    return multi_slices(ctx, n, [=](sylow_b200_ctx* c, size_t, size_t off, size_t m) {
      return sylow_b200_miller_loop_batch(c, g1 + off * 64, adv(g1_inf, off), g2 + off * 128, adv(g2_inf, off), m,
                                          f_out + off * 384);
    });
  ENTER(ctx);
  if (n && (!g1 || !g2 || !f_out)) return SYLOW_B200_ERR_ARG;
  if (!n) return 0;
  return pairing_host(ctx, g1, g1_inf, g2, g2_inf, n, f_out, false);
}

int sylow_b200_miller_product(sylow_b200_ctx* ctx, const uint8_t* g1, const uint8_t* g1_inf, const uint8_t* g2,
                              const uint8_t* g2_inf, size_t n, uint8_t f_out[384]) {
  if (is_multi(ctx) && g1 && g2 && f_out && n)
    return multi_product(ctx, n, [=](sylow_b200_ctx* c, size_t off, size_t m, uint8_t* part) {
      return sylow_b200_miller_product(c, g1 + off * 64, adv(g1_inf, off), g2 + off * 128, adv(g2_inf, off), m, part);
    }, f_out);
  ENTER(ctx);
  if (!f_out || (n && (!g1 || !g2))) return SYLOW_B200_ERR_ARG;
  Staging io(ctx);
  const uint8_t *d2 = io.up(g2, n * 128), *d1 = io.up(g1, n * 64), *d1i = io.up(g1_inf, n), *d2i = io.up(g2_inf, n);
  uint8_t* d_f = io.area(384);
  CKS(io.err);
  CKS(sylow_b200_miller_product_dev(ctx, d1, d1i, d2, d2i, n, d_f, nullptr));
  io.down(f_out, d_f, 384);
  return io.finish();
}

int sylow_b200_final_exp_batch(sylow_b200_ctx* ctx, const uint8_t* f, size_t n, uint8_t* gt_out) {
  if (is_multi(ctx) && f && gt_out && n >= 4096)
    return multi_slices(ctx, n, [=](sylow_b200_ctx* c, size_t, size_t off, size_t m) {
      return sylow_b200_final_exp_batch(c, f + off * 384, m, gt_out + off * 384);
    });
  ENTER(ctx);
  if (n && (!f || !gt_out)) return SYLOW_B200_ERR_ARG;
  if (!n) return 0;
  Staging io(ctx);
  const uint8_t* df = io.up(f, n * 384);
  uint8_t* d_gt = io.area(n * 384);
  CKS(io.err);
  CKS(sylow_b200_final_exp_batch_dev(ctx, df, n, d_gt, nullptr));
  io.down(gt_out, d_gt, n * 384);
  return io.finish();
}

int sylow_b200_fp12_product(sylow_b200_ctx* ctx, const uint8_t* f, size_t n, uint8_t out[384]) {
  ENTER(ctx);
  if (!out || (n && !f)) return SYLOW_B200_ERR_ARG;
  if (!n) {
    memcpy(out, kOneCanonical, 384);
    return 0;
  }
  Staging io(ctx);
  const uint8_t* df = io.up(f, n * 384);
  uint8_t* d_prod = io.area(384);
  CKS(io.err);
  CKS(reserve(ctx, ctx->scratch0, n * 384));
  CKS(reserve(ctx, ctx->scratch1, (n / 4 + 1) * 384));
  k_fp12_convert<<<nblocks(n, 128), 128, 0, ctx->stream>>>(df, n, ctx->scratch0.p, 1);
  LAUNCHED(ctx);
  CKS(product_reduce(ctx, ctx->scratch0.p, ctx->scratch1.p, n, d_prod, 0, ctx->stream));
  io.down(out, d_prod, 384);
  return io.finish();
}

int sylow_b200_pairing_check_batch(sylow_b200_ctx* ctx, const uint8_t* g1, const uint8_t* g1_inf, const uint8_t* g2,
                                   const uint8_t* g2_inf, size_t k, size_t n_checks, uint8_t* ok_out) {
  if (is_multi(ctx) && g1 && g2 && ok_out)
    return multi_slices(ctx, n_checks, [=](sylow_b200_ctx* c, size_t, size_t off, size_t m) {
      return sylow_b200_pairing_check_batch(c, g1 + off * k * 64, adv(g1_inf, off * k), g2 + off * k * 128,
                                            adv(g2_inf, off * k), k, m, ok_out + off);
    });
  ENTER(ctx);
  if (n_checks && !ok_out) return SYLOW_B200_ERR_ARG;
  if (!n_checks) return 0;
  size_t n = k * n_checks;
  if (n && (!g1 || !g2)) return SYLOW_B200_ERR_ARG;
  Staging io(ctx);
  const uint8_t *d2 = io.up(g2, n * 128), *d1 = io.up(g1, n * 64), *d1i = io.up(g1_inf, n), *d2i = io.up(g2_inf, n);
  uint8_t* d_ok = io.area(n_checks);
  CKS(io.err);
  CKS(sylow_b200_pairing_check_batch_dev(ctx, d1, d1i, d2, d2i, k, n_checks, d_ok, nullptr));
  io.down(ok_out, d_ok, n_checks);
  return io.finish();
}

// pts == nullptr: the generator of the group (g1/g2_mul_generator_batch)
static int mul_host(sylow_b200_ctx* ctx, int g2, const uint8_t* pts, const uint8_t* pts_inf, const uint8_t* scalars,
                    size_t n, uint8_t* out, uint8_t* out_inf) {
  if (is_multi(ctx) && scalars && out) {
    const size_t pb = g2 ? 128 : 64;
    return multi_slices(ctx, n, [=](sylow_b200_ctx* c, size_t, size_t off, size_t m) {
      return mul_host(c, g2, adv(pts, off * pb), adv(pts_inf, off), scalars + off * 32, m, out + off * pb,
                      adv(out_inf, off));
    });
  }
  ENTER(ctx);
  if (n && (!scalars || !out)) return SYLOW_B200_ERR_ARG;
  if (!n) return 0;
  size_t pb = g2 ? 128 : 64;
  Staging io(ctx);
  uint8_t* d_out = io.area(n * pb);
  const uint8_t *dp = io.up(pts, n * pb), *dk = io.up(scalars, n * 32), *dpi = io.up(pts_inf, n);
  uint8_t* d_out_inf = io.area(n);
  CKS(io.err);
  if (!pts)
    CKS(mul_gen_dev(ctx, g2, dk, n, d_out, d_out_inf, nullptr));
  else
    CKS(mul_dev(ctx, g2, dp, dpi, dk, n, d_out, d_out_inf, nullptr));
  io.down(out, d_out, n * pb);
  if (out_inf) io.down(out_inf, d_out_inf, n);
  return io.finish();
}
int sylow_b200_g1_mul_batch(sylow_b200_ctx* ctx, const uint8_t* pts, const uint8_t* pts_inf, const uint8_t* scalars,
                            size_t n, uint8_t* out, uint8_t* out_inf) {
  if (n && !pts) return SYLOW_B200_ERR_ARG;
  return mul_host(ctx, 0, pts, pts_inf, scalars, n, out, out_inf);
}
int sylow_b200_g2_mul_batch(sylow_b200_ctx* ctx, const uint8_t* pts, const uint8_t* pts_inf, const uint8_t* scalars,
                            size_t n, uint8_t* out, uint8_t* out_inf) {
  if (n && !pts) return SYLOW_B200_ERR_ARG;
  return mul_host(ctx, 1, pts, pts_inf, scalars, n, out, out_inf);
}
int sylow_b200_g1_mul_generator_batch(sylow_b200_ctx* ctx, const uint8_t* scalars, size_t n, uint8_t* out,
                                      uint8_t* out_inf) {
  return mul_host(ctx, 0, nullptr, nullptr, scalars, n, out, out_inf);
}
int sylow_b200_g2_mul_generator_batch(sylow_b200_ctx* ctx, const uint8_t* scalars, size_t n, uint8_t* out,
                                      uint8_t* out_inf) {
  return mul_host(ctx, 1, nullptr, nullptr, scalars, n, out, out_inf);
}

static int add_host(sylow_b200_ctx* ctx, int g2, const uint8_t* a, const uint8_t* a_inf, const uint8_t* b,
                    const uint8_t* b_inf, size_t n, int subtract, uint8_t* out, uint8_t* out_inf) {
  const size_t pb = g2 ? 128 : 64;
  if (is_multi(ctx) && a && b && out) {
    return multi_slices(ctx, n, [=](sylow_b200_ctx* c, size_t, size_t off, size_t m) {
      return add_host(c, g2, a + off * pb, adv(a_inf, off), b + off * pb, adv(b_inf, off), m, subtract, out + off * pb,
                      adv(out_inf, off));
    });
  }
  ENTER(ctx);
  if (n && (!a || !b || !out)) return SYLOW_B200_ERR_ARG;
  if (!n) return 0;
  Staging io(ctx);
  uint8_t* d_out = io.area(n * pb);
  const uint8_t *da = io.up(a, n * pb), *db = io.up(b, n * pb), *dai = io.up(a_inf, n), *dbi = io.up(b_inf, n);
  uint8_t* d_out_inf = io.area(n);
  CKS(io.err);
  CKS(add_dev(ctx, g2, da, dai, db, dbi, n, subtract, d_out, d_out_inf, nullptr));
  io.down(out, d_out, n * pb);
  if (out_inf) io.down(out_inf, d_out_inf, n);
  return io.finish();
}
int sylow_b200_g1_add_batch(sylow_b200_ctx* ctx, const uint8_t* a, const uint8_t* a_inf, const uint8_t* b,
                            const uint8_t* b_inf, size_t n, int subtract, uint8_t* out, uint8_t* out_inf) {
  return add_host(ctx, 0, a, a_inf, b, b_inf, n, subtract, out, out_inf);
}
int sylow_b200_g2_add_batch(sylow_b200_ctx* ctx, const uint8_t* a, const uint8_t* a_inf, const uint8_t* b,
                            const uint8_t* b_inf, size_t n, int subtract, uint8_t* out, uint8_t* out_inf) {
  return add_host(ctx, 1, a, a_inf, b, b_inf, n, subtract, out, out_inf);
}

// the end of a hashing host form: finishes with the hash-to-curve failure flag, then CannotHashToGroup if it is set
static int check_hash_fail(Staging& io) {
  sylow_b200_ctx* ctx = io.ctx;
  int f = 0;
  io.down(&f, ctx->d_fail, sizeof(int));
  CKS(io.finish());
  if (f) {
    CK(cudaMemsetAsync(ctx->d_fail, 0, sizeof(int), ctx->stream));
    return SYLOW_B200_ERR_CANNOT_HASH;
  }
  return 0;
}

// n messages and their offsets, staged; malformed offsets or a missing message buffer fail the call with ERR_ARG
struct DevMsgs {
  const uint8_t* msgs;
  const uint64_t* offsets;
};
static DevMsgs msgs_to_dev(Staging& io, const uint8_t* msgs, const uint64_t* offsets, size_t n) {
  bool ok = offsets && offsets[0] == 0;
  for (size_t i = 0; ok && i < n; i++) ok = offsets[i + 1] >= offsets[i];
  const size_t total = ok ? (size_t)offsets[n] : 0;
  if (!ok || (total && !msgs)) {
    if (!io.err) io.err = SYLOW_B200_ERR_ARG;
    return {};
  }
  const uint8_t* dm = total ? io.up(msgs, total) : io.area(16);  // all messages empty: still a valid pointer
  return {dm, reinterpret_cast<const uint64_t*>(io.up(offsets, (n + 1) * sizeof(uint64_t)))};
}

int sylow_b200_hash_to_g1_batch(sylow_b200_ctx* ctx, const uint8_t* msgs, const uint64_t* offsets, size_t n,
                                const uint8_t* dst, size_t dst_len, int hash_id, uint8_t* out, uint8_t* out_inf) {
  if (is_multi(ctx) && offsets && out && n)
    return multi_slices(ctx, n, [=](sylow_b200_ctx* c, size_t, size_t off, size_t m) {
      MsgSlice ms(msgs, offsets, off, m);
      return sylow_b200_hash_to_g1_batch(c, ms.msgs, ms.offs.data(), m, dst, dst_len, hash_id, out + off * 64,
                                         adv(out_inf, off));
    });
  ENTER(ctx);
  DstPrime dp;
  CKS(make_dst_prime(ctx, dst, dst_len, hash_id, dp));
  if (!n) return 0;
  if (!out) return SYLOW_B200_ERR_ARG;
  Staging io(ctx);
  uint8_t* d_out = io.area(n * 64);
  const DevMsgs m = msgs_to_dev(io, msgs, offsets, n);
  uint8_t* d_out_inf = io.area(n);
  CKS(io.err);
  CKS(hash_launch(ctx, m.msgs, m.offsets, n, dp, 0, d_out, d_out_inf, ctx->stream));
  io.down(out, d_out, n * 64);
  if (out_inf) io.down(out_inf, d_out_inf, n);
  return check_hash_fail(io);
}

int sylow_b200_sign_batch(sylow_b200_ctx* ctx, const uint8_t* sks, const uint8_t* msgs, const uint64_t* offsets,
                          size_t n, const uint8_t* dst, size_t dst_len, int hash_id, uint8_t* sigs_out,
                          uint8_t* sigs_out_inf) {
  if (is_multi(ctx) && offsets && sks && sigs_out && n)
    return multi_slices(ctx, n, [=](sylow_b200_ctx* c, size_t, size_t off, size_t m) {
      MsgSlice ms(msgs, offsets, off, m);
      return sylow_b200_sign_batch(c, sks + off * 32, ms.msgs, ms.offs.data(), m, dst, dst_len, hash_id,
                                   sigs_out + off * 64, adv(sigs_out_inf, off));
    });
  ENTER(ctx);
  DstPrime dp;
  CKS(make_dst_prime(ctx, dst, dst_len, hash_id, dp));
  if (!n) return 0;
  if (!sks || !sigs_out) return SYLOW_B200_ERR_ARG;
  Staging io(ctx);
  uint8_t *d_hm = io.area(n * 65), *d_sig = io.area(n * 64);  // H(m_i), then their flags; the signatures
  const DevMsgs m = msgs_to_dev(io, msgs, offsets, n);
  const uint8_t* dk = io.up(sks, n * 32);
  uint8_t* d_sig_inf = io.area(n);
  CKS(io.err);
  CKS(hash_launch(ctx, m.msgs, m.offsets, n, dp, 0, d_hm, d_hm + n * 64, ctx->stream));
  CKS(sylow_b200_g1_mul_batch_dev(ctx, d_hm, d_hm + n * 64, dk, n, d_sig, d_sig_inf, nullptr));
  io.down(sigs_out, d_sig, n * 64);
  if (sigs_out_inf) io.down(sigs_out_inf, d_sig_inf, n);
  return check_hash_fail(io);
}

int sylow_b200_verify_batch_partial(sylow_b200_ctx* ctx, const uint8_t* pks, const uint8_t* pks_inf, const uint8_t* msgs,
                                    const uint64_t* offsets, const uint8_t* sigs, const uint8_t* sigs_inf, size_t n,
                                    const uint8_t* dst, size_t dst_len, int hash_id, const uint8_t* weight_seed,
                                    uint64_t first_index, uint8_t f_out[384]) {
  if (is_multi(ctx) && offsets && pks && sigs && f_out && n)
    return multi_product(ctx, n, [=](sylow_b200_ctx* c, size_t off, size_t m, uint8_t* part) {
      MsgSlice ms(msgs, offsets, off, m);
      return sylow_b200_verify_batch_partial(c, pks + off * 128, adv(pks_inf, off), ms.msgs, ms.offs.data(),
                                             sigs + off * 64, adv(sigs_inf, off), m, dst, dst_len, hash_id,
                                             weight_seed, first_index + off, part);
    }, f_out);
  ENTER(ctx);
  if (!f_out) return SYLOW_B200_ERR_ARG;
  DstPrime dp;
  CKS(make_dst_prime(ctx, dst, dst_len, hash_id, dp));
  if (!n) {
    memcpy(f_out, kOneCanonical, 384);
    return 0;
  }
  if (!pks || !sigs) return SYLOW_B200_ERR_ARG;
  Staging io(ctx);
  uint8_t *dpk = io.area(n * 128), *dsg = io.area(n * 64);
  // messages first, on the compute stream: the hash-to-curve kernel starts as soon as they are there, while the keys
  // and signatures (six times the bytes) still travel on the copy stream
  const DevMsgs m = msgs_to_dev(io, msgs, offsets, n);
  uint8_t *dpki = io.area(pks_inf ? n : 0), *dsgi = io.area(sigs_inf ? n : 0), *d_f = io.area(384);
  CKS(io.err);
  CK(cudaMemcpyAsync(dpk, pks, n * 128, cudaMemcpyHostToDevice, ctx->copy_in));
  CK(cudaMemcpyAsync(dsg, sigs, n * 64, cudaMemcpyHostToDevice, ctx->copy_in));
  if (pks_inf) CK(cudaMemcpyAsync(dpki, pks_inf, n, cudaMemcpyHostToDevice, ctx->copy_in));
  if (sigs_inf) CK(cudaMemcpyAsync(dsgi, sigs_inf, n, cudaMemcpyHostToDevice, ctx->copy_in));
  CK(cudaEventRecord(ctx->ev_fork, ctx->copy_in));
  CKS(verify_partial_core(ctx, dpk, dpki, m.msgs, m.offsets, dsg, dsgi, n, dst, dst_len, hash_id, weight_seed,
                          first_index, d_f, nullptr, ctx->ev_fork));
  io.down(f_out, d_f, 384);
  return check_hash_fail(io);
}

int sylow_b200_verify_batch_finish(sylow_b200_ctx* ctx, const uint8_t* partials, size_t n_partials, int* ok) {
  ENTER(ctx);
  if (!ok || (n_partials && !partials)) return SYLOW_B200_ERR_ARG;
  uint8_t prod[384], gt[384];
  CKS(sylow_b200_fp12_product(ctx, partials, n_partials, prod));
  CKS(sylow_b200_final_exp_batch(ctx, prod, 1, gt));
  *ok = memcmp(gt, kOneCanonical, 384) == 0;
  return 0;
}

int sylow_b200_verify_batch(sylow_b200_ctx* ctx, const uint8_t* pks, const uint8_t* pks_inf, const uint8_t* msgs,
                            const uint64_t* offsets, const uint8_t* sigs, const uint8_t* sigs_inf, size_t n,
                            const uint8_t* dst, size_t dst_len, int hash_id, const uint8_t* weight_seed, int* ok) {
  if (!ok) return SYLOW_B200_ERR_ARG;
  uint8_t f[384];
  CKS(sylow_b200_verify_batch_partial(ctx, pks, pks_inf, msgs, offsets, sigs, sigs_inf, n, dst, dst_len, hash_id,
                                      weight_seed, 0, f));
  return sylow_b200_verify_batch_finish(ctx, f, 1, ok);
}

int sylow_b200_verify_each(sylow_b200_ctx* ctx, const uint8_t* pks, const uint8_t* pks_inf, const uint8_t* msgs,
                           const uint64_t* offsets, const uint8_t* sigs, const uint8_t* sigs_inf, size_t n,
                           const uint8_t* dst, size_t dst_len, int hash_id, uint8_t* ok_out) {
  if (is_multi(ctx) && offsets && pks && sigs && ok_out && n)
    return multi_slices(ctx, n, [=](sylow_b200_ctx* c, size_t, size_t off, size_t m) {
      MsgSlice ms(msgs, offsets, off, m);
      return sylow_b200_verify_each(c, pks + off * 128, adv(pks_inf, off), ms.msgs, ms.offs.data(), sigs + off * 64,
                                    adv(sigs_inf, off), m, dst, dst_len, hash_id, ok_out + off);
    });
  ENTER(ctx);
  DstPrime dp;
  CKS(make_dst_prime(ctx, dst, dst_len, hash_id, dp));
  if (!n) return 0;
  if (!pks || !sigs || !ok_out) return SYLOW_B200_ERR_ARG;
  Staging io(ctx);
  const uint8_t *dpk = io.up(pks, n * 128), *dsg = io.up(sigs, n * 64);
  const DevMsgs m = msgs_to_dev(io, msgs, offsets, n);
  const uint8_t *dpki = io.up(pks_inf, n), *dsgi = io.up(sigs_inf, n);
  uint8_t* d_ok = io.area(n);
  CKS(io.err);
  CKS(verify_miller_values(ctx, dpk, dpki, m.msgs, m.offsets, dsg, dsgi, n, dp, ctx->stream));
  CKS(launch_check_products(ctx, ctx->scratch0.p, 1, n, d_ok, ctx->stream));
  io.down(ok_out, d_ok, n);
  return check_hash_fail(io);
}

// ------------------------------------------------------------------------------- precomputed G2
int sylow_b200_g2_precompute(sylow_b200_ctx* ctx, const uint8_t* g2, size_t n, uint8_t* coeffs_out) {
  ENTER(ctx);
  if (n && (!g2 || !coeffs_out)) return SYLOW_B200_ERR_ARG;
  if (!n) return 0;
  Staging io(ctx);
  uint8_t* d_tab = io.area(n * SY_TABLE_BYTES);
  const uint8_t* d2 = io.up(g2, n * 128);
  CKS(io.err);
  k_g2_precompute<<<nblocks(n, SY_GLUED_THREADS), SY_GLUED_THREADS, 0, ctx->stream>>>(d2, n, d_tab, 0);
  LAUNCHED(ctx);
  io.down(coeffs_out, d_tab, n * SY_TABLE_BYTES);
  return io.finish();
}

// uploads k canonical tables and converts them to Montgomery form in ctx->tables
static int tables_to_dev(Staging& io, const uint8_t* coeffs, size_t k) {
  sylow_b200_ctx* ctx = io.ctx;
  const uint8_t* dc = io.up(coeffs, k * SY_TABLE_BYTES);
  CKS(io.err);
  CKS(reserve(ctx, ctx->tables, k * SY_TABLE_BYTES));
  size_t nfp = k * SY_TABLE_BYTES / 32;
  k_fp_convert<<<nblocks(nfp, 128), 128, 0, ctx->stream>>>(dc, nfp, ctx->tables.p, 1);
  LAUNCHED(ctx);
  return 0;
}

int sylow_b200_miller_loop_precomputed(sylow_b200_ctx* ctx, const uint8_t* coeffs, const uint8_t* g1,
                                       const uint8_t* g1_inf, size_t n, uint8_t* f_out) {
  ENTER(ctx);
  if (!coeffs || (n && (!g1 || !f_out))) return SYLOW_B200_ERR_ARG;
  if (!n) return 0;
  Staging io(ctx);
  CKS(tables_to_dev(io, coeffs, 1));
  uint8_t* d_f = io.area(n * 384);
  const uint8_t *d1 = io.up(g1, n * 64), *d1i = io.up(g1_inf, n);
  CKS(io.err);
  CKS(launch_glued(ctx, 0, 1, nullptr, 0, nullptr, nullptr, nullptr, d1, 1, d1i, ctx->tables.p, n, d_f, ctx->stream));
  k_fp12_convert<<<nblocks(n, 128), 128, 0, ctx->stream>>>(d_f, n, d_f, 0);
  LAUNCHED(ctx);
  io.down(f_out, d_f, n * 384);
  return io.finish();
}

int sylow_b200_pairing_check_fixed_batch_dev(sylow_b200_ctx* ctx, const uint8_t* d_g1, const uint8_t* d_g1_inf,
                                             const uint8_t* d_g2_var, const uint8_t* d_g2_var_inf, size_t k_var,
                                             const uint8_t* d_tables, size_t k_fixed, size_t n_checks,
                                             uint8_t* d_ok_out, void* stream) {
  ENTER_DEV(ctx);
  if (n_checks && (!d_g1 || !d_ok_out || !d_tables || (k_var && !d_g2_var))) return SYLOW_B200_ERR_ARG;
  if (!n_checks) return 0;
  cudaStream_t s = pick(ctx, stream);
  size_t k = k_var + k_fixed;
  CKS(reserve(ctx, ctx->scratch0, n_checks * 384));
  const uint8_t* g1f = d_g1 + k_var * 64;
  const uint8_t* g1f_inf = d_g1_inf ? d_g1_inf + k_var : nullptr;
  if (!k_fixed) return SYLOW_B200_ERR_ARG;  // other shapes: use sylow_b200_pairing_check_batch
  CKS(launch_glued(ctx, k_var, k_fixed, d_g1, k, d_g1_inf, d_g2_var, d_g2_var_inf, g1f, k, g1f_inf, d_tables, n_checks,
                   ctx->scratch0.p, s));
  return launch_check_products(ctx, ctx->scratch0.p, 1, n_checks, d_ok_out, s);
}

int sylow_b200_tables_to_device(sylow_b200_ctx* ctx, const uint8_t* coeffs, size_t k, uint8_t* d_tables_out, void* stream) {
  ENTER_DEV(ctx);
  if (!coeffs || !d_tables_out || !k) return SYLOW_B200_ERR_ARG;
  Staging io(ctx);
  CKS(tables_to_dev(io, coeffs, k));
  CKS(io.finish());
  CK(cudaMemcpyAsync(d_tables_out, ctx->tables.p, k * SY_TABLE_BYTES, cudaMemcpyDeviceToDevice, pick(ctx, stream)));
  CK(cudaStreamSynchronize(pick(ctx, stream)));  // ctx->tables is reused by the next call
  return 0;
}

int sylow_b200_pairing_check_fixed_batch(sylow_b200_ctx* ctx, const uint8_t* g1, const uint8_t* g1_inf,
                                         const uint8_t* g2_var, const uint8_t* g2_var_inf, size_t k_var,
                                         const uint8_t* coeffs_fixed, size_t k_fixed, size_t n_checks, uint8_t* ok_out) {
  ENTER(ctx);
  if (n_checks && (!g1 || !ok_out || !coeffs_fixed || (k_var && !g2_var))) return SYLOW_B200_ERR_ARG;
  if (!k_fixed || !glued_shape_ok(k_var, k_fixed)) return SYLOW_B200_ERR_ARG;
  if (!n_checks) return 0;
  size_t k = k_var + k_fixed;
  Staging io(ctx);
  CKS(tables_to_dev(io, coeffs_fixed, k_fixed));
  const uint8_t *d2 = io.up(g2_var, n_checks * k_var * 128), *d1 = io.up(g1, n_checks * k * 64);
  const uint8_t *d1i = io.up(g1_inf, n_checks * k), *d2i = io.up(g2_var_inf, n_checks * k_var);
  uint8_t* d_ok = io.area(n_checks);
  CKS(io.err);
  CKS(sylow_b200_pairing_check_fixed_batch_dev(ctx, d1, d1i, d2, d2i, k_var, ctx->tables.p, k_fixed, n_checks, d_ok,
                                               nullptr));
  io.down(ok_out, d_ok, n_checks);
  return io.finish();
}

// d_out (canonical) = prod over n >= 1 pairs of the Miller loop of g1[k] against table idx[k] (k if idx is null):
// glue_pairs' choice of pairs per thread, the n % glue leftover pairs one per thread, then product_reduce.
static int miller_product_tables(sylow_b200_ctx* ctx, const uint8_t* tables, size_t n_tables, const uint32_t* idx,
                                 const uint8_t* g1, const uint8_t* g1_inf, size_t n, uint8_t* d_out, cudaStream_t s) {
  const int glue = glue_pairs(ctx->sms, n, 6045, kGluedShape);
  const size_t items = n / glue, done = items * glue;
  CKS(reserve(ctx, ctx->scratch0, n * 384));
  CKS(reserve(ctx, ctx->scratch1, (n / 4 + 1) * 384));
  CKS(launch_miller_tables(ctx, glue, tables, n_tables, idx, g1, g1_inf, items, ctx->scratch0.p, 1, s));
  if (done < n) {
    // without an index pair k uses table k: the leftover pairs start at table `done`
    const uint8_t* t = idx ? tables : tables + done * SY_TABLE_BYTES;
    CKS(launch_miller_tables(ctx, 1, t, idx ? n_tables : n_tables - done, idx ? idx + done : nullptr, g1 + done * 64,
                             adv(g1_inf, done), n - done, ctx->scratch0.p + items * 384, 1, s));
  }
  return product_reduce(ctx, ctx->scratch0.p, ctx->scratch1.p, items + (n - done), d_out, 0, s);
}

int sylow_b200_miller_loop_precomputed_batch(sylow_b200_ctx* ctx, const uint8_t* coeffs, const uint8_t* g1,
                                             const uint8_t* g1_inf, size_t n, uint8_t* f_out) {
  if (is_multi(ctx) && coeffs && g1 && f_out)
    return multi_slices(ctx, n, [=](sylow_b200_ctx* c, size_t, size_t off, size_t m) {
      return sylow_b200_miller_loop_precomputed_batch(c, coeffs + off * SY_TABLE_BYTES, g1 + off * 64, adv(g1_inf, off),
                                                      m, f_out + off * 384);
    });
  ENTER(ctx);
  if (n && (!coeffs || !g1 || !f_out)) return SYLOW_B200_ERR_ARG;
  if (!n) return 0;
  Staging io(ctx);
  CKS(tables_to_dev(io, coeffs, n));
  uint8_t* d_f = io.area(n * 384);
  const uint8_t *d1 = io.up(g1, n * 64), *d1i = io.up(g1_inf, n);
  CKS(io.err);
  CKS(launch_miller_tables(ctx, 1, ctx->tables.p, n, nullptr, d1, d1i, n, d_f, 0, ctx->stream));
  io.down(f_out, d_f, n * 384);
  return io.finish();
}

int sylow_b200_miller_product_precomputed(sylow_b200_ctx* ctx, const uint8_t* coeffs, const uint8_t* g1,
                                          const uint8_t* g1_inf, size_t n, uint8_t f_out[384]) {
  if (is_multi(ctx) && coeffs && g1 && f_out && n)
    return multi_product(ctx, n, [=](sylow_b200_ctx* c, size_t off, size_t m, uint8_t* part) {
      return sylow_b200_miller_product_precomputed(c, coeffs + off * SY_TABLE_BYTES, g1 + off * 64, adv(g1_inf, off), m,
                                                   part);
    }, f_out);
  ENTER(ctx);
  if (!f_out || (n && (!coeffs || !g1))) return SYLOW_B200_ERR_ARG;
  if (!n) {
    memcpy(f_out, kOneCanonical, 384);
    return 0;
  }
  Staging io(ctx);
  CKS(tables_to_dev(io, coeffs, n));
  const uint8_t *d1 = io.up(g1, n * 64), *d1i = io.up(g1_inf, n);
  uint8_t* d_f = io.area(384);
  CKS(io.err);
  CKS(miller_product_tables(ctx, ctx->tables.p, n, nullptr, d1, d1i, n, d_f, ctx->stream));
  io.down(f_out, d_f, 384);
  return io.finish();
}

int sylow_b200_g2_precompute_dev(sylow_b200_ctx* ctx, const uint8_t* d_g2, size_t n, uint8_t* d_tables_out,
                                 void* stream) {
  ENTER_DEV(ctx);
  if (n && (!d_g2 || !d_tables_out)) return SYLOW_B200_ERR_ARG;
  if (!n) return 0;
  k_g2_precompute<<<nblocks(n, SY_GLUED_THREADS), SY_GLUED_THREADS, 0, pick(ctx, stream)>>>(d_g2, n, d_tables_out, 1);
  LAUNCHED(ctx);
  return 0;
}

int sylow_b200_miller_product_precomputed_dev(sylow_b200_ctx* ctx, const uint8_t* d_tables, size_t n_tables,
                                              const uint32_t* d_table_idx, const uint8_t* d_g1, const uint8_t* d_g1_inf,
                                              size_t n, uint8_t* d_f_out, void* stream) {
  ENTER_DEV(ctx);
  if (!d_f_out || (n && (!d_tables || !d_g1 || !n_tables || (!d_table_idx && n > n_tables))))
    return SYLOW_B200_ERR_ARG;
  cudaStream_t s = pick(ctx, stream);
  if (!n) {
    CK(cudaMemcpyAsync(d_f_out, kOneCanonical, 384, cudaMemcpyHostToDevice, s));
    return 0;
  }
  return miller_product_tables(ctx, d_tables, n_tables, d_table_idx, d_g1, d_g1_inf, n, d_f_out, s);
}

// ------------------------------------------------------------------------------- validation
int sylow_b200_g1_validate_batch(sylow_b200_ctx* ctx, const uint8_t* g1, const uint8_t* g1_inf, size_t n,
                                 int8_t* status_out) {
  ENTER(ctx);
  if (n && (!g1 || !status_out)) return SYLOW_B200_ERR_ARG;
  if (!n) return 0;
  Staging io(ctx);
  const uint8_t *d1 = io.up(g1, n * 64), *d1i = io.up(g1_inf, n);
  int8_t* d_st = reinterpret_cast<int8_t*>(io.area(n));
  CKS(io.err);
  k_g1_validate<<<nblocks(n, 128), 128, 0, ctx->stream>>>(d1, d1i, n, d_st, 0);
  LAUNCHED(ctx);
  io.down(status_out, d_st, n);
  return io.finish();
}

int sylow_b200_g2_validate_batch(sylow_b200_ctx* ctx, const uint8_t* g2, const uint8_t* g2_inf, size_t n,
                                 int8_t* status_out) {
  if (is_multi(ctx) && g2 && status_out)
    return multi_slices(ctx, n, [=](sylow_b200_ctx* c, size_t, size_t off, size_t m) {
      return sylow_b200_g2_validate_batch(c, g2 + off * 128, adv(g2_inf, off), m, status_out + off);
    });
  ENTER(ctx);
  if (n && (!g2 || !status_out)) return SYLOW_B200_ERR_ARG;
  if (!n) return 0;
  Staging io(ctx);
  const uint8_t *d2 = io.up(g2, n * 128), *d2i = io.up(g2_inf, n);
  int8_t* d_st = reinterpret_cast<int8_t*>(io.area(n));
  CKS(io.err);
  k_g2_validate<<<nblocks(n, SY_MUL_THREADS), SY_MUL_THREADS, 0, ctx->stream>>>(d2, d2i, n, d_st, 0);
  LAUNCHED(ctx);
  io.down(status_out, d_st, n);
  return io.finish();
}

// ------------------------------------------------------------------------------- big-endian codecs
static int from_be(sylow_b200_ctx* ctx, int g2, const uint8_t* be, size_t n, int mode, int validate, uint8_t* out,
                   uint8_t* inf_out, int8_t* status_out) {
  ENTER(ctx);
  if (n && (!be || !out || !inf_out || !status_out)) return SYLOW_B200_ERR_ARG;
  if (!n) return 0;
  size_t w = g2 ? 128 : 64;
  Staging io(ctx);
  const uint8_t* dbe = io.up(be, n * w);
  uint8_t *d_pts = io.area(n * w), *d_inf = io.area(n);
  int8_t* st = reinterpret_cast<int8_t*>(io.area(n));
  CKS(io.err);
  if (g2) {
    k_decode_be<4><<<nblocks(n, 128), 128, 0, ctx->stream>>>(dbe, 128, n, mode, d_pts, d_inf, st);
    LAUNCHED(ctx);
    if (validate) {
      k_g2_validate<<<nblocks(n, SY_MUL_THREADS), SY_MUL_THREADS, 0, ctx->stream>>>(d_pts, d_inf, n, st, 1);
      LAUNCHED(ctx);
    }
  } else {
    k_decode_be<2><<<nblocks(n, 128), 128, 0, ctx->stream>>>(dbe, 64, n, mode, d_pts, d_inf, st);
    LAUNCHED(ctx);
    if (validate) {
      k_g1_validate<<<nblocks(n, 128), 128, 0, ctx->stream>>>(d_pts, d_inf, n, st, 1);
      LAUNCHED(ctx);
    }
  }
  io.down(out, d_pts, n * w);
  io.down(inf_out, d_inf, n);
  io.down(status_out, st, n);
  return io.finish();
}
int sylow_b200_g1_from_be_bytes_batch(sylow_b200_ctx* ctx, const uint8_t* be, size_t n, int eip_mode, uint8_t* g1_out,
                                      uint8_t* inf_out, int8_t* status_out) {
  return from_be(ctx, 0, be, n, eip_mode ? 1 : 0, 1, g1_out, inf_out, status_out);
}
int sylow_b200_g2_from_be_bytes_batch(sylow_b200_ctx* ctx, const uint8_t* be, size_t n, int eip_mode, uint8_t* g2_out,
                                      uint8_t* inf_out, int8_t* status_out) {
  return from_be(ctx, 1, be, n, eip_mode ? 1 : 0, 1, g2_out, inf_out, status_out);
}
static int to_be(sylow_b200_ctx* ctx, int g2, const uint8_t* pts, const uint8_t* inf, size_t n, int scrub, uint8_t* be_out) {
  ENTER(ctx);
  if (n && (!pts || !be_out)) return SYLOW_B200_ERR_ARG;
  if (!n) return 0;
  size_t w = g2 ? 128 : 64;
  Staging io(ctx);
  const uint8_t *dp = io.up(pts, n * w), *di = io.up(inf, n);
  uint8_t* d_be = io.area(n * w);
  CKS(io.err);
  if (g2)
    k_encode_be<4><<<nblocks(n, 128), 128, 0, ctx->stream>>>(dp, di, n, scrub, d_be);
  else
    k_encode_be<2><<<nblocks(n, 128), 128, 0, ctx->stream>>>(dp, di, n, scrub, d_be);
  LAUNCHED(ctx);
  io.down(be_out, d_be, n * w);
  return io.finish();
}
int sylow_b200_g1_to_be_bytes_batch(sylow_b200_ctx* ctx, const uint8_t* g1, const uint8_t* g1_inf, size_t n, int scrubbed,
                                    uint8_t* be_out) {
  return to_be(ctx, 0, g1, g1_inf, n, scrubbed, be_out);
}
int sylow_b200_g2_to_be_bytes_batch(sylow_b200_ctx* ctx, const uint8_t* g2, const uint8_t* g2_inf, size_t n, int scrubbed,
                                    uint8_t* be_out) {
  return to_be(ctx, 1, g2, g2_inf, n, scrubbed, be_out);
}

int sylow_b200_eip197_pairing_check_batch(sylow_b200_ctx* ctx, const uint8_t* input, size_t k, size_t n_checks,
                                          uint8_t* ok_out, int8_t* status_out) {
  ENTER(ctx);
  if (n_checks && (!ok_out || !status_out || (k && !input))) return SYLOW_B200_ERR_ARG;
  if (!n_checks) return 0;
  size_t n = k * n_checks;
  Staging io(ctx);
  const uint8_t* din = io.up(input, n * 192);
  uint8_t *d2 = io.area(n * 128), *d1 = io.area(n * 64), *d1i = io.area(n), *d2i = io.area(n);
  int8_t* st1 = reinterpret_cast<int8_t*>(io.area(2 * n));  // per-pair decode status of G1, then of G2
  int8_t* st2 = st1 + n;
  uint8_t* d_ok = io.area(2 * n_checks + 64);
  CKS(io.err);
  int8_t* d_st = reinterpret_cast<int8_t*>(d_ok + ((n_checks + 15) / 16) * 16);
  if (n) {
    k_decode_be<2><<<nblocks(n, 128), 128, 0, ctx->stream>>>(din, 192, n, 1, d1, d1i, st1);
    LAUNCHED(ctx);
    k_decode_be<4><<<nblocks(n, 128), 128, 0, ctx->stream>>>(din + 64, 192, n, 1, d2, d2i, st2);
    LAUNCHED(ctx);
    k_g1_validate<<<nblocks(n, 128), 128, 0, ctx->stream>>>(d1, d1i, n, st1, 1);
    LAUNCHED(ctx);
    k_g2_validate<<<nblocks(n, SY_MUL_THREADS), SY_MUL_THREADS, 0, ctx->stream>>>(d2, d2i, n, st2, 1);
    LAUNCHED(ctx);
    CKS(sylow_b200_pairing_check_batch_dev(ctx, d1, d1i, d2, d2i, k, n_checks, d_ok, nullptr));
    k_fold_status<<<nblocks(n_checks, 128), 128, 0, ctx->stream>>>(st1, st2, k, n_checks, d_ok, d_st);
    LAUNCHED(ctx);
  } else {
    CK(cudaMemsetAsync(d_ok, 1, n_checks, ctx->stream));  // empty input: success (reth_bn128.rs:173-175)
    CK(cudaMemsetAsync(d_st, 0, n_checks, ctx->stream));
  }
  io.down(ok_out, d_ok, n_checks);
  io.down(status_out, d_st, n_checks);
  return io.finish();
}

// The EIP-196 ecAdd (mul = 0: x1 || y1 || x2 || y2, 128 B) and ecMul (mul = 1: x || y || s, 96 B) bodies over n
// inputs: decode and validate the points, add or multiply, and encode.  A failed input's point decodes to (0, 1) or
// stays off the curve; the group law runs on it as on any other (complete formulas, no memory it does not own) and
// k_eip196_finish discards the result.
static int eip196_host(sylow_b200_ctx* ctx, int mul, const uint8_t* input, size_t n, uint8_t* out, int8_t* status_out) {
  const size_t stride = mul ? 96 : 128;
  if (is_multi(ctx) && input && out && status_out) {
    return multi_slices(ctx, n, [=](sylow_b200_ctx* c, size_t, size_t off, size_t m) {
      return eip196_host(c, mul, input + off * stride, m, out + off * 64, status_out + off);
    });
  }
  ENTER(ctx);
  if (n && (!input || !out || !status_out)) return SYLOW_B200_ERR_ARG;
  if (!n) return 0;
  Staging io(ctx);
  const uint8_t* din = io.up(input, n * stride);
  uint8_t *da = io.area(n * 64), *db = io.area(n * 64), *d_res = io.area(n * 64), *d_be = io.area(n * 64);
  uint8_t* flags = io.area(6 * n);  // a_inf, b_inf, res_inf, then the int8 statuses of a, b and the result
  CKS(io.err);
  uint8_t *a_inf = flags, *b_inf = flags + n, *res_inf = flags + 2 * n;
  int8_t* st_a = reinterpret_cast<int8_t*>(flags + 3 * n);
  int8_t *st_b = mul ? nullptr : st_a + n, *st = st_a + 2 * n;
  const unsigned blocks = nblocks(n, 128);
  k_decode_be<2><<<blocks, 128, 0, ctx->stream>>>(din, stride, n, 1, da, a_inf, st_a);
  LAUNCHED(ctx);
  k_g1_validate<<<blocks, 128, 0, ctx->stream>>>(da, a_inf, n, st_a, 1);
  LAUNCHED(ctx);
  if (mul) {
    k_eip196_scalars<<<blocks, 128, 0, ctx->stream>>>(din + 64, stride, n, db);
    LAUNCHED(ctx);
    CKS(sylow_b200_g1_mul_batch_dev(ctx, da, a_inf, db, n, d_res, res_inf, nullptr));
  } else {
    k_decode_be<2><<<blocks, 128, 0, ctx->stream>>>(din + 64, stride, n, 1, db, b_inf, st_b);
    LAUNCHED(ctx);
    k_g1_validate<<<blocks, 128, 0, ctx->stream>>>(db, b_inf, n, st_b, 1);
    LAUNCHED(ctx);
    CKS(add_dev(ctx, 0, da, a_inf, db, b_inf, n, 0, d_res, res_inf, nullptr));
  }
  k_eip196_finish<<<blocks, 128, 0, ctx->stream>>>(d_res, res_inf, st_a, st_b, n, d_be, st);
  LAUNCHED(ctx);
  io.down(out, d_be, n * 64);
  io.down(status_out, st, n);
  return io.finish();
}
int sylow_b200_eip196_add_batch(sylow_b200_ctx* ctx, const uint8_t* input, size_t n, uint8_t* out, int8_t* status_out) {
  return eip196_host(ctx, 0, input, n, out, status_out);
}
int sylow_b200_eip196_mul_batch(sylow_b200_ctx* ctx, const uint8_t* input, size_t n, uint8_t* out, int8_t* status_out) {
  return eip196_host(ctx, 1, input, n, out, status_out);
}

int sylow_b200_gt_mul_batch(sylow_b200_ctx* ctx, const uint8_t* gt, const uint8_t* scalars, size_t n, uint8_t* out) {
  ENTER(ctx);
  if (n && (!gt || !scalars || !out)) return SYLOW_B200_ERR_ARG;
  if (!n) return 0;
  Staging io(ctx);
  uint8_t* d_out = io.area(n * 384);
  const uint8_t *dg = io.up(gt, n * 384), *dk = io.up(scalars, n * 32);
  CKS(io.err);
  k_gt_pow<<<nblocks(n, SY_FEXP_THREADS), SY_FEXP_THREADS, 0, ctx->stream>>>(dg, dk, n, d_out);
  LAUNCHED(ctx);
  io.down(out, d_out, n * 384);
  return io.finish();
}

// ------------------------------------------------------------------------------- Expander trait
int sylow_b200_expand_message_batch(sylow_b200_ctx* ctx, const uint8_t* msgs, const uint64_t* offsets, size_t n,
                                    const uint8_t* dst, size_t dst_len, int hash_id, size_t len_in_bytes, uint8_t* out) {
  ENTER(ctx);
  DstPrime dp;
  CKS(make_dst_prime(ctx, dst, dst_len, hash_id, dp));
  // XMD: ell = ceil(len / 32) <= 255; both: len < 2^16 (hasher.rs:211-216, i2osp(len, 2))
  if (len_in_bytes == 0 || len_in_bytes > 65535) return SYLOW_B200_ERR_ARG;
  if (hash_id != SYLOW_B200_HASH_SHAKE128 && (len_in_bytes + 31) / 32 > 255) return SYLOW_B200_ERR_ARG;
  if (!n) return 0;
  if (!out) return SYLOW_B200_ERR_ARG;
  Staging io(ctx);
  uint8_t* d_out = io.area(n * len_in_bytes);
  const DevMsgs m = msgs_to_dev(io, msgs, offsets, n);
  CKS(io.err);
  k_expand_message<<<nblocks(n, 128), 128, 0, ctx->stream>>>(m.msgs, m.offsets, n, dp, (uint32_t)len_in_bytes, d_out);
  LAUNCHED(ctx);
  io.down(out, d_out, n * len_in_bytes);
  return io.finish();
}

int sylow_b200_hash_to_field_batch(sylow_b200_ctx* ctx, const uint8_t* msgs, const uint64_t* offsets, size_t n,
                                   const uint8_t* dst, size_t dst_len, int hash_id, uint8_t* out) {
  ENTER(ctx);
  DstPrime dp;
  CKS(make_dst_prime(ctx, dst, dst_len, hash_id, dp));
  if (!n) return 0;
  if (!out) return SYLOW_B200_ERR_ARG;
  Staging io(ctx);
  uint8_t* d_out = io.area(n * 64);
  const DevMsgs m = msgs_to_dev(io, msgs, offsets, n);
  CKS(io.err);
  k_hash_to_field<<<nblocks(n, 128), 128, 0, ctx->stream>>>(m.msgs, m.offsets, n, dp, d_out);
  LAUNCHED(ctx);
  io.down(out, d_out, n * 64);
  return io.finish();
}

// ------------------------------------------------------------------------------- sums / same-signer batches
int sylow_b200_g1_sum(sylow_b200_ctx* ctx, const uint8_t* pts, const uint8_t* pts_inf, size_t n, uint8_t out[64],
                      uint8_t* out_inf) {
  ENTER(ctx);
  if (!out || !out_inf || (n && !pts)) return SYLOW_B200_ERR_ARG;
  if (!n) {
    memset(out, 0, 64);
    out[32] = 1;  // GroupAffine::zero(): (0, 1, infinity)
    *out_inf = 1;
    return 0;
  }
  Staging io(ctx);
  const uint8_t *dp = io.up(pts, n * 64), *di = io.up(pts_inf, n);
  uint8_t* d_sum = io.area(128);  // point, then its flag
  CKS(io.err);
  CKS(g1_sum_reduce(ctx, dp, di, n, 0, d_sum, d_sum + 64, ctx->stream));
  io.down(out, d_sum, 64);
  io.down(out_inf, d_sum + 64, 1);
  return io.finish();
}

#define SY_MSM_BUCKET_MIN 131072
// Bucket MSM on device buffers: d_out = 64-byte affine point, d_out_inf its flag.  window_bits = 0 picks c from n.
static int g1_msm_bucket_dev(sylow_b200_ctx* ctx, const uint8_t* d_pts, const uint8_t* d_inf, const uint8_t* d_scalars,
                             size_t n, int window_bits, uint8_t* d_out, uint8_t* d_out_inf, cudaStream_t s) {
  int c = window_bits;
  if (c <= 0) {
    int lg = 0;
    while (((size_t)1 << (lg + 1)) <= n) lg++;
    c = lg - 10 < 8 ? 8 : lg - 10;  // measured optimum (tools/msm_time.py): 8 up to 2^18 points, 10 at 2^20
  }
  if (c < 4) c = 4;
  if (c > (window_bits > 0 ? 16 : 13)) c = window_bits > 0 ? 16 : 13;  // the automatic choice stops at 13 (64 digits per chunk)
  const int nw = (256 + c - 1) / c;
  const size_t nb = (size_t)nw << c;
  // scratch: counts | offsets | cursors | first item (nb u32 each), item start | length (nw * max_items u32 each), items
  // per window, index lists (nw * n u32), Montgomery points (n * 64), item sums, buckets (nb * 96), chunk partials, result
  const size_t max_items = ((size_t)1 << c) + n / SY_MSM_ITEM + 1;
  const size_t ni = (size_t)nw * max_items;
  size_t o_cnt = 0, o_off = o_cnt + nb * 4, o_cur = o_off + nb * 4, o_ifi = o_cur + nb * 4, o_ist = o_ifi + nb * 4;
  size_t o_iln = o_ist + ni * 4, o_iw = o_iln + ni * 4, o_idx = o_iw + 256;
  size_t o_pts = (o_idx + (size_t)nw * n * 4 + 255) & ~(size_t)255, o_isum = o_pts + n * 64, o_bkt = o_isum + ni * 96;
  size_t o_par = o_bkt + nb * 96, o_res = o_par + (size_t)nw * SY_MSM_CHUNKS * 96, total = o_res + 96;
  CKS(reserve(ctx, ctx->msm, total));
  uint8_t* base = ctx->msm.p;
  uint32_t* cnt = reinterpret_cast<uint32_t*>(base + o_cnt);
  uint32_t* off = reinterpret_cast<uint32_t*>(base + o_off);
  uint32_t* cur = reinterpret_cast<uint32_t*>(base + o_cur);
  uint32_t* ifi = reinterpret_cast<uint32_t*>(base + o_ifi);
  uint32_t* ist = reinterpret_cast<uint32_t*>(base + o_ist);
  uint32_t* iln = reinterpret_cast<uint32_t*>(base + o_iln);
  uint32_t* iw = reinterpret_cast<uint32_t*>(base + o_iw);
  uint32_t* idx = reinterpret_cast<uint32_t*>(base + o_idx);
  CK(cudaMemsetAsync(cnt, 0, nb * 4, s));
  k_msm_count<<<nblocks(n, 256), 256, 0, s>>>(d_scalars, d_inf, n, c, nw, cnt);
  LAUNCHED(ctx);
  k_msm_offsets<<<nblocks(nw, 32), 32, 0, s>>>(cnt, c, nw, max_items, off, cur, ifi, ist, iln, iw);
  LAUNCHED(ctx);
  k_msm_scatter<<<nblocks(n, 256), 256, 0, s>>>(d_scalars, d_inf, n, c, nw, cur, idx);
  LAUNCHED(ctx);
  k_fp_convert<<<nblocks(2 * n, 128), 128, 0, s>>>(d_pts, 2 * n, base + o_pts, 1);
  LAUNCHED(ctx);
  k_msm_item_sum<<<nblocks(ni, SY_MUL_THREADS), SY_MUL_THREADS, 0, s>>>(base + o_pts, n, nw, max_items, ist, iln, iw, idx,
                                                                       base + o_isum);
  LAUNCHED(ctx);
  k_msm_bucket_sum<<<nblocks(nb, SY_MUL_THREADS), SY_MUL_THREADS, 0, s>>>(c, nw, max_items, cnt, ifi, base + o_isum,
                                                                         base + o_bkt);
  LAUNCHED(ctx);
  k_msm_chunk_reduce<<<nblocks((size_t)nw * SY_MSM_CHUNKS, 64), 64, 0, s>>>(base + o_bkt, c, nw, base + o_par);
  LAUNCHED(ctx);
  k_msm_window_sum<<<nblocks(nw, 32), 32, 0, s>>>(base + o_par, nw);
  LAUNCHED(ctx);
  k_msm_window_final<<<1, 1, 0, s>>>(base + o_par, c, nw, base + o_res);
  LAUNCHED(ctx);
  k_g1_finish_sum<<<1, 1, 0, s>>>(base + o_res, 0, d_out, d_out_inf);
  LAUNCHED(ctx);
  return 0;
}

int sylow_b200_g1_msm_bucket(sylow_b200_ctx* ctx, const uint8_t* pts, const uint8_t* pts_inf, const uint8_t* scalars,
                             size_t n, int window_bits, uint8_t out[64], uint8_t* out_inf) {
  ENTER(ctx);
  if (!out || !out_inf || (n && (!pts || !scalars)) || window_bits < 0 || window_bits > 16) return SYLOW_B200_ERR_ARG;
  if (!n) return sylow_b200_g1_sum(ctx, nullptr, nullptr, 0, out, out_inf);
  if (n >= ((size_t)1 << 31)) return SYLOW_B200_ERR_ARG;
  Staging io(ctx);
  const uint8_t *dp = io.up(pts, n * 64), *dk = io.up(scalars, n * 32), *di = io.up(pts_inf, n);
  uint8_t* d_sum = io.area(128);  // point, then its flag
  CKS(io.err);
  CKS(g1_msm_bucket_dev(ctx, dp, di, dk, n, window_bits, d_sum, d_sum + 64, ctx->stream));
  io.down(out, d_sum, 64);
  io.down(out_inf, d_sum + 64, 1);
  return io.finish();
}

int sylow_b200_g1_msm(sylow_b200_ctx* ctx, const uint8_t* pts, const uint8_t* pts_inf, const uint8_t* scalars, size_t n,
                      uint8_t out[64], uint8_t* out_inf) {
  ENTER(ctx);
  if (!out || !out_inf || (n && (!pts || !scalars))) return SYLOW_B200_ERR_ARG;
  if (!n) return sylow_b200_g1_sum(ctx, nullptr, nullptr, 0, out, out_inf);
  // from 2^17 points on the bucket method beats n GLV ladders + tree sum (tools/msm_time.py)
  if (n >= SY_MSM_BUCKET_MIN && n < ((size_t)1 << 31))
    return sylow_b200_g1_msm_bucket(ctx, pts, pts_inf, scalars, n, 0, out, out_inf);
  Staging io(ctx);
  uint8_t* d_kp = io.area(n * 65);  // k_i P_i, then their flags
  const uint8_t *dp = io.up(pts, n * 64), *dk = io.up(scalars, n * 32), *di = io.up(pts_inf, n);
  uint8_t* d_sum = io.area(128);
  CKS(io.err);
  CKS(sylow_b200_g1_mul_batch_dev(ctx, dp, di, dk, n, d_kp, d_kp + n * 64, nullptr));
  CKS(g1_sum_reduce(ctx, d_kp, d_kp + n * 64, n, 0, d_sum, d_sum + 64, ctx->stream));
  io.down(out, d_sum, 64);
  io.down(out_inf, d_sum + 64, 1);
  return io.finish();
}

int sylow_b200_lagrange_coefficients_batch(sylow_b200_ctx* ctx, const uint64_t* ids, size_t n_sets, size_t t,
                                           uint8_t* out) {
  ENTER(ctx);
  if ((n_sets && t) && (!ids || !out)) return SYLOW_B200_ERR_ARG;
  size_t n = n_sets * t;
  if (!n) return 0;
  Staging io(ctx);
  uint8_t* d_lam = io.area(n * 32);
  const uint64_t* d_ids = reinterpret_cast<const uint64_t*>(io.up(ids, n * 8));
  CKS(io.err);
  k_lagrange<<<nblocks(n, 128), 128, 0, ctx->stream>>>(d_ids, n_sets, t, d_lam);
  LAUNCHED(ctx);
  io.down(out, d_lam, n * 32);
  return io.finish();
}

int sylow_b200_threshold_aggregate_batch(sylow_b200_ctx* ctx, const uint64_t* ids, const uint8_t* sigs,
                                         const uint8_t* sigs_inf, size_t n_sets, size_t t, uint8_t* out,
                                         uint8_t* out_inf) {
  ENTER(ctx);
  if (n_sets && (!out || !out_inf || (t && (!ids || !sigs)))) return SYLOW_B200_ERR_ARG;
  if (!n_sets) return 0;
  if (!t) {  // the empty sum: GroupProjective::default() = infinity, encoded (0, 1) + flag
    for (size_t s = 0; s < n_sets; s++) {
      memset(out + s * 64, 0, 64);
      out[s * 64 + 32] = 1;
      out_inf[s] = 1;
    }
    return 0;
  }
  size_t n = n_sets * t;
  Staging io(ctx);
  uint8_t* d_shares = io.area(n * 96);  // lambda_i sig_i, projective
  const uint8_t *d_sigs = io.up(sigs, n * 64), *d_ids = io.up(ids, n * 8), *d_inf = io.up(sigs_inf, n);
  uint8_t* d_agg = io.area(n_sets * 65);  // the n_sets points, then their flags
  CKS(io.err);
  k_lagrange_mul<<<nblocks(n, SY_MUL_THREADS), SY_MUL_THREADS, 0, ctx->stream>>>(
      reinterpret_cast<const uint64_t*>(d_ids), d_sigs, d_inf, n_sets, t, d_shares);
  LAUNCHED(ctx);
  k_g1_segment_sum<<<nblocks(n_sets, 4), 128, 0, ctx->stream>>>(d_shares, n_sets, t, d_agg, d_agg + n_sets * 64);
  LAUNCHED(ctx);
  io.down(out, d_agg, n_sets * 64);
  io.down(out_inf, d_agg + n_sets * 64, n_sets);
  return io.finish();
}

int sylow_b200_verify_batch_same_signer(sylow_b200_ctx* ctx, const uint8_t* pk, int pk_inf, const uint8_t* msgs,
                                        const uint64_t* offsets, const uint8_t* sigs, const uint8_t* sigs_inf, size_t n,
                                        const uint8_t* dst, size_t dst_len, int hash_id, const uint8_t* weight_seed,
                                        int* ok) {
  ENTER(ctx);
  if (!ok) return SYLOW_B200_ERR_ARG;
  DstPrime dp;
  CKS(make_dst_prime(ctx, dst, dst_len, hash_id, dp));
  if (!n) {
    *ok = 1;
    return 0;
  }
  if (!pk || !sigs) return SYLOW_B200_ERR_ARG;
  WeightSeed ws;
  const bool weighted = load_seed(weight_seed, ws);
  uint8_t h_ok = 0;
  Staging io(ctx);
  uint8_t* d_hm = io.area(n * 65);  // H(m_i), then their flags
  const uint8_t* dsg = io.up(sigs, n * 64);
  const DevMsgs m = msgs_to_dev(io, msgs, offsets, n);
  const uint8_t *dsgi = io.up(sigs_inf, n), *dpk = io.up(pk, 128);
  // e(sum r_i sig_i, G2gen) * e(-sum r_i H(m_i), pk) == 1 (r_i = 1 without a seed): two Miller loops for the whole batch
  uint8_t* d_pairs = io.area(1024);     // two G1 points (128 B) + two flags at +128 + the G2 pair at +256
  CKS(io.err);
  uint8_t* d_flags = d_pairs + 128;
  uint8_t* d_g2 = d_pairs + 256;        // G2gen || pk
  uint8_t* d_g2_inf = d_pairs + 520;    // 0, pk_inf
  uint8_t* d_ok = d_pairs + 512;
  cudaStream_t st_ = ctx->stream;
  CKS(hash_launch(ctx, m.msgs, m.offsets, n, dp, 0, d_hm, d_hm + n * 64, st_));
  if (weighted) {
    CKS(reserve(ctx, ctx->proj, n * 96));
    k_g1_mul_weight<<<nblocks(n, SY_MUL_THREADS), SY_MUL_THREADS, 0, st_>>>(dsg, dsgi, ws, 0, n, ctx->proj.p);
    LAUNCHED(ctx);
    CKS(g1_sum_reduce(ctx, ctx->proj.p, nullptr, n, 0, d_pairs, d_flags, st_, 0));
    k_g1_mul_weight<<<nblocks(n, SY_MUL_THREADS), SY_MUL_THREADS, 0, st_>>>(d_hm, d_hm + n * 64, ws, 0, n, ctx->proj.p);
    LAUNCHED(ctx);
    CKS(g1_sum_reduce(ctx, ctx->proj.p, nullptr, n, 1, d_pairs + 64, d_flags + 1, st_, 0));
  } else {
    CKS(g1_sum_reduce(ctx, dsg, dsgi, n, 0, d_pairs, d_flags, st_));
    CKS(g1_sum_reduce(ctx, d_hm, d_hm + n * 64, n, 1, d_pairs + 64, d_flags + 1, st_));
  }
  const uint8_t h_g2_inf[2] = {0, (uint8_t)(pk_inf ? 1 : 0)};
  CK(cudaMemcpyAsync(d_g2, kG2GenWords, 128, cudaMemcpyHostToDevice, st_));
  CK(cudaMemcpyAsync(d_g2 + 128, dpk, 128, cudaMemcpyDeviceToDevice, st_));
  CK(cudaMemcpyAsync(d_g2_inf, h_g2_inf, 2, cudaMemcpyHostToDevice, st_));
  CKS(sylow_b200_pairing_check_batch_dev(ctx, d_pairs, d_flags, d_g2, d_g2_inf, 2, 1, d_ok, nullptr));
  io.down(&h_ok, d_ok, 1);
  int st = check_hash_fail(io);
  *ok = h_ok;
  return st;
}

// ------------------------------------------------------------------------------- diagnostics
int sylow_b200_batch_weights(sylow_b200_ctx* ctx, const uint8_t* weight_seed, uint64_t first_index, size_t n,
                             uint64_t* out) {
  ENTER(ctx);
  if (!weight_seed || (n && !out)) return SYLOW_B200_ERR_ARG;
  if (!n) return 0;
  WeightSeed ws;
  load_seed(weight_seed, ws);
  Staging io(ctx);
  uint64_t* d_w = reinterpret_cast<uint64_t*>(io.area(n * 8));
  CKS(io.err);
  k_batch_weights<<<nblocks(n, 128), 128, 0, ctx->stream>>>(ws, first_index, n, d_w);
  LAUNCHED(ctx);
  io.down(out, d_w, n * 8);
  return io.finish();
}

int sylow_b200_fp_op_batch(sylow_b200_ctx* ctx, int op, const uint8_t* a, const uint8_t* b, size_t n, uint8_t* out) {
  ENTER(ctx);
  if (n && (!a || !b || !out)) return SYLOW_B200_ERR_ARG;
  if (!n) return 0;
  Staging io(ctx);
  const uint8_t *da = io.up(a, n * 32), *db = io.up(b, n * 32);
  uint8_t* d_out = io.area(n * 32);
  CKS(io.err);
  k_fp_op<<<nblocks(n, 128), 128, 0, ctx->stream>>>(op, da, db, n, d_out);
  LAUNCHED(ctx);
  io.down(out, d_out, n * 32);
  return io.finish();
}

int sylow_b200_fp12_op_batch(sylow_b200_ctx* ctx, int op, const uint8_t* a, const uint8_t* b, size_t n, uint8_t* out) {
  ENTER(ctx);
  if (n && (!a || !b || !out)) return SYLOW_B200_ERR_ARG;
  if (!n) return 0;
  Staging io(ctx);
  const uint8_t *da = io.up(a, n * 384), *db = io.up(b, n * 384);
  uint8_t* d_out = io.area(n * 384);
  CKS(io.err);
  k_fp12_op<<<nblocks(n, SY_SMALL_THREADS), SY_SMALL_THREADS, 0, ctx->stream>>>(op, da, db, n, d_out);
  LAUNCHED(ctx);
  io.down(out, d_out, n * 384);
  return io.finish();
}


int sylow_b200_imad_probe(sylow_b200_ctx* ctx, int variant, int blocks, int threads, int iters, float* ms_out,
                          double* ops_out) {
  ENTER(ctx);
  if (!ms_out || !ops_out || blocks <= 0 || threads <= 0 || threads > 1024 || iters <= 0) return SYLOW_B200_ERR_ARG;
  Staging io(ctx);
  uint8_t* d_words = io.area(256);
  CKS(io.err);
  CK(cudaMemsetAsync(d_words, 0x5a, 256, ctx->stream));
  struct Event {
    cudaEvent_t e = nullptr;
    ~Event() {
      if (e) cudaEventDestroy(e);
    }
  } e0, e1;  // released on every return
  CK(cudaEventCreate(&e0.e));
  CK(cudaEventCreate(&e1.e));
  const uint32_t* src = reinterpret_cast<const uint32_t*>(d_words);
  uint32_t* sink = reinterpret_cast<uint32_t*>(d_words) + 32;
  double per_thread_iter = 0;
  for (int rep = 0; rep < 2; rep++) {  // the first pass warms up
    CK(cudaEventRecord(e0.e, ctx->stream));
    switch (variant) {
      case 0: k_imad_probe<1><<<blocks, threads, 0, ctx->stream>>>(iters, src, sink); per_thread_iter = 1; break;
      case 1: k_imad_probe<2><<<blocks, threads, 0, ctx->stream>>>(iters, src, sink); per_thread_iter = 2; break;
      case 2: k_imad_probe<4><<<blocks, threads, 0, ctx->stream>>>(iters, src, sink); per_thread_iter = 4; break;
      case 10: k_pipe_probe<0><<<blocks, threads, 0, ctx->stream>>>(iters, src, sink); per_thread_iter = 64; break;
      case 11: k_pipe_probe<1><<<blocks, threads, 0, ctx->stream>>>(iters, src, sink); per_thread_iter = 64; break;
      case 12: k_pipe_probe<2><<<blocks, threads, 0, ctx->stream>>>(iters, src, sink); per_thread_iter = 64; break;
      case 13: k_dfma_probe<<<blocks, threads, 0, ctx->stream>>>(iters, src, sink); per_thread_iter = 64; break;
      default: return SYLOW_B200_ERR_ARG;
    }
    LAUNCHED(ctx);
    CK(cudaEventRecord(e1.e, ctx->stream));
    CK(cudaEventSynchronize(e1.e));
  }
  CK(cudaEventElapsedTime(ms_out, e0.e, e1.e));
  *ops_out = (double)blocks * threads * (double)iters * per_thread_iter;
  return io.finish();
}

}  // extern "C"

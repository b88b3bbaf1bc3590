/* sylow_b200.h - C ABI of libsylow_b200.so, the B200-native batched BN254 engine.
 *
 * This is the drop-in boundary for sylow's data-parallel hot path.  sylow itself has no FFI
 * (#![deny(unsafe_code)], /root/reference/src/lib.rs:63); these entry points are what a
 * `sylow-cuda-sys` crate binds (INTEGRATION.md) so that a sylow fork can add `pairing_batch`,
 * `verify_batch`, `g1_mul_batch`, ... next to the functions they batch.  Each entry cites the
 * reference interface it replaces.
 *
 * Wire formats (all host or device buffers are caller-owned, contiguous, AoS):
 *   Fp        32 B   little-endian canonical integer in [0, p)  == Fp::value().to_words()  (fp.rs:232-234)
 *   G1 affine 64 B   x || y                                     (groups/group.rs:174-181)
 *   G2 affine 128 B  x.c0 || x.c1 || y.c0 || y.c1
 *   Fp12 / Gt 384 B  12 Fp in tower order c0.c0.c0, c0.c0.c1, ..., c1.c2.c1   (fp12.rs:561-574)
 *   scalar    32 B   little-endian integer < 2^256 (sylow passes an Fp-range value, group.rs:639-649)
 *   infinity  parallel uint8 flag array (mirrors `infinity: Choice`); NULL = no point is infinite.
 *
 * Conventions: return 0 on success, a negative sylow_b200_status otherwise; never aborts; no
 * callee-allocated memory is returned; a context is used by one call at a time.  A context made by
 * sylow_b200_create is bound to ONE CUDA device; one made by sylow_b200_create_multi owns one such
 * context per listed device and shards every batched host-pointer call as contiguous slices, one host
 * thread per GPU, combining the 384-byte Miller partial products of the product forms on the first
 * device (SURVEY.md 8e) - results are bit-identical to the single-device call.  (One process per GPU
 * works too: shard the batch yourself and combine partials with sylow_b200_fp12_product /
 * sylow_b200_verify_batch_finish; bench.py does that over torch.distributed.)  Host-pointer entry
 * points are synchronous (results are in host memory on return).  The `_dev` entry points take
 * DEVICE pointers (16-byte aligned) of a single-device context and enqueue on `stream` (a
 * cudaStream_t passed as void*; NULL = the context's own stream) without synchronising - this is what
 * bench.py times with inputs resident in HBM.  All `_dev` calls on one context share its scratch
 * buffers: enqueue them on ONE stream (or order the streams yourself); the library does not
 * serialise calls issued on different streams.  There is no CPU fallback: every entry point fails
 * with SYLOW_B200_ERR_CUDA if no device is usable.
 *
 * Points are NOT validated by the pairing / BLS entry points (sylow's typed API cannot hold an invalid
 * point; raw bytes can): run sylow_b200_g1_validate_batch / sylow_b200_g2_validate_batch on untrusted
 * input first.  An off-curve or off-subgroup input gives an unspecified (but memory-safe) result.
 */
#ifndef SYLOW_B200_H
#define SYLOW_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct sylow_b200_ctx sylow_b200_ctx;

typedef enum {
  SYLOW_B200_OK = 0,
  SYLOW_B200_ERR_ARG = -1,            /* NULL pointer, bad size, unsupported hash id or shape */
  SYLOW_B200_ERR_CUDA = -2,           /* CUDA runtime error (see sylow_b200_last_cuda_error) */
  SYLOW_B200_ERR_NOT_ON_CURVE = -3,   /* GroupError::NotOnCurve      (groups/group.rs:37-47) */
  SYLOW_B200_ERR_NOT_IN_SUBGROUP = -4,/* GroupError::NotInSubgroup */
  SYLOW_B200_ERR_CANNOT_HASH = -5,    /* GroupError::CannotHashToGroup */
  SYLOW_B200_ERR_DECODE = -6,         /* GroupError::DecodeError: a coordinate >= p */
  SYLOW_B200_ERR_NOMEM = -7
} sylow_b200_status;

#define SYLOW_B200_HASH_KECCAK256 0   /* XMDExpander::<Keccak256>, lib.rs:181,225 */
#define SYLOW_B200_HASH_SHA256 1      /* XMDExpander::<Sha256>, the digest of the reference's RFC 9380 vectors */
#define SYLOW_B200_HASH_SHAKE128 2    /* XOFExpander::<Shake128> (hasher.rs:258-330), security parameter k = 128 */

/* Context: owns its streams and growable device staging buffers on `device_id`. */
int sylow_b200_create(sylow_b200_ctx** out, int device_id);
/* Multi-device context over device_ids[0 .. n_devices) (SURVEY.md 8b): every batched host-pointer entry point shards
 * its batch over the devices; entry points without a sharded form run on device_ids[0].  The same device may be
 * listed more than once (two slices then share that GPU). */
int sylow_b200_create_multi(sylow_b200_ctx** out, const int* device_ids, int n_devices);
/* Number of devices of a context (1 for sylow_b200_create) and the single-device context of device slot i, which the
 * `_dev` entry points need (owned by the parent: do not destroy it). */
int sylow_b200_device_count(const sylow_b200_ctx* ctx);
sylow_b200_ctx* sylow_b200_device_ctx(sylow_b200_ctx* ctx, int i);
int sylow_b200_destroy(sylow_b200_ctx* ctx);
const char* sylow_b200_strerror(int status);
/* cudaError_t of the last failing CUDA call on this context (0 if none). */
int sylow_b200_last_cuda_error(const sylow_b200_ctx* ctx);
/* Number of kernels this context has launched since creation (bench.py's gpu_launches). */
uint64_t sylow_b200_launch_count(const sylow_b200_ctx* ctx);

/* ---- pairing --------------------------------------------------------------------------------- */

/* n independent pairings, gt_out[i] = e(g1[i], g2[i]); an infinite input gives Gt::identity().
 * Replaces a loop over `pairing(&G1Projective, &G2Projective) -> Gt`  (pairing.rs:870-893).
 * Launch shape (same bits either way): one thread per pairing in whole waves of the GPU; batches of at most
 * 148 x 128 pairs, and the remainder of a larger batch after its whole waves, run on two cooperating lanes per
 * pairing (csrc/pairing_lanes.cuh) - about 5 ms for 1 .. 9 472 pairings instead of 8.5 ms.  The environment variable
 * SYLOW_B200_LANES (0: one thread per pairing only, 2: two lanes always) overrides the choice for measurements. */
int sylow_b200_pairing_batch(sylow_b200_ctx* ctx, const uint8_t* g1, const uint8_t* g1_inf, const uint8_t* g2,
                             const uint8_t* g2_inf, size_t n, uint8_t* gt_out /* n*384 */);

/* n independent Miller loops, f_out[i] = G2Affine::precompute(g2[i]).miller_loop(g1[i]), canonical
 * Fp12 (pairing.rs:676-708 composed with :590-619, bit-identical MillerLoopResult).  Infinite pairs give 1. */
int sylow_b200_miller_loop_batch(sylow_b200_ctx* ctx, const uint8_t* g1, const uint8_t* g1_inf, const uint8_t* g2,
                                 const uint8_t* g2_inf, size_t n, uint8_t* f_out /* n*384 */);

/* prod_i miller_loop(g2[i], g1[i]) == glued_miller_loop(&[G2PreComputed], &[G1Affine])  (pairing.rs:970-1022;
 * equal bit-for-bit because Fp12 multiplication is exact and commutative, SURVEY.md 3.2).  Infinite pairs
 * are skipped (contribute 1) - the reference's behaviour there is unpinned (SURVEY Q7).  n = 0 gives 1. */
int sylow_b200_miller_product(sylow_b200_ctx* ctx, const uint8_t* g1, const uint8_t* g1_inf, const uint8_t* g2,
                              const uint8_t* g2_inf, size_t n, uint8_t f_out[384]);

/* gt_out[i] = MillerLoopResult::final_exponentiation(f[i])  (pairing.rs:245-492). */
int sylow_b200_final_exp_batch(sylow_b200_ctx* ctx, const uint8_t* f, size_t n, uint8_t* gt_out /* n*384 */);

/* out = prod_i f[i] in Fp12 (n = 0 gives 1).  Combines per-GPU Miller partial products (the
 * `MulAssign for MillerLoopResult` of pairing.rs:63-68). */
int sylow_b200_fp12_product(sylow_b200_ctx* ctx, const uint8_t* f, size_t n, uint8_t out[384]);

/* n_checks independent product checks of pairs_per_check pairs each:
 * ok_out[c] = (glued_pairing(g1s_c, g2s_c) == Gt::identity())  (pairing.rs:1029-1037; the ecPairing
 * shape of examples/reth_bn128.rs:211-214).  Pair j of check c is element c*pairs_per_check + j.
 * pairs_per_check = 0: every check is the empty product, the identity, so every ok_out[c] is 1 (g1 and g2 may then be
 * NULL; no kernel runs). */
int sylow_b200_pairing_check_batch(sylow_b200_ctx* ctx, const uint8_t* g1, const uint8_t* g1_inf, const uint8_t* g2,
                                   const uint8_t* g2_inf, size_t pairs_per_check, size_t n_checks, uint8_t* ok_out);

/* Pairing checks with a pair count per check: ok_out[c] = (glued_pairing(pairs [offsets[c], offsets[c+1])) ==
 * Gt::identity()).  offsets: n_checks + 1 non-decreasing uint64 values, as for the message offsets of the hashing calls
 * (offsets[0] need not be 0; g1 / g2 / the flags hold offsets[n_checks] pairs).  An empty check is the identity
 * (ok = 1).  Infinite pairs are skipped, as in pairing_check_batch.  Decreasing offsets: SYLOW_B200_ERR_ARG.
 * One set of launches for the whole batch: each check of k pairs runs as k / G glued Miller loops of G = 1, 2 or 4
 * pairs (G chosen once per batch from the total pair count, as for verify_batch) plus one 2-pair and / or one 1-pair
 * loop for its remainder; the values of a check are multiplied in chunks of at most 32 per thread, level by level,
 * then one final exponentiation per check.  A multi-device context cuts the batch at check boundaries into slices of
 * about equal pair counts.  SYLOW_B200_RAGGED_GLUE (1, 2 or 4) fixes G for measurements. */
int sylow_b200_pairing_check_ragged_batch(sylow_b200_ctx* ctx, const uint8_t* g1, const uint8_t* g1_inf,
                                          const uint8_t* g2, const uint8_t* g2_inf, const uint64_t* offsets,
                                          size_t n_checks, uint8_t* ok_out);

/* ---- precomputed G2 (G2PreComputed) --------------------------------------------------------------- */

/* coeffs_out[i] = G2Affine::precompute(g2[i]) (pairing.rs:676-708): the 87 line-coefficient triples
 * Ell(c0, c1, c2), 3 x Fp2 = 192 B each, 16704 B per point, canonical, bit-identical to the reference's
 * G2PreComputed::coeffs. */
int sylow_b200_g2_precompute(sylow_b200_ctx* ctx, const uint8_t* g2, size_t n, uint8_t* coeffs_out /* n*16704 */);

/* f_out[i] = G2PreComputed::miller_loop(g1[i]) (pairing.rs:590-619) for ONE precomputed G2 point against n G1
 * points; the table is staged in shared memory and broadcast to the threads.  Infinite G1 gives 1. */
int sylow_b200_miller_loop_precomputed(sylow_b200_ctx* ctx, const uint8_t* coeffs /* 16704 */, const uint8_t* g1,
                                       const uint8_t* g1_inf, size_t n, uint8_t* f_out /* n*384 */);

/* Product checks where the LAST k_fixed pairs of every check use the same k_fixed G2 points for all checks
 * (Groth16: e(A,B) e(-alpha,beta) e(-L,gamma) e(-C,delta) == 1 with beta, gamma, delta fixed).  g1 holds
 * k_var + k_fixed points per check (variable pairs first), g2_var k_var points per check, coeffs_fixed the
 * k_fixed tables from sylow_b200_g2_precompute.  One multi-Miller loop with a shared squaring per check
 * (glued_miller_loop, pairing.rs:970-1022) + one final exponentiation.  Supported shapes (k_var, k_fixed):
 * (1,1), (1,3), (0,1); anything else returns SYLOW_B200_ERR_ARG (use sylow_b200_pairing_check_batch). */
int sylow_b200_pairing_check_fixed_batch(sylow_b200_ctx* ctx, const uint8_t* g1, const uint8_t* g1_inf,
                                         const uint8_t* g2_var, const uint8_t* g2_var_inf, size_t k_var,
                                         const uint8_t* coeffs_fixed, size_t k_fixed, size_t n_checks, uint8_t* ok_out);

/* One table PER PAIR (sylow_b200_miller_loop_precomputed uses one table for all pairs): pair i is g1[i] against the
 * canonical table coeffs[i*16704 ..] (sylow_b200_g2_precompute output).  A table has no infinity form: drop such pairs
 * or flag them on the G1 side.  These two host entry points move 16.7 KB per pair over the host link; they are there
 * for API parity and moderate batches.  The throughput path keeps the tables resident in device memory
 * (sylow_b200_g2_precompute_dev + sylow_b200_miller_product_precomputed_dev).
 * _batch: f_out[i] = G2PreComputed::miller_loop(g1[i]) (pairing.rs:590-619), canonical; infinite G1 gives 1.
 * product: glued_miller_loop(&[G2PreComputed], &[G1Affine]) (pairing.rs:970-1022), bit-identical to
 *   sylow_b200_miller_product on the same points; infinite G1 pairs are skipped, n = 0 gives 1. */
int sylow_b200_miller_loop_precomputed_batch(sylow_b200_ctx* ctx, const uint8_t* coeffs /* n*16704 */,
                                             const uint8_t* g1, const uint8_t* g1_inf, size_t n,
                                             uint8_t* f_out /* n*384 */);
int sylow_b200_miller_product_precomputed(sylow_b200_ctx* ctx, const uint8_t* coeffs /* n*16704 */, const uint8_t* g1,
                                          const uint8_t* g1_inf, size_t n, uint8_t f_out[384]);

/* ---- input validation (untrusted batches: precompile calldata, aggregated signatures) ------------- */

/* status_out[i] = 0 if g1[i] is a valid point, SYLOW_B200_ERR_DECODE if a coordinate is >= p
 * (Fp::from_be_bytes' range check, fp.rs:686-719), SYLOW_B200_ERR_NOT_ON_CURVE if y^2 != x^3 + 3
 * (G1Affine::new, g1.rs:111-132).  Flagged-infinite points are valid.  The call itself returns 0. */
int sylow_b200_g1_validate_batch(sylow_b200_ctx* ctx, const uint8_t* g1, const uint8_t* g1_inf, size_t n,
                                 int8_t* status_out);
/* As above for G2 plus SYLOW_B200_ERR_NOT_IN_SUBGROUP when (x+1)Q + psi(xQ) + psi^2(xQ) != psi^3(2xQ)
 * (G2Affine::new_unchecked g2.rs:279-297, G2Projective::new g2.rs:460-525). */
int sylow_b200_g2_validate_batch(sylow_b200_ctx* ctx, const uint8_t* g2, const uint8_t* g2_inf, size_t n,
                                 int8_t* status_out);

/* ---- big-endian wire codecs ------------------------------------------------------------------------ */

/* G1Affine::from_be_bytes (g1.rs:151-280) / G2Affine::from_be_bytes (g2.rs:361-433) over a batch: 64 / 128
 * big-endian bytes per point (G2: imaginary parts first, g2.rs:325-328) -> wire form, infinity flags and a
 * status per point (0, SYLOW_B200_ERR_DECODE, _NOT_ON_CURVE, _NOT_IN_SUBGROUP); invalid points decode to
 * (0, 1).  eip_mode = 0: sylow's codec (bit 7 of byte 0 flags infinity, which must be x = 0, y = 1);
 * eip_mode = 1: EIP-196/197 (all-zero = infinity, no flag bit; examples/reth_bn128.rs:118-126,187-194). */
int sylow_b200_g1_from_be_bytes_batch(sylow_b200_ctx* ctx, const uint8_t* be /* n*64 */, size_t n, int eip_mode,
                                      uint8_t* g1_out, uint8_t* inf_out, int8_t* status_out);
int sylow_b200_g2_from_be_bytes_batch(sylow_b200_ctx* ctx, const uint8_t* be /* n*128 */, size_t n, int eip_mode,
                                      uint8_t* g2_out, uint8_t* inf_out, int8_t* status_out);
/* to_be_bytes / to_be_bytes_scrubbed (g1.rs:136-160, g2.rs:319-333). */
int sylow_b200_g1_to_be_bytes_batch(sylow_b200_ctx* ctx, const uint8_t* g1, const uint8_t* g1_inf, size_t n, int scrubbed,
                                    uint8_t* be_out /* n*64 */);
int sylow_b200_g2_to_be_bytes_batch(sylow_b200_ctx* ctx, const uint8_t* g2, const uint8_t* g2_inf, size_t n, int scrubbed,
                                    uint8_t* be_out /* n*128 */);
/* The EIP-197 ecPairing precompile body (examples/reth_bn128.rs:156-217) for n_checks inputs of k pairs each
 * (k * 192 big-endian bytes per input): decode, validate (field range, curve, G2 subgroup), glued_pairing ==
 * identity.  ok_out[c] = 1/0; status_out[c] = 0 or the first decode/validation error of input c (then ok = 0). */
int sylow_b200_eip197_pairing_check_batch(sylow_b200_ctx* ctx, const uint8_t* input, size_t k, size_t n_checks,
                                          uint8_t* ok_out, int8_t* status_out);
/* EIP-197 over n_checks inputs of any length: input c = input[offsets[c] .. offsets[c+1]) (byte offsets, non-decreasing,
 * offsets[0] need not be 0).  A length that is a multiple of 192: decode, validate and check, as in
 * sylow_b200_eip197_pairing_check_batch; an empty input succeeds.  A length that is not: ok = 0 and status =
 * SYLOW_B200_ERR_ARG, and none of its bytes are decoded.  The call itself returns 0 (SYLOW_B200_ERR_ARG for decreasing
 * offsets).  Runs as sylow_b200_pairing_check_ragged_batch, sharded the same way on a multi-device context. */
int sylow_b200_eip197_pairing_check_ragged_batch(sylow_b200_ctx* ctx, const uint8_t* input, const uint64_t* offsets,
                                                 size_t n_checks, uint8_t* ok_out, int8_t* status_out);

/* The EIP-196 precompile bodies (examples/reth_bn128.rs, the adapter ahead of the ecPairing body at :156-217) over
 * n fixed-size inputs.  The caller zero-pads short calldata and truncates long calldata, as the EVM does.
 * add: input i = x1 || y1 || x2 || y2 (128 B big-endian);  mul: input i = x || y || s (96 B; s any 256-bit integer).
 * out[i] = 64 B big-endian result; the point at infinity is all-zero (input and output).
 * status_out[i] = 0, SYLOW_B200_ERR_DECODE (a coordinate >= p) or SYLOW_B200_ERR_NOT_ON_CURVE;
 * a failed input gives out[i] = 64 zero bytes.  The call itself returns 0. */
int sylow_b200_eip196_add_batch(sylow_b200_ctx* ctx, const uint8_t* input /* n*128 */, size_t n, uint8_t* out /* n*64 */,
                                int8_t* status_out);
int sylow_b200_eip196_mul_batch(sylow_b200_ctx* ctx, const uint8_t* input /* n*96 */, size_t n, uint8_t* out /* n*64 */,
                                int8_t* status_out);

/* ---- group law --------------------------------------------------------------------------------- */

/* out[i] = affine(a[i] + b[i]), or affine(a[i] - b[i]) when subtract != 0 (group.rs:528-624, :475-495).
 * Complete: equal, opposite and infinite operands are ordinary inputs.  a_inf, b_inf and out_inf may be NULL. */
int sylow_b200_g1_add_batch(sylow_b200_ctx* ctx, const uint8_t* a /* n*64 */, const uint8_t* a_inf,
                            const uint8_t* b /* n*64 */, const uint8_t* b_inf, size_t n, int subtract,
                            uint8_t* out /* n*64 */, uint8_t* out_inf);
int sylow_b200_g2_add_batch(sylow_b200_ctx* ctx, const uint8_t* a /* n*128 */, const uint8_t* a_inf,
                            const uint8_t* b /* n*128 */, const uint8_t* b_inf, size_t n, int subtract,
                            uint8_t* out /* n*128 */, uint8_t* out_inf);

/* ---- scalar multiplication --------------------------------------------------------------------- */

/* out[i] = affine(scalars[i] * pts[i]);  replaces `&G1Projective * &Fp` + GroupAffine::from
 * (groups/group.rs:639-667, :475-495).  out_inf may be NULL. */
int sylow_b200_g1_mul_batch(sylow_b200_ctx* ctx, const uint8_t* pts /* n*64 */, const uint8_t* pts_inf,
                            const uint8_t* scalars /* n*32 */, size_t n, uint8_t* out /* n*64 */, uint8_t* out_inf);
int sylow_b200_g2_mul_batch(sylow_b200_ctx* ctx, const uint8_t* pts /* n*128 */, const uint8_t* pts_inf,
                            const uint8_t* scalars /* n*32 */, size_t n, uint8_t* out /* n*128 */, uint8_t* out_inf);

/* out[i] = affine(scalars[i] * G) for the G1 / G2 generator: the same bytes as g1_mul_batch / g2_mul_batch on the
 * repeated generator (`G1Projective::generator() * &k`; KeyPair::generate's pk, lib.rs:105-137).  A fixed-base table
 * of the generator, built on the device on a context's first such call, replaces the ladder.  out_inf may be NULL. */
int sylow_b200_g1_mul_generator_batch(sylow_b200_ctx* ctx, const uint8_t* scalars /* n*32 */, size_t n,
                                      uint8_t* out /* n*64 */, uint8_t* out_inf);
int sylow_b200_g2_mul_generator_batch(sylow_b200_ctx* ctx, const uint8_t* scalars /* n*32 */, size_t n,
                                      uint8_t* out /* n*128 */, uint8_t* out_inf);

/* out[i] = gt[i] * scalars[i] in sylow's additive notation, i.e. gt[i]^scalars[i] in Fp12  (`&Gt * &Fr`,
 * groups/gt.rs:188-215).  gt[i] must be a Gt value (a final-exponentiation output: cyclotomic subgroup). */
int sylow_b200_gt_mul_batch(sylow_b200_ctx* ctx, const uint8_t* gt /* n*384 */, const uint8_t* scalars /* n*32 */,
                            size_t n, uint8_t* out /* n*384 */);

/* out = sum_i pts[i] (affine + infinity flag): signature aggregation.  sylow_b200_g1_msm = sum_i scalars[i] * pts[i]
 * (Lagrange-weighted aggregation of examples/dkg.rs:190-236) as a batch of ladders plus the same tree sum - a
 * batch of GLV ladders plus the same tree sum below 2^17 points, the bucket method (sylow_b200_g1_msm_bucket) above. */
int sylow_b200_g1_sum(sylow_b200_ctx* ctx, const uint8_t* pts /* n*64 */, const uint8_t* pts_inf, size_t n,
                      uint8_t out[64], uint8_t* out_inf);
int sylow_b200_g1_msm(sylow_b200_ctx* ctx, const uint8_t* pts /* n*64 */, const uint8_t* pts_inf,
                      const uint8_t* scalars /* n*32 */, size_t n, uint8_t out[64], uint8_t* out_inf);
/* The same sum by the bucket (Pippenger) method: counting sort of the points by (window, digit), one thread per bucket,
 * running sums per window, Horner over the windows.  window_bits = 0 chooses max(8, log2(n) - 10); buckets are cut
 * into work items of at most 256 points, so skewed digits (equal scalars, the short top window) do not serialise.
 * sylow_b200_g1_msm switches to it from 2^17 points on; any 256-bit scalar, infinite points are skipped. */
int sylow_b200_g1_msm_bucket(sylow_b200_ctx* ctx, const uint8_t* pts /* n*64 */, const uint8_t* pts_inf,
                             const uint8_t* scalars /* n*32 */, size_t n, int window_bits, uint8_t out[64],
                             uint8_t* out_inf);

/* Threshold-signature aggregation (examples/dkg.rs:190-226, examples/threshold_signing.rs:124-155).  A batch of
 * `n_sets` independent aggregations of `t` shares each; ids[s*t + i] is the participant id x of share i of set s
 * (`Fr::from(id as u64)`).
 *   lagrange_coefficients_batch: out[s*t + i] = prod_{j != i} x_j / (x_j - x_i) mod r   (32-byte LE canonical Fr)
 *   threshold_aggregate_batch:   out[s] = sum_i lambda[s][i] * sigs[s*t + i]             (affine + infinity flag)
 * Fr::inv(0) = 0 as in the reference (fields/fp.rs:418-424), so a repeated id gives a zero coefficient instead of a
 * failure; the reference's HashMap keys cannot repeat. */
int sylow_b200_lagrange_coefficients_batch(sylow_b200_ctx* ctx, const uint64_t* ids /* n_sets*t */, size_t n_sets,
                                           size_t t, uint8_t* out /* n_sets*t*32 */);
int sylow_b200_threshold_aggregate_batch(sylow_b200_ctx* ctx, const uint64_t* ids /* n_sets*t */,
                                         const uint8_t* sigs /* n_sets*t*64 */, const uint8_t* sigs_inf, size_t n_sets,
                                         size_t t, uint8_t* out /* n_sets*64 */, uint8_t* out_inf /* n_sets */);

/* ---- hash to curve / BLS ------------------------------------------------------------------------ */

/* out[i] = affine(G1Projective::hash_to_curve(XMDExpander::<Keccak256>::new(dst, 128), msg_i))
 * (groups/g1.rs:307-331, hasher.rs:84-128,201-250, svdw.rs:180-262).  msg_i = msgs[offsets[i]..offsets[i+1]). */
int sylow_b200_hash_to_g1_batch(sylow_b200_ctx* ctx, const uint8_t* msgs, const uint64_t* offsets /* n+1 */, size_t n,
                                const uint8_t* dst, size_t dst_len, int hash_id, uint8_t* out /* n*64 */,
                                uint8_t* out_inf /* may be NULL */);

/* The `Expander` trait (hasher.rs:55-129) for XMDExpander<D>, D in {Keccak-256, SHA-256}, security parameter 128;
 * a DST longer than 255 bytes is replaced by H("H2C-OVERSIZE-DST-" || DST) as XMDExpander::new does (:157-172).
 * expand_message: out[i] = len_in_bytes bytes (ceil(len/32) <= 255, hasher.rs:201-250);
 * hash_to_field: out[i] = two canonical Fp (count 2, L 48, hasher.rs:84-128). */
int sylow_b200_expand_message_batch(sylow_b200_ctx* ctx, const uint8_t* msgs, const uint64_t* offsets, size_t n,
                                    const uint8_t* dst, size_t dst_len, int hash_id, size_t len_in_bytes,
                                    uint8_t* out /* n*len_in_bytes */);
int sylow_b200_hash_to_field_batch(sylow_b200_ctx* ctx, const uint8_t* msgs, const uint64_t* offsets, size_t n,
                                   const uint8_t* dst, size_t dst_len, int hash_id, uint8_t* out /* n*64 */);

/* sigs[i] = affine(sign(sk[i], msg_i)) = sk[i] * H(msg_i)   (lib.rs:179-187).  sigs_out_inf (may be NULL) flags the
 * identity, which sk = 0 mod r produces. */
int sylow_b200_sign_batch(sylow_b200_ctx* ctx, const uint8_t* sks /* n*32 */, const uint8_t* msgs,
                          const uint64_t* offsets, size_t n, const uint8_t* dst, size_t dst_len, int hash_id,
                          uint8_t* sigs_out /* n*64 */, uint8_t* sigs_out_inf /* n, may be NULL */);

/* ok_out[i] = verify(pk[i], msg_i, sig[i]) = (e(sig, G2gen) == e(H(msg), pk))  (lib.rs:223-236),
 * one boolean per signature.  pks_inf / sigs_inf (may be NULL) flag identity keys / signatures: that side's pairing
 * is Gt::identity(), as in pairing() (pairing.rs:876-886). */
int sylow_b200_verify_each(sylow_b200_ctx* ctx, const uint8_t* pks /* n*128 */, const uint8_t* pks_inf,
                           const uint8_t* msgs, const uint64_t* offsets, const uint8_t* sigs /* n*64 */,
                           const uint8_t* sigs_inf, size_t n, const uint8_t* dst, size_t dst_len, int hash_id,
                           uint8_t* ok_out);

/* The product check of examples/verify_multiple_messages_same_signer.rs:40-60 over n (key, message, signature)
 * triples:   prod_i e(r_i sig_i, G2gen) e(-r_i H(msg_i), pk_i) == 1.
 *   weight_seed == NULL: r_i = 1, exactly the reference example.  This is AGGREGATE verification: it proves the
 *     product, not each factor - errors that cancel (sig_1 + D, sig_2 - D) pass.  Use it when the signatures come
 *     from one aggregator, or use sylow_b200_verify_each for per-signature verdicts.
 *   weight_seed != NULL (32 secret random bytes drawn AFTER the batch is fixed): BATCH verification with
 *     r_i = the first 8 bytes of Keccak-256(seed || LE64(first_index + i)) | 1; a batch with any invalid signature
 *     passes with probability <= 2^-63.  Costs two 64-bit G1 ladders per signature on top.
 * _partial: this GPU's 384-byte share f_out = miller(sum_i r_i sig_i, G2gen) * prod_i miller(-r_i H(msg_i), pk_i)
 *   (prod_i e(sig_i, G2gen) = e(sum_i sig_i, G2gen), so the product of all shares has the same final exponentiation
 *   as the reference's 2n-pair glued loop); first_index = global index of the slice's first triple.
 * _finish: *ok = (final_exponentiation(prod_i partials[i]) == Gt::identity()).  n_partials = number of GPUs.
 * sylow_b200_verify_batch = partial + finish (on a multi-device context: one partial per GPU). */
int sylow_b200_verify_batch_partial(sylow_b200_ctx* ctx, const uint8_t* pks, const uint8_t* pks_inf, const uint8_t* msgs,
                                    const uint64_t* offsets, const uint8_t* sigs, const uint8_t* sigs_inf, size_t n,
                                    const uint8_t* dst, size_t dst_len, int hash_id,
                                    const uint8_t* weight_seed /* 32 B or NULL */, uint64_t first_index,
                                    uint8_t f_out[384]);
int sylow_b200_verify_batch_finish(sylow_b200_ctx* ctx, const uint8_t* partials /* n_partials*384 */,
                                   size_t n_partials, int* ok);
int sylow_b200_verify_batch(sylow_b200_ctx* ctx, const uint8_t* pks, const uint8_t* pks_inf, const uint8_t* msgs,
                            const uint64_t* offsets, const uint8_t* sigs, const uint8_t* sigs_inf, size_t n,
                            const uint8_t* dst, size_t dst_len, int hash_id,
                            const uint8_t* weight_seed /* 32 B or NULL */, int* ok);

/* The reference example's exact setting - many messages, ONE signer (examples/verify_multiple_messages_same_signer.rs:
 * 40-60): prod e(sig_i, G2gen) e(-H(m_i), pk) = e(sum sig_i, G2gen) e(-sum H(m_i), pk), i.e. n hashes, 2n point
 * additions and two Miller loops for the whole batch.  Same verdict as the product form; weight_seed as above. */
int sylow_b200_verify_batch_same_signer(sylow_b200_ctx* ctx, const uint8_t* pk /* 128 */, int pk_inf, const uint8_t* msgs,
                                        const uint64_t* offsets, const uint8_t* sigs /* n*64 */, const uint8_t* sigs_inf,
                                        size_t n, const uint8_t* dst, size_t dst_len, int hash_id,
                                        const uint8_t* weight_seed /* 32 B or NULL */, int* ok);

/* ---- Groth16 proof verification ------------------------------------------------------------------ */

/* Verification of Groth16 proofs over BN254 under one verifying key with l = n_public public inputs (l may be 0):
 *   e(A, B) e(-alpha, beta) e(-L, gamma) e(-C, delta) == 1,   L = IC_0 + sum_{i=1..l} x_i IC_i.
 * Formats (wire form above, little-endian):
 *   verifying key, host:  alpha (G1) || beta || gamma || delta (G2) || IC_0 .. IC_l (G1): 448 + 64 (l + 1) bytes.
 *                         No point of the key can be infinite.
 *   proof:                A (G1) || B (G2) || C (G1), 256 bytes.  proofs_inf: n x 3 flags (A, B, C) or NULL; a flagged
 *                         A or B drops the pair e(A, B), a flagged C drops e(-C, delta).
 *   public inputs:        n x l canonical Fr values, 32 bytes each (proof j's inputs at inputs + j*l*32).  An input >= r
 *                         makes that proof INVALID; it is never reduced mod r (a reduced alias would let anyone change
 *                         the public input without changing the proof; the snarkjs / Solidity verifiers reject it too).
 *   prepared key, device: SYLOW_B200_GROTH16_VK_DEV_BYTES(l) bytes of caller-owned device memory (16-byte aligned):
 *                         the beta, gamma, delta line tables in the device form of sylow_b200_tables_to_device
 *                         (3 x 16704 B), -alpha (64 B, canonical affine), IC_0 (64 B), then one fixed-base table per
 *                         IC_i, i = 1 .. l (32 windows x 128 affine multiples, Montgomery form: 262144 B each).
 * Proof points are NOT validated, as in every pairing entry point: run sylow_b200_g1_validate_batch (A, C) and
 * sylow_b200_g2_validate_batch (B) on untrusted proofs first.  The key is validated by prepare_vk and by the host forms.
 * prepare_vk: validates the host key (G1 points on the curve, beta / gamma / delta on the curve and in the subgroup) and
 *   returns the first failing status in key order (SYLOW_B200_ERR_DECODE, _NOT_ON_CURVE, _NOT_IN_SUBGROUP); otherwise
 *   builds the device form at d_vk_out on the device.  Synchronous.
 * verify_each: ok_out[j] = proof j verifies.  The host form prepares the key itself (on every device of a multi-device
 *   context, which shards the proofs as usual).
 * verify_batch: *ok = prod_j check_j^{r_j} == 1 with r_j = batch_weight(weight_seed, first_index + j) as for
 *   sylow_b200_verify_batch: ONE final exponentiation, one fused Miller loop (r_j A_j, B_j) per proof and three table
 *   pairs for the whole batch.  weight_seed (32 secret random bytes drawn after the batch is fixed) is REQUIRED: NULL
 *   returns SYLOW_B200_ERR_ARG.  A batch with an invalid proof passes with probability <= 2^-63 (for validated points);
 *   an input >= r always fails it.  n = 0 gives *ok = 1.
 * verify_batch_partial_dev: the 384-byte share of a slice whose first proof has the global index first_index; combine
 *   the shares with sylow_b200_verify_batch_finish.  An input >= r makes the share zero, so the batch fails. */
#define SYLOW_B200_GROTH16_VK_DEV_BYTES(n_public) ((size_t)50240 + (size_t)(n_public) * (size_t)262144)
int sylow_b200_groth16_prepare_vk(sylow_b200_ctx* ctx, const uint8_t* vk, size_t n_public, uint8_t* d_vk_out,
                                  void* stream);
int sylow_b200_groth16_verify_each(sylow_b200_ctx* ctx, const uint8_t* vk, size_t n_public, const uint8_t* proofs,
                                   const uint8_t* proofs_inf, const uint8_t* inputs, size_t n, uint8_t* ok_out);
int sylow_b200_groth16_verify_each_dev(sylow_b200_ctx* ctx, const uint8_t* d_vk, size_t n_public,
                                       const uint8_t* d_proofs, const uint8_t* d_proofs_inf, const uint8_t* d_inputs,
                                       size_t n, uint8_t* d_ok_out, void* stream);
int sylow_b200_groth16_verify_batch(sylow_b200_ctx* ctx, const uint8_t* vk, size_t n_public, const uint8_t* proofs,
                                    const uint8_t* proofs_inf, const uint8_t* inputs, size_t n,
                                    const uint8_t* weight_seed /* 32 B, required */, int* ok);
int sylow_b200_groth16_verify_batch_partial_dev(sylow_b200_ctx* ctx, const uint8_t* d_vk, size_t n_public,
                                                const uint8_t* d_proofs, const uint8_t* d_proofs_inf,
                                                const uint8_t* d_inputs, size_t n,
                                                const uint8_t* weight_seed /* host, 32 B, required */,
                                                uint64_t first_index, uint8_t* d_f_out /* 384 */, void* stream);

/* ---- device-resident variants (DEVICE pointers, asynchronous on `stream`) ----------------------- */

int sylow_b200_pairing_batch_dev(sylow_b200_ctx* ctx, const uint8_t* d_g1, const uint8_t* d_g1_inf,
                                 const uint8_t* d_g2, const uint8_t* d_g2_inf, size_t n, uint8_t* d_gt_out,
                                 void* stream);
int sylow_b200_miller_loop_batch_dev(sylow_b200_ctx* ctx, const uint8_t* d_g1, const uint8_t* d_g1_inf,
                                     const uint8_t* d_g2, const uint8_t* d_g2_inf, size_t n, uint8_t* d_f_out,
                                     void* stream);
int sylow_b200_miller_product_dev(sylow_b200_ctx* ctx, const uint8_t* d_g1, const uint8_t* d_g1_inf,
                                  const uint8_t* d_g2, const uint8_t* d_g2_inf, size_t n, uint8_t* d_f_out,
                                  void* stream);
int sylow_b200_final_exp_batch_dev(sylow_b200_ctx* ctx, const uint8_t* d_f, size_t n, uint8_t* d_gt_out,
                                   void* stream);
int sylow_b200_pairing_check_batch_dev(sylow_b200_ctx* ctx, const uint8_t* d_g1, const uint8_t* d_g1_inf,
                                       const uint8_t* d_g2, const uint8_t* d_g2_inf, size_t pairs_per_check,
                                       size_t n_checks, uint8_t* d_ok_out, void* stream);
/* Device points, flags and verdicts; offsets in HOST memory: the launch plan is built on the host from them.  The plan's
 * device copy belongs to the call (a stream-ordered allocation freed on `stream` after its last kernel), so nothing of
 * it is shared with the next call. */
int sylow_b200_pairing_check_ragged_batch_dev(sylow_b200_ctx* ctx, const uint8_t* d_g1, const uint8_t* d_g1_inf,
                                              const uint8_t* d_g2, const uint8_t* d_g2_inf,
                                              const uint64_t* offsets /* host, n_checks + 1 */, size_t n_checks,
                                              uint8_t* d_ok_out, void* stream);
/* d_tables: k_fixed tables in the library's device form, produced by sylow_b200_tables_to_device. */
int sylow_b200_pairing_check_fixed_batch_dev(sylow_b200_ctx* ctx, const uint8_t* d_g1, const uint8_t* d_g1_inf,
                                             const uint8_t* d_g2_var, const uint8_t* d_g2_var_inf, size_t k_var,
                                             const uint8_t* d_tables, size_t k_fixed, size_t n_checks,
                                             uint8_t* d_ok_out, void* stream);
/* Converts k canonical host tables (sylow_b200_g2_precompute output) to the device form at d_tables_out
 * (k*16704 B of device memory). */
int sylow_b200_tables_to_device(sylow_b200_ctx* ctx, const uint8_t* coeffs, size_t k, uint8_t* d_tables_out, void* stream);
/* G2Affine::precompute of n device-resident points straight into caller-owned device memory, in the device form
 * (d_tables_out: n*16704 B).  No host round trip and no staging buffer: 2^20 tables take 17.5 GB once. */
int sylow_b200_g2_precompute_dev(sylow_b200_ctx* ctx, const uint8_t* d_g2, size_t n, uint8_t* d_tables_out,
                                 void* stream);
/* d_f_out (384 B, canonical) = the Miller product over n pairs, pair i = d_g1[i] against device-form table
 * d_table_idx[i] of d_tables (n_tables tables).  d_table_idx NULL: pair i uses table i, and n > n_tables is
 * SYLOW_B200_ERR_ARG.  An index >= n_tables makes the product the Fp12 zero (its final exponentiation is zero, never
 * the identity, so a check built on it fails closed); nothing is read out of bounds.  Infinite G1 pairs are skipped,
 * n = 0 gives 1.  1, 2 or 4 pairs share one thread's Fp12 squarings, by the fewest-wave-times rule. */
int sylow_b200_miller_product_precomputed_dev(sylow_b200_ctx* ctx, const uint8_t* d_tables, size_t n_tables,
                                              const uint32_t* d_table_idx, const uint8_t* d_g1,
                                              const uint8_t* d_g1_inf, size_t n, uint8_t* d_f_out /* 384 */,
                                              void* stream);
int sylow_b200_g1_mul_batch_dev(sylow_b200_ctx* ctx, const uint8_t* d_pts, const uint8_t* d_pts_inf,
                                const uint8_t* d_scalars, size_t n, uint8_t* d_out, uint8_t* d_out_inf, void* stream);
int sylow_b200_g2_mul_batch_dev(sylow_b200_ctx* ctx, const uint8_t* d_pts, const uint8_t* d_pts_inf,
                                const uint8_t* d_scalars, size_t n, uint8_t* d_out, uint8_t* d_out_inf, void* stream);
int sylow_b200_g1_add_batch_dev(sylow_b200_ctx* ctx, const uint8_t* d_a, const uint8_t* d_a_inf, const uint8_t* d_b,
                                const uint8_t* d_b_inf, size_t n, int subtract, uint8_t* d_out, uint8_t* d_out_inf,
                                void* stream);
int sylow_b200_g2_add_batch_dev(sylow_b200_ctx* ctx, const uint8_t* d_a, const uint8_t* d_a_inf, const uint8_t* d_b,
                                const uint8_t* d_b_inf, size_t n, int subtract, uint8_t* d_out, uint8_t* d_out_inf,
                                void* stream);
int sylow_b200_g1_mul_generator_batch_dev(sylow_b200_ctx* ctx, const uint8_t* d_scalars, size_t n, uint8_t* d_out,
                                          uint8_t* d_out_inf, void* stream);
int sylow_b200_g2_mul_generator_batch_dev(sylow_b200_ctx* ctx, const uint8_t* d_scalars, size_t n, uint8_t* d_out,
                                          uint8_t* d_out_inf, void* stream);
int sylow_b200_hash_to_g1_batch_dev(sylow_b200_ctx* ctx, const uint8_t* d_msgs, const uint64_t* d_offsets, size_t n,
                                    const uint8_t* dst, size_t dst_len /* host */, int hash_id, uint8_t* d_out,
                                    uint8_t* d_out_inf, void* stream);
int sylow_b200_verify_batch_partial_dev(sylow_b200_ctx* ctx, const uint8_t* d_pks, const uint8_t* d_pks_inf,
                                        const uint8_t* d_msgs, const uint64_t* d_offsets, const uint8_t* d_sigs,
                                        const uint8_t* d_sigs_inf, size_t n, const uint8_t* dst,
                                        size_t dst_len /* host */, int hash_id,
                                        const uint8_t* weight_seed /* host, 32 B or NULL */, uint64_t first_index,
                                        uint8_t* d_f_out /* 384 */, void* stream);
/* The hashing `_dev` calls (hash_to_g1_batch_dev, verify_batch_partial_dev) cannot return GroupError::CannotHashToGroup
 * themselves: this synchronises `stream`, sets *failed = 1 if a hash-to-curve of the LAST such call failed (SvdW's
 * square-root check, svdw.rs:253-261), and clears the flag.  Every hashing call clears the flag when it starts. */
int sylow_b200_hash_failed_dev(sylow_b200_ctx* ctx, void* stream, int* failed);

/* ---- diagnostics used by the parity tests and the roofline microbenchmark ---------------------- */

/* out[i] = a[i] (op) b[i] on canonical Fp values; op: 0 mul, 1 add, 2 sub, 3 inv(a) (binary GCD), 4 a/2, 5 -a,
 * 6 inv(a) by the Fermat ladder, 7 raw output (a / p) + 1 from the Jacobi iteration, + 4 if a^((p-1)/2) disagrees. */
int sylow_b200_fp_op_batch(sylow_b200_ctx* ctx, int op, const uint8_t* a, const uint8_t* b, size_t n, uint8_t* out);
/* out[i] = a[i] (op) b[i] on Fp12; op: 0 mul, 1 sqr(a), 2 inv(a), 3/4/5 frobenius^{1,2,3}(a),
 * 6 cyclotomic_squared(a), 7 a.sparse_mul(b.c0.c0, b.c0.c1, b.c0.c2).  The lower tower levels on their own, operands in
 * the leading coefficients (a2 = a.c0.c0, a6 = a.c0) and zeros elsewhere in the output: 8 Fp2 mul, 9 Fp2 sqr, 10 Fp6 mul,
 * 11 Fp6 sqr, 12 Fp2 inv, 13 (xi a2, b2 + xi a2, b2 - xi a2), 14 Fp6 inv, 15 (a2 * b.c0.c0.c0, a2 / 2, conj(a2)). */
int sylow_b200_fp12_op_batch(sylow_b200_ctx* ctx, int op, const uint8_t* a, const uint8_t* b, size_t n, uint8_t* out);
/* out[i] = the batch-verification weight r_(first_index + i) derived from weight_seed (tests). */
int sylow_b200_batch_weights(sylow_b200_ctx* ctx, const uint8_t* weight_seed /* 32 B */, uint64_t first_index, size_t n,
                             uint64_t* out);
/* Register-resident throughput probes (the IMAD roofline denominator, SURVEY.md 8d).  Every thread
 * runs `iters` loop iterations.  variant 0/1/2: 1/2/4 interleaved dependent Montgomery multiplications
 * per iteration (*ops_out = Fp multiplications; x136 = limb products).  variant 10: independent
 * mad.wide.u32; 11: independent 32-bit mad.lo.u32; 12: mad.lo.cc/madc.hi.cc carry chains (the
 * IMAD.WIDE.U32.X form fp_mul uses); 13: independent fma.rn.f64 (the FP64 pipe, for comparison) - *ops_out =
 * multiply-add instructions issued per thread x threads.
 * *ms_out = device time of the second of two launches.  Any other variant returns SYLOW_B200_ERR_ARG. */
int sylow_b200_imad_probe(sylow_b200_ctx* ctx, int variant, int blocks, int threads, int iters, float* ms_out,
                          double* ops_out);

#ifdef __cplusplus
}
#endif
#endif /* SYLOW_B200_H */

//! `src/batch.rs` of a sylow fork: the batched entry points BASELINE.json's north_star asks for
//! (`pairing_batch`, `verify_batch`, `g1_mul_batch`, ...), implemented on top of `sylow-cuda-sys`.
//!
//! It must live INSIDE sylow because `Gt(pub(crate) Fp12)`, `MillerLoopResult(pub(crate) Fp12)` and the
//! fields of `GroupAffine` are crate-private (src/groups/gt.rs:115, src/pairing.rs:72,
//! src/groups/group.rs:174-181).  `lib.rs` adds:
//!
//! ```ignore
//! mod batch;
//! pub use crate::batch::{final_exponentiation_batch, g1_add_batch, g1_generator_mul_batch, g1_mul_batch, g2_add_batch,
//!                        g2_generator_mul_batch, g2_mul_batch, glued_miller_loop_batch,
//!                        glued_miller_loop_precomputed_batch, glued_pairing_batch, pairing_batch, pairing_check_batch, pairing_check_ragged_batch,
//!                        sign_batch,
//!                        threshold_aggregate_batch, verify_batch, verify_each, groth16_verify_each,
//!                        groth16_verify_batch, Groth16Proof, Groth16VerifyingKey, BatchError, Engine};
//! ```
//!
//! All slicing over GPUs, the per-GPU host threads and the combination of the 384-byte Miller partial products live
//! behind the C ABI (`sylow_b200_create_multi`): every function here is ONE call on ONE context, so this file, the
//! C++ header and the Python binding cannot drift apart.
//!
//! NOT COMPILED in the build image (no Rust toolchain).  `tests/test_rust_boundary.py` checks statically that
//! every name in the `pub use` list above is defined here, that every `sys::` symbol exists in
//! `sylow-cuda-sys/src/lib.rs` and that every call passes as many arguments as the declaration takes; the C ABI
//! underneath is what the parity tests exercise (Python ctypes + include/sylow_b200.hpp).
use crate::fields::fp::Fp;
use crate::fields::fp12::Fp12;
use crate::fields::fp2::Fp2;
use crate::fields::fp6::Fp6;
use crate::groups::g1::{G1Affine, G1Projective};
use crate::groups::g2::{G2Affine, G2Projective};
use crate::groups::group::GroupError;
use crate::groups::gt::Gt;
use crate::pairing::{G2PreComputed, MillerLoopResult};
use crypto_bigint::U256;
use subtle::Choice;
use sylow_cuda_sys as sys;

/// Errors of the batched entry points: sylow's own `GroupError` where the library reports one, and the failures a
/// CPU library cannot have.
#[derive(Debug)]
pub enum BatchError {
    /// NotOnCurve / NotInSubgroup / CannotHashToGroup / DecodeError, as the reference's typed API would raise them
    Group(GroupError),
    /// mismatched batch lengths, unsupported shape
    InvalidArgument,
    /// device or host allocation failed
    OutOfMemory,
    /// a CUDA runtime call failed; `code` is the `cudaError_t` (`sylow_b200_last_cuda_error`)
    Cuda { code: i32 },
}

impl From<GroupError> for BatchError {
    fn from(e: GroupError) -> Self {
        BatchError::Group(e)
    }
}

/// One context over the listed GPUs.  `Engine::new(&[0, 1, .., 7])` for an 8xB200 box; a batch is cut into
/// contiguous slices inside the library (SURVEY.md 8e) and results are bit-identical to a single GPU's.
pub struct Engine {
    ctx: *mut sys::SylowB200Ctx,
}

// A context is used by one call at a time; `&mut self` on every entry point enforces it.
unsafe impl Send for Engine {}

impl Engine {
    pub fn new(devices: &[i32]) -> Result<Self, BatchError> {
        let mut ctx = core::ptr::null_mut();
        let st = unsafe { sys::sylow_b200_create_multi(&mut ctx, devices.as_ptr(), devices.len() as i32) };
        if st != sys::SYLOW_B200_OK {
            return Err(map_status(st, 0));
        }
        Ok(Engine { ctx })
    }
    pub fn device_count(&self) -> usize {
        unsafe { sys::sylow_b200_device_count(self.ctx) as usize }
    }
    fn check(&self, st: i32) -> Result<(), BatchError> {
        if st == sys::SYLOW_B200_OK {
            return Ok(());
        }
        Err(map_status(st, unsafe { sys::sylow_b200_last_cuda_error(self.ctx) }))
    }
}

impl Drop for Engine {
    fn drop(&mut self) {
        unsafe { sys::sylow_b200_destroy(self.ctx) };
    }
}

fn map_status(st: i32, cuda: i32) -> BatchError {
    match st {
        sys::SYLOW_B200_ERR_NOT_ON_CURVE => BatchError::Group(GroupError::NotOnCurve),
        sys::SYLOW_B200_ERR_NOT_IN_SUBGROUP => BatchError::Group(GroupError::NotInSubgroup),
        sys::SYLOW_B200_ERR_CANNOT_HASH => BatchError::Group(GroupError::CannotHashToGroup),
        sys::SYLOW_B200_ERR_DECODE => BatchError::Group(GroupError::DecodeError),
        sys::SYLOW_B200_ERR_NOMEM => BatchError::OutOfMemory,
        sys::SYLOW_B200_ERR_CUDA => BatchError::Cuda { code: cuda },
        _ => BatchError::InvalidArgument,
    }
}

fn same_len(a: usize, b: usize) -> Result<usize, BatchError> {
    if a == b {
        Ok(a)
    } else {
        Err(BatchError::InvalidArgument)
    }
}

// ---- marshalling: Fp <-> 32 little-endian bytes of `value().to_words()` (src/fields/fp.rs:232-234) ----
fn put_fp(out: &mut Vec<u8>, x: &Fp) {
    for w in x.value().to_words() {
        out.extend_from_slice(&w.to_le_bytes());
    }
}
fn get_fp(b: &[u8]) -> Fp {
    let mut w = [0u64; 4];
    for (i, c) in b.chunks_exact(8).enumerate() {
        w[i] = u64::from_le_bytes(c.try_into().unwrap());
    }
    Fp::new(U256::from_words(w))
}
fn get_fp2(b: &[u8]) -> Fp2 {
    Fp2::new(&[get_fp(&b[0..32]), get_fp(&b[32..64])])
}
fn get_fp12(b: &[u8]) -> Fp12 {
    let c: Vec<Fp2> = b.chunks_exact(64).map(get_fp2).collect();
    Fp12::new(&[Fp6::new(&[c[0], c[1], c[2]]), Fp6::new(&[c[3], c[4], c[5]])])
}
fn put_fp12(out: &mut Vec<u8>, f: &Fp12) {
    // tower order c0.c0.c0, c0.c0.c1, ..., c1.c2.c1 (src/fields/fp12.rs:561-574)
    for c6 in f.0.iter() {
        for c2 in c6.0.iter() {
            for c in c2.0.iter() {
                put_fp(out, c);
            }
        }
    }
}
fn get_g1(b: &[u8], inf: u8) -> G1Affine {
    G1Affine { x: get_fp(&b[..32]), y: get_fp(&b[32..64]), infinity: Choice::from(inf) }
}
fn get_g2(b: &[u8], inf: u8) -> G2Affine {
    G2Affine { x: get_fp2(&b[..64]), y: get_fp2(&b[64..128]), infinity: Choice::from(inf) }
}
fn marshal_g1(p: &[G1Projective]) -> (Vec<u8>, Vec<u8>) {
    let (mut v, mut inf) = (Vec::with_capacity(p.len() * 64), Vec::with_capacity(p.len()));
    for q in p {
        let a = G1Affine::from(q); // src/groups/group.rs:475-495
        put_fp(&mut v, &a.x);
        put_fp(&mut v, &a.y);
        inf.push(a.is_zero() as u8);
    }
    (v, inf)
}
fn marshal_g2(p: &[G2Projective]) -> (Vec<u8>, Vec<u8>) {
    let (mut v, mut inf) = (Vec::with_capacity(p.len() * 128), Vec::with_capacity(p.len()));
    for q in p {
        let a = G2Affine::from(q);
        for c in [a.x.0[0], a.x.0[1], a.y.0[0], a.y.0[1]] {
            put_fp(&mut v, &c);
        }
        inf.push(a.is_zero() as u8);
    }
    (v, inf)
}
fn marshal_scalars(k: &[Fp]) -> Vec<u8> {
    let mut v = Vec::with_capacity(k.len() * 32);
    k.iter().for_each(|x| put_fp(&mut v, x));
    v
}
fn pack_msgs(msgs: &[&[u8]]) -> (Vec<u8>, Vec<u64>) {
    let mut offs = Vec::with_capacity(msgs.len() + 1);
    let mut buf = Vec::new();
    offs.push(0u64);
    for m in msgs {
        buf.extend_from_slice(m);
        offs.push(buf.len() as u64);
    }
    if buf.is_empty() {
        buf.push(0); // a valid pointer for an all-empty batch
    }
    (buf, offs)
}

/// `p.iter().zip(q).map(|(p, q)| pairing(p, q))` on the GPUs (src/pairing.rs:870-893).
pub fn pairing_batch(e: &mut Engine, p: &[G1Projective], q: &[G2Projective]) -> Result<Vec<Gt>, BatchError> {
    let n = same_len(p.len(), q.len())?;
    let (g1, g1i) = marshal_g1(p);
    let (g2, g2i) = marshal_g2(q);
    let mut out = vec![0u8; n * 384];
    e.check(unsafe {
        sys::sylow_b200_pairing_batch(e.ctx, g1.as_ptr(), g1i.as_ptr(), g2.as_ptr(), g2i.as_ptr(), n, out.as_mut_ptr())
    })?;
    Ok(out.chunks_exact(384).map(|b| Gt(get_fp12(b))).collect())
}

/// `glued_miller_loop` over the batch (src/pairing.rs:970-1022): the product of the per-pair Miller values, equal
/// bit for bit to the shared-squaring loop.  Infinite pairs contribute 1.
pub fn glued_miller_loop_batch(e: &mut Engine, p: &[G1Projective], q: &[G2Projective]) -> Result<MillerLoopResult, BatchError> {
    let n = p.len().min(q.len()); // zip truncation, like the reference (:975)
    let (g1, g1i) = marshal_g1(&p[..n]);
    let (g2, g2i) = marshal_g2(&q[..n]);
    let mut out = [0u8; 384];
    e.check(unsafe {
        sys::sylow_b200_miller_product(e.ctx, g1.as_ptr(), g1i.as_ptr(), g2.as_ptr(), g2i.as_ptr(), n, out.as_mut_ptr())
    })?;
    Ok(MillerLoopResult(get_fp12(&out)))
}

/// `glued_miller_loop(&[G2PreComputed], &[G1Affine])` itself (src/pairing.rs:970-1022): the 87 `Ell` triples of every
/// table go over canonically, one table per pair.  Pairs with an infinite G1 point, or a table of the identity,
/// contribute 1.  This moves 16.7 KB per pair to the device; keep hot tables resident with
/// `sylow_b200_g2_precompute_dev` + `sylow_b200_miller_product_precomputed_dev` instead.
pub fn glued_miller_loop_precomputed_batch(e: &mut Engine, q: &[G2PreComputed], p: &[G1Affine]) -> Result<MillerLoopResult, BatchError> {
    let n = p.len().min(q.len()); // zip truncation, like the reference (:975)
    let (mut coeffs, mut g1, mut g1i) = (Vec::with_capacity(n * 16704), Vec::with_capacity(n * 64), Vec::with_capacity(n));
    for (pc, a) in q[..n].iter().zip(&p[..n]) {
        if pc.coeffs.len() != 87 {
            return Err(BatchError::InvalidArgument);
        }
        for (c0, c1, c2) in pc.coeffs.iter() {
            for c in [c0.0[0], c0.0[1], c1.0[0], c1.0[1], c2.0[0], c2.0[1]] {
                put_fp(&mut coeffs, &c);
            }
        }
        put_fp(&mut g1, &a.x);
        put_fp(&mut g1, &a.y);
        g1i.push((a.is_zero() || pc.q.is_zero()) as u8);
    }
    let mut out = [0u8; 384];
    e.check(unsafe {
        sys::sylow_b200_miller_product_precomputed(e.ctx, coeffs.as_ptr(), g1.as_ptr(), g1i.as_ptr(), n, out.as_mut_ptr())
    })?;
    Ok(MillerLoopResult(get_fp12(&out)))
}

/// `MillerLoopResult::final_exponentiation` (src/pairing.rs:245-492) over a batch.
pub fn final_exponentiation_batch(e: &mut Engine, f: &[MillerLoopResult]) -> Result<Vec<Gt>, BatchError> {
    let n = f.len();
    let mut inp = Vec::with_capacity(n * 384);
    f.iter().for_each(|x| put_fp12(&mut inp, &x.0));
    let mut out = vec![0u8; n * 384];
    e.check(unsafe { sys::sylow_b200_final_exp_batch(e.ctx, inp.as_ptr(), n, out.as_mut_ptr()) })?;
    Ok(out.chunks_exact(384).map(|b| Gt(get_fp12(b))).collect())
}

/// `glued_pairing(g1s, g2s)` (src/pairing.rs:1029-1037): one Miller product, one final exponentiation.
pub fn glued_pairing_batch(e: &mut Engine, p: &[G1Projective], q: &[G2Projective]) -> Result<Gt, BatchError> {
    let f = glued_miller_loop_batch(e, p, q)?;
    Ok(final_exponentiation_batch(e, &[f])?.remove(0))
}

/// `p.len() / pairs_per_check` independent checks `glued_pairing(..) == Gt::identity()` (the ecPairing / Groth16
/// shape, examples/reth_bn128.rs:211-214).
pub fn pairing_check_batch(e: &mut Engine, p: &[G1Projective], q: &[G2Projective], pairs_per_check: usize) -> Result<Vec<bool>, BatchError> {
    let n = same_len(p.len(), q.len())?;
    if pairs_per_check == 0 || n % pairs_per_check != 0 {
        return Err(BatchError::InvalidArgument);
    }
    let (g1, g1i) = marshal_g1(p);
    let (g2, g2i) = marshal_g2(q);
    let mut ok = vec![0u8; n / pairs_per_check];
    e.check(unsafe {
        sys::sylow_b200_pairing_check_batch(e.ctx, g1.as_ptr(), g1i.as_ptr(), g2.as_ptr(), g2i.as_ptr(), pairs_per_check,
                                            n / pairs_per_check, ok.as_mut_ptr())
    })?;
    Ok(ok.into_iter().map(|b| b != 0).collect())
}

/// Checks with a pair count each: check c is `glued_pairing(p[o_c..o_{c+1}], q[o_c..o_{c+1}]) == Gt::identity()` with
/// `o = offsets` (`offsets.len()` = checks + 1, non-decreasing, ending at `p.len()`); an empty check holds.  One call
/// for a block's ecPairing inputs of every length.
pub fn pairing_check_ragged_batch(e: &mut Engine, p: &[G1Projective], q: &[G2Projective], offsets: &[u64]) -> Result<Vec<bool>, BatchError> {
    let n = same_len(p.len(), q.len())?;
    if offsets.is_empty() || offsets[offsets.len() - 1] != n as u64 {
        return Err(BatchError::InvalidArgument);
    }
    let (g1, g1i) = marshal_g1(p);
    let (g2, g2i) = marshal_g2(q);
    let mut ok = vec![0u8; offsets.len() - 1];
    e.check(unsafe {
        sys::sylow_b200_pairing_check_ragged_batch(e.ctx, g1.as_ptr(), g1i.as_ptr(), g2.as_ptr(), g2i.as_ptr(),
                                                   offsets.as_ptr(), offsets.len() - 1, ok.as_mut_ptr())
    })?;
    Ok(ok.into_iter().map(|b| b != 0).collect())
}

/// `scalars[i] * pts[i]` (src/groups/group.rs:639-667), returned affine.
pub fn g1_mul_batch(e: &mut Engine, pts: &[G1Projective], scalars: &[Fp]) -> Result<Vec<G1Affine>, BatchError> {
    let n = same_len(pts.len(), scalars.len())?;
    let (g1, g1i) = marshal_g1(pts);
    let ks = marshal_scalars(scalars);
    let (mut out, mut inf) = (vec![0u8; n * 64], vec![0u8; n]);
    e.check(unsafe {
        sys::sylow_b200_g1_mul_batch(e.ctx, g1.as_ptr(), g1i.as_ptr(), ks.as_ptr(), n, out.as_mut_ptr(), inf.as_mut_ptr())
    })?;
    Ok(out.chunks_exact(64).zip(&inf).map(|(b, &i)| get_g1(b, i)).collect())
}

/// `&a[i] + &b[i]`, or `&a[i] - &b[i]` when `subtract` (src/groups/group.rs:528-624), followed by the affine conversion.
pub fn g1_add_batch(e: &mut Engine, a: &[G1Projective], b: &[G1Projective], subtract: bool) -> Result<Vec<G1Affine>, BatchError> {
    let n = same_len(a.len(), b.len())?;
    let ((pa, ia), (pb, ib)) = (marshal_g1(a), marshal_g1(b));
    let (mut out, mut inf) = (vec![0u8; n * 64], vec![0u8; n]);
    e.check(unsafe {
        sys::sylow_b200_g1_add_batch(e.ctx, pa.as_ptr(), ia.as_ptr(), pb.as_ptr(), ib.as_ptr(), n, subtract as i32,
                                     out.as_mut_ptr(), inf.as_mut_ptr())
    })?;
    Ok(out.chunks_exact(64).zip(&inf).map(|(b, &i)| get_g1(b, i)).collect())
}

/// The same on the twist.
pub fn g2_add_batch(e: &mut Engine, a: &[G2Projective], b: &[G2Projective], subtract: bool) -> Result<Vec<G2Affine>, BatchError> {
    let n = same_len(a.len(), b.len())?;
    let ((pa, ia), (pb, ib)) = (marshal_g2(a), marshal_g2(b));
    let (mut out, mut inf) = (vec![0u8; n * 128], vec![0u8; n]);
    e.check(unsafe {
        sys::sylow_b200_g2_add_batch(e.ctx, pa.as_ptr(), ia.as_ptr(), pb.as_ptr(), ib.as_ptr(), n, subtract as i32,
                                     out.as_mut_ptr(), inf.as_mut_ptr())
    })?;
    Ok(out.chunks_exact(128).zip(&inf).map(|(b, &i)| get_g2(b, i)).collect())
}

/// The same on the twist.
pub fn g2_mul_batch(e: &mut Engine, pts: &[G2Projective], scalars: &[Fp]) -> Result<Vec<G2Affine>, BatchError> {
    let n = same_len(pts.len(), scalars.len())?;
    let (g2, g2i) = marshal_g2(pts);
    let ks = marshal_scalars(scalars);
    let (mut out, mut inf) = (vec![0u8; n * 128], vec![0u8; n]);
    e.check(unsafe {
        sys::sylow_b200_g2_mul_batch(e.ctx, g2.as_ptr(), g2i.as_ptr(), ks.as_ptr(), n, out.as_mut_ptr(), inf.as_mut_ptr())
    })?;
    Ok(out.chunks_exact(128).zip(&inf).map(|(b, &i)| get_g2(b, i)).collect())
}

/// `G1Projective::generator() * &scalars[i]`, returned affine: the values of `g1_mul_batch` on the repeated generator,
/// from a fixed-base table of the generator.
pub fn g1_generator_mul_batch(e: &mut Engine, scalars: &[Fp]) -> Result<Vec<G1Affine>, BatchError> {
    let n = scalars.len();
    let ks = marshal_scalars(scalars);
    let (mut out, mut inf) = (vec![0u8; n * 64], vec![0u8; n]);
    e.check(unsafe { sys::sylow_b200_g1_mul_generator_batch(e.ctx, ks.as_ptr(), n, out.as_mut_ptr(), inf.as_mut_ptr()) })?;
    Ok(out.chunks_exact(64).zip(&inf).map(|(b, &i)| get_g1(b, i)).collect())
}

/// The same on the twist: `KeyPair::generate`'s public keys (src/lib.rs:105-137).
pub fn g2_generator_mul_batch(e: &mut Engine, scalars: &[Fp]) -> Result<Vec<G2Affine>, BatchError> {
    let n = scalars.len();
    let ks = marshal_scalars(scalars);
    let (mut out, mut inf) = (vec![0u8; n * 128], vec![0u8; n]);
    e.check(unsafe { sys::sylow_b200_g2_mul_generator_batch(e.ctx, ks.as_ptr(), n, out.as_mut_ptr(), inf.as_mut_ptr()) })?;
    Ok(out.chunks_exact(128).zip(&inf).map(|(b, &i)| get_g2(b, i)).collect())
}

/// `sign(&sk[i], msgs[i])` (src/lib.rs:179-187): hash-to-curve and one scalar multiplication per message.
pub fn sign_batch(e: &mut Engine, sks: &[Fp], msgs: &[&[u8]]) -> Result<Vec<G1Affine>, BatchError> {
    let n = same_len(sks.len(), msgs.len())?;
    let ks = marshal_scalars(sks);
    let (buf, offs) = pack_msgs(msgs);
    let (mut out, mut inf) = (vec![0u8; n * 64], vec![0u8; n]);
    e.check(unsafe {
        sys::sylow_b200_sign_batch(e.ctx, ks.as_ptr(), buf.as_ptr(), offs.as_ptr(), n, crate::DST.as_ptr(), crate::DST.len(),
                                   sys::SYLOW_B200_HASH_KECCAK256, out.as_mut_ptr(), inf.as_mut_ptr())
    })?;
    Ok(out.chunks_exact(64).zip(&inf).map(|(b, &i)| get_g1(b, i)).collect())
}

/// `verify(&pks[i], msgs[i], &sigs[i])` per signature (src/lib.rs:223-236), identity keys and signatures included
/// (the library applies `pairing`'s infinity rule, src/pairing.rs:876-886).
pub fn verify_each(e: &mut Engine, pks: &[G2Projective], msgs: &[&[u8]], sigs: &[G1Projective]) -> Result<Vec<bool>, BatchError> {
    let n = same_len(pks.len(), same_len(msgs.len(), sigs.len())?)?;
    let (pk, pki) = marshal_g2(pks);
    let (sg, sgi) = marshal_g1(sigs);
    let (buf, offs) = pack_msgs(msgs);
    let mut ok = vec![0u8; n];
    e.check(unsafe {
        sys::sylow_b200_verify_each(e.ctx, pk.as_ptr(), pki.as_ptr(), buf.as_ptr(), offs.as_ptr(), sg.as_ptr(), sgi.as_ptr(), n,
                                    crate::DST.as_ptr(), crate::DST.len(), sys::SYLOW_B200_HASH_KECCAK256, ok.as_mut_ptr())
    })?;
    Ok(ok.into_iter().map(|b| b != 0).collect())
}

/// prod e(r_i sig_i, G2gen) * e(-r_i H(m_i), pk_i) == 1 with ONE final exponentiation
/// (examples/verify_multiple_messages_same_signer.rs:40-60, generalised to per-message keys).
/// `weight_seed = None` is the reference example's unweighted product (aggregate verification: cancelling errors
/// pass); `Some(seed)` with 32 secret random bytes drawn after the batch is fixed is batch verification with random
/// 64-bit weights, sound for every signature.
pub fn verify_batch(e: &mut Engine, pks: &[G2Projective], msgs: &[&[u8]], sigs: &[G1Projective], weight_seed: Option<&[u8; 32]>) -> Result<bool, BatchError> {
    let n = same_len(pks.len(), same_len(msgs.len(), sigs.len())?)?;
    let (pk, pki) = marshal_g2(pks);
    let (sg, sgi) = marshal_g1(sigs);
    let (buf, offs) = pack_msgs(msgs);
    let seed = weight_seed.map_or(core::ptr::null(), |s| s.as_ptr());
    let mut ok = 0i32;
    e.check(unsafe {
        sys::sylow_b200_verify_batch(e.ctx, pk.as_ptr(), pki.as_ptr(), buf.as_ptr(), offs.as_ptr(), sg.as_ptr(), sgi.as_ptr(), n,
                                     crate::DST.as_ptr(), crate::DST.len(), sys::SYLOW_B200_HASH_KECCAK256, seed, &mut ok)
    })?;
    Ok(ok != 0)
}

/// A Groth16 verifying key over BN254: a proof (A, B, C) with public inputs x_1 .. x_l holds when
/// e(A, B) e(-alpha, beta) e(-L, gamma) e(-C, delta) == 1 with L = ic[0] + sum_i x_i ic[i]; `ic` has l + 1 points.
pub struct Groth16VerifyingKey {
    pub alpha: G1Projective,
    pub beta: G2Projective,
    pub gamma: G2Projective,
    pub delta: G2Projective,
    pub ic: Vec<G1Projective>,
}
/// A Groth16 proof.  Its points are not validated here: decode untrusted proofs with the checked constructors.
pub struct Groth16Proof {
    pub a: G1Projective,
    pub b: G2Projective,
    pub c: G1Projective,
}
// key, proofs with their n x 3 infinity flags, and the public inputs (l canonical 32-byte little-endian Fr per proof) in
// the wire form of include/sylow_b200.h; InvalidArgument if a proof does not carry l inputs
fn marshal_groth16(vk: &Groth16VerifyingKey, proofs: &[Groth16Proof], inputs: &[&[[u8; 32]]])
                   -> Result<(Vec<u8>, usize, Vec<u8>, Vec<u8>, Vec<u8>), BatchError> {
    if vk.ic.is_empty() || same_len(proofs.len(), inputs.len()).is_err() {
        return Err(BatchError::InvalidArgument);
    }
    let l = vk.ic.len() - 1;
    let mut key = marshal_g1(core::slice::from_ref(&vk.alpha)).0;
    key.extend(marshal_g2(&[vk.beta, vk.gamma, vk.delta]).0);
    key.extend(marshal_g1(&vk.ic).0);
    let (mut pr, mut inf, mut x) = (Vec::with_capacity(proofs.len() * 256), Vec::with_capacity(proofs.len() * 3),
                                    Vec::with_capacity(proofs.len() * l * 32));
    for (p, xs) in proofs.iter().zip(inputs) {
        if xs.len() != l {
            return Err(BatchError::InvalidArgument);
        }
        let (a, ai) = marshal_g1(core::slice::from_ref(&p.a));
        let (b, bi) = marshal_g2(core::slice::from_ref(&p.b));
        let (c, ci) = marshal_g1(core::slice::from_ref(&p.c));
        pr.extend(a);
        pr.extend(b);
        pr.extend(c);
        inf.extend([ai[0], bi[0], ci[0]]);
        for v in xs.iter() {
            x.extend_from_slice(v);
        }
    }
    Ok((key, l, pr, inf, x))
}

/// One verdict per Groth16 proof under `vk`; `inputs[j]` are proof j's public inputs.  An input >= r fails its proof.
pub fn groth16_verify_each(e: &mut Engine, vk: &Groth16VerifyingKey, proofs: &[Groth16Proof], inputs: &[&[[u8; 32]]])
                           -> Result<Vec<bool>, BatchError> {
    let (key, l, pr, inf, x) = marshal_groth16(vk, proofs, inputs)?;
    let mut ok = vec![0u8; proofs.len()];
    e.check(unsafe {
        sys::sylow_b200_groth16_verify_each(e.ctx, key.as_ptr(), l, pr.as_ptr(), inf.as_ptr(), x.as_ptr(), proofs.len(),
                                            ok.as_mut_ptr())
    })?;
    Ok(ok.into_iter().map(|b| b != 0).collect())
}

/// One verdict for a batch of Groth16 proofs under `vk`: prod_j check_j^{r_j} == 1 with random 64-bit weights from
/// `weight_seed` (32 secret random bytes drawn after the batch is fixed) and ONE final exponentiation.
pub fn groth16_verify_batch(e: &mut Engine, vk: &Groth16VerifyingKey, proofs: &[Groth16Proof], inputs: &[&[[u8; 32]]],
                            weight_seed: &[u8; 32]) -> Result<bool, BatchError> {
    let (key, l, pr, inf, x) = marshal_groth16(vk, proofs, inputs)?;
    let mut ok = 0i32;
    e.check(unsafe {
        sys::sylow_b200_groth16_verify_batch(e.ctx, key.as_ptr(), l, pr.as_ptr(), inf.as_ptr(), x.as_ptr(), proofs.len(),
                                             weight_seed.as_ptr(), &mut ok)
    })?;
    Ok(ok != 0)
}

/// Threshold aggregation (examples/dkg.rs:190-226): `ids.len() / t` independent sets of `t` partial signatures;
/// `out[s] = sum_i lambda_i * sigs[s*t + i]` with the Lagrange coefficients at 0 computed on the device.
pub fn threshold_aggregate_batch(e: &mut Engine, ids: &[u64], sigs: &[G1Projective], t: usize) -> Result<Vec<G1Affine>, BatchError> {
    if t == 0 || ids.len() != sigs.len() || ids.len() % t != 0 {
        return Err(BatchError::InvalidArgument);
    }
    let n_sets = ids.len() / t;
    let (sg, sgi) = marshal_g1(sigs);
    let (mut out, mut inf) = (vec![0u8; n_sets * 64], vec![0u8; n_sets]);
    e.check(unsafe {
        sys::sylow_b200_threshold_aggregate_batch(e.ctx, ids.as_ptr(), sg.as_ptr(), sgi.as_ptr(), n_sets, t, out.as_mut_ptr(),
                                                  inf.as_mut_ptr())
    })?;
    Ok(out.chunks_exact(64).zip(&inf).map(|(b, &i)| get_g1(b, i)).collect())
}

// sylow_b200.hpp - header-only C++ host mirror of sylow's hot-path API over the C ABI (sylow_b200.h).
//
// The reference is Rust (compiled); there is no Rust toolchain in the build image, so the compiled-language
// host side that can actually be built and run here is this header (INTEGRATION.md section 4).  Names and
// argument meaning follow /root/reference/src/lib.rs:71-84: Fp, Fp2, Fp12, G1Affine, G2Affine, Gt, pairing,
// glued_pairing, sign, verify - plus the batched entry points the north star adds.  No field arithmetic
// happens here: every call goes to the CUDA library and throws sylow::Error on failure (no CPU fallback).
#pragma once
#include <array>
#include <cstdint>
#include <cstring>
#include <memory>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "sylow_b200.h"

namespace sylow {

// Canonical little-endian residue in [0, p): the 4 u64 words of `Fp::value().to_words()` (fp.rs:232-234).
struct Fp {
  std::array<std::uint64_t, 4> w{};
  static Fp from_u64(std::uint64_t v) { Fp f; f.w[0] = v; return f; }
  bool operator==(const Fp& o) const { return w == o.w; }
};
struct Fp2 { Fp c0, c1; bool operator==(const Fp2& o) const { return c0 == o.c0 && c1 == o.c1; } };
// Tower order c0.c0.c0, c0.c0.c1, ..., c1.c2.c1 (fp12.rs:561-574)
struct Fp12 {
  std::array<Fp, 12> c{};
  bool operator==(const Fp12& o) const { return c == o.c; }
  static Fp12 one() { Fp12 f; f.c[0] = Fp::from_u64(1); return f; }
};
struct G1Affine { Fp x, y; bool infinity = false; };   // groups/group.rs:174-181
struct G2Affine { Fp2 x, y; bool infinity = false; };
struct Gt { Fp12 v; bool operator==(const Gt& o) const { return v == o.v; } static Gt identity() { return Gt{Fp12::one()}; } };
struct MillerLoopResult { Fp12 v; };
// Groth16 (sylow_b200.h): e(A, B) e(-alpha, beta) e(-L, gamma) e(-C, delta) == 1, L = ic[0] + sum_i x_i ic[i]
struct Groth16VerifyingKey { G1Affine alpha; G2Affine beta, gamma, delta; std::vector<G1Affine> ic; };
struct Groth16Proof { G1Affine a; G2Affine b; G1Affine c; };
using FrBytes = std::array<std::uint8_t, 32>;  // canonical little-endian public input

static_assert(sizeof(Fp) == 32 && sizeof(Fp2) == 64 && sizeof(Fp12) == 384, "wire layout");

// lib.rs:90
inline const std::string& DST() { static const std::string d = "WARLOCK-CHAOS-V01-CS01-SHA-256"; return d; }

struct Error : std::runtime_error {
  int status;
  Error(int s, const char* where) : std::runtime_error(std::string(where) + ": " + sylow_b200_strerror(s)), status(s) {}
};

class Engine {
 public:
  explicit Engine(int device = 0) { ck(sylow_b200_create(&ctx_, device), "sylow_b200_create"); }
  // One context over several GPUs (sylow_b200_create_multi): every batched call below shards its batch as
  // contiguous slices inside the library; results are bit-identical to the single-device call.
  explicit Engine(const std::vector<int>& devices) {
    ck(sylow_b200_create_multi(&ctx_, devices.data(), (int)devices.size()), "sylow_b200_create_multi");
  }
  size_t device_count() const { return (size_t)sylow_b200_device_count(ctx_); }
  ~Engine() { if (ctx_) sylow_b200_destroy(ctx_); }
  Engine(const Engine&) = delete;
  Engine& operator=(const Engine&) = delete;

  // pairing(&G1Projective, &G2Projective) -> Gt over a batch (pairing.rs:870-893)
  std::vector<Gt> pairing_batch(const std::vector<G1Affine>& p, const std::vector<G2Affine>& q) {
    size_t n = same(p.size(), q.size());
    Packed a = pack(p), b = pack(q);
    std::vector<Gt> out(n);
    ck(sylow_b200_pairing_batch(ctx_, a.pts.data(), a.inf.data(), b.pts.data(), b.inf.data(), n, bytes(out)), "pairing_batch");
    return out;
  }
  Gt pairing(const G1Affine& p, const G2Affine& q) { return pairing_batch({p}, {q})[0]; }

  // glued_miller_loop / glued_pairing (pairing.rs:970-1037)
  MillerLoopResult glued_miller_loop(const std::vector<G1Affine>& p, const std::vector<G2Affine>& q) {
    size_t n = p.size() < q.size() ? p.size() : q.size();  // zip truncation like the reference (:975)
    Packed a = pack(p), b = pack(q);
    MillerLoopResult r;
    ck(sylow_b200_miller_product(ctx_, a.pts.data(), a.inf.data(), b.pts.data(), b.inf.data(), n,
                                 reinterpret_cast<std::uint8_t*>(&r.v)), "miller_product");
    return r;
  }
  Gt final_exponentiation(const MillerLoopResult& f) {
    Gt g;
    ck(sylow_b200_final_exp_batch(ctx_, reinterpret_cast<const std::uint8_t*>(&f.v), 1,
                                  reinterpret_cast<std::uint8_t*>(&g.v)), "final_exp_batch");
    return g;
  }
  Gt glued_pairing(const std::vector<G1Affine>& p, const std::vector<G2Affine>& q) {
    return final_exponentiation(glued_miller_loop(p, q));
  }
  // n_checks product checks of k pairs each (ecPairing / Groth16 shape)
  std::vector<bool> pairing_check_batch(const std::vector<G1Affine>& p, const std::vector<G2Affine>& q, size_t k) {
    size_t n = same(p.size(), q.size());
    if (k == 0 || n % k) throw Error(SYLOW_B200_ERR_ARG, "pairing_check_batch");
    Packed a = pack(p), b = pack(q);
    std::vector<std::uint8_t> ok(n / k);
    ck(sylow_b200_pairing_check_batch(ctx_, a.pts.data(), a.inf.data(), b.pts.data(), b.inf.data(), k, n / k, ok.data()),
       "pairing_check_batch");
    return std::vector<bool>(ok.begin(), ok.end());
  }
  // check c multiplies pairs [offsets[c], offsets[c+1]); offsets.size() = n_checks + 1, non-decreasing, ending at p.size()
  std::vector<bool> pairing_check_ragged_batch(const std::vector<G1Affine>& p, const std::vector<G2Affine>& q,
                                               const std::vector<std::uint64_t>& offsets) {
    size_t n = same(p.size(), q.size());
    if (offsets.empty() || offsets.back() != n) throw Error(SYLOW_B200_ERR_ARG, "pairing_check_ragged_batch");
    Packed a = pack(p), b = pack(q);
    std::vector<std::uint8_t> ok(offsets.size() - 1);
    ck(sylow_b200_pairing_check_ragged_batch(ctx_, a.pts.data(), a.inf.data(), b.pts.data(), b.inf.data(), offsets.data(),
                                             ok.size(), ok.data()),
       "pairing_check_ragged_batch");
    return std::vector<bool>(ok.begin(), ok.end());
  }
  // EIP-197 ecPairing bodies over calldata of any length: (ok, status) per input; see the C header
  std::pair<std::vector<bool>, std::vector<std::int8_t>> eip197_pairing_check_ragged_batch(
      const std::vector<std::vector<std::uint8_t>>& inputs) {
    std::vector<std::uint64_t> offs(inputs.size() + 1, 0);
    for (size_t i = 0; i < inputs.size(); i++) offs[i + 1] = offs[i] + inputs[i].size();
    std::vector<std::uint8_t> buf;
    buf.reserve(offs.back());
    for (const auto& in : inputs) buf.insert(buf.end(), in.begin(), in.end());
    std::vector<std::uint8_t> ok(inputs.size());
    std::vector<std::int8_t> st(inputs.size());
    ck(sylow_b200_eip197_pairing_check_ragged_batch(ctx_, buf.data(), offs.data(), inputs.size(), ok.data(), st.data()),
       "eip197_pairing_check_ragged_batch");
    return {std::vector<bool>(ok.begin(), ok.end()), st};
  }

  // &GroupProjective * &Fp (group.rs:639-667) + GroupAffine::from (:475-495)
  std::vector<G1Affine> g1_mul_batch(const std::vector<G1Affine>& pts, const std::vector<Fp>& k) {
    size_t n = same(pts.size(), k.size());
    Packed a = pack(pts);
    std::vector<std::uint8_t> out(n * 64), inf(n);
    ck(sylow_b200_g1_mul_batch(ctx_, a.pts.data(), a.inf.data(), reinterpret_cast<const std::uint8_t*>(k.data()), n,
                               out.data(), inf.data()), "g1_mul_batch");
    std::vector<G1Affine> r(n);
    for (size_t i = 0; i < n; i++) { std::memcpy(&r[i].x, &out[64 * i], 64); r[i].infinity = inf[i]; }
    return r;
  }
  // &a[i] + &b[i], or &a[i] - &b[i] when subtract (group.rs:528-624), + GroupAffine::from (:475-495)
  std::vector<G1Affine> g1_add_batch(const std::vector<G1Affine>& a, const std::vector<G1Affine>& b,
                                     bool subtract = false) {
    size_t n = same(a.size(), b.size());
    Packed pa = pack(a), pb = pack(b);
    std::vector<std::uint8_t> out(n * 64), inf(n);
    ck(sylow_b200_g1_add_batch(ctx_, pa.pts.data(), pa.inf.data(), pb.pts.data(), pb.inf.data(), n, subtract ? 1 : 0,
                               out.data(), inf.data()), "g1_add_batch");
    std::vector<G1Affine> r(n);
    for (size_t i = 0; i < n; i++) { std::memcpy(&r[i].x, &out[64 * i], 64); r[i].infinity = inf[i]; }
    return r;
  }
  std::vector<G2Affine> g2_add_batch(const std::vector<G2Affine>& a, const std::vector<G2Affine>& b,
                                     bool subtract = false) {
    size_t n = same(a.size(), b.size());
    Packed pa = pack(a), pb = pack(b);
    std::vector<std::uint8_t> out(n * 128), inf(n);
    ck(sylow_b200_g2_add_batch(ctx_, pa.pts.data(), pa.inf.data(), pb.pts.data(), pb.inf.data(), n, subtract ? 1 : 0,
                               out.data(), inf.data()), "g2_add_batch");
    std::vector<G2Affine> r(n);
    for (size_t i = 0; i < n; i++) { std::memcpy(&r[i].x, &out[128 * i], 128); r[i].infinity = inf[i]; }
    return r;
  }
  // Threshold aggregation: `n_sets` sets of `t` shares; ids[s*t + i] is the participant id of share i of set s.
  // out[s] = sum_i lambda_i * sigs[s*t + i] with the Lagrange coefficients at 0 (examples/dkg.rs:190-226).
  std::vector<G1Affine> threshold_aggregate_batch(const std::vector<std::uint64_t>& ids,
                                                  const std::vector<G1Affine>& sigs, size_t t) {
    size_t n = same(ids.size(), sigs.size());
    if (!t || n % t) throw std::invalid_argument("threshold_aggregate_batch: n must be a multiple of t");
    size_t n_sets = n / t;
    Packed a = pack(sigs);
    std::vector<std::uint8_t> out(n_sets * 64), inf(n_sets);
    ck(sylow_b200_threshold_aggregate_batch(ctx_, ids.data(), a.pts.data(), a.inf.data(), n_sets, t, out.data(),
                                            inf.data()), "threshold_aggregate_batch");
    std::vector<G1Affine> r(n_sets);
    for (size_t i = 0; i < n_sets; i++) { std::memcpy(&r[i].x, &out[64 * i], 64); r[i].infinity = inf[i]; }
    return r;
  }
  std::vector<G2Affine> g2_mul_batch(const std::vector<G2Affine>& pts, const std::vector<Fp>& k) {
    size_t n = same(pts.size(), k.size());
    Packed a = pack(pts);
    std::vector<std::uint8_t> out(n * 128), inf(n);
    ck(sylow_b200_g2_mul_batch(ctx_, a.pts.data(), a.inf.data(), reinterpret_cast<const std::uint8_t*>(k.data()), n,
                               out.data(), inf.data()), "g2_mul_batch");
    std::vector<G2Affine> r(n);
    for (size_t i = 0; i < n; i++) { std::memcpy(&r[i].x, &out[128 * i], 128); r[i].infinity = inf[i]; }
    return r;
  }

  // G1Projective::generator() * &k[i] and G2Projective::generator() * &k[i] (KeyPair::generate's pk, lib.rs:105-137):
  // the values of g1_mul_batch / g2_mul_batch on the repeated generator, from a fixed-base table
  std::vector<G1Affine> g1_mul_generator_batch(const std::vector<Fp>& k) {
    std::vector<std::uint8_t> out(k.size() * 64), inf(k.size());
    ck(sylow_b200_g1_mul_generator_batch(ctx_, reinterpret_cast<const std::uint8_t*>(k.data()), k.size(), out.data(),
                                         inf.data()), "g1_mul_generator_batch");
    std::vector<G1Affine> r(k.size());
    for (size_t i = 0; i < k.size(); i++) { std::memcpy(&r[i].x, &out[64 * i], 64); r[i].infinity = inf[i]; }
    return r;
  }
  std::vector<G2Affine> g2_mul_generator_batch(const std::vector<Fp>& k) {
    std::vector<std::uint8_t> out(k.size() * 128), inf(k.size());
    ck(sylow_b200_g2_mul_generator_batch(ctx_, reinterpret_cast<const std::uint8_t*>(k.data()), k.size(), out.data(),
                                         inf.data()), "g2_mul_generator_batch");
    std::vector<G2Affine> r(k.size());
    for (size_t i = 0; i < k.size(); i++) { std::memcpy(&r[i].x, &out[128 * i], 128); r[i].infinity = inf[i]; }
    return r;
  }

  // G1Projective::hash_to_curve(&XMDExpander::<Keccak256>::new(dst, 128), msg) (g1.rs:307-331)
  std::vector<G1Affine> hash_to_g1_batch(const std::vector<std::string>& msgs, const std::string& dst = DST()) {
    Msgs m(msgs);
    std::vector<std::uint8_t> out(msgs.size() * 64), inf(msgs.size());
    ck(sylow_b200_hash_to_g1_batch(ctx_, m.buf.data(), m.offs.data(), msgs.size(), udata(dst), dst.size(),
                                   SYLOW_B200_HASH_KECCAK256, out.data(), inf.data()), "hash_to_g1_batch");
    std::vector<G1Affine> r(msgs.size());
    for (size_t i = 0; i < r.size(); i++) { std::memcpy(&r[i].x, &out[64 * i], 64); r[i].infinity = inf[i]; }
    return r;
  }
  // sign(&Fp, &[u8]) (lib.rs:179-187)
  std::vector<G1Affine> sign_batch(const std::vector<Fp>& sks, const std::vector<std::string>& msgs,
                                   const std::string& dst = DST()) {
    size_t n = same(sks.size(), msgs.size());
    Msgs m(msgs);
    std::vector<std::uint8_t> out(n * 64), inf(n + 1);
    ck(sylow_b200_sign_batch(ctx_, reinterpret_cast<const std::uint8_t*>(sks.data()), m.buf.data(), m.offs.data(), n,
                             udata(dst), dst.size(), SYLOW_B200_HASH_KECCAK256, out.data(), inf.data()), "sign_batch");
    std::vector<G1Affine> r(n);
    for (size_t i = 0; i < n; i++) { std::memcpy(&r[i].x, &out[64 * i], 64); r[i].infinity = inf[i]; }
    return r;
  }
  // verify(&G2Projective, &[u8], &G1Projective) per signature (lib.rs:223-236); identity keys / signatures follow
  // pairing()'s infinity rule (pairing.rs:876-886) inside the library
  std::vector<bool> verify_each(const std::vector<G2Affine>& pks, const std::vector<std::string>& msgs,
                                const std::vector<G1Affine>& sigs, const std::string& dst = DST()) {
    size_t n = same(pks.size(), same(msgs.size(), sigs.size()));
    Msgs m(msgs);
    Packed pk = pack(pks), sg = pack(sigs);
    std::vector<std::uint8_t> ok(n);
    ck(sylow_b200_verify_each(ctx_, pk.pts.data(), pk.inf.data(), m.buf.data(), m.offs.data(), sg.pts.data(),
                              sg.inf.data(), n, udata(dst), dst.size(), SYLOW_B200_HASH_KECCAK256, ok.data()),
       "verify_each");
    return std::vector<bool>(ok.begin(), ok.end());
  }
  // The product check with one final exponentiation (examples/verify_multiple_messages_same_signer.rs:40-60).
  // weight_seed == nullptr: the reference example's unweighted product (aggregate verification);
  // 32 secret random bytes: batch verification with random 64-bit weights (sound per signature).
  bool verify_batch(const std::vector<G2Affine>& pks, const std::vector<std::string>& msgs,
                    const std::vector<G1Affine>& sigs, const std::string& dst = DST(),
                    const std::array<std::uint8_t, 32>* weight_seed = nullptr) {
    size_t n = same(pks.size(), same(msgs.size(), sigs.size()));
    Msgs m(msgs);
    Packed pk = pack(pks), sg = pack(sigs);
    int ok = 0;
    ck(sylow_b200_verify_batch(ctx_, pk.pts.data(), pk.inf.data(), m.buf.data(), m.offs.data(), sg.pts.data(),
                               sg.inf.data(), n, udata(dst), dst.size(), SYLOW_B200_HASH_KECCAK256,
                               weight_seed ? weight_seed->data() : nullptr, &ok), "verify_batch");
    return ok != 0;
  }
  bool verify(const G2Affine& pk, const std::string& msg, const G1Affine& sig) { return verify_each({pk}, {msg}, {sig})[0]; }

  // Groth16 verdicts under vk: inputs[j] holds proof j's vk.ic.size() - 1 public inputs; an input >= r fails its proof.
  // Proof points are not validated (g1/g2_validate_batch first).
  std::vector<bool> groth16_verify_each(const Groth16VerifyingKey& vk, const std::vector<Groth16Proof>& proofs,
                                        const std::vector<std::vector<FrBytes>>& inputs) {
    G16 g(vk, proofs, inputs);
    std::vector<std::uint8_t> ok(proofs.size());
    ck(sylow_b200_groth16_verify_each(ctx_, g.vk.data(), g.l, g.proofs.data(), g.inf.data(), g.x.data(), proofs.size(),
                                      ok.data()), "groth16_verify_each");
    return std::vector<bool>(ok.begin(), ok.end());
  }
  // one verdict for the batch, with random 64-bit weights from weight_seed (32 secret random bytes)
  bool groth16_verify_batch(const Groth16VerifyingKey& vk, const std::vector<Groth16Proof>& proofs,
                            const std::vector<std::vector<FrBytes>>& inputs, const std::array<std::uint8_t, 32>& weight_seed) {
    G16 g(vk, proofs, inputs);
    int ok = 0;
    ck(sylow_b200_groth16_verify_batch(ctx_, g.vk.data(), g.l, g.proofs.data(), g.inf.data(), g.x.data(), proofs.size(),
                                       weight_seed.data(), &ok), "groth16_verify_batch");
    return ok != 0;
  }

  sylow_b200_ctx* raw() { return ctx_; }

 private:
  struct Packed { std::vector<std::uint8_t> pts, inf; };
  struct Msgs {
    std::vector<std::uint8_t> buf;
    std::vector<std::uint64_t> offs;
    explicit Msgs(const std::vector<std::string>& m) {
      offs.push_back(0);
      for (const auto& s : m) { buf.insert(buf.end(), s.begin(), s.end()); offs.push_back(buf.size()); }
      if (buf.empty()) buf.push_back(0);
    }
  };
  // key, proofs, their n x 3 infinity flags and inputs in the wire form of sylow_b200.h
  struct G16 {
    std::vector<std::uint8_t> vk, proofs, inf, x;
    size_t l;
    G16(const Groth16VerifyingKey& k, const std::vector<Groth16Proof>& p, const std::vector<std::vector<FrBytes>>& in) {
      if (k.ic.empty() || p.size() != in.size()) throw Error(SYLOW_B200_ERR_ARG, "groth16 arguments");
      l = k.ic.size() - 1;
      auto put = [](std::vector<std::uint8_t>& v, const void* a, size_t b) {
        v.insert(v.end(), static_cast<const std::uint8_t*>(a), static_cast<const std::uint8_t*>(a) + b);
      };
      put(vk, &k.alpha.x, 64);
      for (const G2Affine* q : {&k.beta, &k.gamma, &k.delta}) put(vk, &q->x, 128);
      for (const G1Affine& q : k.ic) put(vk, &q.x, 64);
      for (size_t j = 0; j < p.size(); j++) {
        if (in[j].size() != l) throw Error(SYLOW_B200_ERR_ARG, "groth16 public inputs");
        put(proofs, &p[j].a.x, 64);
        put(proofs, &p[j].b.x, 128);
        put(proofs, &p[j].c.x, 64);
        inf.insert(inf.end(), {p[j].a.infinity, p[j].b.infinity, p[j].c.infinity});
        for (const FrBytes& v : in[j]) put(x, v.data(), 32);
      }
      x.resize(x.size() + 16);  // a valid pointer for l = 0
      proofs.resize(proofs.size() + 16);
      inf.resize(inf.size() + 1);
    }
  };
  template <class P>
  static Packed pack(const std::vector<P>& v) {
    constexpr size_t W = sizeof(P::x) * 2;
    Packed r;
    r.pts.resize(v.size() * W + 16);
    r.inf.resize(v.size() + 1);
    for (size_t i = 0; i < v.size(); i++) { std::memcpy(&r.pts[W * i], &v[i].x, W); r.inf[i] = v[i].infinity; }
    return r;
  }
  template <class T> static std::uint8_t* bytes(std::vector<T>& v) { return reinterpret_cast<std::uint8_t*>(v.data()); }
  static const std::uint8_t* udata(const std::string& s) { return reinterpret_cast<const std::uint8_t*>(s.data()); }
  static size_t same(size_t a, size_t b) { if (a != b) throw Error(SYLOW_B200_ERR_ARG, "batch sizes differ"); return a; }
  void ck(int st, const char* where) { if (st != 0) throw Error(st, where); }
  sylow_b200_ctx* ctx_ = nullptr;
};

// One context over several GPUs (SURVEY 8e).  The slicing, the per-GPU host threads and the combination of the
// 384-byte Miller partials live inside the library (sylow_b200_create_multi), so this is the same class.
class MultiEngine : public Engine {
 public:
  explicit MultiEngine(const std::vector<int>& devices) : Engine(devices) {}
  size_t size() const { return device_count(); }
};

}  // namespace sylow

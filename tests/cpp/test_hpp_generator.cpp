// Exercises the generator multiplications of include/sylow_b200.hpp on the GPU: KeyPair::generate's public key
// (lib.rs:105-137) derived with g2_mul_generator_batch must equal g2_mul_batch({g2}, {sk}); the G1 form likewise, and a
// two-slot MultiEngine must agree.  Prints one tag per check for tests/test_gpu_generator_mul.py.
#include <cstdio>

#include "../../include/sylow_b200.hpp"

using namespace sylow;

static bool same(const G1Affine& a, const G1Affine& b) { return a.x == b.x && a.y == b.y && a.infinity == b.infinity; }
static bool same(const G2Affine& a, const G2Affine& b) { return a.x == b.x && a.y == b.y && a.infinity == b.infinity; }

int main() {
  try {
    Engine eng(0);
    G1Affine g1{Fp::from_u64(1), Fp::from_u64(2), false};
    G2Affine g2;  // src/groups/g2.rs:47-77
    g2.x.c0.w = {5106727233969649389ull, 7440829307424791261ull, 4785637993704342649ull, 1729627375292849782ull};
    g2.x.c1.w = {10945020018377822914ull, 17413811393473931026ull, 8241798111626485029ull, 1841571559660931130ull};
    g2.y.c0.w = {5541340697920699818ull, 16416156555105522555ull, 5380518976772849807ull, 1353435754470862315ull};
    g2.y.c1.w = {6173549831154472795ull, 13567992399387660019ull, 17050234209342075797ull, 650358724130500725ull};
    // KeyPair::generate: pk = sk * G2gen
    Fp sk = Fp::from_u64(0x1234567890abcdefull);
    sk.w[3] = 0x0123456789abcdefull;
    G2Affine pk = eng.g2_mul_generator_batch({sk})[0];
    std::printf("PK %d\n", (int)same(pk, eng.g2_mul_batch({g2}, {sk})[0]));
    // a batch with 0 and the group order r (both give the point at infinity) between ordinary scalars
    Fp r;
    r.w = {0x43e1f593f0000001ull, 0x2833e84879b97091ull, 0xb85045b68181585dull, 0x30644e72e131a029ull};
    std::vector<Fp> ks = {Fp::from_u64(1), Fp::from_u64(0), sk, r, Fp::from_u64(987654321)};
    std::vector<G1Affine> p = eng.g1_mul_generator_batch(ks), p_ref = eng.g1_mul_batch(std::vector<G1Affine>(5, g1), ks);
    std::vector<G2Affine> q = eng.g2_mul_generator_batch(ks), q_ref = eng.g2_mul_batch(std::vector<G2Affine>(5, g2), ks);
    bool g1_ok = true, g2_ok = true;
    for (size_t i = 0; i < ks.size(); i++) {
      g1_ok = g1_ok && same(p[i], p_ref[i]);
      g2_ok = g2_ok && same(q[i], q_ref[i]);
    }
    std::printf("G1 %d\nG2 %d\nINF %d %d\n", (int)g1_ok, (int)g2_ok, (int)(p[1].infinity && q[3].infinity),
                (int)(!p[0].infinity && !q[4].infinity));
    MultiEngine multi({0, 0});
    std::vector<G2Affine> m = multi.g2_mul_generator_batch(ks);
    bool multi_ok = true;
    for (size_t i = 0; i < ks.size(); i++) multi_ok = multi_ok && same(m[i], q[i]);
    std::printf("MULTI %d\n", (int)multi_ok);
    std::printf("EMPTY %d\n", (int)eng.g1_mul_generator_batch({}).empty());
  } catch (const std::exception& e) {
    std::printf("ERROR %s\n", e.what());
    return 1;
  }
  return 0;
}

// Exercises the pointwise additions of include/sylow_b200.hpp on the GPU: a + b and a - b for a = k1 G, b = k2 G must
// equal g*_mul_batch(G, k1 +- k2) in both groups, a - a must be the point at infinity, and a two-slot MultiEngine must
// agree.  Prints one tag per check for tests/test_gpu_group_law.py.
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
    // k1 > k2 so that k1 - k2 needs no reduction mod r
    std::vector<Fp> k1 = {Fp::from_u64(1000), Fp::from_u64(77), Fp::from_u64(5)};
    std::vector<Fp> k2 = {Fp::from_u64(1), Fp::from_u64(77), Fp::from_u64(2)};
    std::vector<Fp> ks, kd;
    for (size_t i = 0; i < k1.size(); i++) {
      ks.push_back(Fp::from_u64(k1[i].w[0] + k2[i].w[0]));
      kd.push_back(Fp::from_u64(k1[i].w[0] - k2[i].w[0]));
    }
    std::vector<G1Affine> G1s(3, g1);
    std::vector<G2Affine> G2s(3, g2);
    auto a1 = eng.g1_mul_batch(G1s, k1), b1 = eng.g1_mul_batch(G1s, k2);
    auto a2 = eng.g2_mul_batch(G2s, k1), b2 = eng.g2_mul_batch(G2s, k2);
    auto s1 = eng.g1_add_batch(a1, b1), d1 = eng.g1_add_batch(a1, b1, true);
    auto s2 = eng.g2_add_batch(a2, b2), d2 = eng.g2_add_batch(a2, b2, true);
    auto rs1 = eng.g1_mul_batch(G1s, ks), rd1 = eng.g1_mul_batch(G1s, kd);
    auto rs2 = eng.g2_mul_batch(G2s, ks), rd2 = eng.g2_mul_batch(G2s, kd);
    bool ok1 = true, ok2 = true;
    for (size_t i = 0; i < ks.size(); i++) {
      ok1 = ok1 && same(s1[i], rs1[i]) && same(d1[i], rd1[i]);
      ok2 = ok2 && same(s2[i], rs2[i]) && same(d2[i], rd2[i]);
    }
    std::printf("G1 %d\nG2 %d\n", (int)ok1, (int)ok2);
    std::printf("INF %d\n", (int)(d1[1].infinity && d2[1].infinity && !s1[1].infinity && !s2[1].infinity));
    MultiEngine multi({0, 0});
    auto m1 = multi.g1_add_batch(a1, b1, true);
    auto m2 = multi.g2_add_batch(a2, b2);
    bool multi_ok = true;
    for (size_t i = 0; i < ks.size(); i++) multi_ok = multi_ok && same(m1[i], d1[i]) && same(m2[i], s2[i]);
    std::printf("MULTI %d\n", (int)multi_ok);
  } catch (const std::exception& e) {
    std::printf("ERROR %s\n", e.what());
    return 1;
  }
  return 0;
}

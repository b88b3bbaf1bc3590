// TEST-ONLY: the launch policy of csrc/launch_plan.h with the block shapes of csrc/kernels_pairing.cuh, compiled for the
// host.  Used by tests/test_launch_plan.py.
#include "../../sylow_b200/csrc/kernels_pairing.cuh"
#include "../../sylow_b200/csrc/launch_plan.h"

#include <cstdint>

// kernels_pairing.cuh's two-lane code is compiled for the host here but never run: its barrier only has to link
extern "C" void sylow_hostsim_lane_sync() {}

static constexpr BlockShape kMiller{SY_MILLER_THREADS, SY_MILLER_MINB}, kFexp{SY_FEXP_THREADS, SY_FEXP_MINB},
    kLanes{SY_LANES_THREADS, SY_LANES_MINB}, kGlued{SY_GLUED_THREADS, SY_GLUED_MINB};

static void put(const Segment& g, uint64_t* out) {
  out[0] = g.first;
  out[1] = g.count;
  out[2] = g.blocks;
  out[3] = g.threads;
  out[4] = g.lanes;
}

extern "C" {

// The launches of launch_miller (kernel 0) or launch_final_exp (kernel 1) for n items: (first, count, blocks, threads,
// lanes) per launch in out, returns the number of launches.
int lp_batch(int kernel, int sms, uint64_t n, int lanes_mode, uint64_t* out) {
  int k = 0;
  for (const Segment& g : batch_plan(sms, n, kernel ? kFexp : kMiller, kLanes, lanes_mode)) put(g, out + 5 * k++);
  return k;
}

// launch_check_products' final-exponentiation launch for n_checks checks, as above
void lp_check(int sms, uint64_t n_checks, int lanes_mode, uint64_t* out) {
  put(check_products_segment(sms, n_checks, kFexp, kLanes, lanes_mode), out);
}

int lp_glue(int sms, uint64_t n, uint64_t pair_cost) { return glue_pairs(sms, n, pair_cost, kGlued); }

}  // extern "C"

// Launch policy of the batch kernels (sylow_b200.cu): which launches cover a batch of n items, as pure host functions of
// the SM count, the batch size, the kernels' block shapes and the SYLOW_B200_LANES mode.  Host-only, so that
// tests/hostsim/launch_plan.cu can pin the launches without a GPU.
#pragma once
#include <cstddef>

// block size and resident blocks per SM of a kernel (its __launch_bounds__)
struct BlockShape {
  unsigned threads, per_sm;
};
// items [first, first + count) as blocks x threads; lanes: the two-lane kernel, threads / 2 items per block
struct Segment {
  size_t first, count;
  unsigned blocks, threads;
  bool lanes;
};
// at most two launches, in order
struct LaunchPlan {
  Segment seg[2];
  int size = 0;
  void add(const Segment& s) { seg[size++] = s; }
  const Segment* begin() const { return seg; }
  const Segment* end() const { return seg + size; }
};

inline unsigned nblocks(size_t n, size_t threads) { return (unsigned)((n + threads - 1) / threads); }
// items of one full wave of a one-thread kernel, and of a two-lane kernel (two threads per item)
inline size_t wave_items(int sms, BlockShape b) { return (size_t)sms * b.threads * b.per_sm; }
inline size_t lane_wave(int sms, BlockShape lanes) { return (size_t)sms * (lanes.threads / 2) * lanes.per_sm; }

// Launch shapes that do not waste the last wave.  Both pairing kernels run one item per thread for several
// milliseconds, so a batch that is not a whole number of waves (k_miller keeps 256 threads resident per SM,
// k_final_exp 384) ends with a partly filled wave that takes as long as a full one - at 2^17 items per GPU (a 2^20
// batch sharded over 8) that is 3.46 and 2.31 waves.  The whole waves are launched as usual; a remainder of less than
// 0.6 wave is launched separately as one (k_final_exp) or two (k_miller) SMALL blocks per SM, so that every SM works
// on it at low occupancy - a lone warp per scheduler runs 1.5x (Miller) to 2x (final exponentiation) faster than one of
// two or three co-resident warps (profiles/r01_overlap_probe.md), and the remainder finishes in that much less time.
// (Cutting the last 1 + r waves into two rounds of equal, reduced occupancy instead was measured and is not better:
// profiles/r02g_policy_sweep.jsonl, tail_split 2.)
inline LaunchPlan wave_split(int sms, size_t n, BlockShape b) {
  LaunchPlan p;
  const size_t wave = wave_items(sms, b), r = n % wave;
  if (r == 0 || r * 10 >= wave * 6) {
    p.add({0, n, nblocks(n, b.threads), b.threads, false});
    return p;
  }
  const size_t slots = (size_t)sms * b.per_sm;
  unsigned t = (unsigned)(((r + slots - 1) / slots + 31) / 32 * 32);
  if (t > b.threads) t = b.threads;
  if (n > r) p.add({0, n - r, nblocks(n - r, b.threads), b.threads, false});
  p.add({n - r, r, nblocks(r, t), t, false});
  return p;
}

// A two-lane launch of items [first, first + n) spread over every SM: pairs per block = n / (SMs x resident blocks), in
// whole warps (16 pairs), at most lanes.threads / 2.
inline Segment lanes_segment(int sms, size_t first, size_t n, BlockShape lanes) {
  const size_t slots = (size_t)sms * lanes.per_sm;
  size_t pairs = ((n + slots - 1) / slots + 15) / 16 * 16;
  if (pairs > lanes.threads / 2) pairs = lanes.threads / 2;
  return {first, n, nblocks(n, pairs), (unsigned)pairs * 2, true};
}

// Two lanes per item (k_miller_lanes, k_final_exp_lanes, csrc/pairing_lanes.cuh): the same values in 0.55-0.6 of the
// time per item when the items alone cannot fill the GPU, 0.88 of the one-thread kernels' throughput when they can
// (profiles/r02f_lanes_kbench.jsonl, r02g_policy_sweep.jsonl).  Used for batches of at most one two-lane wave
// (148 x 128 items) and for the remainder of a larger batch after its whole one-thread waves when that remainder fits one
// two-lane wave: 1 .. 9 472 pairings 8.5 -> 5.0 ms, 2^17 pairings (a 2^20 batch over 8 GPUs) 46.3 -> 44.3 ms.
// lanes_mode (SYLOW_B200_LANES): 0 never, 1 automatic, 2 always.  Otherwise wave_split of the one-thread kernel.
inline LaunchPlan batch_plan(int sms, size_t n, BlockShape one, BlockShape lanes, int lanes_mode) {
  LaunchPlan p;
  const size_t lw = lane_wave(sms, lanes);
  if (lanes_mode == 2 || (lanes_mode == 1 && n <= lw)) {
    p.add(lanes_segment(sms, 0, n, lanes));
    return p;
  }
  const size_t r = n % wave_items(sms, one);
  if (lanes_mode == 1 && r && r <= lw) {
    p.add({0, n - r, nblocks(n - r, one.threads), one.threads, false});
    p.add(lanes_segment(sms, n - r, r, lanes));
    return p;
  }
  return wave_split(sms, n, one);
}

// ok[c] = final_exp(product of check c's Miller values) == 1.  Batches that fit one two-lane wave go through
// k_final_exp_lanes (group products, exponentiation, comparison as three launches: about half the latency) in any mode
// but 0 - mode 2 does not force larger ones onto two lanes; larger ones through the fused one-thread kernel
// (k_check_products, shape `fexp`), in blocks small enough to reach every SM.
inline Segment check_products_segment(int sms, size_t n_checks, BlockShape fexp, BlockShape lanes, int lanes_mode) {
  if (lanes_mode != 0 && n_checks <= lane_wave(sms, lanes)) return lanes_segment(sms, 0, n_checks, lanes);
  unsigned t = (unsigned)(((n_checks + sms - 1) / sms + 31) / 32 * 32);
  if (t > fexp.threads) t = fexp.threads;
  return {0, n_checks, nblocks(n_checks, t), t, false};
}

// Whether pairing_check_batch runs each of n_checks checks of k pairs as ONE glued loop (k_glued<k, 0>, shape `glued`)
// rather than k separate Miller loops multiplied by launch_check_products: 2- and 4-pair checks (ecPairing, Groth16
// without fixed tables), once there are enough checks to fill the GPU - a whole glued wave of 2-pair checks, half of one
// of 4-pair checks.
inline bool glued_checks(int sms, size_t k, size_t n_checks, BlockShape glued) {
  const size_t wave = wave_items(sms, glued);
  return (k == 2 && n_checks >= wave) || (k == 4 && n_checks >= wave / 2);
}

// Pairs per thread (1, 2 or 4) for n >= 1 pairs whose Miller loops only meet as a product, glued into one loop per
// thread (k_glued<M, 0>, k_miller_tables<M>, shape `glued`): the glue of fewest wave-times, i.e. whole waves of n / g
// threads times the Fp multiplications of g glued pairs.  pair_cost is one pair's count (8 444 fused, 6 045 from a
// table); every pair after the first saves its Fp12 squarings, 63 x 36 multiplications.
inline int glue_pairs(int sms, size_t n, size_t pair_cost, BlockShape glued) {
  const size_t wave = wave_items(sms, glued), save = 63 * 36;
  const size_t cost[3] = {pair_cost, 2 * pair_cost - save, 4 * pair_cost - 3 * save};
  int glue = 0;
  size_t best = ~(size_t)0;
  for (int j = 0; j < 3; j++) {
    const size_t g = (size_t)1 << j, waves = (n / g + wave - 1) / wave;
    if (n >= g && waves * cost[j] < best) {
      best = waves * cost[j];
      glue = (int)g;
    }
  }
  return glue;
}

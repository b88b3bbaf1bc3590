// TEST-ONLY: the ragged-check plan of csrc/ragged_plan.h with the glued block shape of csrc/kernels_pairing.cuh,
// compiled for the host.  Used by tests/test_ragged_plan.py.
#include "../../sylow_b200/csrc/kernels_pairing.cuh"
#include "../../sylow_b200/csrc/ragged_plan.h"

#include <cstdint>
#include <cstring>

// kernels_pairing.cuh's two-lane code is compiled for the host here but never run: its barrier only has to link
extern "C" void sylow_hostsim_lane_sync() {}

static constexpr BlockShape kGlued{SY_GLUED_THREADS, SY_GLUED_MINB};

extern "C" {

// The plan of n_checks checks (glue 0: glue_pairs' choice).  head[0 .. 7] = glue, n_pairs, items of 4, 2 and 1 pairs,
// n_values, number of levels, number of words; then (n_chunks, at) per level.  Returns the plan; rp_words copies its
// words, rp_free releases it.
void* rp_build(int sms, const uint64_t* offsets, uint64_t n_checks, int glue, uint64_t* head, uint64_t head_cap) {
  RaggedPlan* p = new RaggedPlan(ragged_plan(sms, offsets, n_checks, kGlued, glue));
  const uint64_t h[8] = {(uint64_t)p->glue, p->n_pairs, p->n_items[0], p->n_items[1], p->n_items[2], p->n_values,
                         p->levels.size(), p->words.size()};
  memcpy(head, h, sizeof(h));
  for (size_t l = 0; l < p->levels.size() && 8 + 2 * l + 1 < head_cap; l++) {
    head[8 + 2 * l] = p->levels[l].n_chunks;
    head[9 + 2 * l] = p->levels[l].at;
  }
  return p;
}
void rp_words(void* p, uint32_t* out) {
  const std::vector<uint32_t>& w = static_cast<RaggedPlan*>(p)->words;
  memcpy(out, w.data(), w.size() * 4);
}
void rp_free(void* p) { delete static_cast<RaggedPlan*>(p); }

// ragged_cuts for D devices into cut (D + 1 entries)
void rp_cuts(const uint64_t* offsets, uint64_t n_checks, uint64_t D, uint64_t* cut) {
  std::vector<size_t> c = ragged_cuts(offsets, n_checks, D);
  for (size_t g = 0; g <= D; g++) cut[g] = c[g];
}

int rp_offsets_ok(const uint64_t* offsets, uint64_t n_checks) { return ragged_offsets_ok(offsets, n_checks); }

uint64_t rp_chunk() { return kRaggedChunk; }

}  // extern "C"

// Launch plan of the ragged pairing checks (sylow_b200_pairing_check_ragged_batch): check c holds the pairs
// [offsets[c], offsets[c + 1]), and every check may hold a different number of them.  A pure host function of the
// offsets, the SM count and the glued block shape, so that tests/hostsim/ragged_plan.cu can check it without a GPU.
//
// The plan turns the checks into launches of the existing kernels:
//   1. items: each check of k pairs becomes k / G items of G consecutive pairs (G = glue_pairs, once per batch), and its
//      remainder one 2-pair and/or one 1-pair item.  No item crosses a check boundary and none is padded.
//   2. gather: the source pair of every position of the gathered arrays, the 4-pair items first, then the 2-pair items,
//      then the 1-pair items, each class in check order; k_glued<4, 0>, k_glued<2, 0> and launch_miller then run on three
//      contiguous arrays, and item v of the classes in that order writes value v.
//   3. products: per level, chunks of at most kRaggedChunk value indices, one thread each (k_fp12_segment_products).
//      A check of at most kRaggedChunk values is one chunk that writes the check's product to final slot c; a longer
//      one is cut into chunks whose products are appended to the value array and multiplied at the next level.
//   4. device cuts (ragged_cuts): check boundaries that give each device of a multi-device context about n_pairs / D
//      pairs.
#pragma once
#include <cstddef>
#include <cstdint>
#include <vector>

#include "launch_plan.h"

// Values one thread of k_fp12_segment_products multiplies at most.  An Fp12 product is 18 Fp2 products, about 1/150 of
// one pair's 8 444 Fp multiplications in a Miller loop, so a chunk of 32 costs a fifth of the Miller loop of one of its
// values, while a check of 2^20 glued pairs (2^18 values) needs only four levels (32^4 >= 2^18).
static constexpr size_t kRaggedChunk = 32;
// one fused pair's Fp multiplications for glue_pairs (verify_partial_core and the uniform checks count the same)
static constexpr size_t kRaggedPairCost = 8444;
// bit of a chunk's destination that names a final slot (the check index below it) rather than a value index
static constexpr uint32_t kRaggedFinal = 0x80000000u;

// one level of products: the words at `at` hold chunk (n_chunks + 1 starts into idx), dst (n_chunks), idx
struct RaggedLevel {
  size_t n_chunks, at;
};

struct RaggedPlan {
  int glue = 1;                  // G: pairs per glued item of the batch
  size_t n_pairs = 0;            // offsets[n_checks] - offsets[0]
  size_t n_items[3] = {0, 0, 0}; // items of 4, 2 and 1 pairs, in value order
  size_t n_values = 0;           // the items' values and every non-final chunk product
  std::vector<RaggedLevel> levels;
  // gather (n_pairs pair indices relative to offsets[0]), then each level's chunk / dst / idx arrays.  uint32: the
  // pairs of one device's batch (194 bytes each) stay far below 2^32, and the entry point rejects more.
  std::vector<uint32_t> words;
  size_t n_items_total() const { return n_items[0] + n_items[1] + n_items[2]; }
};

// false if the offsets decrease anywhere
inline bool ragged_offsets_ok(const uint64_t* offsets, size_t n_checks) {
  for (size_t c = 0; c < n_checks; c++)
    if (offsets[c + 1] < offsets[c]) return false;
  return true;
}

// The plan of n_checks >= 1 checks over n_pairs >= 1 pairs.  glue: 0 for glue_pairs' choice, else 1, 2 or 4.
inline RaggedPlan ragged_plan(int sms, const uint64_t* offsets, size_t n_checks, BlockShape glued, int glue = 0) {
  RaggedPlan p;
  const uint64_t o0 = offsets[0];
  p.n_pairs = (size_t)(offsets[n_checks] - o0);
  p.glue = glue ? glue : glue_pairs(sms, p.n_pairs, kRaggedPairCost, glued);
  const size_t G = (size_t)p.glue;
  // items per check of each class
  auto split = [G](size_t k, size_t& i4, size_t& i2, size_t& i1) {
    i4 = G == 4 ? k / 4 : 0;
    const size_t rem = k - 4 * i4;
    i2 = G >= 2 ? rem / 2 : 0;
    i1 = rem - 2 * i2;
  };
  for (size_t c = 0; c < n_checks; c++) {
    size_t i4, i2, i1;
    split((size_t)(offsets[c + 1] - offsets[c]), i4, i2, i1);
    p.n_items[0] += i4;
    p.n_items[1] += i2;
    p.n_items[2] += i1;
  }
  const size_t n_items = p.n_items_total();
  p.words.resize(p.n_pairs);
  // level 0: check c's values, listed in cur[cb[c] .. cb[c + 1])
  std::vector<uint32_t> cur(n_items);
  std::vector<size_t> cb(n_checks + 1);
  {
    size_t pos[3] = {0, 4 * p.n_items[0], 4 * p.n_items[0] + 2 * p.n_items[1]};
    size_t val[3] = {0, p.n_items[0], p.n_items[0] + p.n_items[1]};
    size_t at = 0;
    for (size_t c = 0; c < n_checks; c++) {
      size_t cnt[3];
      split((size_t)(offsets[c + 1] - offsets[c]), cnt[0], cnt[1], cnt[2]);
      uint32_t src = (uint32_t)(offsets[c] - o0);
      cb[c] = at;
      for (int j = 0; j < 3; j++) {
        const size_t width = (size_t)4 >> j;
        for (size_t i = 0; i < cnt[j]; i++) {
          for (size_t v = 0; v < width; v++) p.words[pos[j]++] = src++;
          cur[at++] = (uint32_t)val[j]++;
        }
      }
    }
    cb[n_checks] = at;
  }
  p.n_values = n_items;
  // levels: every check is live at level 0 (an empty one as one empty chunk that writes 1); a check stays live while its
  // list is longer than one chunk
  std::vector<size_t> live(n_checks);
  for (size_t c = 0; c < n_checks; c++) live[c] = c;
  while (!live.empty()) {
    std::vector<uint32_t> chunk(1, 0), dst, idx, next;
    std::vector<size_t> next_cb(1, 0), next_live;
    for (size_t c : live) {
      const size_t b = cb[c], m = cb[c + 1] - b;
      if (m <= kRaggedChunk) {
        idx.insert(idx.end(), cur.begin() + b, cur.begin() + b + m);
        chunk.push_back((uint32_t)idx.size());
        dst.push_back(kRaggedFinal | (uint32_t)c);
        continue;
      }
      for (size_t s = 0; s < m; s += kRaggedChunk) {
        const size_t e = s + kRaggedChunk < m ? s + kRaggedChunk : m;
        idx.insert(idx.end(), cur.begin() + b + s, cur.begin() + b + e);
        chunk.push_back((uint32_t)idx.size());
        dst.push_back((uint32_t)p.n_values);
        next.push_back((uint32_t)p.n_values++);
      }
      next_live.push_back(c);
      next_cb.push_back(next.size());
    }
    p.levels.push_back({dst.size(), p.words.size()});
    p.words.insert(p.words.end(), chunk.begin(), chunk.end());
    p.words.insert(p.words.end(), dst.begin(), dst.end());
    p.words.insert(p.words.end(), idx.begin(), idx.end());
    // the live checks' lists of the next level, indexed by check again
    cur.swap(next);
    for (size_t i = 0; i < next_live.size(); i++) {
      cb[next_live[i]] = next_cb[i];
      cb[next_live[i] + 1] = next_cb[i + 1];
    }
    live.swap(next_live);
  }
  return p;
}

// Check boundaries cut[0] = 0 <= cut[1] <= ... <= cut[D] = n_checks for D devices: cut[g] is the first check that
// starts at or past g n_pairs / D pairs, so device g's pair count is within one check of n_pairs / D.
inline std::vector<size_t> ragged_cuts(const uint64_t* offsets, size_t n_checks, size_t D) {
  std::vector<size_t> cut(D + 1, n_checks);
  const uint64_t o0 = offsets[0], n_pairs = offsets[n_checks] - o0;
  size_t c = 0;
  cut[0] = 0;
  for (size_t g = 1; g < D; g++) {
    // (offsets[c] - o0) D >= g n_pairs, in 128 bits so that no 64-bit offsets overflow
    while (c < n_checks && (unsigned __int128)(offsets[c] - o0) * D < (unsigned __int128)g * n_pairs) c++;
    cut[g] = c;
  }
  return cut;
}

// How abc_heads_fused shares the persistent CTAs among the head pairs. Every pair runs the same conv1 (N = 256) on every
// tile, but its conv2 chunks and logit stores differ a lot (v2 heads: pair (4,5) = 1 + 360 channels, four chunks; pair
// (0,1) = 1 + 14, two chunks of 16), so an equal split leaves the light pairs idle while the heaviest one sets the time.
// Host-only; tests/test_heads_split_cpu.py calls it through a probe.
#pragma once
#include <cstdint>

namespace abc {

// Cost of one 128-pixel tile of a pair in tensor-pipe cycles of one SM, a model rather than a measurement:
//   conv1      : 2 x 9 x 4 MMAs of 128 x 256 x 16 at 8192 bf16 FLOP/clk = 128 clk each;
//   conv2      : 8 MMAs of 128 x nc x 16 per chunk, nc / 2 clk each plus the fixed per-MMA cost of ~60 clk (DESIGN.md 4.1);
//   logits     : 128 pixels x channels x 4 bytes at 64 B/clk -- the stores overlap the MMAs of the next tile only in part,
//                because the next chunk waits for the drain of the previous one.
inline int64_t hf_pair_tile_cost(int n_chunks, const int* nc, int logit_channels) {
  int64_t c = 72 * 128;
  for (int i = 0; i < n_chunks; ++i) c += 8 * (nc[i] / 2 + 60);
  return c + static_cast<int64_t>(128) * 4 * logit_channels / 64;
}

// ctas[p] for pairs p = 0 .. pairs-1: at least one each, then every further CTA (up to `sms` in total) to the pair with the
// largest cost per CTA -- the split that minimises the largest per-CTA share. A pair never gets more CTAs than tiles.
// Returns the total.
inline int hf_split_ctas(int pairs, const int64_t* cost, int sms, int num_tiles, int* ctas) {
  int total = 0;
  for (int p = 0; p < pairs; ++p) {
    ctas[p] = 1;
    ++total;
  }
  while (total < sms) {
    int best = -1;
    for (int p = 0; p < pairs; ++p) {
      if (ctas[p] >= num_tiles) continue;
      if (best < 0 || cost[p] * ctas[best] > cost[best] * ctas[p]) best = p;
    }
    if (best < 0) break;
    ++ctas[best];
    ++total;
  }
  return total;
}

}  // namespace abc

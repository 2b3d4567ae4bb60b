// Launch geometry of the BatchNorm-side passes of train_ops.cu: statistics, normalise + activation (+ max-pool), backward
// reduce / apply, and the fp32 NCHW -> P8 conversion with bias sums. All of them use one decomposition: grid.y = 8-channel
// plane, grid.z = image, grid.x strides over the pixels (or 2x2 pixel blocks) of that plane.
#pragma once
#include <algorithm>
#include <cstdlib>

#include "common.cuh"

namespace abc {

constexpr int kBnThreads = 256;        // 8 warps; the block reductions of these passes rely on it
constexpr int kBnBlocksPerSm = 12;     // grid cap, profiles/r02_train_ab_bn_grid.txt; ABCNET_BN_BLOCKS_PER_SM overrides it

// What a thread handles per grid-stride step, and how many such steps a block takes at least.
enum class BnPass {
  kStats,    // bn_stats: one 16-byte vector (8 channels of one pixel), 4 per thread
  kPixels,   // bn_act, backward reduce / apply, nchw_to_p8_ex: one vector, 2 per thread
  kPool,     // the fused 2x2 max-pool variants: one 2x2 block of vectors, 1 per thread
};

struct BnLaunch {
  dim3 grid;
  int block;
};

// grid.x: enough blocks to fill the machine, few enough that every thread streams several vectors and the per-block atomics
// stay negligible. The kernels stride over the plane, so any grid.x >= 1 is correct.
inline BnLaunch bn_launch_config(BnPass pass, int N, int planes, int H, int W, int sms = sm_count()) {
  static const long long per_sm = [] {
    const char* e = getenv("ABCNET_BN_BLOCKS_PER_SM");
    return e && atoi(e) > 0 ? atoi(e) : kBnBlocksPerSm;
  }();
  const long long items = pass == BnPass::kPool ? static_cast<long long>(H / 2) * (W / 2) : static_cast<long long>(H) * W;
  const long long per_block = kBnThreads * (pass == BnPass::kStats ? 4ll : pass == BnPass::kPixels ? 2ll : 1ll);
  const long long blocks = static_cast<long long>(planes) * N;
  const long long need = (items + per_block - 1) / per_block, cap = (sms * per_sm + blocks - 1) / blocks;
  return {dim3(static_cast<unsigned>(std::max(1ll, std::min(need, cap))), planes, N), kBnThreads};
}

}  // namespace abc

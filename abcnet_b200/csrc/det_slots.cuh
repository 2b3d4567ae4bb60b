// Slot layout of the deterministic reductions (torch.use_deterministic_algorithms): instead of adding its partial sums to
// the output with atomics, every producer (a CTA, or a fixed owner inside one) stores them with plain stores into a slot of
// its own in a caller-owned workspace, ws[slot * n + e] for output element e < n; then det_reduce (common.cu) sums the slots
// of each element in slot-index order. Slot counts follow the launch geometry, so one rule serves the launchers, the
// *_workspace_bytes queries of the C-ABI and tests/test_det_slots_cpu.py, which probes this header on the host.
#pragma once
#include <cstddef>
#include <cstdint>

#include "bn_launch.cuh"

#if defined(__CUDACC__)
#define ABC_DET_FN __host__ __device__ __forceinline__
#else
#define ABC_DET_FN inline
#endif

namespace abc {

ABC_DET_FN size_t det_slot_index(int slot, int n, int e) { return static_cast<size_t>(slot) * n + e; }
inline size_t det_ws_bytes(long long slots, long long n, size_t elem) { return static_cast<size_t>(slots * n) * elem; }

// wgrad_kernel: split-K over grid.x CTAs (each takes pixel tiles blockIdx.x, + gridDim.x, ...), grid.y = (co tile, ci tile,
// tap group). One slot per grid.x index; a slot holds the whole fp32 [ntaps][cout][cin] gradient, every element of it written
// by exactly one CTA of that grid.x column.
inline int wgrad_grid_x(int sms, int gy, int num_tiles) {
  int gx = (sms > 0 ? sms : 148) / gy;
  if (gx < 1) gx = 1;
  return gx > num_tiles ? num_tiles : gx;
}

// The BatchNorm-side passes (bn_launch.cuh): one slot per (image, grid.x block) of a channel plane, slot = z * grid.x + x.
inline int bn_slots(const BnLaunch& l) { return static_cast<int>(l.grid.x * l.grid.z); }
ABC_DET_FN int bn_slot(unsigned bx, unsigned bz, unsigned gx) { return static_cast<int>(bz * gx + bx); }

// Fused statistics of the convolution epilogue: 8 owners per CTA -- the 8 epilogue warps of the row-folded 16-channel
// variant, or (epilogue half, folded row) of the operand-swap variant -- so slot = blockIdx.x * 8 + owner.
constexpr int kConvStatOwners = 8;
inline int conv_stat_slots(int gx) { return gx * kConvStatOwners; }

// Stem weight gradients (conv_c1_wgrad*): one slot per block, 144 values (16 output channels x 9 taps) per input channel.
constexpr int kC1WgradBlocksDense = 148 * 4, kC1WgradBlocksSparse = 148 * 8;

// Loss kernels: one slot per block. The sparse-bias layout of loss_kernel_v2_p8 per slot: the 16 sums, the bias gradients of
// the two centre heads, then heads 1, 2, 3 (14 + 3 + 2 channels) and 5, 6, 7 (6 n_omega + n_omega + n_omega channels).
ABC_DET_FN int loss_elems(bool p8, int n_omega) { return p8 ? 16 + 2 + 19 + 8 * n_omega : 16; }
constexpr int kLossMaxOmegaDet = 64;   // shared-memory bound of the deterministic per-block bias sums (8 n_omega + 19 channels)

}  // namespace abc

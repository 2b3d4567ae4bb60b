// Implicit-GEMM convolution for sm_100a: TMA halo tiles -> tcgen05.mma (bf16 x bf16 -> fp32 in TMEM) -> fused epilogue.
//
// Replaces the cuDNN calls behind nn.Conv2d(3x3, pad 1) / nn.Conv2d(1x1) / nn.ConvTranspose2d(k3, s2) + crop of the
// reference U-Net (/root/reference/src/unet.py:12-17, :44-55, :66-70), with BatchNorm (eval) folded into the weights,
// ReLU / LeakyReLU, the 2x2 max-pool of Down (:30) and the channel concatenation of Up (:59) fused into the epilogue.
//
// Data layout ("P8"): activations are bf16 [N][C/8][H][W][8]. For one 8-channel plane, consecutive pixels are
// consecutive 16-byte vectors, which is exactly the SWIZZLE_NONE K-major core-matrix layout of the tcgen05 shared
// memory descriptor (8 rows x 16 bytes, contiguous). A (TH+2) x (TW+2) halo tile of KP planes is brought in by ONE
// 4-D TMA box (zero fill outside the image = conv padding) and the nine 3x3 taps are nine descriptors whose start
// address is shifted by (dy*(TW+2) + dx) * 16 bytes: the activation tile is read from L2 once per K-chunk, not 9 times.
//
//   GEMM M = 128 output pixels = 16 rows x 8 columns of one image (8-row core-matrix groups = tile rows, SBO = row pitch)
//   GEMM N = n_tile output channels (runtime, multiple of 16, <= 256)
//   GEMM K = 16 channels per MMA (two planes, LBO = plane pitch), KC = min(cin, 64) channels per pipeline stage
//
// Warp roles (384 threads, 1 CTA / SM, persistent over M tiles, blockIdx.y = N tile):
//   warp 0 : TMA producer for activation halo tiles (A ring)
//   warp 3 : bulk-copy producer for packed weight blocks (B ring, or resident when the layer's weights fit in smem)
//   warp 1 : MMA issuer (one thread), accumulators double-buffered in TMEM
//   warp 2 : TMEM allocation / release
//   warps 4-11 : epilogue (tcgen05.ld -> bias + activation -> bf16 P8 / fp32 NCHW stores, optional fused max-pool)
#include <cstdlib>
#include <cuda.h>
#include <cuda_bf16.h>

#include "common.cuh"
#include "det_slots.cuh"
#include "p8_device.cuh"
#include "ptx_sm100.cuh"

namespace abc {

constexpr int kMaxNA = 8;
constexpr int kMaxAcc = 8;           // accumulator stages in TMEM: 512 / (mt * n_tile) columns each, 2..8
constexpr int kMaxNB = 16;
constexpr uint32_t kHeaderBytes = 2048;
constexpr uint32_t kSmemBudget = 232448;   // 227 KB opt-in limit per CTA
constexpr int kThreads = 384;          // warps 0-3: producers / MMA / TMEM, warps 4-11: epilogue
constexpr int kTmemCols = 512;
// operand-swap mode: per epilogue warp a [16 pixels][32 channels] bf16 transposition buffer, rows padded to 80 bytes so
// that both the 2-byte column writes and the 16-byte row reads are bank-conflict free
constexpr uint32_t kSwapRowBytes = 80;
constexpr uint32_t kSwapWarpBytes = 16 * kSwapRowBytes;
constexpr uint32_t kSwapStageBytes = 8 * kSwapWarpBytes;   // 10240

struct ConvKParams {
  int N, H, W, tiles_x, tiles_y, groups_x, num_groups;   // a group = mt horizontally adjacent 16x8 tiles
  int in_plane_off, kp, nkc, ntaps, halo, n_tile, resident_b, na, nb, mt, nacc, acc_cols;
  int chunks_per_seg, blocks_per_ntile;      // K segments: chunk kc uses taps [seg_tap0[s], seg_tap0[s] + seg_ntaps[s]), s = kc / chunks_per_seg
  int seg_tap0[4], seg_ntaps[4];
  uint32_t a_stage_bytes, a_tile_bytes, a_plane_bytes, a_row_bytes, b_block_bytes;
  uint32_t tap_off[18];
  int dbg;                                   // experiments only (ABCNET_PAIR_DBG)
  int fold;                                  // row folding J (1, 2, 4): GEMM column = (16-channel block, row j, channel)
  int tile_rows;                             // image rows per tile: 16 * fold, or 32 in operand-swap mode
  uint32_t smem_a_off, smem_b_off;
  const uint8_t* wpack;
  const float* bias;
  int cout, act, out_mode;
  void* out;
  int out_planes, out_plane_off, out_H, out_W, out_sy, out_oy, out_sx, out_ox;
  void* pool_out;
  int pool_planes, pool_plane_off;
  int subpixel;                              // channels per sub-pixel phase (AbcConvDesc.subpixel), 0 = off
  int fp16;                                  // activations / weights are IEEE fp16 instead of bf16 (AbcConvDesc.act_fp16)
  // fused train-mode BatchNorm statistics (AbcConvDesc.stat_sum / stat_sq): per output channel sum / sum of squares of the
  // bf16-rounded outputs, accumulated per thread over the CTA's whole tile loop, one fp64 atomic per thread at the end
  double* stat_sum;
  double* stat_sq;
  // DET: the same per-thread / per-warp sums stored to slot blockIdx.x * 8 + owner of [slots][2 cout] (sums, then squares)
  // instead of the atomics (det_slots.cuh)
  double* stat_ws;
};

__device__ __forceinline__ float apply_act(float v, int act) {
  if (act == 1) return fmaxf(v, 0.f);
  if (act == 2) return v > 0.f ? v : 0.01f * v;
  return v;
}

__device__ __forceinline__ uint4 pack8_bf16(const float* v) {
  __nv_bfloat162 a = __floats2bfloat162_rn(v[0], v[1]);
  __nv_bfloat162 b = __floats2bfloat162_rn(v[2], v[3]);
  __nv_bfloat162 c = __floats2bfloat162_rn(v[4], v[5]);
  __nv_bfloat162 d = __floats2bfloat162_rn(v[6], v[7]);
  uint4 r;
  r.x = *reinterpret_cast<uint32_t*>(&a);
  r.y = *reinterpret_cast<uint32_t*>(&b);
  r.z = *reinterpret_cast<uint32_t*>(&c);
  r.w = *reinterpret_cast<uint32_t*>(&d);
  return r;
}

// 2x2 max-pool helpers on packed 16-bit pairs (bf16 or fp16: f16)
__device__ __forceinline__ uint32_t pool_max_bf16x2(uint32_t a, bool f16) {
  uint32_t b = __shfl_xor_sync(0xffffffffu, a, 1);
  a = max2_act16(a, b, f16);
  b = __shfl_xor_sync(0xffffffffu, a, 8);
  return max2_act16(a, b, f16);
}

__device__ __forceinline__ uint4 hmax_bf16x8(uint4 a, uint4 b, bool f16) {
  return make_uint4(max2_act16(a.x, b.x, f16), max2_act16(a.y, b.y, f16), max2_act16(a.z, b.z, f16), max2_act16(a.w, b.w, f16));
}

// max with the horizontally adjacent pixel (lane ^ 1)
__device__ __forceinline__ uint4 pool_hmax_x(uint4 q, bool f16) {
  uint4 o;
  o.x = __shfl_xor_sync(0xffffffffu, q.x, 1);
  o.y = __shfl_xor_sync(0xffffffffu, q.y, 1);
  o.z = __shfl_xor_sync(0xffffffffu, q.z, 1);
  o.w = __shfl_xor_sync(0xffffffffu, q.w, 1);
  return hmax_bf16x8(q, o, f16);
}

__device__ __forceinline__ uint4 pool_max_bf16x8(uint4 q, bool f16) {
  q.x = pool_max_bf16x2(q.x, f16);
  q.y = pool_max_bf16x2(q.y, f16);
  q.z = pool_max_bf16x2(q.z, f16);
  q.w = pool_max_bf16x2(q.w, f16);
  return q;
}

// KSTEPS: K-steps of 16 channels per pipeline stage = kp / 2 (1, 2, 3 or 4). RESIDENT: the layer's weights of one n-tile
// stay in shared memory (no B ring). Both are compile-time so that the MMA-issuing warp -- for the 16/32-channel layers
// THE pacing resource: 9 small MMAs per 128-pixel tile -- runs a branch-free, fully unrolled tap loop.
// CG2: CTA-pair mode (cta_group::2, launched as (2,1,1) clusters): the two CTAs of a pair take two consecutive groups,
// each loads its own activation tiles and HALF of every weight block (n_tile / 2 rows), the leader's MMA warp issues
// M = 256 instructions for both, and each CTA's epilogue drains its own 128 TMEM lanes. See ptx_sm100.cuh.
// SWAP: operand-swap mode (AbcConvDesc.swap_mn): M = the 128 output channels of the n-tile (the weight block is the A
// operand), N = 256 pixels (one 32 x 8 tile per pipeline stage is the B operand); accumulator = [channel][pixel].
// STATS: the non-swap epilogue of the row-folded 16-channel layers also accumulates the fused BatchNorm statistics (32 extra
// registers per epilogue thread, hence its own instantiation); the operand-swap epilogue does so behind a runtime flag.
// DET: the fused statistics go to the deterministic slots of p.stat_ws instead of fp64 atomics.
template <int KSTEPS, bool RESIDENT, bool CG2, bool SWAP = false, bool STATS = false, bool DET = false>
__global__ void __launch_bounds__(kThreads, 1)
conv_igemm_kernel(const __grid_constant__ CUtensorMap tmap, const ConvKParams p) {
  static_assert(!(CG2 && RESIDENT), "the CTA-pair variant streams its weights");
  static_assert(!(CG2 && SWAP), "operand swap is a single-CTA mode");
  static_assert(!(STATS && (SWAP || CG2)), "STATS is the non-swap, single-CTA variant");
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t sbase = smem_u32(smem);
  const int warp = static_cast<int>(warp_id_uniform());   // provably warp-uniform
  const int lane = threadIdx.x & 31;
  const uint32_t cta_rank = CG2 ? cluster_ctarank() : 0u;
  const bool leader = cta_rank == 0;

  // barrier slots (8 bytes each)
  const uint32_t bar_a_full = sbase;                        // [kMaxNA]
  const uint32_t bar_a_empty = sbase + 8 * kMaxNA;          // [kMaxNA]
  const uint32_t bar_b_full = sbase + 8 * (2 * kMaxNA);     // [kMaxNB]
  const uint32_t bar_b_empty = bar_b_full + 8 * kMaxNB;     // [kMaxNB]
  const uint32_t bar_acc_full = bar_b_empty + 8 * kMaxNB;   // [kMaxAcc]
  const uint32_t bar_acc_empty = bar_acc_full + 8 * kMaxAcc;   // [kMaxAcc]
  static_assert(8 * (2 * kMaxNA + 2 * kMaxNB + 2 * kMaxAcc) <= 768, "barrier slots overflow the header");
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + 768);
  float* bias_s = reinterpret_cast<float*>(smem + 1024);    // [256]

  if (threadIdx.x == 0) {
    // pair mode: the leader's "full" barriers also collect one relayed arrival from the peer CTA (its data has landed),
    // and its "accumulator empty" barriers the epilogue warps of both CTAs
    const uint32_t full_count = (CG2 && leader && !(p.dbg & 1)) ? 2 : 1;
    for (int i = 0; i < kMaxNA; ++i) {
      mbar_init(bar_a_full + 8 * i, full_count);
      mbar_init(bar_a_empty + 8 * i, 1);
    }
    for (int i = 0; i < kMaxNB; ++i) {
      mbar_init(bar_b_full + 8 * i, full_count);
      mbar_init(bar_b_empty + 8 * i, 1);
    }
    for (int i = 0; i < kMaxAcc; ++i) {
      mbar_init(bar_acc_full + 8 * i, 1);
      mbar_init(bar_acc_empty + 8 * i, CG2 ? 16 : 8);
    }
    fence_mbar_init();
    tma_prefetch_desc(&tmap);
  }
  if (CG2) cluster_sync_all();              // both CTAs' barriers exist before the pair-wide TMEM allocation / any remote arrival
  if (warp == 2) {
    if (CG2) tmem_alloc_pair<kTmemCols>(smem_u32(tmem_slot));
    else tmem_alloc<kTmemCols>(smem_u32(tmem_slot));
  }
  for (int i = threadIdx.x; i < p.n_tile; i += kThreads) bias_s[i] = p.bias[blockIdx.y * p.n_tile + i];
  uint32_t* utab = reinterpret_cast<uint32_t*>(smem + 800);   // [<= 32] per-unit constants of the epilogue
  uint32_t* utab2 = reinterpret_cast<uint32_t*>(smem + 928);  // [<= 16] sub-pixel mode: (output plane of the unit) << 16 | pixel offset
  if (threadIdx.x < ((p.mt * p.n_tile) >> 4)) {
    const int col = threadIdx.x << 4;
    const int ti = col / p.n_tile;
    const int ul = (col - ti * p.n_tile) >> 4;               // 16-column unit within the tile = bias unit
    const int b16 = ul / p.fold;
    utab[threadIdx.x] = static_cast<uint32_t>(ti) | (ul << 8) | (b16 << 16) | ((ul - b16 * p.fold) << 24);
    if (p.subpixel > 0 && threadIdx.x < 16) {
      // GEMM column c = phase * subpixel + channel: the unit goes to output pixel (2y + py, 2x + px), plane channel / 8
      const int c0 = blockIdx.y * p.n_tile + (b16 << 4);
      const int ph = c0 / p.subpixel, chn = c0 - ph * p.subpixel;
      utab2[threadIdx.x] = (static_cast<uint32_t>(chn >> 3) << 16) | static_cast<uint32_t>((ph >> 1) * p.out_W + (ph & 1));
    }
  }
  tc_fence_before();
  if (CG2) cluster_sync_all();
  else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_slot);
  // groups: a CTA takes g_first, g_first + gridDim.x, ...; in pair mode both CTAs iterate over the leader's sequence and
  // the peer takes the following group (clamped to the last one when the count is odd: computed, not stored)
  const int g_first = CG2 ? static_cast<int>(blockIdx.x & ~1u) : static_cast<int>(blockIdx.x);

  const int groups_per_img = p.groups_x * p.tiles_y;
  const uint32_t a_region = sbase + p.smem_a_off;
  const uint32_t b_region = sbase + p.smem_b_off;
  const int blocks_per_ntile = p.blocks_per_ntile;

  if (warp == 0) {
    // ------------------------------------------------------------------ A producer (TMA halo tiles)
    int stage = 0;
    uint32_t phase = 0;
    for (int gp = g_first; gp < p.num_groups; gp += gridDim.x) {
      const int g = CG2 ? min(gp + static_cast<int>(cta_rank), p.num_groups - 1) : gp;
      const int n = g / groups_per_img;
      const int rem = g - n * groups_per_img;
      const int ty = rem / p.groups_x;
      const int tx0 = (rem - ty * p.groups_x) * p.mt;
      const int c1 = ty * p.tile_rows - p.halo;
      for (int kc = 0; kc < p.nkc; ++kc) {
        mbar_wait(bar_a_empty + 8 * stage, phase ^ 1);
        if (elect_one()) {
          mbar_arrive_expect_tx(bar_a_full + 8 * stage, p.a_stage_bytes);
          for (int i = 0; i < p.mt; ++i)
            tma_load_4d(a_region + stage * p.a_stage_bytes + i * p.a_tile_bytes, &tmap, bar_a_full + 8 * stage,
                        ((tx0 + i) * 8 - p.halo) * 8, c1, p.in_plane_off + kc * p.kp, n);
        }
        __syncwarp();
        if (++stage == p.na) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else if (warp == 3) {
    // ------------------------------------------------------------------ B producer (packed weight blocks)
    // pair mode: p.b_block_bytes is this CTA's half block; the pack holds [block][half] (see abc_conv_igemm)
    const size_t b_src_stride = CG2 ? 2 * static_cast<size_t>(p.b_block_bytes) : p.b_block_bytes;
    const uint8_t* wsrc = p.wpack + static_cast<size_t>(blockIdx.y) * blocks_per_ntile * b_src_stride +
                          (CG2 ? cta_rank * p.b_block_bytes : 0u);
    if (RESIDENT) {
      if (blockIdx.x < p.num_groups && elect_one()) {
        mbar_arrive_expect_tx(bar_b_full, static_cast<uint32_t>(blocks_per_ntile) * p.b_block_bytes);
        for (int blk = 0; blk < blocks_per_ntile; ++blk)
          bulk_load_1d(b_region + blk * p.b_block_bytes, wsrc + static_cast<size_t>(blk) * p.b_block_bytes,
                       p.b_block_bytes, bar_b_full);
      }
      __syncwarp();
    } else {
      int stage = 0;
      uint32_t phase = 0;
      for (int g = g_first; g < p.num_groups; g += gridDim.x) {
        for (int blk = 0; blk < blocks_per_ntile; ++blk) {
          mbar_wait(bar_b_empty + 8 * stage, phase ^ 1);
          if (elect_one()) {
            mbar_arrive_expect_tx(bar_b_full + 8 * stage, p.b_block_bytes);
            bulk_load_1d(b_region + stage * p.b_block_bytes, wsrc + static_cast<size_t>(blk) * b_src_stride,
                         p.b_block_bytes, bar_b_full + 8 * stage);
          }
          __syncwarp();
          if (++stage == p.nb) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1 && CG2 && !leader) {
    // ------------------------------------------------------------------ peer CTA: relay "my operands have landed" to the
    // leader's full barriers (same stage sequence as the leader's MMA loop; one arrival per stage use)
    int a_stage = 0, b_stage = 0;
    uint32_t a_phase = 0, b_phase = 0;
    for (int g = g_first; g < p.num_groups; g += gridDim.x) {
      for (int kc = 0; kc < p.nkc; ++kc) {
        mbar_wait(bar_a_full + 8 * a_stage, a_phase);
        if (!(p.dbg & 1) && elect_one()) mbar_arrive_cluster(mapa_cluster(bar_a_full + 8 * a_stage, 0));
        __syncwarp();
        if (++a_stage == p.na) {
          a_stage = 0;
          a_phase ^= 1;
        }
        for (int t = 0; t < p.ntaps; ++t) {
          mbar_wait(bar_b_full + 8 * b_stage, b_phase);
          if (!(p.dbg & 1) && elect_one()) mbar_arrive_cluster(mapa_cluster(bar_b_full + 8 * b_stage, 0));
          __syncwarp();
          if (++b_stage == p.nb) {
            b_stage = 0;
            b_phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    const bool f16 = p.fp16 != 0;
    const uint32_t idesc = SWAP ? umma_idesc_16(128, 256, 0, 0, f16) : umma_idesc_16(CG2 ? 256 : 128, p.n_tile, 0, 0, f16);
    const int b_rows = CG2 ? p.n_tile >> 1 : p.n_tile;          // weight rows held by this CTA
    auto mma = [&](uint32_t d, uint32_t a_lo, uint32_t a_hi_, uint32_t b_lo, uint32_t b_hi_, uint32_t acc_) {
      if (CG2) umma_bf16_lohi_pair(d, a_lo, a_hi_, b_lo, b_hi_, idesc, acc_);
      else if (SWAP) umma_bf16_lohi(d, b_lo, b_hi_, a_lo, a_hi_, idesc, acc_);     // weights = A (M), pixels = B (N)
      else umma_bf16_lohi(d, a_lo, a_hi_, b_lo, b_hi_, idesc, acc_);
    };
    auto commit = [&](uint32_t bar) {
      if (CG2) umma_commit_pair(bar);
      else umma_commit(bar);
    };
    // descriptors as (lo, hi) halves: hi is constant, lo = (smem address >> 4) advances by plain 32-bit adds
    const uint64_t a_hi64 = umma_desc_hi(p.a_plane_bytes, p.a_row_bytes * p.fold);   // LBO = plane pitch, SBO = pitch of J tile rows
    // weights: planar (SWIZZLE_NONE) blocks [kc/8][rows][8]; in pair mode 128-byte-swizzled rows of 64 channels -- the half
    // of B that the peer SM fetches from this CTA's shared memory moves in 128-byte rows instead of 16-byte pieces
    // (measured: 344 clk per N = 256 MMA with planar blocks, i.e. ~12 B/clk across the pair)
    const uint64_t b_hi64 = CG2 ? umma_desc_hi_sw128() : umma_desc_hi(b_rows * 16, 128);   // LBO = plane pitch, SBO = 8 rows * 16 B
    const uint32_t a_hi = static_cast<uint32_t>(a_hi64 >> 32), b_hi = static_cast<uint32_t>(b_hi64 >> 32);
    const uint32_t a_lo0 = static_cast<uint32_t>(a_hi64) | (a_region >> 4);
    const uint32_t b_lo0 = static_cast<uint32_t>(b_hi64) | (b_region >> 4);
    const uint32_t a_kstep = (2 * p.a_plane_bytes) >> 4, b_kstep = CG2 ? 2u : (2 * b_rows * 16) >> 4;
    const uint32_t a_tile16 = p.a_tile_bytes >> 4, a_stage16 = p.a_stage_bytes >> 4, b_block16 = p.b_block_bytes >> 4;
    int a_stage = 0, b_stage = 0, acc = 0;
    uint32_t a_phase = 0, b_phase = 0, acc_phase = 0;
    if (RESIDENT && blockIdx.x < p.num_groups) {
      mbar_wait(bar_b_full, 0);
      tc_fence_after();
    }
    if (p.chunks_per_seg == p.nkc) {
      // ---- fast path (one K segment = every layer of the forward pass and every 3x3 data gradient)
      uint32_t tap16[18];
#pragma unroll
      for (int t = 0; t < 18; ++t) tap16[t] = p.tap_off[t] >> 4;
      const int ntaps = p.ntaps, nkc = p.nkc, mt = p.mt, n_tile = p.n_tile, na = p.na, nb = p.nb, nacc = p.nacc;
      const uint32_t acc_cols = p.acc_cols;
      for (int g = g_first; g < p.num_groups; g += gridDim.x) {
        mbar_wait(bar_acc_empty + 8 * acc, acc_phase ^ 1);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + acc * acc_cols;
        uint32_t b_res = b_lo0;                               // resident weights: blocks in (chunk, tap) order
        for (int kc = 0; kc < nkc; ++kc) {
          mbar_wait(bar_a_full + 8 * a_stage, a_phase);
          tc_fence_after();
          const uint32_t a_base = a_lo0 + a_stage * a_stage16;
#pragma unroll
          for (int t = 0; t < 18; ++t) {
            if (t < ntaps) {                                  // warp-uniform
              uint32_t b_base;
              if (RESIDENT) {
                b_base = b_res;
                b_res += b_block16;
              } else {
                mbar_wait(bar_b_full + 8 * b_stage, b_phase);
                tc_fence_after();
                b_base = b_lo0 + b_stage * b_block16;
              }
              const uint32_t a_tap = a_base + tap16[t];
              const uint32_t acc0 = (kc | t) != 0 ? 1u : 0u;
              if (elect_one()) {
                uint32_t d_col = tmem_d, a_t = a_tap;
                for (int i = 0; i < mt; ++i, d_col += n_tile, a_t += a_tile16) {
#pragma unroll
                  for (int j = 0; j < KSTEPS; ++j)
                    mma(d_col, a_t + j * a_kstep, a_hi, b_base + j * b_kstep, b_hi, j != 0 ? 1u : acc0);
                }
                if (!RESIDENT) commit(bar_b_empty + 8 * b_stage);
              }
              __syncwarp();
              if (!RESIDENT) {
                if (++b_stage == nb) {
                  b_stage = 0;
                  b_phase ^= 1;
                }
              }
            }
          }
          if (elect_one()) commit(bar_a_empty + 8 * a_stage);
          __syncwarp();
          if (++a_stage == na) {
            a_stage = 0;
            a_phase ^= 1;
          }
        }
        if (elect_one()) commit(bar_acc_full + 8 * acc);
        __syncwarp();
        if (++acc == nacc) {
          acc = 0;
          acc_phase ^= 1;
        }
      }
    } else
    for (int g = blockIdx.x; g < p.num_groups; g += gridDim.x) {
      mbar_wait(bar_acc_empty + 8 * acc, acc_phase ^ 1);
      tc_fence_after();
      const uint32_t tmem_d = tmem_base + acc * p.acc_cols;
      int blk = 0;
      for (int kc = 0; kc < p.nkc; ++kc) {
        mbar_wait(bar_a_full + 8 * a_stage, a_phase);
        tc_fence_after();
        const uint32_t a_base = a_lo0 + a_stage * a_stage16;
        const int seg = kc / p.chunks_per_seg;
        const int t_begin = p.seg_tap0[seg], t_end = t_begin + p.seg_ntaps[seg];
        for (int t = t_begin; t < t_end; ++t, ++blk) {
          uint32_t b_base;
          if (RESIDENT) {
            b_base = b_lo0 + blk * b_block16;
          } else {
            mbar_wait(bar_b_full + 8 * b_stage, b_phase);
            tc_fence_after();
            b_base = b_lo0 + b_stage * b_block16;
          }
          const uint32_t a_tap = a_base + (p.tap_off[t] >> 4);
          const uint32_t acc0 = (kc | (t - t_begin)) != 0 ? 1u : 0u;
          if (elect_one()) {
#pragma unroll 2
            for (int i = 0; i < p.mt; ++i) {
#pragma unroll
              for (int j = 0; j < KSTEPS; ++j)
                umma_bf16_lohi(tmem_d + i * p.n_tile, a_tap + i * a_tile16 + j * a_kstep, a_hi, b_base + j * b_kstep, b_hi,
                               idesc, j != 0 ? 1u : acc0);
            }
            if (!RESIDENT) umma_commit(bar_b_empty + 8 * b_stage);
          }
          __syncwarp();
          if (!RESIDENT) {
            if (++b_stage == p.nb) {
              b_stage = 0;
              b_phase ^= 1;
            }
          }
        }
        if (elect_one()) umma_commit(bar_a_empty + 8 * a_stage);
        __syncwarp();
        if (++a_stage == p.na) {
          a_stage = 0;
          a_phase ^= 1;
        }
      }
      if (elect_one()) umma_commit(bar_acc_full + 8 * acc);
      __syncwarp();
      if (++acc == p.nacc) {
        acc = 0;
        acc_phase ^= 1;
      }
    }
  } else if (warp >= 4 && SWAP) {
    // ------------------------------------------------------------------ epilogue, operand-swap mode
    // Accumulator: TMEM lane = output channel of the n-tile, column = pixel r * 8 + c of the 32 x 8 tile. Warp (q, eh)
    // drains channels [32 q, 32 q + 32) of tile rows [16 eh, 16 eh + 16): 16 columns (two tile rows) per TMEM load with
    // the next load in flight, bias + activation, bf16, then an 8 x 8 (channel x pixel) transposition through the warp's
    // private shared-memory buffer: lane (g, i) ends up with the 8 channels of plane g for pixel column i -> one 16-byte
    // store per lane, 128 contiguous bytes per (plane, tile row).
    const int q = warp & 3;
    const int eh = (warp - 4) >> 2;
    const int n0 = blockIdx.y * p.n_tile;
    const float bias = bias_s[q * 32 + lane];
    const float slope = p.act == 1 ? 0.f : (p.act == 2 ? 0.01f : 1.f);     // act(v) = max(v, slope * v)
    const int g8 = lane >> 3, i8 = lane & 7;
    // row folding J: GEMM row m = j * (128 / J) + channel, pixel column (r, c) = image row (ty * 32 + r) * J + j. The 8-channel
    // group this lane stores after the transposition starts at GEMM row m0.
    const int J = p.fold, cpj = 128 / J;
    const int m0 = q * 32 + g8 * 8;
    const int fj = m0 / cpj, ch0 = m0 - fj * cpj;
    uint8_t* stage = smem + kHeaderBytes + (warp - 4) * kSwapWarpBytes;
    unsigned short* st_w = reinterpret_cast<unsigned short*>(stage) + lane;                 // + pixel * (kSwapRowBytes / 2)
    const bool f16 = p.fp16 != 0;
    const uint4* st_r = reinterpret_cast<const uint4*>(stage + i8 * kSwapRowBytes + g8 * 16);  // + row * 8 * kSwapRowBytes / 16
    const bool plane_ok = (n0 + ch0) < p.cout;
    const size_t out_plane_px = static_cast<size_t>(p.out_H) * p.out_W;
    // fused statistics: this thread's own GEMM row (before the transposition) = (folded row fj_own, channel)
    const bool do_stats = p.stat_sum != nullptr;
    const int m_own = q * 32 + lane;
    const int fj_own = m_own / cpj;
    float st_s = 0.f, st_q = 0.f;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int g = g_first; g < p.num_groups; g += gridDim.x) {
      const int n = g / groups_per_img;
      const int rem = g - n * groups_per_img;
      const int ty = rem / p.groups_x;
      const int tx = rem - ty * p.groups_x;
      const int x = tx * 8 + i8;
      const int y0 = (ty * 32 + eh * 16) * J + fj;
      uint4* obase = reinterpret_cast<uint4*>(p.out) +
                     (static_cast<size_t>(n) * p.out_planes + p.out_plane_off + ((n0 + ch0) >> 3)) * out_plane_px +
                     static_cast<size_t>(p.out_oy) * p.out_W + (x * p.out_sx + p.out_ox);
      const bool col_ok = plane_ok && x < p.W;
      const uint32_t tbase = tmem_base + acc * p.acc_cols + (static_cast<uint32_t>(q * 32) << 16) + eh * 128;
      // statistics: validity of the 8 pixel columns of this tile (bit c: column tx * 8 + c is inside the image)
      const int x_left = p.W - tx * 8;
      const uint32_t xmask8 = x_left >= 8 ? 0xffu : ((1u << (x_left > 0 ? x_left : 0)) - 1u);
      const int yo0 = (ty * 32 + eh * 16) * J + fj_own;
      mbar_wait(bar_acc_full + 8 * acc, acc_phase);
      tc_fence_after();
      auto process = [&](uint32_t (&raw)[16], int it) {
        uint32_t vmask = 0;
        if (do_stats)
          vmask = ((yo0 + (it * 2) * J) < p.H ? xmask8 : 0u) | ((yo0 + (it * 2 + 1) * J) < p.H ? (xmask8 << 8) : 0u);
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          const float t = __uint_as_float(raw[i]) + bias;
          const unsigned short hv = to_act16(fmaxf(t, t * slope), f16);
          st_w[i * (kSwapRowBytes / 2)] = hv;
          if (do_stats && ((vmask >> i) & 1u)) {              // training (bf16 only, checked on the host)
            const float r = __uint_as_float(static_cast<uint32_t>(hv) << 16);
            st_s += r;
            st_q = fmaf(r, r, st_q);
          }
        }
        __syncwarp();
#pragma unroll
        for (int rr = 0; rr < 2; ++rr) {
          const uint4 val = st_r[rr * (8 * kSwapRowBytes / 16)];
          const int y = y0 + (it * 2 + rr) * J;
          if (col_ok && y < p.H) obase[static_cast<size_t>(y * p.out_sy) * p.out_W] = val;
        }
        __syncwarp();
      };
      uint32_t raw_a[16], raw_b[16];
      tmem_ld16(tbase, raw_a);
#pragma unroll 1
      for (int it = 0; it < 8; it += 2) {
        tmem_ld_wait();
        tmem_ld16(tbase + (it + 1) * 16, raw_b);
        process(raw_a, it);
        tmem_ld_wait();
        if (it + 2 < 8) tmem_ld16(tbase + (it + 2) * 16, raw_a);
        process(raw_b, it + 1);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_acc_empty + 8 * acc);
      if (++acc == p.nacc) {
        acc = 0;
        acc_phase ^= 1;
      }
    }
    if (do_stats) {
      const int ch = n0 + (m_own - fj_own * cpj);
      if (ch < p.cout) {
        if constexpr (DET) {            // owner = (epilogue half, folded row)
          const int slot = blockIdx.x * kConvStatOwners + eh * J + fj_own;
          p.stat_ws[det_slot_index(slot, 2 * p.cout, ch)] = static_cast<double>(st_s);
          p.stat_ws[det_slot_index(slot, 2 * p.cout, p.cout + ch)] = static_cast<double>(st_q);
        } else {
          atomicAdd(p.stat_sum + ch, static_cast<double>(st_s));
          atomicAdd(p.stat_sq + ch, static_cast<double>(st_q));
        }
      }
    }
  } else if (warp >= 4) {
    // ------------------------------------------------------------------ epilogue (8 warps: two per TMEM lane quarter)
    // The accumulators of one group are mt * n_tile contiguous TMEM columns. They are drained in 16-column units, two
    // units per 32-column load; the two warps of a lane quarter take alternate loads and each keeps the next load in
    // flight while it converts / stores the current one. For the 16 / 32-channel layers and the 1x1 heads this loop, not
    // the MMA, paces the kernel (ncu source view), so per-unit integer work is table-driven: utab[u] holds what depends on
    // the unit index only, everything that depends on the group is hoisted out of the unit loop.
    const int q = warp & 3;                 // TMEM lane quarter == warp_id % 4
    const int eh = (warp - 4) >> 2;         // which of the two interleaved chunk streams
    const int m = q * 32 + lane;            // GEMM row = pixel within the 16 x 8 tile
    const int r = m >> 3, c = m & 7;
    const int n0 = blockIdx.y * p.n_tile;
    const int units = (p.mt * p.n_tile) >> 4;
    const int nchunks = (units + 1) >> 1;
    const float slope = p.act == 1 ? 0.f : (p.act == 2 ? 0.01f : 1.f);     // act(v) = max(v, slope * v)
    const bool f16 = p.fp16 != 0;
    const float4* bias4 = reinterpret_cast<const float4*>(bias_s);
    const size_t out_plane_px = static_cast<size_t>(p.out_H) * p.out_W;
    const int ph = p.H >> 1, pw = p.W >> 1;
    const size_t pool_plane_px = static_cast<size_t>(ph) * pw;
    int acc = 0;
    uint32_t acc_phase = 0;
    float sacc[STATS ? 16 : 1], qacc[STATS ? 16 : 1];       // fused statistics of the 16 channels (cout == 16, row-folded)
#pragma unroll
    for (int i = 0; i < (STATS ? 16 : 1); ++i) sacc[i] = qacc[i] = 0.f;
    const uint32_t acc_empty_base = CG2 ? mapa_cluster(bar_acc_empty, 0) : bar_acc_empty;   // the leader's barriers
    for (int gp = g_first; gp < p.num_groups; gp += gridDim.x) {
      const int g = CG2 ? min(gp + static_cast<int>(cta_rank), p.num_groups - 1) : gp;
      const bool g_valid = !CG2 || (gp + static_cast<int>(cta_rank) < p.num_groups);   // odd group count: the peer's last group is a dummy
      const int n = g / groups_per_img;
      const int rem = g - n * groups_per_img;
      const int ty = rem / p.groups_x;
      const int tx0 = (rem - ty * p.groups_x) * p.mt;
      const int ybase = (ty * 16 + r) * p.fold;            // row of this thread's pixel (fold: of its first pixel)
      const int xbase = tx0 * 8 + c;
      // pixel offset of (ybase, xbase) in one output plane, and the plane index of channel n0 of image n
      const size_t out_px0 = static_cast<size_t>(ybase * p.out_sy + p.out_oy) * p.out_W + (xbase * p.out_sx + p.out_ox);
      const size_t out_pl0 = static_cast<size_t>(n) * p.out_planes + p.out_plane_off + (n0 >> 3);
      const size_t pool_px0 = static_cast<size_t>(ybase >> 1) * pw + (xbase >> 1);
      const size_t pool_pl0 = static_cast<size_t>(n) * p.pool_planes + p.pool_plane_off + (n0 >> 3);
      const uint32_t tbase = tmem_base + acc * p.acc_cols + (static_cast<uint32_t>(q * 32) << 16);
      mbar_wait(bar_acc_full + 8 * acc, acc_phase);
      tc_fence_after();

      auto load = [&](uint32_t (&raw)[2][16], int ch) {
        tmem_ld16(tbase + ch * 32, raw[0]);
        if (2 * ch + 1 < units) tmem_ld16(tbase + ch * 32 + 16, raw[1]);
      };
      auto process = [&](uint32_t (&raw)[2][16], int ch) {
        uint4 keep0 = make_uint4(0, 0, 0, 0), keep1 = keep0;    // fold + pool: the even row's packed values
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          const int u = 2 * ch + half;
          if (u >= units) break;                            // warp-uniform
          // utab[u] = (tile ti | bias unit << 8 | 16-channel block b << 16 | folded row j << 24); without folding j == 0
          const uint32_t info = utab[u];
          const int ti = info & 0xff, bu = (info >> 8) & 0xff, b16 = (info >> 16) & 0xff, j = info >> 24;
          if (tx0 + ti >= p.tiles_x) continue;              // warp-uniform
          const int ch0 = n0 + (b16 << 4);
          const int y = ybase + j;
          const int x = xbase + ti * 8;
          const bool valid = (y < p.H) && (x < p.W) && (ch0 < p.cout) && g_valid;
          const bool two = (ch0 + 8) < p.cout;
          float v[16];
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const float4 bb = bias4[bu * 4 + i];
            float t0 = __uint_as_float(raw[half][4 * i + 0]) + bb.x, t1 = __uint_as_float(raw[half][4 * i + 1]) + bb.y;
            float t2 = __uint_as_float(raw[half][4 * i + 2]) + bb.z, t3 = __uint_as_float(raw[half][4 * i + 3]) + bb.w;
            v[4 * i + 0] = fmaxf(t0, t0 * slope);
            v[4 * i + 1] = fmaxf(t1, t1 * slope);
            v[4 * i + 2] = fmaxf(t2, t2 * slope);
            v[4 * i + 3] = fmaxf(t3, t3 * slope);
          }
          if (p.out_mode == 0) {
            uint4 q0 = pack8_act16(v, f16), q1 = pack8_act16(v + 8, f16);
            if constexpr (STATS) {
              if (valid) {
                float r[16];
                unpack8u(q0, r);
                unpack8u(q1, r + 8);
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                  sacc[i] += r[i];
                  qacc[i] = fmaf(r[i], r[i], qacc[i]);
                }
              }
            }
            if (p.out != nullptr && valid) {
              uint4* o;
              if (p.subpixel > 0) {
                const uint32_t t2 = utab2[u];
                o = reinterpret_cast<uint4*>(p.out) +
                    (static_cast<size_t>(n) * p.out_planes + p.out_plane_off + (t2 >> 16)) * out_plane_px + out_px0 + (t2 & 0xffffu) +
                    ti * 8 * p.out_sx;
              } else {
                o = reinterpret_cast<uint4*>(p.out) + (out_pl0 + 2 * b16) * out_plane_px + out_px0 +
                    static_cast<size_t>(j * p.out_sy) * p.out_W + ti * 8 * p.out_sx;
              }
              o[0] = q0;
              if (two) o[out_plane_px] = q1;
            }
            if (p.pool_out != nullptr) {
              // 2x2 max-pool on the packed bf16 pairs (rounding is monotonic: max of rounded == rounded max).
              bool write;
              if (p.fold == 1) {
                // lane <-> pixel: xor 1 = x neighbour, xor 8 = y neighbour
                q0 = pool_max_bf16x8(q0, f16);
                q1 = pool_max_bf16x8(q1, f16);
                write = !(c & 1) && !(r & 1);
              } else {
                // folded rows: the vertical neighbour (j ^ 1) is the other half of this chunk, in the same thread
                if (half == 0) {
                  keep0 = q0;
                  keep1 = q1;
                  continue;
                }
                q0 = pool_hmax_x(hmax_bf16x8(q0, keep0, f16), f16);
                q1 = pool_hmax_x(hmax_bf16x8(q1, keep1, f16), f16);
                write = !(c & 1);
              }
              if (valid && write) {
                uint4* o = reinterpret_cast<uint4*>(p.pool_out) + (pool_pl0 + 2 * b16) * pool_plane_px + pool_px0 +
                           static_cast<size_t>(j >> 1) * pw + ti * 4;
                o[0] = q0;
                if (two) o[pool_plane_px] = q1;
              }
            }
          } else if (p.out_mode == 2) {
            // fp32 planar-8 logits [N][planes][H][W][8]: 32 contiguous bytes per thread and plane
            if (valid) {
              float4* o = reinterpret_cast<float4*>(p.out) + 2 * ((out_pl0 + 2 * b16) * out_plane_px + out_px0 + ti * 8 * p.out_sx);
              o[0] = make_float4(v[0], v[1], v[2], v[3]);
              o[1] = make_float4(v[4], v[5], v[6], v[7]);
              if (two) {
                o += 2 * out_plane_px;
                o[0] = make_float4(v[8], v[9], v[10], v[11]);
                o[1] = make_float4(v[12], v[13], v[14], v[15]);
              }
            }
          } else if (valid) {
            float* o = reinterpret_cast<float*>(p.out) + (static_cast<size_t>(n) * p.cout + ch0) * out_plane_px + out_px0 +
                       ti * 8 * p.out_sx;
#pragma unroll
            for (int i = 0; i < 16; ++i)
              if (ch0 + i < p.cout) o[i * out_plane_px] = v[i];
          }
        }
      };

      uint32_t raw_a[2][16], raw_b[2][16];
      int ch = eh;
      if (ch < nchunks) {
        load(raw_a, ch);
        while (true) {
          tmem_ld_wait();
          if (ch + 2 < nchunks) load(raw_b, ch + 2);
          process(raw_a, ch);
          ch += 2;
          if (ch >= nchunks) break;
          tmem_ld_wait();
          if (ch + 2 < nchunks) load(raw_a, ch + 2);
          process(raw_b, ch);
          ch += 2;
          if (ch >= nchunks) break;
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (CG2) mbar_arrive_cluster(acc_empty_base + 8 * acc);
        else mbar_arrive(bar_acc_empty + 8 * acc);
      }
      if (++acc == p.nacc) {
        acc = 0;
        acc_phase ^= 1;
      }
    }
    if constexpr (STATS) {
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        float a = sacc[i], b = qacc[i];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          a += __shfl_xor_sync(0xffffffffu, a, o);
          b += __shfl_xor_sync(0xffffffffu, b, o);
        }
        if (lane == 0 && n0 + i < p.cout) {
          if constexpr (DET) {          // owner = epilogue warp
            const int slot = blockIdx.x * kConvStatOwners + (warp - 4);
            p.stat_ws[det_slot_index(slot, 2 * p.cout, n0 + i)] = static_cast<double>(a);
            p.stat_ws[det_slot_index(slot, 2 * p.cout, p.cout + n0 + i)] = static_cast<double>(b);
          } else {
            atomicAdd(p.stat_sum + n0 + i, static_cast<double>(a));
            atomicAdd(p.stat_sq + n0 + i, static_cast<double>(b));
          }
        }
      }
    }
  }

  tc_fence_before();
  if (CG2) cluster_sync_all();          // the peer may still be reading its accumulators / this CTA's barriers
  else __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    if (CG2) tmem_dealloc_pair<kTmemCols>(tmem_base);
    else tmem_dealloc<kTmemCols>(tmem_base);
  }
}

// ----------------------------------------------------------------------------------------------- host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() { return reinterpret_cast<EncodeTiledFn>(tensor_map_encode_fn()); }

static int conv_kc(int cin) { return cin < 64 ? cin : 64; }

// Tuning / experiment knobs from the environment, read ONCE per process (thread-safe static initialisation; the launch
// path itself never calls getenv).
struct ConvEnv {
  int pair_dbg, mt256, mt, nacc;
  ConvEnv() {
    auto num = [](const char* name, int dflt) { const char* e = getenv(name); return e ? atoi(e) : dflt; };
    pair_dbg = num("ABCNET_PAIR_DBG", 0);
    mt256 = num("ABCNET_MT256", 0);
    mt = num("ABCNET_MT", 0);
    nacc = num("ABCNET_NACC", 0);
  }
};
static const ConvEnv& conv_env() {
  static const ConvEnv e;
  return e;
}

}  // namespace abc

extern "C" int64_t abc_conv_wpack_bytes(int cin, int cout, int ntaps, int n_tile) {
  if (cin <= 0 || cin % 16 || n_tile < 16 || n_tile > 256 || n_tile % 16 || ntaps < 1 || ntaps > 18 || cout < 1) return -1;
  const int n_tiles = (cout + n_tile - 1) / n_tile;
  return static_cast<int64_t>(n_tiles) * n_tile * cin * ntaps * 2;
}

extern "C" int abc_conv_igemm(const AbcConvDesc* d, void* stream_) {
  using namespace abc;
  if (int rc = device_check()) return rc;
  ABC_REQUIRE(d != nullptr, "abc_conv_igemm: null descriptor");
  ABC_REQUIRE(d->in && d->wpack && d->bias, "abc_conv_igemm: null input / weights / bias");
  ABC_REQUIRE(d->out || d->pool_out, "abc_conv_igemm: no output buffer");
  ABC_REQUIRE(d->N > 0 && d->H > 0 && d->W > 0, "abc_conv_igemm: bad geometry N=%d H=%d W=%d", d->N, d->H, d->W);
  ABC_REQUIRE(d->cin >= 16 && d->cin % 16 == 0 && (d->cin <= 64 || d->cin % 64 == 0),
              "abc_conv_igemm: cin=%d must be 16, 32, 48, 64 or a multiple of 64", d->cin);
  ABC_REQUIRE(d->in_plane_off >= 0 && d->in_plane_off + d->cin / 8 <= d->in_planes, "abc_conv_igemm: input plane range");
  ABC_REQUIRE(d->n_tile >= 16 && d->n_tile <= 256 && d->n_tile % 16 == 0, "abc_conv_igemm: n_tile=%d", d->n_tile);
  ABC_REQUIRE(d->ntaps >= 1 && d->ntaps <= 9, "abc_conv_igemm: ntaps=%d", d->ntaps);
  ABC_REQUIRE(d->cout >= 1, "abc_conv_igemm: cout=%d", d->cout);
  ABC_REQUIRE(d->out_mode >= 0 && d->out_mode <= 2, "abc_conv_igemm: out_mode=%d", d->out_mode);
  ABC_REQUIRE((reinterpret_cast<uintptr_t>(d->in) & 15) == 0 && (reinterpret_cast<uintptr_t>(d->wpack) & 15) == 0,
              "abc_conv_igemm: input / weights must be 16-byte aligned");
  const int fold = d->row_fold > 1 ? d->row_fold : 1;
  if (fold > 1) {
    // Row folding (16 / 32-channel layers): J vertically adjacent output pixels share one GEMM row, GEMM N = J * cout.
    ABC_REQUIRE(fold == 2 || fold == 4, "abc_conv_igemm: row_fold=%d must be 1, 2 or 4", fold);
    ABC_REQUIRE(d->ntaps == 9 && d->k_segments <= 1, "abc_conv_igemm: row_fold needs the plain 3x3 tap set");
    ABC_REQUIRE(d->cout % 16 == 0 && d->n_tile == fold * d->cout, "abc_conv_igemm: row_fold needs n_tile == row_fold * cout (cout %% 16 == 0)");
    ABC_REQUIRE(d->out_mode == 0 && d->out_sy == 1 && d->out_sx == 1 && d->out_oy == 0 && d->out_ox == 0,
                "abc_conv_igemm: row_fold supports plain P8 outputs only");
  }
  const bool swap = d->swap_mn != 0;
  if (swap) {
    // with row folding the 128 GEMM rows are (folded row j, channel): row_fold * cout == 128, weight pack rows ordered j * cout + co
    ABC_REQUIRE(d->n_tile == 128 && (fold == 1 || fold == 2 || fold == 4) && d->k_segments <= 1 && !d->cta_pair,
                "abc_conv_igemm: swap_mn needs n_tile == 128 and no k_segments / cta_pair");
    ABC_REQUIRE(d->out_mode == 0 && d->out != nullptr && d->pool_out == nullptr,
                "abc_conv_igemm: swap_mn supports plain P8 outputs only (no pool_out)");
  }
  int halo = 0;
  for (int t = 0; t < d->ntaps; ++t) {
    ABC_REQUIRE(d->tap_dy[t] >= -1 && d->tap_dy[t] <= 1 && d->tap_dx[t] >= -1 && d->tap_dx[t] <= 1,
                "abc_conv_igemm: tap %d offset out of [-1,1]", t);
    if (d->tap_dy[t] || d->tap_dx[t]) halo = 1;
  }
  if (d->out_mode == 0) {
    ABC_REQUIRE(d->cout % 8 == 0, "abc_conv_igemm: P8 output needs cout %% 8 == 0 (got %d)", d->cout);
    // sub-pixel mode: the four phases share the plane range of ONE phase
    const int out_ch = d->subpixel > 0 ? d->subpixel : d->cout;
    if (d->out) ABC_REQUIRE(d->out_plane_off >= 0 && d->out_plane_off + out_ch / 8 <= d->out_planes, "abc_conv_igemm: output plane range");
  } else {
    ABC_REQUIRE(d->out != nullptr && d->pool_out == nullptr, "abc_conv_igemm: fp32 output modes need out and no pool_out");
    if (d->out_mode == 2)
      ABC_REQUIRE(d->out_plane_off >= 0 && d->out_plane_off + (d->cout + 7) / 8 <= d->out_planes,
                  "abc_conv_igemm: planar fp32 output plane range");
  }
  const int subpixel = d->subpixel > 0 ? d->subpixel : 0;
  if (subpixel) {
    // four sub-pixel phases of a stride-2 transposed convolution as blocks of the GEMM N axis (see the header)
    ABC_REQUIRE(d->out_mode == 0 && d->out != nullptr && d->pool_out == nullptr && !swap && fold == 1 && !d->cta_pair,
                "abc_conv_igemm: subpixel needs a plain P8 output without pool / swap / fold / pair");
    ABC_REQUIRE(subpixel % 16 == 0 && d->cout == 4 * subpixel && d->out_sy == 2 && d->out_sx == 2,
                "abc_conv_igemm: subpixel needs cout == 4 * subpixel (multiple of 16) and out_sy == out_sx == 2");
    ABC_REQUIRE(d->n_tile / 16 <= 16 && d->out_W < 32768 && d->out_plane_off + subpixel / 8 <= d->out_planes,
                "abc_conv_igemm: subpixel: n_tile <= 256, out_W < 32768, plane range");
    ABC_REQUIRE((d->H - 1) * 2 + d->out_oy + 1 < d->out_H && (d->W - 1) * 2 + d->out_ox + 1 < d->out_W,
                "abc_conv_igemm: subpixel output mapping exceeds out_H x out_W");
  }
  if (d->out) {
    ABC_REQUIRE(d->out_sy >= 1 && d->out_sx >= 1 && d->out_oy >= 0 && d->out_ox >= 0 &&
                    (d->H - 1) * d->out_sy + d->out_oy < d->out_H && (d->W - 1) * d->out_sx + d->out_ox < d->out_W,
                "abc_conv_igemm: output mapping exceeds out_H x out_W");
  }
  if (d->pool_out) {
    ABC_REQUIRE(d->H % 2 == 0 && d->W % 2 == 0, "abc_conv_igemm: fused max-pool needs even H, W");
    ABC_REQUIRE(d->pool_plane_off >= 0 && d->pool_plane_off + d->cout / 8 <= d->pool_planes, "abc_conv_igemm: pool plane range");
  }

  ConvKParams p{};
  p.N = d->N; p.H = d->H; p.W = d->W;
  p.tiles_x = (d->W + 7) / 8;
  p.fold = fold;
  const ConvEnv& env = conv_env();
  p.dbg = env.pair_dbg;
  p.tile_rows = swap ? 32 * fold : 16 * fold;
  p.tiles_y = (d->H + p.tile_rows - 1) / p.tile_rows;
  p.in_plane_off = d->in_plane_off;
  // K chunk = channels per pipeline stage; 0 = the default min(cin, 64). A smaller chunk halves the activation stage and the
  // weight blocks, i.e. deepens both rings (AbcConvDesc.k_chunk)
  const int kc = d->k_chunk > 0 ? d->k_chunk : conv_kc(d->cin);
  ABC_REQUIRE((kc == 16 || kc == 32 || kc == 48 || kc == 64) && kc <= d->cin && d->cin % kc == 0 && !(d->cta_pair && kc != 64),
              "abc_conv_igemm: k_chunk=%d must be 16, 32 or 64 and divide cin=%d", kc, d->cin);
  p.kp = kc / 8;
  p.nkc = d->cin / kc;
  p.ntaps = fold > 1 ? 3 * (fold + 2) : d->ntaps;
  p.halo = halo;
  p.n_tile = d->n_tile;
  const int rows = p.tile_rows + 2 * halo, cols = 8 + 2 * halo;
  p.a_row_bytes = cols * 16;
  p.a_plane_bytes = rows * p.a_row_bytes;
  p.a_tile_bytes = p.kp * p.a_plane_bytes;
  p.b_block_bytes = static_cast<uint32_t>(d->n_tile) * kc * 2;
  if (fold > 1) {
    // folded taps in (row offset 0..J+1, column offset 0..2) order = the block order of the folded weight pack
    for (int t = 0; t < p.ntaps; ++t) p.tap_off[t] = static_cast<uint32_t>(((t / 3) * cols + (t % 3)) * 16);
  } else {
    for (int t = 0; t < d->ntaps; ++t)
      p.tap_off[t] = static_cast<uint32_t>(((d->tap_dy[t] + halo) * cols + (d->tap_dx[t] + halo)) * 16);
  }
  ABC_REQUIRE((p.a_tile_bytes & 127u) == 0, "abc_conv_igemm: internal: A tile not a 128-byte multiple");
  const int nseg = d->k_segments > 1 ? d->k_segments : 1;
  ABC_REQUIRE(nseg <= 4 && p.nkc % nseg == 0, "abc_conv_igemm: k_segments=%d must divide the %d K chunks (<= 4)", nseg, p.nkc);
  p.chunks_per_seg = p.nkc / nseg;
  p.blocks_per_ntile = 0;
  for (int sgi = 0; sgi < nseg; ++sgi) {
    p.seg_tap0[sgi] = nseg > 1 ? d->seg_tap0[sgi] : 0;
    p.seg_ntaps[sgi] = nseg > 1 ? d->seg_ntaps[sgi] : p.ntaps;
    ABC_REQUIRE(p.seg_tap0[sgi] >= 0 && p.seg_ntaps[sgi] >= 1 && p.seg_tap0[sgi] + p.seg_ntaps[sgi] <= p.ntaps,
                "abc_conv_igemm: segment %d tap range", sgi);
    p.blocks_per_ntile += p.chunks_per_seg * p.seg_ntaps[sgi];
  }
  // CTA-pair mode (AbcConvDesc.cta_pair): only for layers whose weights are streamed (Cin >= 128) -- decided below
  const bool want_pair = d->cta_pair != 0;
  if (want_pair) {
    ABC_REQUIRE(fold == 1 && nseg == 1 && kc == 64 && d->n_tile % 32 == 0,
                "abc_conv_igemm: cta_pair needs cin %% 64 == 0, n_tile %% 32 == 0, no row folding / K segments");
    p.b_block_bytes /= 2;                                  // this CTA's half of every weight block
  }
  const uint32_t total_b = want_pair ? (1u << 30) : static_cast<uint32_t>(p.blocks_per_ntile) * p.b_block_bytes;
  p.smem_a_off = kHeaderBytes + (swap ? kSwapStageBytes : 0u);
  const uint32_t hdr = p.smem_a_off;
  // mt = tiles per pipeline stage: amortises the per-stage barrier round trips and puts more bytes in flight per SM.
  // Bounded by TMEM (two accumulator stages of mt * n_tile <= 256 columns each) and by shared memory.
  int mt_max = swap ? 1 : 256 / d->n_tile;
  // n_tile = 256: with one tile per stage every CTA streams the layer's full weight set per 128 pixels (64 B/clk/SM at
  // the MMA rate, above the ~43 B/clk/SM the L2 delivers); two tiles per weight block halve that at the price of a
  // single accumulator stage (512 TMEM columns): the epilogue no longer overlaps the next group's MMAs.
  if (d->n_tile == 256 && env.mt256 > 0) mt_max = env.mt256 >= 2 ? 2 : 1;
  if (mt_max > 8) mt_max = 8;
  if (mt_max > p.tiles_x) mt_max = p.tiles_x;
  if (env.mt >= 1 && env.mt < mt_max) mt_max = env.mt;
  uint32_t smem_bytes = 0;
  p.mt = 0;
  for (int mt = mt_max; mt >= 1 && !p.mt; --mt) {          // prefer resident weights
    const uint32_t a_stage = mt * p.a_tile_bytes;
    if (total_b < (1u << 20) && hdr + 2 * a_stage + total_b <= kSmemBudget) {
      p.mt = mt; p.resident_b = 1; p.nb = 1;
      int na = static_cast<int>((kSmemBudget - hdr - total_b) / a_stage);
      p.na = na > kMaxNA ? kMaxNA : na;
      p.a_stage_bytes = a_stage;
      p.smem_b_off = hdr + p.na * a_stage;
      smem_bytes = p.smem_b_off + total_b;
    }
  }
  for (int mt = mt_max; mt >= 1 && !p.mt; --mt) {          // otherwise stream weight blocks through a ring
    const uint32_t a_stage = mt * p.a_tile_bytes;
    // at least 4 weight blocks in the ring; the folded swap tiles of the 64-channel layers (2 x 84 KB of activations) leave room for 3
    if (hdr + 2 * a_stage + (swap && fold > 1 ? 3 : 4) * p.b_block_bytes <= kSmemBudget) {
      p.mt = mt; p.resident_b = 0; p.na = 2;
      if (hdr + 3 * a_stage + 6 * p.b_block_bytes <= kSmemBudget) p.na = 3;
      p.a_stage_bytes = a_stage;
      p.smem_b_off = hdr + p.na * a_stage;
      if (want_pair) p.smem_b_off = (p.smem_b_off + 1023u) & ~1023u;   // swizzled blocks start on 1024-byte boundaries
      int nb = static_cast<int>((kSmemBudget - p.smem_b_off) / p.b_block_bytes);
      p.nb = nb > kMaxNB ? kMaxNB : nb;
      smem_bytes = p.smem_b_off + p.nb * p.b_block_bytes;
    }
  }
  ABC_REQUIRE(p.mt >= 1, "abc_conv_igemm: cin=%d n_tile=%d does not fit in shared memory", d->cin, d->n_tile);
  p.acc_cols = swap ? 256 : p.mt * d->n_tile;
  p.nacc = kTmemCols / p.acc_cols;
  if (p.nacc > kMaxAcc) p.nacc = kMaxAcc;
  if (env.nacc >= 2 && env.nacc < p.nacc) p.nacc = env.nacc;
  p.groups_x = (p.tiles_x + p.mt - 1) / p.mt;
  const int64_t groups = static_cast<int64_t>(d->N) * p.groups_x * p.tiles_y;
  ABC_REQUIRE(groups < (1ll << 31), "abc_conv_igemm: too many tiles");
  p.num_groups = static_cast<int>(groups);
  if (smem_bytes < 120 * 1024) smem_bytes = 120 * 1024;   // keep 1 CTA / SM: the kernel owns all 512 TMEM columns
  p.wpack = static_cast<const uint8_t*>(d->wpack);
  p.bias = d->bias;
  p.cout = d->cout; p.act = d->act; p.out_mode = d->out_mode;
  p.out = d->out;
  p.out_planes = d->out_planes; p.out_plane_off = d->out_plane_off;
  p.out_H = d->out_H; p.out_W = d->out_W;
  p.out_sy = d->out_sy; p.out_oy = d->out_oy; p.out_sx = d->out_sx; p.out_ox = d->out_ox;
  p.pool_out = d->pool_out; p.pool_planes = d->pool_planes; p.pool_plane_off = d->pool_plane_off;
  p.subpixel = subpixel;
  p.fp16 = d->act_fp16 ? 1 : 0;
  ABC_REQUIRE(!(p.fp16 && (want_pair || d->stat_sum)), "abc_conv_igemm: act_fp16 is an inference mode (no cta_pair, no fused statistics)");
  cudaStream_t st_ = static_cast<cudaStream_t>(stream_);
  // fused BatchNorm statistics (training forward)
  const bool stats = d->stat_sum != nullptr || d->stat_sq != nullptr;
  if (stats) {
    ABC_REQUIRE(d->stat_sum && d->stat_sq, "abc_conv_igemm: stat_sum and stat_sq go together");
    ABC_REQUIRE(d->out_mode == 0 && d->out != nullptr && d->pool_out == nullptr && !want_pair,
                "abc_conv_igemm: fused statistics need a plain P8 output");
    ABC_REQUIRE(swap || (fold == 4 && d->cout == 16 && d->n_tile == 64 && d->cin == 16),
                "abc_conv_igemm: fused statistics are built for operand-swap launches and the row-folded 16 -> 16 layers "
                "(use abc_bn_stats otherwise)");
    p.stat_sum = d->stat_sum;
    p.stat_sq = d->stat_sq;
    p.stat_ws = d->stat_ws;
    if (d->stat_ws)            // slots no owner writes (unused folded rows) must read as zero in the ordered sum
      ABC_CUDA(cudaMemsetAsync(d->stat_ws, 0, abc_conv_stat_workspace_bytes(d), st_));
    else {
      ABC_CUDA(cudaMemsetAsync(d->stat_sum, 0, d->cout * sizeof(double), st_));
      ABC_CUDA(cudaMemsetAsync(d->stat_sq, 0, d->cout * sizeof(double), st_));
    }
  }

  EncodeTiledFn encode = get_encode_fn();
  if (!encode) {
    set_error("cuTensorMapEncodeTiled driver entry point not available");
    return ABC_ERR_NO_DEVICE;
  }
  CUtensorMap tmap;
  const cuuint64_t gdim[4] = {static_cast<cuuint64_t>(d->W) * 8, static_cast<cuuint64_t>(d->H),
                              static_cast<cuuint64_t>(d->in_planes), static_cast<cuuint64_t>(d->N)};
  const cuuint64_t gstride[3] = {static_cast<cuuint64_t>(d->W) * 16, static_cast<cuuint64_t>(d->W) * d->H * 16,
                                 static_cast<cuuint64_t>(d->W) * d->H * 16 * d->in_planes};
  const cuuint32_t box[4] = {static_cast<cuuint32_t>(cols * 8), static_cast<cuuint32_t>(rows),
                             static_cast<cuuint32_t>(p.kp), 1};
  const cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult cr = encode(&tmap, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(d->in), gdim, gstride, box, estr,
                       CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                       CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (cr != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed with CUresult %d (W=%d H=%d planes=%d N=%d box=%ux%ux%u)", static_cast<int>(cr),
              d->W, d->H, d->in_planes, d->N, box[0], box[1], box[2]);
    return ABC_ERR_CUDA;
  }

  typedef void (*KernelFn)(const CUtensorMap, const ConvKParams);
  KernelFn kernels[2][5] = {{nullptr, conv_igemm_kernel<1, false, false>, conv_igemm_kernel<2, false, false>,
                             conv_igemm_kernel<3, false, false>, conv_igemm_kernel<4, false, false>},
                            {nullptr, conv_igemm_kernel<1, true, false>, conv_igemm_kernel<2, true, false>,
                             conv_igemm_kernel<3, true, false>, conv_igemm_kernel<4, true, false>}};
  KernelFn swap_kernels[2][5] = {{nullptr, conv_igemm_kernel<1, false, false, true>, conv_igemm_kernel<2, false, false, true>,
                                  conv_igemm_kernel<3, false, false, true>, conv_igemm_kernel<4, false, false, true>},
                                 {nullptr, conv_igemm_kernel<1, true, false, true>, conv_igemm_kernel<2, true, false, true>,
                                  conv_igemm_kernel<3, true, false, true>, conv_igemm_kernel<4, true, false, true>}};
  KernelFn swap_det_kernels[2][5] = {{nullptr, conv_igemm_kernel<1, false, false, true, false, true>,
                                      conv_igemm_kernel<2, false, false, true, false, true>, conv_igemm_kernel<3, false, false, true, false, true>,
                                      conv_igemm_kernel<4, false, false, true, false, true>},
                                     {nullptr, conv_igemm_kernel<1, true, false, true, false, true>,
                                      conv_igemm_kernel<2, true, false, true, false, true>, conv_igemm_kernel<3, true, false, true, false, true>,
                                      conv_igemm_kernel<4, true, false, true, false, true>}};
  KernelFn pair_kernel = conv_igemm_kernel<4, false, true>;
  KernelFn stats_kernel = conv_igemm_kernel<1, true, false, false, true>;      // row-folded 16 -> 16 with fused statistics
  KernelFn stats_det_kernel = conv_igemm_kernel<1, true, false, false, true, true>;
  static PerDeviceOnce attr_once;
  ABC_CUDA(attr_once.run([&]() -> cudaError_t {
    for (int r = 0; r < 2; ++r)
      for (int k = 1; k <= 4; ++k) {
        if (cudaError_t e = cudaFuncSetAttribute(kernels[r][k], cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBudget)) return e;
        if (cudaError_t e = cudaFuncSetAttribute(swap_kernels[r][k], cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBudget)) return e;
        if (cudaError_t e = cudaFuncSetAttribute(swap_det_kernels[r][k], cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBudget)) return e;
      }
    if (cudaError_t e = cudaFuncSetAttribute(stats_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBudget)) return e;
    if (cudaError_t e = cudaFuncSetAttribute(stats_det_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBudget)) return e;
    return cudaFuncSetAttribute(pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBudget);
  }));
  const int ksteps = p.kp / 2;
  ABC_REQUIRE(ksteps >= 1 && ksteps <= 4, "abc_conv_igemm: internal: ksteps=%d", ksteps);
  const int n_tiles = (d->cout + d->n_tile - 1) / d->n_tile;
  int sms = sm_count();
  if (sms <= 0) sms = 148;
  int gx = sms / n_tiles;
  if (gx < 1) gx = 1;
  if (want_pair) {
    // (2,1,1) clusters: the two CTAs of a pair sit on one TPC and share every tcgen05.mma (M = 256)
    ABC_REQUIRE(!p.resident_b && ksteps == 4, "abc_conv_igemm: internal: cta_pair with resident weights");
    const int need = (p.num_groups + 1) & ~1;
    gx &= ~1;
    if (gx > need) gx = need;
    if (gx < 2) gx = 2;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(gx, n_tiles, 1);
    cfg.blockDim = dim3(kThreads, 1, 1);
    cfg.dynamicSmemBytes = smem_bytes;
    cfg.stream = static_cast<cudaStream_t>(stream_);
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    ABC_CUDA(cudaLaunchKernelEx(&cfg, pair_kernel, tmap, p));
    return launch_check("conv_igemm_kernel<pair>");
  }
  if (gx > p.num_groups) gx = p.num_groups;
  dim3 grid(gx, n_tiles, 1);
  const bool det = stats && p.stat_ws;
  KernelFn fn = (swap ? (det ? swap_det_kernels : swap_kernels) : kernels)[p.resident_b ? 1 : 0][ksteps];
  if (stats && !swap) {
    ABC_REQUIRE(p.resident_b && ksteps == 1, "abc_conv_igemm: internal: fused statistics variant");
    fn = det ? stats_det_kernel : stats_kernel;
  }
  fn<<<grid, kThreads, smem_bytes, st_>>>(tmap, p);
  if (int rc = launch_check(swap ? "conv_igemm_kernel<swap>" : "conv_igemm_kernel")) return rc;
  return det ? det_reduce(p.stat_ws, conv_stat_slots(gx), 2 * d->cout, det_out2(d->stat_sum, d->stat_sq, d->cout), 0, st_) : ABC_OK;
}

// Workspace of the deterministic fused statistics (AbcConvDesc.stat_ws): the grid.x of the launch above, 8 owners per CTA.
extern "C" size_t abc_conv_stat_workspace_bytes(const AbcConvDesc* d) {
  using namespace abc;
  if (!d || d->cout <= 0 || d->n_tile <= 0) return 0;
  const int n_tiles = (d->cout + d->n_tile - 1) / d->n_tile;
  int sms = sm_count();
  if (sms <= 0) sms = 148;
  const int gx = sms / n_tiles < 1 ? 1 : sms / n_tiles;      // an upper bound of the launch's grid.x (it is capped by the groups)
  return det_ws_bytes(conv_stat_slots(gx), 2ll * d->cout, sizeof(double));
}

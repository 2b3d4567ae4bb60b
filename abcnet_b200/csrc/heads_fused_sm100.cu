// Fused output heads for sm_100a: for every head of the U-Net, conv3x3(128 -> 128) + BatchNorm(eval, folded) +
// LeakyReLU(0.01) + conv1x1(128 -> h) in ONE kernel -- OutConv of /root/reference/src/unet.py:63-74, applied to the shared
// trunk at :116-118. The 128-channel hidden map of a head never leaves tensor memory:
//
//   conv1 : implicit GEMM as in conv_igemm_sm100.cu (TMA halo tile, 9 shifted descriptors, tcgen05.mma M = 128 pixels,
//           N = 256 = TWO heads per CTA, K = 2 chunks x 9 taps x 64 channels), accumulators in TMEM;
//   epilogue phase 1 : TMEM -> registers -> bias + LeakyReLU -> 16-bit -> back to TMEM (tcgen05.st), two values per
//           32-bit column, lane = pixel: the A-operand layout of tcgen05.mma kind::f16 with A in tensor memory;
//   conv2 : 8 MMAs per chunk of <= 128 output channels (A = hidden map from TMEM, B = the head's 1x1 weights, one chunk
//           at a time in a shared-memory slot of their own), accumulating into the TMEM columns phase 1 has just drained;
//   epilogue phase 2 : TMEM -> + bias -> fp32 logits (NCHW, or planar-8 for the fused inference + decode path).
//
// TMEM: two buffers of 256 columns (tile t uses buffer t & 1). In buffer b, conv1 accumulates head A in columns [0, 128) and
// head B in [128, 256); phase 1 writes hidden A to [0, 64) and hidden B to [64, 128); the conv2 chunks then accumulate one
// after another in [128, 256). The buffer returns to conv1 (tile t + 2) once its last chunk is drained.
//
// Compared with conv_igemm(conv1) + 8 x conv_igemm(conv2) this removes the write and re-read of the hidden maps
// (2 x 8.6 GB per 256-image batch) and nine launches. conv1 and conv2 have an issuing warp each, so the conv1 MMA stream
// waits on the epilogue only for a free TMEM buffer (the one of tile t - 2), never for a logit drain: each conv2 chunk
// waits for the drain of the one before, and with one issuer that wait stalled conv1 too. The hidden maps take no shared
// memory, which leaves room for a 4-block conv1 weight ring next to the conv2 slot.
//
// Warp roles (384 threads, 1 CTA / SM, persistent over M tiles; the CTAs are split among the head pairs by
// hf_split_ctas in heads_split.cuh):
//   warp 0 : TMA producer (activation halo tiles)      warp 3 : bulk-copy producer (conv1 weight blocks)
//   warp 1 : conv1 MMA issuer                          warp 2 : TMEM allocation, then conv2 weight loads + MMA issuer
//   warps 4-11 : epilogue (two per TMEM lane quarter)
#include <cuda.h>
#include <cuda_bf16.h>

#include "common.cuh"
#include "heads_split.cuh"
#include "p8_device.cuh"
#include "ptx_sm100.cuh"

namespace abc {

constexpr int kHfThreads = 384;
constexpr int kHfMaxPairs = 8, kHfMaxItems = 6;
constexpr uint32_t kHfHeader = 4096;
constexpr uint32_t kHfARow = 10 * 16, kHfAPlane = 18 * kHfARow, kHfAStage = 8 * kHfAPlane;   // 64 channels = 8 planes
constexpr uint32_t kHfBBlock = 256 * 64 * 2;
constexpr uint32_t kHfSmemLimit = 232448;
constexpr uint32_t kHfW2Slot = 128 * 16 * 8 * 2;   // one conv2 chunk: [16 K planes][<= 128 channels][8] 16-bit
constexpr int kHfNA = 2;
constexpr int kHfNB = static_cast<int>((kHfSmemLimit - kHfHeader - kHfNA * kHfAStage - kHfW2Slot) / kHfBBlock);   // 4 conv1 blocks
constexpr uint32_t kHfSmem = kHfHeader + kHfNA * kHfAStage + kHfNB * kHfBBlock + kHfW2Slot;
static_assert(kHfSmem <= kHfSmemLimit, "shared memory budget");

struct HfItem {          // one conv2 chunk: <= 128 output channels of one head
  int head_slot;         // 0 / 1: first / second head of the pair
  int nc;                // GEMM N of this chunk (multiple of 16, <= 128)
  int ch0;               // first output channel of the head covered by this chunk
  int w2_off;            // byte offset of the packed [16][nc][8] 16-bit weight block in w2
  int bias_off;          // offset (floats) of the chunk's bias in the pair's bias2 block
};

struct HfParams {
  int N, H, W, tiles_x, tiles_y, num_tiles, in_plane_off;
  const uint8_t* w1;     // packed conv1 weights [pair][chunk 2][tap 9][8][256][8] 16-bit
  const float* bias1;    // [pairs * 256]
  const uint8_t* w2;
  const float* bias2;    // per pair: bias2_off[pair] .. (+ bias2_len[pair])
  int pairs;
  int cta0[kHfMaxPairs + 1];   // CTAs [cta0[p], cta0[p + 1]) work on pair p
  int bias2_off[kHfMaxPairs], bias2_len[kHfMaxPairs];
  int n_items[kHfMaxPairs];
  HfItem items[kHfMaxPairs][kHfMaxItems];
  void* out[2 * kHfMaxPairs];      // per head
  int out_mode[2 * kHfMaxPairs];   // 1: NCHW fp32, 2: planar-8 fp32
  int cout[2 * kHfMaxPairs];
  int out_planes[2 * kHfMaxPairs];
  uint32_t tap16[9];
  unsigned long long* trace;       // kHfTraceWords per CTA (kTrace instantiation only)
};

// Per-CTA timeline record of the kTrace instantiation (tools/heads_trace.py reads it): clock64 cycles spent in each wait.
enum HfTraceWord {
  kHtPair, kHtTiles, kHtStartNs, kHtEndNs, kHtCycles,
  kHtC1BFull, kHtC1AFull, kHtC1AccEmpty,                    // conv1 issuer
  kHtC2HidFull, kHtC2C2Empty, kHtC2WFull, kHtC2WEmpty,      // conv2 issuer
  kHtEpAccFull, kHtEpPhase1, kHtEpC2Full, kHtEpPhase2,      // epilogue warp 4: waits and busy cycles of the two phases
  kHfTraceWords
};

__device__ __forceinline__ unsigned long long global_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

// mbar_wait that, in the kTrace instantiation, adds the cycles it waited to `acc`
template <bool kTrace>
__device__ __forceinline__ void mbar_wait_t(uint32_t bar, uint32_t parity, unsigned long long& acc) {
  if constexpr (kTrace) {
    const long long t0 = clock64();
    mbar_wait(bar, parity);
    acc += static_cast<unsigned long long>(clock64() - t0);
  } else {
    mbar_wait(bar, parity);
  }
}

// kF16: activations and weights are IEEE fp16 (UNet(act_dtype="fp16")), else bf16. kTrace: write p.trace (HfTraceWord)
template <bool kF16, bool kTrace>
__global__ void __launch_bounds__(kHfThreads, 1)
heads_fused_kernel(const __grid_constant__ CUtensorMap tmap, const __grid_constant__ HfParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t sbase = smem_u32(smem);
  const int warp = static_cast<int>(warp_id_uniform());
  const int lane = threadIdx.x & 31;
  int pair = 0;
  while (pair + 1 < p.pairs && static_cast<int>(blockIdx.x) >= p.cta0[pair + 1]) ++pair;
  const int cta_rank = blockIdx.x - p.cta0[pair], cta_stride = p.cta0[pair + 1] - p.cta0[pair];

  // barrier slots (8 bytes each)
  const uint32_t bar_a_full = sbase, bar_a_empty = sbase + 8 * kHfNA;
  const uint32_t bar_b_full = sbase + 8 * 2 * kHfNA, bar_b_empty = bar_b_full + 8 * kHfNB;
  const uint32_t bar_acc_full = bar_b_empty + 8 * kHfNB;       // [2] conv1 accumulators of a buffer complete
  const uint32_t bar_acc_empty = bar_acc_full + 16;            // [2] buffer fully drained (after the conv2 logits)
  const uint32_t bar_hid_full = bar_acc_empty + 16;            // both hidden operands of a tile written to TMEM
  const uint32_t bar_c2_full = bar_hid_full + 8;               // a conv2 chunk is complete in TMEM
  const uint32_t bar_c2_empty = bar_c2_full + 8;               // ... and has been drained
  const uint32_t bar_w2_full = bar_c2_empty + 8;               // a conv2 chunk's weights are in the conv2 slot
  const uint32_t bar_w2_empty = bar_w2_full + 8;               // ... and its MMAs have read them
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + 512);
  HfItem* items_s = reinterpret_cast<HfItem*>(smem + 576);     // [kHfMaxItems]
  float* bias1_s = reinterpret_cast<float*>(smem + 1024);      // [256]
  float* bias2_s = reinterpret_cast<float*>(smem + 2048);      // [512]
  const int n_items = p.n_items[pair];

  if (threadIdx.x == 0) {
    for (int i = 0; i < kHfNA; ++i) {
      mbar_init(bar_a_full + 8 * i, 1);
      mbar_init(bar_a_empty + 8 * i, 1);
    }
    for (int i = 0; i < kHfNB; ++i) {
      mbar_init(bar_b_full + 8 * i, 1);
      mbar_init(bar_b_empty + 8 * i, 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(bar_acc_full + 8 * i, 1);
      mbar_init(bar_acc_empty + 8 * i, 8);
    }
    mbar_init(bar_hid_full, 8);
    mbar_init(bar_c2_full, 1);
    mbar_init(bar_c2_empty, 8);
    mbar_init(bar_w2_full, 1);
    mbar_init(bar_w2_empty, 1);
    fence_mbar_init();
    tma_prefetch_desc(&tmap);
  }
  if (warp == 2) tmem_alloc<512>(smem_u32(tmem_slot));
  for (int i = threadIdx.x; i < 256; i += kHfThreads) bias1_s[i] = p.bias1[pair * 256 + i];
  for (int i = threadIdx.x; i < p.bias2_len[pair]; i += kHfThreads) bias2_s[i] = p.bias2[p.bias2_off[pair] + i];
  if (threadIdx.x < n_items) items_s[threadIdx.x] = p.items[pair][threadIdx.x];
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_slot);
  unsigned long long* const trace = kTrace ? p.trace + static_cast<size_t>(blockIdx.x) * kHfTraceWords : nullptr;
  unsigned long long t_start_ns = 0;
  long long t_start_clk = 0;
  if constexpr (kTrace) {
    t_start_ns = global_ns();
    t_start_clk = clock64();
  }

  const uint32_t a_region = sbase + kHfHeader;
  const uint32_t b_region = a_region + kHfNA * kHfAStage;
  const uint32_t w2_region = b_region + kHfNB * kHfBBlock;
  const int tiles_per_img = p.tiles_x * p.tiles_y;
  // tiles of this CTA: cta_rank, cta_rank + cta_stride, ...
  const int my_tiles = (p.num_tiles > cta_rank) ? (p.num_tiles - cta_rank + cta_stride - 1) / cta_stride : 0;

  if (warp == 0) {
    // ------------------------------------------------------------------ A producer
    int stage = 0;
    uint32_t phase = 0;
    for (int it = 0; it < my_tiles; ++it) {
      const int g = cta_rank + it * cta_stride;
      const int n = g / tiles_per_img;
      const int rem = g - n * tiles_per_img;
      const int ty = rem / p.tiles_x, tx = rem - ty * p.tiles_x;
      for (int kc = 0; kc < 2; ++kc) {
        mbar_wait(bar_a_empty + 8 * stage, phase ^ 1);
        if (elect_one()) {
          mbar_arrive_expect_tx(bar_a_full + 8 * stage, kHfAStage);
          tma_load_4d(a_region + stage * kHfAStage, &tmap, bar_a_full + 8 * stage, (tx * 8 - 1) * 8, ty * 16 - 1,
                      p.in_plane_off + kc * 8, n);
        }
        __syncwarp();
        if (++stage == kHfNA) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else if (warp == 3) {
    // ------------------------------------------------------------------ B producer: conv1 weight blocks
    const uint8_t* w1 = p.w1 + static_cast<size_t>(pair) * 18 * kHfBBlock;
    int stage = 0;
    uint32_t phase = 0;
    for (int it = 0; it < my_tiles; ++it) {
      for (int step = 0; step < 18; ++step) {
        mbar_wait(bar_b_empty + 8 * stage, phase ^ 1);
        if (elect_one()) {
          mbar_arrive_expect_tx(bar_b_full + 8 * stage, kHfBBlock);
          bulk_load_1d(b_region + stage * kHfBBlock, w1 + static_cast<size_t>(step) * kHfBBlock, kHfBBlock, bar_b_full + 8 * stage);
        }
        __syncwarp();
        if (++stage == kHfNB) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ conv1 MMA issuer
    const uint32_t idesc1 = umma_idesc_16(128, 256, 0, 0, kF16);
    const uint64_t a_hi64 = umma_desc_hi(kHfAPlane, kHfARow);
    const uint64_t b_hi64 = umma_desc_hi(256 * 16, 128);
    const uint32_t a_hi = static_cast<uint32_t>(a_hi64 >> 32), b_hi = static_cast<uint32_t>(b_hi64 >> 32);
    const uint32_t a_lo0 = static_cast<uint32_t>(a_hi64) | (a_region >> 4);
    const uint32_t b_lo0 = static_cast<uint32_t>(b_hi64) | (b_region >> 4);
    constexpr uint32_t a_kstep = (2 * kHfAPlane) >> 4, b_kstep = (2 * 256 * 16) >> 4;
    int a_stage = 0, b_stage = 0;
    uint32_t a_phase = 0, b_phase = 0;
    uint32_t acc_empty_phase = 0;   // one phase bit per buffer
    unsigned long long w_b = 0, w_a = 0, w_acc = 0;
    for (int it = 0; it < my_tiles; ++it) {
      const int s = it & 1;
      const uint32_t tmem_d = tmem_base + s * 256;
      // the only wait on the epilogue: buffer s is free once tile it - 2's last conv2 chunk has been drained
      mbar_wait_t<kTrace>(bar_acc_empty + 8 * s, ((acc_empty_phase >> s) & 1u) ^ 1u, w_acc);
      acc_empty_phase ^= 1u << s;
      tc_fence_after();
      uint32_t a_base = 0;
      for (int step = 0; step < 18; ++step) {
        const int t = step >= 9 ? step - 9 : step;
        if (t == 0) {
          mbar_wait_t<kTrace>(bar_a_full + 8 * a_stage, a_phase, w_a);
          tc_fence_after();
          a_base = a_lo0 + a_stage * (kHfAStage >> 4);
        }
        mbar_wait_t<kTrace>(bar_b_full + 8 * b_stage, b_phase, w_b);
        tc_fence_after();
        const uint32_t b_base = b_lo0 + b_stage * (kHfBBlock >> 4);
        const uint32_t a_tap = a_base + p.tap16[t];
        if (elect_one()) {
#pragma unroll
          for (int j = 0; j < 4; ++j)
            umma_bf16_lohi(tmem_d, a_tap + j * a_kstep, a_hi, b_base + j * b_kstep, b_hi, idesc1, (step | j) != 0 ? 1u : 0u);
          umma_commit(bar_b_empty + 8 * b_stage);
          if (t == 8) umma_commit(bar_a_empty + 8 * a_stage);
        }
        __syncwarp();
        if (++b_stage == kHfNB) {
          b_stage = 0;
          b_phase ^= 1;
        }
        if (t == 8 && ++a_stage == kHfNA) {
          a_stage = 0;
          a_phase ^= 1;
        }
      }
      if (elect_one()) umma_commit(bar_acc_full + 8 * s);
      __syncwarp();
    }
    if constexpr (kTrace) {
      if (lane == 0) {
        trace[kHtC1BFull] = w_b;
        trace[kHtC1AFull] = w_a;
        trace[kHtC1AccEmpty] = w_acc;
      }
    }
  } else if (warp == 2) {
    // ------------------------------------------------------------------ conv2 MMA issuer (after the TMEM allocation)
    // Per chunk: load its weights into the conv2 slot once the previous chunk's MMAs have read it (this overlaps the
    // previous chunk's drain), wait for the drain, issue. tcgen05.commit tracks only this thread's MMAs, so the conv1
    // warp's commits are independent of these.
    uint32_t hid_full_phase = 0, c2_empty_phase = 0, w2_phase = 0;
    unsigned long long w_hid = 0, w_c2e = 0, w_wf = 0, w_we = 0;
    for (int it = 0; it < my_tiles; ++it) {
      const uint32_t tbuf = tmem_base + (it & 1) * 256;
      for (int i = 0; i < n_items; ++i) {
        const HfItem item = items_s[i];
        const uint32_t bytes = static_cast<uint32_t>(item.nc) * 256u;
        mbar_wait_t<kTrace>(bar_w2_empty, w2_phase ^ 1u, w_we);
        if (elect_one()) {
          mbar_arrive_expect_tx(bar_w2_full, bytes);
          bulk_load_1d(w2_region, p.w2 + item.w2_off, bytes, bar_w2_full);
        }
        __syncwarp();
        if (i == 0) {                                          // both hidden operands of this tile are in TMEM
          mbar_wait_t<kTrace>(bar_hid_full, hid_full_phase, w_hid);
          hid_full_phase ^= 1u;
        }
        mbar_wait_t<kTrace>(bar_c2_empty, c2_empty_phase ^ 1u, w_c2e);   // the previous chunk has been drained
        c2_empty_phase ^= 1u;
        mbar_wait_t<kTrace>(bar_w2_full, w2_phase, w_wf);
        w2_phase ^= 1u;
        tc_fence_after();
        const uint32_t idesc2 = umma_idesc_16(128, item.nc, 0, 0, kF16);
        const uint64_t w_hi64 = umma_desc_hi(static_cast<uint32_t>(item.nc) * 16, 128);
        const uint32_t w_hi = static_cast<uint32_t>(w_hi64 >> 32);
        const uint32_t w_lo = static_cast<uint32_t>(w_hi64) | (w2_region >> 4);
        const uint32_t a2 = tbuf + item.head_slot * 64;
        const uint32_t d2 = tbuf + 128;
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < 8; ++k)
            umma_16_ts(d2, a2 + k * 8, w_lo + k * 2 * item.nc, w_hi, idesc2, k != 0 ? 1u : 0u);
          umma_commit(bar_w2_empty);
          umma_commit(bar_c2_full);
        }
        __syncwarp();
      }
    }
    if constexpr (kTrace) {
      if (lane == 0) {
        trace[kHtC2HidFull] = w_hid;
        trace[kHtC2C2Empty] = w_c2e;
        trace[kHtC2WFull] = w_wf;
        trace[kHtC2WEmpty] = w_we;
      }
    }
  } else if (warp >= 4) {
    // ------------------------------------------------------------------ epilogue
    const int q = warp & 3;
    const int eh = (warp - 4) >> 2;
    const int m = q * 32 + lane;
    const int r = m >> 3, c = m & 7;
    const float4* bias1_4 = reinterpret_cast<const float4*>(bias1_s);
    const float4* bias2_4 = reinterpret_cast<const float4*>(bias2_s);
    const size_t plane_px = static_cast<size_t>(p.H) * p.W;
    uint32_t acc_full_phase = 0, c2_full_phase = 0;        // acc_full: one phase bit per buffer
    unsigned long long w_acc = 0, w_c2 = 0, busy1 = 0, busy2 = 0;
    long long t_mark = 0;
    for (int it = 0; it < my_tiles; ++it) {
      const int g = cta_rank + it * cta_stride;
      const int n = g / tiles_per_img;
      const int rem = g - n * tiles_per_img;
      const int ty = rem / p.tiles_x, tx = rem - ty * p.tiles_x;
      const int y = ty * 16 + r, x = tx * 8 + c;
      const bool valid = (y < p.H) && (x < p.W);
      const size_t px = static_cast<size_t>(y) * p.W + x;
      const int s = it & 1;
      const uint32_t tstage = tmem_base + s * 256 + (static_cast<uint32_t>(q * 32) << 16);
      mbar_wait_t<kTrace>(bar_acc_full + 8 * s, (acc_full_phase >> s) & 1u, w_acc);
      acc_full_phase ^= 1u << s;
      tc_fence_after();
      if constexpr (kTrace) t_mark = clock64();
      // ---- phase 1: conv1 accumulators -> bias + LeakyReLU -> 16-bit hidden operand, back into TMEM. This warp takes
      // channels [64 eh, 64 eh + 64) of each head: accumulator columns hs * 128 + 64 eh + [0, 64) -> packed columns
      // hs * 64 + 32 eh + [0, 32). Hidden A and B overwrite head A's accumulators, which BOTH warps of the lane quarter
      // must have loaded first (the named barrier); head B's accumulators are not overwritten in this phase.
#pragma unroll 1
      for (int hs = 0; hs < 2; ++hs) {
        uint32_t raw[4][16];
#pragma unroll
        for (int i = 0; i < 4; ++i) tmem_ld16(tstage + hs * 128 + eh * 64 + i * 16, raw[i]);
        tmem_ld_wait();
        if (hs == 0) {
          tc_fence_before();
          named_bar_sync(1 + q, 64);
          tc_fence_after();
        }
        uint32_t packed[32];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          float v[16];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float4 bb = bias1_4[hs * 32 + eh * 16 + i * 4 + j];
            const float t0 = __uint_as_float(raw[i][4 * j + 0]) + bb.x, t1 = __uint_as_float(raw[i][4 * j + 1]) + bb.y;
            const float t2 = __uint_as_float(raw[i][4 * j + 2]) + bb.z, t3 = __uint_as_float(raw[i][4 * j + 3]) + bb.w;
            v[4 * j + 0] = fmaxf(t0, 0.01f * t0);
            v[4 * j + 1] = fmaxf(t1, 0.01f * t1);
            v[4 * j + 2] = fmaxf(t2, 0.01f * t2);
            v[4 * j + 3] = fmaxf(t3, 0.01f * t3);
          }
          const uint4 u0 = pack8_act16(v, kF16), u1 = pack8_act16(v + 8, kF16);
          packed[8 * i + 0] = u0.x; packed[8 * i + 1] = u0.y; packed[8 * i + 2] = u0.z; packed[8 * i + 3] = u0.w;
          packed[8 * i + 4] = u1.x; packed[8 * i + 5] = u1.y; packed[8 * i + 6] = u1.z; packed[8 * i + 7] = u1.w;
        }
        tmem_st16(tstage + hs * 64 + eh * 32, packed);
        tmem_st16(tstage + hs * 64 + eh * 32 + 16, packed + 16);
      }
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_hid_full);
      if constexpr (kTrace) {
        busy1 += static_cast<unsigned long long>(clock64() - t_mark);
        t_mark = clock64();
      }
      // ---- phase 2: conv2 accumulators of this tile, chunk by chunk -> + bias -> fp32 logits
#pragma unroll 1
      for (int ii = 0; ii < n_items; ++ii) {
        const HfItem item = items_s[ii];
        const int head = 2 * pair + item.head_slot;
        mbar_wait_t<kTrace>(bar_c2_full, c2_full_phase, w_c2);
        c2_full_phase ^= 1u;
        tc_fence_after();
        const int units = item.nc >> 4;
        const int cout = p.cout[head];
        const int mode = p.out_mode[head];
        uint32_t raw[16];
#pragma unroll 1
        for (int u = eh; u < units; u += 2) {
          tmem_ld16(tstage + 128 + u * 16, raw);
          tmem_ld_wait();
          const int ch0 = item.ch0 + u * 16;
          float v[16];
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const float4 bb = bias2_4[(item.bias_off >> 2) + u * 4 + i];
            v[4 * i + 0] = __uint_as_float(raw[4 * i + 0]) + bb.x;
            v[4 * i + 1] = __uint_as_float(raw[4 * i + 1]) + bb.y;
            v[4 * i + 2] = __uint_as_float(raw[4 * i + 2]) + bb.z;
            v[4 * i + 3] = __uint_as_float(raw[4 * i + 3]) + bb.w;
          }
          if (valid && ch0 < cout) {
            if (mode == 2) {
              float4* o = reinterpret_cast<float4*>(p.out[head]) +
                          2 * ((static_cast<size_t>(n) * p.out_planes[head] + (ch0 >> 3)) * plane_px + px);
              o[0] = make_float4(v[0], v[1], v[2], v[3]);
              o[1] = make_float4(v[4], v[5], v[6], v[7]);
              if (ch0 + 8 < cout) {
                o += 2 * plane_px;
                o[0] = make_float4(v[8], v[9], v[10], v[11]);
                o[1] = make_float4(v[12], v[13], v[14], v[15]);
              }
            } else {
              float* o = reinterpret_cast<float*>(p.out[head]) + (static_cast<size_t>(n) * cout + ch0) * plane_px + px;
#pragma unroll
              for (int i = 0; i < 16; ++i)
                if (ch0 + i < cout) o[i * plane_px] = v[i];
            }
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_c2_empty);
      }
      if (lane == 0) mbar_arrive(bar_acc_empty + 8 * s);
      if constexpr (kTrace) busy2 += static_cast<unsigned long long>(clock64() - t_mark);
    }
    if constexpr (kTrace) {
      if (warp == 4 && lane == 0) {
        trace[kHtEpAccFull] = w_acc;
        trace[kHtEpPhase1] = busy1;
        trace[kHtEpC2Full] = w_c2;
        trace[kHtEpPhase2] = busy2 - w_c2;
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc<512>(tmem_base);
  }
  if constexpr (kTrace) {
    if (threadIdx.x == 0) {
      trace[kHtPair] = pair;
      trace[kHtTiles] = my_tiles;
      trace[kHtStartNs] = t_start_ns;
      trace[kHtEndNs] = global_ns();
      trace[kHtCycles] = static_cast<unsigned long long>(clock64() - t_start_clk);
    }
  }
}

typedef CUresult (*HfEncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                    const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static HfEncodeTiledFn hf_encode_fn() { return reinterpret_cast<HfEncodeTiledFn>(tensor_map_encode_fn()); }

}  // namespace abc

extern "C" int abc_heads_fused(const AbcHeadsFusedDesc* d, void* stream_) {
  using namespace abc;
  if (int rc = device_check()) return rc;
  ABC_REQUIRE(d != nullptr, "abc_heads_fused: null descriptor");
  ABC_REQUIRE(d->in && d->w1pack && d->bias1 && d->w2pack && d->bias2, "abc_heads_fused: null input / weights / bias");
  ABC_REQUIRE(d->N > 0 && d->H > 0 && d->W > 0, "abc_heads_fused: bad geometry N=%d H=%d W=%d", d->N, d->H, d->W);
  ABC_REQUIRE(d->in_plane_off >= 0 && d->in_plane_off + 16 <= d->in_planes, "abc_heads_fused: the trunk has 128 channels = 16 planes");
  ABC_REQUIRE(d->n_heads >= 1 && d->n_heads <= 2 * kHfMaxPairs, "abc_heads_fused: n_heads=%d (1..%d)", d->n_heads, 2 * kHfMaxPairs);
  ABC_REQUIRE((reinterpret_cast<uintptr_t>(d->in) & 15) == 0 && (reinterpret_cast<uintptr_t>(d->w1pack) & 15) == 0 &&
                  (reinterpret_cast<uintptr_t>(d->w2pack) & 15) == 0 && (reinterpret_cast<uintptr_t>(d->bias2) & 15) == 0,
              "abc_heads_fused: buffers must be 16-byte aligned");
  const int pairs = (d->n_heads + 1) / 2;
  HfParams p{};
  p.N = d->N; p.H = d->H; p.W = d->W;
  p.tiles_x = (d->W + 7) / 8;
  p.tiles_y = (d->H + 15) / 16;
  const int64_t tiles = static_cast<int64_t>(d->N) * p.tiles_x * p.tiles_y;
  ABC_REQUIRE(tiles < (1ll << 31), "abc_heads_fused: too many tiles");
  p.num_tiles = static_cast<int>(tiles);
  p.in_plane_off = d->in_plane_off;
  p.w1 = static_cast<const uint8_t*>(d->w1pack);
  p.bias1 = d->bias1;
  p.w2 = static_cast<const uint8_t*>(d->w2pack);
  p.bias2 = d->bias2;
  for (int t = 0; t < 9; ++t) p.tap16[t] = static_cast<uint32_t>((t / 3) * 10 + (t % 3));   // (ky, kx) order, 16-byte units
  // conv2 chunks: channels [128 c, 128 (c + 1)) of every head, N rounded up to 16; the weight / bias packs hold them in
  // (head, chunk) order, each pair's bias block padded to the chunk widths
  int w2_off = 0, bias_off_total = 0;
  for (int pr = 0; pr < pairs; ++pr) {
    int ni = 0, bias_len = 0;
    p.bias2_off[pr] = bias_off_total;
    for (int hs = 0; hs < 2; ++hs) {
      const int head = 2 * pr + hs;
      if (head >= d->n_heads) break;
      const int cout = d->cout[head];
      ABC_REQUIRE(cout >= 1 && d->out[head] != nullptr, "abc_heads_fused: head %d: cout=%d / null output", head, cout);
      ABC_REQUIRE(d->out_mode[head] == 1 || d->out_mode[head] == 2, "abc_heads_fused: head %d: out_mode must be 1 (NCHW) or 2 (planar-8)", head);
      if (d->out_mode[head] == 2)
        ABC_REQUIRE(d->out_planes[head] >= (cout + 7) / 8, "abc_heads_fused: head %d: planar output needs %d planes", head, (cout + 7) / 8);
      p.out[head] = d->out[head];
      p.out_mode[head] = d->out_mode[head];
      p.cout[head] = cout;
      p.out_planes[head] = d->out_planes[head];
      const int chunks = (cout + 127) / 128;
      for (int cidx = 0; cidx < chunks; ++cidx) {
        ABC_REQUIRE(ni < kHfMaxItems, "abc_heads_fused: pair %d needs more than %d conv2 chunks", pr, kHfMaxItems);
        const int cnt = cout - 128 * cidx < 128 ? cout - 128 * cidx : 128;
        HfItem& it = p.items[pr][ni];
        it.head_slot = hs;
        it.nc = (cnt + 15) / 16 * 16;
        it.ch0 = 128 * cidx;
        it.w2_off = w2_off;
        it.bias_off = bias_len;
        w2_off += it.nc * 256;
        bias_len += it.nc;
        ++ni;
      }
    }
    ABC_REQUIRE(bias_len <= 512, "abc_heads_fused: pair %d: %d conv2 output columns exceed the 512 supported", pr, bias_len);
    p.n_items[pr] = ni;
    p.bias2_len[pr] = bias_len;
    bias_off_total += bias_len;
  }
  ABC_REQUIRE(w2_off == d->w2pack_bytes && bias_off_total == d->bias2_len,
              "abc_heads_fused: pack sizes differ (weights %d vs %lld bytes, bias %d vs %d floats); use abc_heads_fused_pack_sizes",
              w2_off, static_cast<long long>(d->w2pack_bytes), bias_off_total, d->bias2_len);

  HfEncodeTiledFn encode = hf_encode_fn();
  if (!encode) {
    set_error("cuTensorMapEncodeTiled driver entry point not available");
    return ABC_ERR_NO_DEVICE;
  }
  CUtensorMap tmap;
  const cuuint64_t gdim[4] = {static_cast<cuuint64_t>(d->W) * 8, static_cast<cuuint64_t>(d->H),
                              static_cast<cuuint64_t>(d->in_planes), static_cast<cuuint64_t>(d->N)};
  const cuuint64_t gstride[3] = {static_cast<cuuint64_t>(d->W) * 16, static_cast<cuuint64_t>(d->W) * d->H * 16,
                                 static_cast<cuuint64_t>(d->W) * d->H * 16 * d->in_planes};
  const cuuint32_t box[4] = {80, 18, 8, 1};
  const cuuint32_t estr[4] = {1, 1, 1, 1};
  const bool f16 = d->act_fp16 != 0;
  CUresult cr = encode(&tmap, f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(d->in), gdim, gstride, box, estr,
                       CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                       CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (cr != CUDA_SUCCESS) {
    set_error("abc_heads_fused: cuTensorMapEncodeTiled failed with CUresult %d", static_cast<int>(cr));
    return ABC_ERR_CUDA;
  }
  static PerDeviceOnce attr_once;
  ABC_CUDA(attr_once.run([] {
    void (*const kernels[4])(const CUtensorMap, const HfParams) = {heads_fused_kernel<false, false>, heads_fused_kernel<true, false>,
                                                                   heads_fused_kernel<false, true>, heads_fused_kernel<true, true>};
    for (auto k : kernels)
      if (cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, kHfSmem); e != cudaSuccess) return e;
    return cudaSuccess;
  }));
  int sms = sm_count();
  if (sms <= 0) sms = 148;
  int64_t cost[kHfMaxPairs];
  for (int pr = 0; pr < pairs; ++pr) {
    int nc[kHfMaxItems], channels = 0;
    for (int i = 0; i < p.n_items[pr]; ++i) nc[i] = p.items[pr][i].nc;
    for (int hs = 0; hs < 2 && 2 * pr + hs < d->n_heads; ++hs) channels += d->cout[2 * pr + hs];
    cost[pr] = hf_pair_tile_cost(p.n_items[pr], nc, channels);
  }
  int ctas[kHfMaxPairs];
  const int total = hf_split_ctas(pairs, cost, sms, p.num_tiles, ctas);
  p.pairs = pairs;
  p.cta0[0] = 0;
  for (int pr = 0; pr < pairs; ++pr) p.cta0[pr + 1] = p.cta0[pr] + ctas[pr];
  p.trace = static_cast<unsigned long long*>(d->trace);
  cudaStream_t st = static_cast<cudaStream_t>(stream_);
  if (d->trace)
    (f16 ? heads_fused_kernel<true, true> : heads_fused_kernel<false, true>)<<<total, kHfThreads, kHfSmem, st>>>(tmap, p);
  else if (f16)
    heads_fused_kernel<true, false><<<total, kHfThreads, kHfSmem, st>>>(tmap, p);
  else
    heads_fused_kernel<false, false><<<total, kHfThreads, kHfSmem, st>>>(tmap, p);
  return launch_check("heads_fused_kernel");
}

extern "C" int abc_heads_fused_pack_sizes(int n_heads, const int* cout, int64_t* w2pack_bytes, int* bias2_len) {
  using namespace abc;
  ABC_REQUIRE(n_heads >= 1 && n_heads <= 2 * kHfMaxPairs && cout && w2pack_bytes && bias2_len, "abc_heads_fused_pack_sizes: bad arguments");
  int64_t wb = 0;
  int bl = 0;
  for (int h = 0; h < n_heads; ++h) {
    ABC_REQUIRE(cout[h] >= 1, "abc_heads_fused_pack_sizes: cout[%d]=%d", h, cout[h]);
    for (int c0 = 0; c0 < cout[h]; c0 += 128) {
      const int cnt = cout[h] - c0 < 128 ? cout[h] - c0 : 128;
      const int nc = (cnt + 15) / 16 * 16;
      wb += nc * 256;
      bl += nc;
    }
  }
  *w2pack_bytes = wb;
  *bias2_len = bl;
  return ABC_OK;
}

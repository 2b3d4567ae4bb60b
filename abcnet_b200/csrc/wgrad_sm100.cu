// Weight-gradient implicit GEMM for sm_100a (tcgen05, accumulators resident in TMEM across the whole pixel loop).
//
// Replaces cuDNN's backward-filter behind autograd of nn.Conv2d / nn.ConvTranspose2d (/root/reference/src/train.py:140):
//   dW[tap][co][ci] = sum over (n, y, x) of dz[n, co, y, x] * a[n, ci, y + dy(tap), x + dx(tap)]
// GEMM view per tap: D[M = co][N = ci], K = pixels. Both operands come straight from the P8 activation layout
// ([N][C/8][H][W][8] bf16) as MN-major SWIZZLE_NONE core matrices: 8 consecutive pixels of one 8-channel plane are
// 8 K-rows x 16 bytes = 128 contiguous bytes; the next 8 channels are one plane pitch away (SBO) and the next 8 pixels
// are the next tile row (LBO). A K = 16 MMA therefore consumes two rows of the 16 x 8 pixel tile; the 3x3 taps are
// start-address shifts inside the activation halo tile, exactly as in the forward kernel.
//
// Each CTA owns one (co tile, ci tile, tap group) and a strided subset of the pixel tiles; it accumulates
// taps_per_cta x [128 x n_tile] fp32 blocks in TMEM (taps_per_cta * n_tile <= 512 columns) over all its tiles and adds
// them to the global fp32 gradient with atomicAdd at the end (split-K over CTAs). The deterministic variant (DET) stores the
// block to the CTA's split-K slot of a workspace instead, and det_reduce adds the slots to the gradient in slot order.
#include <cuda.h>
#include <cuda_bf16.h>

#include "common.cuh"
#include "det_slots.cuh"
#include "ptx_sm100.cuh"

namespace abc {

constexpr int kWgThreads = 192;          // warp 0: TMA producer, warp 1: MMA issuer + TMEM owner, warps 2-5: epilogue
constexpr uint32_t kWgHeader = 1024;
constexpr int kWgStages = 3;           // maximum; the launch picks 2 or 3 from the shared-memory budget

struct WgradParams {
  int N, H, W, tiles_x, tiles_y, num_tiles;
  int dz_plane_off, a_plane_off;
  int m_planes;            // planes of dz loaded per tile (<= 16)
  int n_tile;              // ci per CTA (multiple of 16, <= 256)
  int n_ci_tiles, n_co_tiles, tap_groups, taps_per_cta, ntaps, halo;
  int cout, cin, stages;
  uint32_t a_stage_bytes, dz_tile_bytes, in_tile_bytes, in_plane_bytes, in_row_bytes;
  uint32_t tap_off[9];
  // tap-folded mode (cin <= 32): every tap's shifted 16 x 8 box of the input is loaded as its own smem block, so that the
  // taps line up on the GEMM N axis (N = taps * cin) and ONE MMA per K step replaces `ntaps` N = cin MMAs whose cost is
  // bounded below by the A-operand read, not by N.
  // row-box mode (fold == 2; the plain 3x3 tap set, cin <= 32): only the THREE row-shifted 16 x 10 boxes are loaded (the dy taps on
  // the GEMM N axis, N = 3 * cin) and the dx taps are 16-byte start-address shifts inside them: three MMAs per K step, but
  // 19 KB instead of 40 KB of L2 -> shared-memory traffic per 128 pixels, which is what bounded the 9-box variant.
  int fold, fold_groups, fold_tap0[2], fold_ntaps[2];
  int tap_dy[9], tap_dx[9];
  int tap_col[9];          // row-box mode: accumulator column block of tap t = (dx + 1) * 3 + (dy + 1)
  float* dw;               // [ntaps][cout][cin] fp32, accumulated with atomicAdd
  float* ws;               // DET: [gridDim.x][ntaps][cout][cin] fp32 split-K slots (det_slots.cuh)
};

template <bool DET = false>
__global__ void __launch_bounds__(kWgThreads, 1)
wgrad_kernel(const __grid_constant__ CUtensorMap tmap_dz, const __grid_constant__ CUtensorMap tmap_in, const WgradParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t sbase = smem_u32(smem);
  const int warp = static_cast<int>(warp_id_uniform());
  const int lane = threadIdx.x & 31;
  const uint32_t bar_full = sbase, bar_empty = sbase + 8 * kWgStages, bar_done = sbase + 16 * kWgStages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + 512);

  // blockIdx.y -> (co tile, ci tile, tap group)
  int by = blockIdx.y;
  const int tg = by % p.tap_groups;
  by /= p.tap_groups;
  const int ci_t = by % p.n_ci_tiles;
  const int co_t = by / p.n_ci_tiles;
  const int tap0 = tg * p.taps_per_cta;
  const int ntap = min(p.taps_per_cta, p.ntaps - tap0);

  if (threadIdx.x == 0) {
    for (int i = 0; i < kWgStages; ++i) {
      mbar_init(bar_full + 8 * i, 1);
      mbar_init(bar_empty + 8 * i, 1);
    }
    mbar_init(bar_done, 1);
    fence_mbar_init();
    tma_prefetch_desc(&tmap_dz);
    tma_prefetch_desc(&tmap_in);
  }
  if (warp == 1) tmem_alloc<512>(smem_u32(tmem_slot));
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_slot);
  const uint32_t stage0 = sbase + kWgHeader;
  const int tiles_per_img = p.tiles_x * p.tiles_y;
  const bool has_work = static_cast<int>(blockIdx.x) < p.num_tiles;

  if (warp == 0) {
    int stage = 0;
    uint32_t phase = 0;
    for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
      const int n = tile / tiles_per_img;
      const int rem = tile - n * tiles_per_img;
      const int ty = rem / p.tiles_x;
      const int tx = rem - ty * p.tiles_x;
      mbar_wait(bar_empty + 8 * stage, phase ^ 1);
      if (elect_one()) {
        const uint32_t dst = stage0 + stage * p.a_stage_bytes;
        mbar_arrive_expect_tx(bar_full + 8 * stage, p.dz_tile_bytes + p.in_tile_bytes);
        tma_load_4d(dst, &tmap_dz, bar_full + 8 * stage, tx * 64, ty * 16, p.dz_plane_off + co_t * 16, n);
        if (p.fold == 2) {
          const uint32_t blk = static_cast<uint32_t>(p.n_tile >> 3) * 2560u;      // one dy box: planes x 16 rows x 10 pixels x 16 B
          for (int j = 0; j < 3; ++j)
            tma_load_4d(dst + 32768 + j * blk, &tmap_in, bar_full + 8 * stage, (tx * 8 - 1) * 8, ty * 16 + j - 1,
                        p.a_plane_off + ci_t * (p.n_tile >> 3), n);
        } else if (p.fold) {
          const uint32_t blk = static_cast<uint32_t>(p.n_tile >> 3) * 2048u;
          for (int t = 0; t < ntap; ++t)
            tma_load_4d(dst + 32768 + t * blk, &tmap_in, bar_full + 8 * stage, (tx * 8 + p.tap_dx[tap0 + t]) * 8,
                        ty * 16 + p.tap_dy[tap0 + t], p.a_plane_off + ci_t * (p.n_tile >> 3), n);
        } else {
          tma_load_4d(dst + 32768, &tmap_in, bar_full + 8 * stage, (tx * 8 - p.halo) * 8, ty * 16 - p.halo,
                      p.a_plane_off + ci_t * (p.n_tile >> 3), n);
        }
      }
      __syncwarp();
      if (++stage == p.stages) {
        stage = 0;
        phase ^= 1;
      }
    }
  } else if (warp == 1) {
    // A = dz^T (M = co): MN-major, LBO = next 8 pixels = next tile row (128 B), SBO = next 8 channels = plane pitch (2048 B)
    // B = a     (N = ci): MN-major, LBO = halo row pitch, SBO = halo plane pitch
    const uint32_t idesc = umma_idesc_bf16(128, p.n_tile, 1, 1);
    const uint32_t idesc_f0 = umma_idesc_bf16(128, p.fold == 2 ? 3 * p.n_tile : (p.fold ? p.fold_ntaps[0] * p.n_tile : 16), 1, 1);
    const uint32_t idesc_f1 = umma_idesc_bf16(128, (p.fold && p.fold_groups > 1) ? p.fold_ntaps[1] * p.n_tile : 16, 1, 1);
    const uint64_t a_hi64 = umma_desc_hi(128, 2048);
    const uint64_t b_hi64 = p.fold == 2 ? umma_desc_hi(160, 2560) : (p.fold ? umma_desc_hi(128, 2048) : umma_desc_hi(p.in_row_bytes, p.in_plane_bytes));
    const uint32_t a_hi = static_cast<uint32_t>(a_hi64 >> 32), b_hi = static_cast<uint32_t>(b_hi64 >> 32);
    const uint32_t a_lo0 = static_cast<uint32_t>(a_hi64) | (stage0 >> 4);
    const uint32_t b_lo0 = static_cast<uint32_t>(b_hi64) | ((stage0 + 32768) >> 4);
    const uint32_t stage16 = p.a_stage_bytes >> 4;
    const uint32_t a_kstep = (2 * 128) >> 4, b_kstep = p.fold == 2 ? (2 * 160) >> 4 : (p.fold ? a_kstep : (2 * p.in_row_bytes) >> 4);
    const uint32_t fold_blk16 = (static_cast<uint32_t>(p.n_tile >> 3) * 2048u) >> 4;
    int stage = 0;
    uint32_t phase = 0, first = 0;
    for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
      mbar_wait(bar_full + 8 * stage, phase);
      tc_fence_after();
      if (elect_one()) {
        const uint32_t a_base = a_lo0 + stage * stage16, b_base = b_lo0 + stage * stage16;
        if (p.fold == 2) {
#pragma unroll
          for (int s = 0; s < 8; ++s)
#pragma unroll
            for (int j = 0; j < 3; ++j)          // dx = j - 1: one pixel = 16 bytes further into the 10-pixel rows
              umma_bf16_lohi(tmem_base + j * 3 * p.n_tile, a_base + s * a_kstep, a_hi, b_base + j + s * b_kstep, b_hi, idesc_f0,
                             s != 0 ? 1u : first);
        } else if (p.fold) {
#pragma unroll
          for (int s = 0; s < 8; ++s) {
            umma_bf16_lohi(tmem_base, a_base + s * a_kstep, a_hi, b_base + s * b_kstep, b_hi, idesc_f0, s != 0 ? 1u : first);
            if (p.fold_groups > 1)
              umma_bf16_lohi(tmem_base + p.fold_tap0[1] * p.n_tile, a_base + s * a_kstep, a_hi,
                             b_base + p.fold_tap0[1] * fold_blk16 + s * b_kstep, b_hi, idesc_f1, s != 0 ? 1u : first);
          }
        } else
        for (int t = 0; t < ntap; ++t) {
          const uint32_t b_tap = b_base + (p.tap_off[tap0 + t] >> 4);
#pragma unroll
          for (int s = 0; s < 8; ++s)
            umma_bf16_lohi(tmem_base + t * p.n_tile, a_base + s * a_kstep, a_hi, b_tap + s * b_kstep, b_hi, idesc,
                           s != 0 ? 1u : first);
        }
        umma_commit(bar_empty + 8 * stage);
      }
      __syncwarp();
      first = 1;
      if (++stage == p.stages) {
        stage = 0;
        phase ^= 1;
      }
    }
    if (has_work && elect_one()) umma_commit(bar_done);
    __syncwarp();
  } else if (has_work) {
    // epilogue: warps 2..5 -> TMEM lane quarter = warp % 4
    const int q = warp & 3;
    const int co = co_t * 128 + q * 32 + lane;
    mbar_wait(bar_done, 0);
    tc_fence_after();
    for (int t = 0; t < ntap; ++t) {
      const size_t off = (static_cast<size_t>(tap0 + t) * p.cout + co) * p.cin + ci_t * p.n_tile;
      float* dst = DET ? p.ws + det_slot_index(blockIdx.x, p.ntaps * p.cout * p.cin, 0) + off : p.dw + off;
      const uint32_t taddr = tmem_base + (p.fold == 2 ? p.tap_col[tap0 + t] : t) * p.n_tile + (static_cast<uint32_t>(q * 32) << 16);
      for (int c0 = 0; c0 < p.n_tile; c0 += 16) {
        uint32_t raw[16];
        tmem_ld16(taddr + c0, raw);
        tmem_ld_wait();
        if (co < p.cout) {
#pragma unroll
          for (int i = 0; i < 16; ++i)
            if (ci_t * p.n_tile + c0 + i < p.cin) {
              if constexpr (DET) dst[c0 + i] = __uint_as_float(raw[i]);
              else atomicAdd(dst + c0 + i, __uint_as_float(raw[i]));
            }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<512>(tmem_base);
  }
}

typedef CUresult (*EncodeTiledFn2)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                   const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                   CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn2 wg_encode_fn() { return reinterpret_cast<EncodeTiledFn2>(tensor_map_encode_fn()); }

static int make_map(CUtensorMap* m, const void* base, int W, int H, int planes, int N, int box_cols, int box_rows, int box_planes) {
  EncodeTiledFn2 enc = wg_encode_fn();
  if (!enc) {
    set_error("cuTensorMapEncodeTiled driver entry point not available");
    return ABC_ERR_NO_DEVICE;
  }
  const cuuint64_t gdim[4] = {static_cast<cuuint64_t>(W) * 8, static_cast<cuuint64_t>(H), static_cast<cuuint64_t>(planes),
                              static_cast<cuuint64_t>(N)};
  const cuuint64_t gstride[3] = {static_cast<cuuint64_t>(W) * 16, static_cast<cuuint64_t>(W) * H * 16,
                                 static_cast<cuuint64_t>(W) * H * 16 * planes};
  const cuuint32_t box[4] = {static_cast<cuuint32_t>(box_cols * 8), static_cast<cuuint32_t>(box_rows),
                             static_cast<cuuint32_t>(box_planes), 1};
  const cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult cr = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(base), gdim, gstride, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (cr != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed with CUresult %d", static_cast<int>(cr));
    return ABC_ERR_CUDA;
  }
  return ABC_OK;
}

// Launch parameters of abc_conv_wgrad (everything but the tensor maps): grid, shared memory, kernel parameters.
static int wgrad_setup(const AbcWgradDesc* d, WgradParams& p, dim3& grid, uint32_t& smem_launch) {
  ABC_REQUIRE(d && d->dz && d->in && d->dw, "abc_conv_wgrad: null argument");
  ABC_REQUIRE(d->N > 0 && d->H > 0 && d->W > 0, "abc_conv_wgrad: bad geometry");
  ABC_REQUIRE(d->cout >= 8 && d->cout % 8 == 0 && d->cin >= 16 && d->cin % 16 == 0, "abc_conv_wgrad: cout %% 8, cin %% 16 (cout=%d cin=%d)",
              d->cout, d->cin);
  ABC_REQUIRE(d->ntaps >= 1 && d->ntaps <= 9, "abc_conv_wgrad: ntaps");
  ABC_REQUIRE(d->dz_plane_off >= 0 && d->dz_plane_off + d->cout / 8 <= d->dz_planes && d->in_plane_off >= 0 &&
                  d->in_plane_off + d->cin / 8 <= d->in_planes, "abc_conv_wgrad: plane ranges");
  int halo = 0;
  for (int t = 0; t < d->ntaps; ++t) {
    ABC_REQUIRE(d->tap_dy[t] >= -1 && d->tap_dy[t] <= 1 && d->tap_dx[t] >= -1 && d->tap_dx[t] <= 1, "abc_conv_wgrad: tap offset");
    if (d->tap_dy[t] || d->tap_dx[t]) halo = 1;
  }
  p = WgradParams{};
  p.N = d->N; p.H = d->H; p.W = d->W;
  p.tiles_x = (d->W + 7) / 8; p.tiles_y = (d->H + 15) / 16;
  const int64_t tiles = static_cast<int64_t>(d->N) * p.tiles_x * p.tiles_y;
  ABC_REQUIRE(tiles < (1ll << 31), "abc_conv_wgrad: too many tiles");
  p.num_tiles = static_cast<int>(tiles);
  p.dz_plane_off = d->dz_plane_off; p.a_plane_off = d->in_plane_off;
  p.cout = d->cout; p.cin = d->cin; p.ntaps = d->ntaps; p.halo = halo;
  p.n_tile = d->cin < 128 ? d->cin : 128;
  ABC_REQUIRE(d->cin % p.n_tile == 0, "abc_conv_wgrad: cin=%d must be <= 128 or a multiple of 128", d->cin);
  p.n_ci_tiles = d->cin / p.n_tile;
  p.n_co_tiles = (d->cout + 127) / 128;
  p.m_planes = d->cout < 128 ? d->cout / 8 : 16;
  int tpc = 512 / p.n_tile;
  if (tpc > d->ntaps) tpc = d->ntaps;
  if (d->ntaps == 9 && tpc < 9) tpc = tpc >= 3 ? 3 : 1;       // balanced tap groups for 3x3
  if (d->ntaps == 4 && tpc < 4) tpc = tpc >= 2 ? 2 : 1;
  p.taps_per_cta = tpc;
  p.tap_groups = (d->ntaps + tpc - 1) / tpc;
  const int rows = 16 + 2 * halo, cols = 8 + 2 * halo;
  p.in_row_bytes = cols * 16;
  p.in_plane_bytes = rows * p.in_row_bytes;
  p.in_tile_bytes = (p.n_tile / 8) * p.in_plane_bytes;
  p.dz_tile_bytes = p.m_planes * 2048;
  p.fold = (d->cin <= 32 && d->ntaps > 1 && p.tap_groups == 1) ? 1 : 0;
  if (p.fold) {
    p.in_tile_bytes = static_cast<uint32_t>(d->ntaps) * (p.n_tile / 8) * 2048u;
    const int per = 256 / p.n_tile;                       // taps per MMA (N <= 256)
    if (d->ntaps <= per) {
      p.fold_groups = 1; p.fold_tap0[0] = 0; p.fold_ntaps[0] = d->ntaps;
    } else {
      ABC_REQUIRE(d->ntaps <= 2 * per, "abc_conv_wgrad: internal: fold groups");
      p.fold_groups = 2; p.fold_tap0[0] = 0; p.fold_ntaps[0] = (d->ntaps + 1) / 2;
      p.fold_tap0[1] = p.fold_ntaps[0]; p.fold_ntaps[1] = d->ntaps - p.fold_ntaps[0];
    }
  }
  // Opt-in (AbcWgradDesc.row_boxes): measured equal to the 9-box variant on the whole training step (1744 vs 1745 img/s,
  // profiles/r02_train_ab_wgrad_rowbox.txt) -- the halved L2 fill is paid back by three A-operand reads per K step -- so the
  // default stays the 9-box variant; both are covered by tests/test_train_ops_gpu.py::test_wgrad_conv3x3.
  if (p.fold && d->ntaps == 9 && d->row_boxes) {
    bool seen[9] = {false, false, false, false, false, false, false, false, false};
    bool plain = true;
    for (int t = 0; t < 9; ++t) {
      const int cb = (d->tap_dx[t] + 1) * 3 + (d->tap_dy[t] + 1);
      plain = plain && !seen[cb];
      seen[cb] = true;
      p.tap_col[t] = cb;
    }
    if (plain) {                       // the 9 distinct taps of a 3x3 kernel, in any order
      p.fold = 2;
      p.in_tile_bytes = 3u * (p.n_tile / 8) * 2560u;
    }
  }
  p.a_stage_bytes = 32768 + ((p.in_tile_bytes + 1023u) & ~1023u);
  for (int t = 0; t < d->ntaps; ++t) {
    p.tap_off[t] = static_cast<uint32_t>(((d->tap_dy[t] + halo) * cols + (d->tap_dx[t] + halo)) * 16);
    p.tap_dy[t] = d->tap_dy[t];
    p.tap_dx[t] = d->tap_dx[t];
  }
  p.dw = d->dw;
  p.stages = static_cast<int>((232448 - kWgHeader) / p.a_stage_bytes);
  if (p.stages > kWgStages) p.stages = kWgStages;
  ABC_REQUIRE(p.stages >= 2, "abc_conv_wgrad: shared memory budget exceeded");
  const uint32_t smem_bytes = kWgHeader + p.stages * p.a_stage_bytes;
  const int gy = p.n_co_tiles * p.n_ci_tiles * p.tap_groups;
  grid = dim3(wgrad_grid_x(sm_count(), gy, p.num_tiles), gy);
  smem_launch = smem_bytes < 120 * 1024 ? 120 * 1024 : smem_bytes;   // 1 CTA / SM (owns all TMEM columns)
  return ABC_OK;
}

}  // namespace abc

extern "C" int abc_conv_wgrad(const AbcWgradDesc* d, void* stream) {
  using namespace abc;
  if (int rc = device_check()) return rc;
  WgradParams p;
  dim3 grid;
  uint32_t smem_launch;
  if (int rc = wgrad_setup(d, p, grid, smem_launch)) return rc;
  const int rows = 16 + 2 * p.halo, cols = 8 + 2 * p.halo;
  CUtensorMap map_dz, map_in;
  if (int rc = make_map(&map_dz, d->dz, d->W, d->H, d->dz_planes, d->N, 8, 16, p.m_planes)) return rc;
  if (int rc = make_map(&map_in, d->in, d->W, d->H, d->in_planes, d->N, p.fold == 2 ? 10 : (p.fold ? 8 : cols), p.fold ? 16 : rows, p.n_tile / 8))
    return rc;
  static PerDeviceOnce attr_once;
  ABC_CUDA(attr_once.run([] {
    if (cudaError_t e = cudaFuncSetAttribute(wgrad_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448)) return e;
    return cudaFuncSetAttribute(wgrad_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448);
  }));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (d->ws) {        // deterministic: every CTA stores its block to slot blockIdx.x, then dw += the slots in slot order
    p.ws = d->ws;
    wgrad_kernel<true><<<grid, kWgThreads, smem_launch, st>>>(map_dz, map_in, p);
    if (int rc = launch_check("wgrad_kernel")) return rc;
    const int n = d->ntaps * d->cout * d->cin;
    return det_reduce(d->ws, static_cast<int>(grid.x), n, det_out1(d->dw, n), 1, st);
  }
  wgrad_kernel<false><<<grid, kWgThreads, smem_launch, st>>>(map_dz, map_in, p);
  return launch_check("wgrad_kernel");
}

extern "C" size_t abc_conv_wgrad_workspace_bytes(const AbcWgradDesc* d) {
  using namespace abc;
  WgradParams p;
  dim3 grid;
  uint32_t smem_launch;
  if (wgrad_setup(d, p, grid, smem_launch) != ABC_OK) return 0;
  return det_ws_bytes(grid.x, static_cast<long long>(d->ntaps) * d->cout * d->cin, sizeof(float));
}

/*
 * abcnet_b200 -- C-ABI of the B200-native ABC-Net hot path (U-Net pass + heat-map decoding + losses).
 *
 * The reference (zhang-xuan1314/ABC-Net) has no FFI / plugin API of its own: every GPU instruction it
 * executes is issued by PyTorch library kernels (SURVEY.md section 2.2). Each entry point below therefore
 * replaces a *call site* of the reference, cited as file:line relative to /root/reference.
 *
 * Conventions
 *   - plain C, no torch / CUDA types in the signatures: device pointers are void*, the CUDA stream is a
 *     void* holding a cudaStream_t (NULL = legacy default stream);
 *   - every function returns 0 on success or a negative AbcStatus; abc_last_error() gives a thread-local
 *     message. Nothing throws across the ABI. Nothing allocates device memory: the caller owns all buffers;
 *   - there is NO CPU fallback: without a CUDA device of compute capability 10.x the compute entry points
 *     return ABC_ERR_NO_DEVICE.
 *
 * Activation layout "P8" (planar-8, a.k.a. NC/8HWC8): bf16 tensor [N][C/8][H][W][8]. Channel c lives in
 * plane c/8, slot c%8. A concatenation along channels is a plane offset into a wider buffer, so the
 * reference's F.pad + torch.cat (src/unet.py:51-59) cost nothing.
 */
#ifndef ABCNET_B200_H_
#define ABCNET_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ABC_API __attribute__((visibility("default")))

typedef enum AbcStatus {
  ABC_OK = 0,
  ABC_ERR_INVALID = -1,    /* bad argument (shape / alignment / range) */
  ABC_ERR_NO_DEVICE = -2,  /* no sm_100 device, or driver entry point missing */
  ABC_ERR_CUDA = -3,       /* a CUDA call failed; see abc_last_error() */
  ABC_ERR_CAPACITY = -4    /* caller-provided capacity too small (decode); counts still valid */
} AbcStatus;

ABC_API const char* abc_last_error(void);
ABC_API int abc_version(void);
/* 1 if the current device can run the kernels (compute capability 10.x), else 0. */
ABC_API int abc_device_ok(void);
/* Number of SMs of the current device (grid sizing), or a negative status. */
ABC_API int abc_sm_count(void);
/* Kernels launched by this library in the calling process so far (bench.py's gpu_launches). */
ABC_API int64_t abc_launch_count(void);

/* ---------------------------------------------------------------------------------------------------
 * First convolution: 1 -> 16 channels, 3x3, pad 1, BatchNorm folded, ReLU.
 * Replaces nn.Conv2d + BatchNorm2d + ReLU of inc1 (src/unet.py:12-14 via :83,:101) for in_channels = 1.
 *   img   fp32 [N][1][H][W] (values {0,1}: src/utils.py:80-81, src/utils_for_test.py:22-27)
 *   w     fp32 [16][9] folded weights, b fp32 [16] folded bias
 *   out   P8 bf16 [N][out_planes][H][W][8], channels written to planes [out_plane_off, out_plane_off+2)
 */
ABC_API int abc_conv3x3_c1(const float* img, const float* w, const float* b, void* out, int N, int H, int W,
                           int out_planes, int out_plane_off, void* stream);
/* Same with the binarised image held as uint8 {0,1} (what src/utils_for_test.py:22-24 computes before its float cast):
 * 4x fewer bytes over PCIe and HBM. */
ABC_API int abc_conv3x3_c1_u8(const uint8_t* img, const float* w, const float* b, void* out, int N, int H, int W,
                              int out_planes, int out_plane_off, void* stream);
/* The stem with every option: img fp32 [N][cin][H][W] (img_is_u8 = 0) or uint8 {0,1} [N][1][H][W] (img_is_u8 = 1, cin = 1);
 * flags bit 0: ReLU (eval) / raw conv + bias (train), bit 1: fp16 output instead of bf16 (AbcConvDesc.act_fp16). */
ABC_API int abc_conv3x3_stem(const void* img, int img_is_u8, int cin, const float* w, const float* b, void* out, int N, int H, int W,
                             int out_planes, int out_plane_off, int flags, void* stream);
/* General stem for in_channels = cin in 1..8 real-valued fp32 channels (src/unet.py:77,83 with in_channels != 1; the reference's
 * self-check builds UNet(in_channels=3), unet.py:127): img fp32 NCHW [N][cin][H][W], w fp32 [16][cin][9], b fp32 [16];
 * relu = 1: (BatchNorm-folded) conv + ReLU for eval, relu = 0: raw conv + bias for the training pass. Output as above. */
ABC_API int abc_conv3x3_cn(const float* img, int cin, const float* w, const float* b, void* out, int N, int H, int W,
                           int out_planes, int out_plane_off, int relu, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * Implicit-GEMM convolution on tcgen05 tensor cores (bf16 x bf16 -> fp32 in TMEM).
 * One kernel covers: 3x3 pad-1 convolutions (src/unet.py:12,15,66), the 1x1 head convolutions (:70), and,
 * phase by phase, the stride-2 transposed convolution followed by the crop of Up.forward (:44,:49-55).
 *
 * GEMM view: M = output pixels (tiles of 16 rows x 8 columns of one image), N = output channels
 * (tiles of n_tile), K = cin * ntaps. For every tap t the input pixel of output grid position (y, x) is
 * (y + tap_dy[t], x + tap_dx[t]); out-of-image pixels read as zero.
 *
 * Packed weights: bf16 [n_tiles][cin/kc][ntaps][kc/8][n_tile][8] with kc = min(cin, 64); element
 * (nt, c, t, p, r, e) multiplies input channel c*kc + p*8 + e and produces output channel nt*n_tile + r
 * (rows past cout are zero). bias: fp32 [n_tiles*n_tile].
 */
typedef struct AbcConvDesc {
  const void* in;        /* P8 bf16 [N][in_planes][H][W][8] */
  int N, H, W;           /* input grid */
  int in_planes;         /* planes of the input buffer */
  int in_plane_off;      /* first plane read */
  int cin;               /* channels read: multiple of 16 */
  const void* wpack;     /* packed weights (see above), 16-byte aligned */
  const float* bias;
  int cout;              /* valid output channels */
  int n_tile;            /* multiple of 16, 16..256 */
  int ntaps;             /* 1..9 */
  int tap_dy[9];
  int tap_dx[9];         /* each in [-1, 1] */
  int act;               /* 0 none, 1 ReLU, 2 LeakyReLU(0.01) */
  int out_mode;          /* 0: P8 bf16, 1: NCHW fp32 [N][cout][out_H][out_W], 2: planar-8 fp32 [N][out_planes][out_H][out_W][8] */
  void* out;             /* may be NULL when only the pooled output is wanted */
  int out_planes;        /* P8: planes of the output buffer */
  int out_plane_off;     /* P8: first plane written (concat slot) */
  int out_H, out_W;      /* output grid; output pixel = (y*out_sy + out_oy, x*out_sx + out_ox) */
  int out_sy, out_oy, out_sx, out_ox;
  void* pool_out;        /* optional fused MaxPool2d(2) (src/unet.py:30): P8 bf16 [N][pool_planes][H/2][W/2][8] */
  int pool_planes, pool_plane_off;
  /* Optional K segmentation (0 / 1 = off): the cin channels are split into k_segments equal segments and segment s only
   * uses taps [seg_tap0[s], seg_tap0[s] + seg_ntaps[s]); packed weights then hold, per n-tile, the blocks in consumption
   * order (chunk-major, that chunk's taps). Used for the data gradient of the up-sampling convolution, whose four
   * sub-pixel phases (stacked on the plane axis by abc_deinterleave2) each see their own taps. */
  int k_segments;
  int seg_tap0[4];
  int seg_ntaps[4];
  /* Optional row folding for the 16 / 32-channel layers (0 / 1 = off; 2 or 4): the tensor pipe of an N <= 32 MMA is
   * bound by the shared-memory read of its 128 x 16 activation operand, so J vertically adjacent output pixels are made
   * ONE GEMM row with N = J * cout columns (a Toeplitz expansion of the 3x3 kernel along y): 3 * (J + 2) MMAs per
   * 128 * J pixels instead of 9 * J. Needs the plain 3x3 tap set (ntaps = 9), out_mode 0 without output scaling,
   * n_tile == J * cout, and a folded weight pack: per K chunk the blocks of the 3 * (J + 2) folded taps
   * t' = 3 * r + c (input row offset r - 1 from the first of the J rows, column offset c - 1); block row
   * n = (b * J + j) * 16 + i holds W[co = 16 b + i][ci][ky = r - j][kx = c] (zero unless 0 <= r - j <= 2);
   * bias[n] = bias of channel 16 b + i. */
  int row_fold;
  /* Optional CTA-pair mode (0 = off) for layers with cin >= 128: the kernel is launched as (2,1,1) clusters and every
   * tcgen05.mma is a cta_group::2 instruction with M = 256 (two 128-pixel tiles, one per SM of a TPC); each CTA loads half
   * of every weight block, which halves the shared-memory operand traffic and the L2 -> SM weight stream per SM. The
   * weight pack must hold, for every (n-tile, K chunk, tap) block, first the rows [0, n_tile / 2) then [n_tile / 2, n_tile),
   * each half in the 128-byte swizzle layout of a K-major tcgen05 operand: bf16 [n_tiles][cin/64][ntaps][2][n_tile/2][64]
   * where the 16-byte chunk c (channels 8c .. 8c+7) of row r is stored at chunk position c ^ (r % 8).
   * Needs cin % 64 == 0, n_tile % 32 == 0, no row_fold / k_segments. */
  int cta_pair;
  /* Optional operand swap (0 = off) for layers with n_tile == 128 (the mid-U-Net 128 -> 128 convolutions and their data
   * gradients): the GEMM is issued as D^T = W * A^T, i.e. M = the 128 output channels of the n-tile (weights = tcgen05 A
   * operand) and N = 256 pixels (a 32 x 8 pixel tile = B operand). A tcgen05.mma pays a fixed cost for fetching its
   * 128 x 16 A operand from shared memory, so one N = 256 instruction replaces two N = 128 ones (measured on the same
   * kernel: N = 256 layers reach 1.38 - 1.64 PFLOP/s stand-alone, N = 128 layers 1.22). The accumulator then holds
   * [channel = TMEM lane][pixel = column]; the epilogue transposes 8 channels x 8 pixels through shared memory so that the
   * bf16 P8 stores stay 16 bytes per pixel and 128 contiguous bytes per tile row. Same weight pack, same results as the
   * unswapped kernel bit for bit (identical K order per output element). Needs out_mode 0, no pool_out, no k_segments /
   * cta_pair. May be combined with row_fold = J in {2, 4} for cout = 128 / J (the 64- and 32-channel layers): the 128 GEMM rows
   * are then (folded row j, channel) -- weight pack rows ordered j * cout + co instead of row_fold's (16-channel block, j,
   * channel) order, bias[j * cout + co] = bias of channel co -- and a pixel column stands for J vertically adjacent pixels. */
  int swap_mn;
  /* Optional fused train-mode BatchNorm statistics (src/unet.py:13,16,67 in train() mode): per output channel the sum and sum
   * of squares of the bf16-rounded outputs, fp64 [cout], zeroed by the call. Built for swap_mn launches and for the row-folded
   * 16 -> 16 layers (row_fold = 4, cin = cout = 16); other layers use abc_bn_stats. Replaces one full read of the conv output. */
  double* stat_sum;
  double* stat_sq;
  /* Optional sub-pixel output blocks (0 = off; else the channel count of ONE phase, multiple of 16): the stride-2 transposed
   * convolution + crop of Up.forward (src/unet.py:44,49-55) as ONE launch instead of four. cout must be 4 * subpixel; GEMM
   * column c = phase * subpixel + channel with phase = 2 * py + px is stored at output pixel
   * (y * 2 + out_oy + py, x * 2 + out_ox + px), plane out_plane_off + channel / 8 (out_sy = out_sx = 2). The tap list is the
   * union of the input offsets any phase uses (<= 4); the weight pack holds zero blocks where a phase does not use a tap
   * (SURVEY.md App. A.3: 9 of the 16 (tap, phase) blocks are non-zero). The input tile is read once instead of four times and
   * a thread writes both px phases of a pixel = one full 32-byte sector. */
  int subpixel;
  /* Optional K chunk (0 = min(cin, 64)): channels per pipeline stage, 16 / 32 / 64, dividing cin. The weight pack is laid out
   * with the same kc ([n_tiles][cin/kc][ntaps][kc/8][n_tile][8]). Halving it halves the activation stage and the weight blocks and
   * so deepens both shared-memory rings: for the 64-channel layers at 128 x 128, which are bound by pipeline depth rather than
   * by the tensor pipe or HBM (profiles/r01_down2_3_swapfold_v33.summary.txt). The K order of the accumulation changes with it. */
  int k_chunk;
  /* Optional IEEE fp16 activations and weights (0 = bf16, the default and the only training format): input, packed weights and
   * P8 outputs of this launch are fp16 (same 16-bit P8 layout, same tcgen05 rate; fp32 accumulation and fp32 logits as before).
   * fp16 carries 11 significand bits against bf16's 8, so the rounding error of every stored activation is 8 x smaller -- the
   * "decision-stable" inference mode (UNet(..., act_dtype="fp16")): fewer threshold / NMS / omega ties flip against the fp32
   * reference. Outputs saturate at +-65504. Inference only (no fused statistics, no cta_pair). */
  int act_fp16;
  /* Optional (NULL = fp64 atomics): workspace of abc_conv_stat_workspace_bytes(desc) bytes for the fused statistics. Each
   * epilogue owner stores its partial sums to a slot of its own and a second kernel sums the slots in a fixed order, so that
   * stat_sum / stat_sq are bit-reproducible (torch.use_deterministic_algorithms). */
  double* stat_ws;
} AbcConvDesc;

ABC_API int abc_conv_igemm(const AbcConvDesc* desc, void* stream);
ABC_API size_t abc_conv_stat_workspace_bytes(const AbcConvDesc* desc);
/* Bytes of packed weights for a layer (host-side helper for allocation). */
ABC_API int64_t abc_conv_wpack_bytes(int cin, int cout, int ntaps, int n_tile);

/* ---------------------------------------------------------------------------------------------------
 * Fused output heads (inference): for every head conv3x3(128 -> 128) + BatchNorm (folded) + LeakyReLU(0.01) +
 * conv1x1(128 -> cout[h]) in one kernel -- OutConv, src/unet.py:63-74, applied to the shared trunk at :116-118. The hidden
 * 128-channel maps stay in tensor memory (csrc/heads_fused_sm100.cu). Two heads share one CTA; the CTAs are split among
 * the head pairs in proportion to their work (csrc/heads_split.cuh).
 *   w1pack / bias1 : conv1 of all heads concatenated on the output-channel axis, packed as for abc_conv_igemm with
 *                    n_tile = 256 and the 3x3 taps in (ky, kx) order (zero-padded to a multiple of 256 channels)
 *   w2pack / bias2 : conv2 in (head, chunk) order, chunk c = output channels [128 c, 128 (c + 1)) of the head with
 *                    nc = count rounded up to 16: 16-bit [16 (K planes)][nc][8] (zero rows past the count), bias fp32 [nc];
 *                    total sizes from abc_heads_fused_pack_sizes
 *   out[h]         : fp32 logits, out_mode[h] = 1: NCHW [N][cout][H][W]; 2: planar-8 [N][out_planes][H][W][8]
 *   act_fp16       : 0: bf16 trunk and weights; 1: IEEE fp16 (AbcConvDesc.act_fp16), hidden maps rounded to fp16
 *   trace          : NULL, or a device buffer of 16 uint64 per CTA: the kernel then records, per CTA, its head pair, tile
 *                    count, start / end %globaltimer and the clock64 cycles each issuing warp and the epilogue spent
 *                    waiting on each barrier (tools/heads_trace.py). For profiling; the logits are unchanged.
 * Limits: n_heads <= 16, at most 6 chunks and 512 padded conv2 channels per pair of heads.
 */
typedef struct AbcHeadsFusedDesc {
  const void* in;          /* trunk: P8 bf16 [N][in_planes][H][W][8], 128 channels from plane in_plane_off */
  int N, H, W;
  int in_planes, in_plane_off;
  const void* w1pack;
  const float* bias1;
  int n_heads;
  int cout[16];
  const void* w2pack;
  int64_t w2pack_bytes;
  const float* bias2;
  int bias2_len;
  void* out[16];
  int out_mode[16];
  int out_planes[16];
  int act_fp16;
  void* trace;
} AbcHeadsFusedDesc;
ABC_API int abc_heads_fused(const AbcHeadsFusedDesc* desc, void* stream);
ABC_API int abc_heads_fused_pack_sizes(int n_heads, const int* cout, int64_t* w2pack_bytes, int* bias2_len);

/* ---------------------------------------------------------------------------------------------------
 * Heat-map decoding: threshold + 3x3 NMS on the atom / bond centre maps, ordered peak compaction, per-peak
 * class / offset gather. Replaces src/img2smiles.py:62-80 (dense NMS / omega NMS), :115-124 (dense argmax
 * maps) and the gather part of :134-182 (one .cpu().item() sync per scalar in the reference).
 *
 * Inputs are the 8 head outputs as the reference returns them: fp32 NCHW, contiguous
 *   0 atom centre [N,1,H,W]   1 atom type [N,c_type,H,W]  2 charge [N,c_charge,H,W]  3 H-count [N,c_hs,H,W]
 *   4 bond centre [N,1,H,W]   5 bond type [N,n_btype*n_omega,H,W] (channel = type*n_omega + omega)
 *   6 rho [N,n_omega,H,W]     7 omega [N,n_omega,H,W]
 * Outputs (caller allocated):
 *   atoms  AbcAtomRec[N][atom_cap]  every atom-centre peak in row-major order (x = row, y = column);
 *                                   the greedy < 2 px de-duplication of :183-187 is left to the caller
 *   bonds  AbcBondRec[N][bond_cap]  every surviving (bond peak, omega) pair in the reference's
 *                                   enumeration order (row-major peaks, ascending omega, :134-171)
 *   counts int32[N][4] = (atom peaks, bond records, bond-centre peaks, 0); when a count exceeds its
 *          capacity the list is truncated and ABC_ERR_CAPACITY is NOT raised here (no sync) -- the caller
 *          compares counts with capacities after its D2H copy.
 * omega_mode 0: candidates = circular 3-tap NMS & (z > thr) (img2smiles.py:74-80, img2smiles3.py)
 *            1: candidates = every omega whose logit != 0 (img2smiles2.py:139)
 * thr is the logit threshold (-1 in the reference, img2smiles.py:64), or a probability when centre_prob = 1.
 */
typedef struct AbcAtomRec {
  uint16_t x, y;
  uint8_t type, charge, hs, pad;
} AbcAtomRec;
typedef struct AbcBondRec {
  uint16_t x, y;
  uint8_t omega, type;
  uint16_t pad;
  float rho;               /* |z_rho| (img2smiles.py:70) */
} AbcBondRec;
typedef struct AbcDecodeDesc {
  const float* maps[8];
  int N, H, W;
  int c_type, c_charge, c_hs, n_omega, n_btype;
  float thr;
  int omega_mode;
  AbcAtomRec* atoms;
  int atom_cap;
  AbcBondRec* bonds;
  int bond_cap;
  int32_t* counts;
  int p8f_mask;            /* bit k set: maps[k] is planar-8 fp32 [N][ceil(C/8)][H][W][8] (abc_conv_igemm out_mode 2)
                              instead of NCHW: 8 channels of a pixel share one 32-byte sector, so the per-peak gathers
                              of the fused inference+decode path touch ~8x fewer sectors */
  int centre_prob;         /* 0: threshold + 3x3 NMS on the raw centre logits (img2smiles.py:62-68, thr = -1).
                              1: on p = clamp(sigmoid(z), 1e-5, 1 - 1e-5), the training-time metric definition
                              (train.py:95,100,145-151, thr = 0.25); the omega candidates (mode 0) keep using thr_omega */
  float thr_omega;         /* logit threshold of the omega NMS when centre_prob = 1 (ignored otherwise: thr is used) */
  /* Sparse heads (SURVEY.md section 8f, N4; 0 = off): the class / offset maps are only read at peaks, so the fused
   * inference + decode path may evaluate those heads only there. Slot s = (n * 2 + which) * peak_cap + i is peak i
   * (row-major) of image n, which = 0 atom centres / 1 bond centres; P = 2 * N * peak_cap slots.
   *   sparse_mode 1 ("find")  : only maps[0] and maps[4] are read; writes peak_pix[N][2][peak_cap] (pixel index y * W + x,
   *                             truncated at peak_cap) and the untruncated counts peak_cnt[N][2]; no records.
   *   sparse_mode 2 ("finish"): maps[1..3] and maps[5..7] are COMPACT logits over the slots -- [1][C][P] fp32, or planar-8
   *                             [1][ceil(C/8)][P][8] where p8f_mask says so -- as produced by running the heads on the
   *                             output of abc_gather_patches; records and counts as in mode 0 (counts[0] / counts[2] are
   *                             the untruncated peak counts: the caller checks them against peak_cap).
   * Pooled slot layout (pool_slots > 0; peak_cap is then ignored): the whole batch shares one pool of P = pool_slots slots.
   * Slot s = peak_off[n * 2 + which] + i is peak i of image n, where peak_off[2N + 1] holds the exclusive prefix sums of the
   * untruncated counts peak_cnt[N][2] in (n, which) order and peak_off[2N] is their total. An image may have any number of
   * peaks; a peak whose slot would be >= pool_slots gets none, so the records are complete exactly when the total
   * (counts[0] + counts[2] summed over the batch) is <= pool_slots.
   *   sparse_mode 1 writes the UNTRUNCATED lists peak_pix[N][2][H * W], peak_cnt and peak_off (a deterministic scan,
   *                 no atomics: the same counts always give the same slots);
   *   sparse_mode 2 reads the slots through peak_off; the compact logits are [1][C][pool_slots] (or planar-8), as produced
   *                 from the output of abc_gather_patches_pooled. */
  int32_t* peak_pix;
  int32_t* peak_cnt;
  int peak_cap;            /* multiple of 64, <= 1024 */
  int sparse_mode;
  int32_t* peak_off;       /* pooled layout: [2N + 1] slot offsets (written by sparse_mode 1, read by sparse_mode 2) */
  int pool_slots;          /* 0: the fixed layout above; > 0: the pooled layout, a multiple of 64 (2 * N * H * W < 2^31) */
} AbcDecodeDesc;
ABC_API int abc_decode_peaks(const AbcDecodeDesc* desc, void* stream);
/* Sparse heads, step 2: for every valid slot the 3x3 neighbourhood of the trunk (P8 bf16 [N][planes][H][W][8], zero outside the
 * image) becomes one pixel of the compact P8 tensor out = [1][9 * planes][P / 8][8][8], planes ordered (64-channel chunk, tap,
 * plane) = the K order of the dense 3x3 abc_conv_igemm. A 1x1 abc_conv_igemm over `out` (cin = 72 * planes, H = P / 8, W = 8)
 * with the packed weights of the dense 3x3 layer then reproduces that layer's outputs at the peaks bit for bit. */
ABC_API int abc_gather_patches(const void* trunk, int N, int H, int W, int planes, const int32_t* peak_pix, const int32_t* peak_cnt,
                               int peak_cap, void* out, void* stream);
/* The same gather in the pooled slot layout (AbcDecodeDesc.pool_slots): peak_pix [N][2][H * W], peak_cnt [N][2] and peak_off
 * [2N + 1] as written by sparse_mode 1, out = [1][9 * planes][pool_slots / 8][8][8]. Slots past the batch's total keep their
 * old contents; no slot at or past pool_slots is written. */
ABC_API int abc_gather_patches_pooled(const void* trunk, int N, int H, int W, int planes, const int32_t* peak_pix,
                                      const int32_t* peak_cnt, const int32_t* peak_off, int pool_slots, void* out, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * Host-side assembly of the decoded records into V2000 MOL-block text (HOST memory in, HOST memory out, no GPU work):
 * the per-image Python loop of src/img2smiles.py:183-318 (atom de-duplication, bond -> atom assignment by the anisotropic
 * float64 distance, pair de-duplication, valence repair, re-indexing, implicit-H list) followed by the text builder of
 * src/generate_smiles.py:18-105, multi-threaded over images. Byte-identical to the Python path on the same records.
 *   atoms / bonds / counts : the arrays abc_decode_peaks filled, after the device -> host copy
 *   cos_tab / sin_tab      : cos / sin of omega_w = w * (pi / (n_omega / 2)) + pi / n_omega - pi / 2, w < n_omega (float64,
 *                            computed by the caller with the same library call as its Python path)
 *   text                   : [N][text_stride] NUL-terminated MOL blocks; text_len[i] = strlen, or -1 when image i has no
 *                            molecule (no atom or no bond-centre peak, img2smiles.py:126-129)
 *   n_threads              : 0 = one per hardware thread
 * Returns ABC_ERR_CAPACITY when a text does not fit text_stride (text_len then holds the required length). */
ABC_API int abc_assemble_molblocks(const AbcAtomRec* atoms, int atom_cap, const AbcBondRec* bonds, int bond_cap,
                                   const int32_t* counts, int N, const double* cos_tab, const double* sin_tab, int n_omega,
                                   int n_threads, char* text, int64_t text_stride, int32_t* text_len);

/* ---------------------------------------------------------------------------------------------------
 * Fused training losses, forward + backward in one pass. Replaces the ~60 ATen kernels (+ autograd) of
 * src/train.py:95-137 (= src/multi_gpu_train2.py:140-192 with class_weights = 0).
 * Pass 1 (abc_loss_partials) accumulates the 8 numerators and 8 denominators in fp64; when all eight dlogits pointers
 * are given it also writes the UNSCALED gradient in the same pass ("fused mode": the per-loss factor u_k / denom_k is
 * applied by the consumer, abc_nchw_to_p8_ex), which saves the second pass over the dense targets;
 * pass 2 (abc_loss_backward) writes dL/dlogits for the 8 maps given the per-loss scale factors
 * u_k / denom_k computed by the host wrapper from `s` (train.py:127-135).
 * Logits and dlogits: fp32 NCHW as returned by UNet.forward. Targets: fp32 dense maps in the reference's
 * layout (bond types [N,6,n_omega,H,W]); rho / omega targets may be fp32 or fp64 (tgt_f64 = 1: utils.py:91-92).
 */
typedef struct AbcLossDesc {
  const float* logits[8];
  const void* targets[8];   /* atom, type, charge, hs, bond, btype, rho, omega */
  int tgt_f64;              /* 1: targets[6], targets[7] are float64 */
  int N, H, W;
  int c_type, c_charge, c_hs, n_omega, n_btype;
  const float* type_weights; /* [c_type] device pointer or NULL (multi_gpu_train2.py:156) */
  double* sums;             /* [16] device: numerators 0..7, denominators 8..15 (order of AbcLossIndex) */
  const float* scale;       /* [8] device: dL/dnum_k = u_k / denom_k (backward pass only) */
  float* dlogits[8];        /* backward pass only */
  double* ws;               /* optional (NULL = fp64 atomics): abc_loss_workspace_bytes(desc, p8) bytes; the sums (and, in
                               abc_loss_partials_p8, the bias gradients) are then added in a fixed order: bit-reproducible */
} AbcLossDesc;
enum AbcLossIndex { ABC_L_ATOM = 0, ABC_L_BOND, ABC_L_TYPE, ABC_L_CHARGE, ABC_L_BTYPE, ABC_L_RHO, ABC_L_OMEGA, ABC_L_HS };
ABC_API int abc_loss_partials(const AbcLossDesc* desc, void* stream);
ABC_API int abc_loss_backward(const AbcLossDesc* desc, void* stream);
/* abc_loss_partials in fused mode with the UNSCALED gradient written directly as the tensor-core operand of the head
 * weight- / data-gradient GEMMs: bf16 P8 [N][planes[k]][H][W][8] for head k (order of `logits`; planes[k] * 8 >= channels of the
 * head; channel padding and padding planes are written as zeros = the K padding of the GEMM), and dbias[k][c] = sum over
 * (n, y, x) of the unscaled fp32 gradient (fp64, zeroed by this call) = the bias gradient of the 1x1 head convolutions
 * (src/unet.py:70) up to the per-loss factor. `dlogits` / `scale` of the descriptor are ignored. Saves the fp32 round trip
 * of the 501-channel gradient and the abc_nchw_to_p8_ex pass. v2 head list only (14 / 3 / 2 / 6 classes, n_omega % 4 == 0);
 * any other head list returns ABC_ERR_INVALID and the caller uses abc_loss_partials + abc_nchw_to_p8_ex. */
typedef struct AbcLossP8Out {
  void* dz[8];
  int planes[8];
  double* dbias[8];
} AbcLossP8Out;
ABC_API int abc_loss_partials_p8(const AbcLossDesc* desc, const AbcLossP8Out* out, void* stream);
/* Workspace of the deterministic mode of abc_loss_partials (p8 = 0) or abc_loss_partials_p8 (p8 = 1; n_omega <= 64). */
ABC_API size_t abc_loss_workspace_bytes(const AbcLossDesc* desc, int p8);

/* ---------------------------------------------------------------------------------------------------
 * Training-mode building blocks (autograd of src/unet.py as used by src/train.py:94,139-140).
 *
 * BatchNorm2d in train mode (unet.py:13,16,67): abc_bn_stats accumulates per-channel sum / sum-of-squares of a conv
 * output z (P8 bf16) in fp64; abc_bn_finalize turns them into scale = gamma * invstd, shift = beta - mean * scale and
 * updates the running statistics (momentum 0.1, unbiased variance); abc_bn_act applies
 * a = act(z * scale + shift) [* dropout mask / (1 - p), unet.py:69] with an optional fused MaxPool2d(2) output (:30).
 * abc_bn_act_backward is the backward of that chain: the incoming gradient is dA (full resolution) and / or dP
 * (gradient of the pooled output, routed to the first maximum of each 2x2 window); outputs dz (P8 bf16),
 * s1[c] = sum g = dL/dbeta and s2[c] = sum g * xhat = dL/dgamma.
 */
ABC_API int abc_bn_stats(const void* z, int N, int H, int W, int planes, int plane_off, int C, double* sum, double* sumsq, void* stream);
ABC_API int abc_bn_finalize(const double* sum, const double* sumsq, int C, double count, const float* gamma, const float* beta,
                            float eps, float momentum, float* running_mean, float* running_var, float* scale, float* shift,
                            float* mean, float* invstd, void* stream);
typedef struct AbcBnActDesc {
  const void* z; int z_planes, z_plane_off;
  void* out; int out_planes, out_plane_off;        /* may be NULL */
  void* pool; int pool_planes, pool_plane_off;     /* may be NULL; [N][pool_planes][H/2][W/2][8] */
  int N, H, W, C;
  const float* scale; const float* shift;
  int act;                                         /* 0 none, 1 ReLU, 2 LeakyReLU(0.01) */
  float drop_p; uint64_t seed;                     /* counter-based dropout, p = 0 disables */
  const uint64_t* seed_dev;                        /* optional device word added to seed at run time (CUDA-graph replays) */
  void* drop_mask;                                 /* optional uint8 [N][C/8][H][W]: with dropout (no pool) the keep bits of each P8
                                                      vector are also stored (bit i = channel 8 * plane + i kept), so that
                                                      abc_bn_act_backward reads 1 byte per vector instead of re-hashing */
} AbcBnActDesc;
ABC_API int abc_bn_act(const AbcBnActDesc* desc, void* stream);
typedef struct AbcBnActBwdDesc {
  const void* z; int z_planes, z_plane_off;
  const void* dA; int dA_planes, dA_plane_off;     /* may be NULL */
  const void* dP; int dP_planes, dP_plane_off;     /* may be NULL */
  void* dz; int dz_planes, dz_plane_off;
  int N, H, W, C;
  const float* scale; const float* shift; const float* mean; const float* invstd;
  int act; float drop_p; uint64_t seed;
  double* s1; double* s2;                          /* [C] each */
  const uint64_t* seed_dev;                        /* as in AbcBnActDesc */
  const float* gscale;                             /* [C] device or NULL: dA is multiplied by gscale[c] first (a per-channel
                                                      factor the producer of dA left out, e.g. the per-loss scale of the heads) */
  const void* drop_mask;                           /* the bytes abc_bn_act stored (AbcBnActDesc.drop_mask) or NULL = regenerate */
  double* ws;                                      /* optional (NULL = fp64 atomics): abc_bn_act_backward_workspace_bytes(desc)
                                                      bytes; s1 / s2 are then summed in a fixed order (bit-reproducible) */
} AbcBnActBwdDesc;
ABC_API int abc_bn_act_backward(const AbcBnActBwdDesc* desc, void* stream);
ABC_API size_t abc_bn_act_backward_workspace_bytes(const AbcBnActBwdDesc* desc);
/* Deterministic forms of abc_bn_stats / abc_channel_sum / abc_nchw_to_p8_ex (torch.use_deterministic_algorithms): the
 * per-block sums are stored to slots of the caller's workspace `ws` and summed in a fixed order instead of added with fp64
 * atomics, so the results are bit-reproducible for a given device and shape. ws: the bytes the *_workspace_bytes queries
 * return. */
ABC_API int abc_bn_stats_det(const void* z, int N, int H, int W, int planes, int plane_off, int C, double* sum, double* sumsq,
                             double* ws, void* stream);
ABC_API int abc_channel_sum_det(const void* x, int N, int H, int W, int planes, int plane_off, int C, double* sum, double* scratch,
                                double* ws, void* stream);
ABC_API size_t abc_bn_stats_workspace_bytes(int N, int H, int W, int C);    /* also abc_channel_sum_det */
ABC_API int abc_nchw_to_p8_ex_det(const float* src, void* dst, int N, int C, int H, int W, int dst_planes, const float* scale,
                                  double* dbias, double* ws, void* stream);
ABC_API size_t abc_nchw_to_p8_ex_workspace_bytes(int N, int C, int H, int W, int dst_planes);
/* fp32 NCHW -> bf16 P8 with zero-padded channels (dlogits -> tensor-core operand). */
ABC_API int abc_nchw_to_p8(const float* src, void* dst, int N, int C, int H, int W, void* stream);
/* Same in one pass with: a device-side scalar scale (NULL = 1), dst_planes >= ceil(C/8) planes written (padding planes
 * zero: the K padding of the data-gradient GEMM) and, if dbias != NULL, dbias[c] = sum over (n, y, x) of the scaled values
 * (fp64; the bias gradient of the 1x1 head convolutions, src/unet.py:70). */
ABC_API int abc_nchw_to_p8_ex(const float* src, void* dst, int N, int C, int H, int W, int dst_planes, const float* scale,
                              double* dbias, void* stream);
/* per-channel sum of a P8 tensor (bias gradients of convolutions that are not followed by BatchNorm). */
ABC_API int abc_channel_sum(const void* x, int N, int H, int W, int planes, int plane_off, int C, double* sum, double* scratch, void* stream);
/* P8 [N][planes][2H][2W][8] -> [N][4*C/8][H][W][8], phase (py, px) stacked on the plane axis (backward of the
 * sub-pixel phases of the up-sampling convolution, unet.py:44). */
ABC_API int abc_deinterleave2(const void* src, int src_planes, int src_plane_off, int C, void* dst, int N, int H, int W, void* stream);
/* Dense training targets on the device (SURVEY.md section 8f, N2): the stamping part of src/utils.py:83-228. The host parses
 * the label strings (abcnet_b200/targets.py: same float64 arithmetic as utils.py:94-160) into records; this call clears
 * (zero_first) and stamps the eight target maps of a batch in HBM, items in label order, later stamps overwriting earlier
 * ones exactly as the reference's Python loop does. All pointers are DEVICE pointers.
 *   atoms    int32 [total atoms][5] = (x, y, type index, charge index, hs); hs outside {0, 1} leaves the H-count map alone
 *   bonds    int32 [total bonds][6] = (x, y, type index, number of omega bins 1 | 2, bin0, bin1); bond_rho float64 [total]
 *   atom_off / bond_off  int32 [N + 1] prefix offsets of the images into the record arrays
 *   maps     atom_target [N][1][H][W], atom_type [N][c_type][H][W], atom_charge [N][c_charge][H][W], atom_hs [N][c_hs][H][W],
 *            bond_target [N][1][H][W], bond_type [N][n_btype][n_omega][H][W] fp32; bond_rho_map / bond_omega
 *            [N][n_omega][H][W] float64 (f64 = 1, the reference's dtype, utils.py:91-92) or float32 (f64 = 0)
 * Coordinates / bins must be in range (the Python wrapper checks; the reference raises IndexError there). */
typedef struct AbcTargetsDesc {
  int N, H, W, n_omega, n_btype, c_type, c_charge, c_hs;
  const int32_t* atoms; const int32_t* atom_off;
  const int32_t* bonds; const double* bond_rho; const int32_t* bond_off;
  float* atom_target; float* atom_type; float* atom_charge; float* atom_hs; float* bond_target; float* bond_type;
  void* bond_rho_map; void* bond_omega;
  int f64;
  int zero_first;
} AbcTargetsDesc;
ABC_API int abc_rasterise_targets(const AbcTargetsDesc* desc, void* stream);

/* Per-step weight re-layout (SURVEY.md section 8f, N3): out[i] = src_ptrs[code >> 22][code & 0x3FFFFF] converted to bf16
 * (out_is_bf16 = 1) or copied as fp32 (0); code 0xFFFFFFFF writes 0. src_ptrs is a DEVICE array of fp32 parameter base
 * pointers, codes a DEVICE uint32 array (n entries, n % 8 == 0, 16-byte aligned like out). One launch rebuilds the packed
 * weight blocks of every convolution of the forward and backward pass from the fp32 master parameters. */
ABC_API int abc_gather_pack(const void* src_ptrs, const void* codes, void* out, int64_t n, int out_is_bf16, void* stream);
/* torch.optim.Adam(lr, betas, eps, weight_decay) of src/train.py:55,141 (L2 decay added to the gradient, bias-corrected
 * moments) over all parameter tensors in one launch. p/g/m/v_ptrs: DEVICE arrays of per-tensor base pointers (fp32,
 * contiguous), sizes: DEVICE int64 element counts, chunks: DEVICE int32 pairs (tensor index, chunk index) -- one thread
 * block per pair handles elements [chunk * abc_adam_chunk_elems(), ...) of that tensor; hyper: DEVICE fp32
 * {lr, beta1, beta2, eps, weight_decay}; step_dev: DEVICE fp32 count of completed steps, incremented by the call
 * (CUDA-graph replayable). */
ABC_API int abc_adam_chunk_elems(void);
ABC_API int abc_adam_step(const void* p_ptrs, const void* g_ptrs, const void* m_ptrs, const void* v_ptrs, const int64_t* sizes,
                          const int32_t* chunks, int n_chunks, const float* hyper, float* step_dev, void* stream);
/* Weight gradient of a convolution on tcgen05 tensor cores (cuDNN backward-filter of the reference's autograd):
 * dw[tap][co][ci] (fp32, caller-zeroed, accumulated with atomicAdd) = sum_pixels dz[co](y, x) * in[ci](y + dy, x + dx).
 * With ws (abc_conv_wgrad_workspace_bytes(desc) bytes) every split-K CTA stores its block to a slot of its own and the
 * slots are added to dw in slot order: bit-reproducible for a given device and shape. */
typedef struct AbcWgradDesc {
  const void* dz; int dz_planes, dz_plane_off; int cout;    /* P8 bf16 gradient of the conv output */
  const void* in; int in_planes, in_plane_off; int cin;     /* P8 bf16 conv input */
  int N, H, W;
  int ntaps; int tap_dy[9]; int tap_dx[9];
  float* dw;
  int row_boxes;   /* 0 (default) / 1: tap-folded launches (cin <= 32, the plain 3x3 tap set) load three row-shifted 16 x 10 boxes and
                      take the dx taps as operand start offsets instead of loading nine shifted 16 x 8 boxes: half the L2 ->
                      shared-memory traffic, three MMAs per K step instead of one; same result, measured equally fast */
  float* ws;       /* optional, NULL = atomics: deterministic split-K workspace */
} AbcWgradDesc;
ABC_API int abc_conv_wgrad(const AbcWgradDesc* desc, void* stream);
ABC_API size_t abc_conv_wgrad_workspace_bytes(const AbcWgradDesc* desc);
/* First convolution without folded BN / activation (training mode): z = conv(img) + b. */
ABC_API int abc_conv3x3_c1_raw(const void* img, int img_is_u8, const float* w, const float* b, void* out, int N, int H, int W,
                               int out_planes, int out_plane_off, void* stream);
/* dw[16][9] of the first 1 -> 16 convolution (img fp32 or uint8). */
ABC_API int abc_conv3x3_c1_wgrad(const void* img, int img_is_u8, const void* dz, int dz_planes, int dz_plane_off, int N, int H, int W,
                                 float* dw, void* stream);
/* Same for the general stem: dw fp32 [16][cin][9] (zeroed by the call). */
ABC_API int abc_conv3x3_cn_wgrad(const float* img, int cin, const void* dz, int dz_planes, int dz_plane_off, int N, int H, int W,
                                 float* dw, void* stream);
/* Deterministic forms of the two (per-block slots of ws, summed in block order; dw is written, not accumulated) and their
 * workspace (cin = 1 for abc_conv3x3_c1_wgrad_det). */
ABC_API int abc_conv3x3_c1_wgrad_det(const void* img, int img_is_u8, const void* dz, int dz_planes, int dz_plane_off, int N, int H,
                                     int W, float* dw, float* ws, void* stream);
ABC_API int abc_conv3x3_cn_wgrad_det(const float* img, int cin, const void* dz, int dz_planes, int dz_plane_off, int N, int H, int W,
                                     float* dw, float* ws, void* stream);
ABC_API size_t abc_conv3x3_wgrad_workspace_bytes(int cin);

/* ---------------------------------------------------------------------------------------------------
 * Whole-network inference (SURVEY.md section 8b: abc_unet_forward_infer) -- UNet.forward of src/unet.py:100-119 in eval mode
 * behind one call, for hosts without the Python layer.
 *
 *   AbcUNetConfig cfg = {1, 8, {1, 14, 3, 2, 1, 360, 60, 60}, 1};
 *   wpack = device_alloc(abc_unet_wpack_bytes(&cfg));                       caller-owned, lives as long as the handle
 *   abc_unet_create(&cfg, tensors, n, wpack, bytes, stream, &net);          tensors: the checkpoint's fp32 state_dict entries
 *   ws = device_alloc(abc_unet_workspace_bytes(&cfg, N, H, W));             caller-owned activations (bf16 P8), 256-byte aligned
 *   abc_unet_forward_infer(net, img, 0, N, H, W, ws, ws_bytes, outs, 1, stream);   outs[i]: fp32 [N][heads[i]][H/4][W/4]
 *   abc_decode_peaks(...) on the same stream; abc_unet_destroy(net);
 *
 * abc_unet_create reads HOST pointers: for every key of the reference's state_dict ("inc1.double_conv.0.weight", ...,
 * "up1.up.weight" [Cin][Cout][3][3], "out_modules.5.conv2.weight", BatchNorm "running_mean" / "running_var"; an optional
 * "module." prefix is ignored, "s" and "num_batches_tracked" are not needed) the fp32 data in the checkpoint's own layout. It
 * folds BatchNorm (running statistics) into the convolutions, packs them for the kernels and uploads the result into wpack
 * (one synchronising copy; nothing else in this library allocates or synchronises). logits_layout 1 = the reference's NCHW fp32
 * tensors, 2 = planar-8 fp32 for heads with more than one channel (what abc_decode_peaks reads fastest, p8f_mask).
 * img: [N][in_channels][H][W] fp32, or uint8 {0,1} (img_is_u8, in_channels = 1). H, W multiples of 32. */
typedef struct AbcUNetConfig {
  int in_channels;     /* 1..8 */
  int n_heads;         /* 1..16 */
  int heads[16];       /* output channels per head (v2: 1, 14, 3, 2, 1, 360, 60, 60) */
  int crop_first;      /* 1: torch >= 1.13 semantics of unet.py:54-55 (drop the FIRST row / column of the up-sampled map) */
  int act_fp16;        /* 0: bf16 activations / weights (default); 1: IEEE fp16 (AbcConvDesc.act_fp16) */
} AbcUNetConfig;
typedef struct AbcNamedTensor {
  const char* name;
  const float* data;   /* host pointer */
  int64_t numel;
} AbcNamedTensor;
typedef struct AbcUNet AbcUNet;   /* opaque */
ABC_API int64_t abc_unet_wpack_bytes(const AbcUNetConfig* cfg);
ABC_API int64_t abc_unet_workspace_bytes(const AbcUNetConfig* cfg, int N, int H, int W);
ABC_API int abc_unet_create(const AbcUNetConfig* cfg, const AbcNamedTensor* tensors, int n_tensors, void* wpack_dev, int64_t wpack_bytes,
                            void* stream, AbcUNet** out);
ABC_API int abc_unet_forward_infer(AbcUNet* net, const void* img, int img_is_u8, int N, int H, int W, void* workspace,
                                   int64_t workspace_bytes, void* const* out_ptrs, int logits_layout, void* stream);
ABC_API int abc_unet_destroy(AbcUNet* net);
/* The packed weight arena in HOST memory -- exactly the bytes abc_unet_create uploads (out_bytes >= abc_unet_wpack_bytes); no
 * CUDA call, usable without a GPU (offline packing, caching, and the CPU test that compares it with the Python packing). */
ABC_API int abc_unet_pack_host(const AbcUNetConfig* cfg, const AbcNamedTensor* tensors, int n_tensors, void* out, int64_t out_bytes,
                               int64_t* used);

#ifdef __cplusplus
}
#endif
#endif /* ABCNET_B200_H_ */

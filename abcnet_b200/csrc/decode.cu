// Fused heat-map decoder: threshold + 3x3 NMS on the atom / bond centre maps, ordered (row-major) peak compaction,
// per-peak class arg-max, circular omega NMS + half-circle test, rho / bond-type gather.
// Kernels: decode_split_kernel (default: one CTA for the atoms and one for the bonds of every image; also the peak-list
// step of the sparse-heads path), decode_kernel (v1: one CTA per image, ABCNET_DECODE_V1=1), gather_patches_kernel and
// decode_finish_kernel (sparse heads, with peak_offsets_kernel in the pooled slot layout of peak_slots.cuh).
//
// Replaces, bit-exactly, the dense tensor statements and the per-scalar .cpu().item() loop of
// /root/reference/src/img2smiles.py:62-80, :115-124 and the gather part of :134-182 (see include/abcnet_b200.h).
// Only the two centre maps are read densely (2 x H x W x 4 B); every other map is touched at peaks only.
#include <cstdlib>

#include "common.cuh"
#include "peak_slots.cuh"

namespace abc {

constexpr int kDecThreads = 1024;
constexpr int kDecWarps = kDecThreads / 32;

struct DecParams {
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
  int p8f_mask;
  int centre_prob;
  float thr_omega;
  // sparse-heads path (AbcDecodeDesc.sparse_mode): peak lists [N][2][slots.list_stride] / raw counts [N][2]; hw_gather =
  // pixels per "image" of the maps the gathers read: H * W, or the number of compact slots in finish mode
  int32_t* peak_pix;
  int32_t* peak_cnt;
  SlotLayout slots;
  int mode;
  int hw_gather;
};

// Element (image n, channel ch, pixel pix) of map k with C channels: NCHW fp32, or planar-8 fp32 [N][ceil(C/8)][HW][8].
__device__ __forceinline__ float ldmap(const DecParams& p, int k, int n, int ch, int pix, int C) {
  const size_t hw = static_cast<size_t>(p.hw_gather);
  if ((p.p8f_mask >> k) & 1)
    return p.maps[k][((static_cast<size_t>(n) * ((C + 7) >> 3) + (ch >> 3)) * hw + pix) * 8 + (ch & 7)];
  return p.maps[k][(static_cast<size_t>(n) * C + ch) * hw + pix];
}

__device__ __forceinline__ int argmax_map(const DecParams& p, int k, int n, int ch0, int chstride, int C, int Ctot, int pix) {
  float best = ldmap(p, k, n, ch0, pix, Ctot);
  int bi = 0;
  for (int c0 = 1; c0 < C; c0 += 8) {             // eight independent loads in flight, then the ordered comparison
    float v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = (c0 + i < C) ? ldmap(p, k, n, ch0 + (c0 + i) * chstride, pix, Ctot) : 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      if (c0 + i < C && v[i] > best) {            // first maximum wins (torch.argmax)
        best = v[i];
        bi = c0 + i;
      }
    }
  }
  return bi;
}

// Exclusive block scan of one int per thread (1024 threads). Returns the exclusive prefix; *total = block sum.
__device__ __forceinline__ int block_exscan(int v, int* warp_sums, int* total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    int t = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += t;
  }
  if (lane == 31) warp_sums[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    int w = warp_sums[lane];
    int winc = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      int t = __shfl_up_sync(0xffffffffu, winc, o);
      if (lane >= o) winc += t;
    }
    warp_sums[lane] = winc - w;          // exclusive warp offsets
    if (lane == 31) warp_sums[32] = winc;
  }
  __syncthreads();
  const int res = warp_sums[warp] + inc - v;
  *total = warp_sums[32];
  __syncthreads();
  return res;
}

// Centre-map value as the NMS sees it: the raw logit (img2smiles.py:62-68) or, in centre_prob mode, the clamped
// probability clamp(sigmoid(z), 1e-5, 1 - 1e-5) of the training-time metric (train.py:95,100,145-151): saturated
// logits then tie at the clamp and plateau into several peaks exactly as max_pool2d(p) == p does.
__device__ __forceinline__ float centre_value(float z, int prob) {
  if (!prob) return z;
  const float s = 1.f / (1.f + expf(-z));
  return fminf(fmaxf(s, 1e-5f), 1.f - 1e-5f);
}

__device__ __forceinline__ bool is_peak(const float* m, int y, int x, int H, int W, float thr) {
  const float v = m[y * W + x];
  if (!(v > thr)) return false;
  const int y0 = y > 0 ? y - 1 : 0, y1 = y < H - 1 ? y + 1 : H - 1;
  const int x0 = x > 0 ? x - 1 : 0, x1 = x < W - 1 ? x + 1 : W - 1;
  for (int yy = y0; yy <= y1; ++yy)
    for (int xx = x0; xx <= x1; ++xx)
      if (m[yy * W + xx] > v) return false;     // max_pool2d(z) == z  <=>  no neighbour is larger
  return true;
}

// Survivor mask of the omega bins of one bond peak, evaluated by a full warp on the n_omega (<= 64) logits in `z`.
// Bit layout: lo = bins 0..31, hi = bins 32..63.
__device__ __forceinline__ void omega_survivors(const float* z, int n, float thr, int mode, uint32_t* lo, uint32_t* hi) {
  const int lane = threadIdx.x & 31;
  const int h = n >> 1;
  bool keep[2];
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const int w = lane + 32 * k;
    bool s = false;
    if (w < n) {
      const float v = z[w];
      bool cand;
      if (mode == 1) {
        cand = (v != 0.f);
      } else {
        const float l = z[w == 0 ? n - 1 : w - 1], r = z[w == n - 1 ? 0 : w + 1];
        cand = (v > thr) && !(l > v) && !(r > v);
      }
      if (cand) {
        if (w <= h - 2) s = !(v < fmaxf(z[w + h - 1], z[w + h]));
        else if (w == h - 1) s = !(v < z[w + h - 1] || v < z[0]);
        else if (w == h) s = !(v <= z[0] || v <= z[n - 1]);
        else s = !(v <= fmaxf(z[w - h - 1], z[w - h]));
      }
    }
    keep[k] = s;
  }
  *lo = __ballot_sync(0xffffffffu, keep[0]);
  *hi = __ballot_sync(0xffffffffu, keep[1]);
}

__global__ void __launch_bounds__(kDecThreads, 1) decode_kernel(const DecParams p) {
  extern __shared__ __align__(16) uint8_t dsm[];
  const int HW = p.H * p.W;
  float* map = reinterpret_cast<float*>(dsm);                                  // [HW]  (later: per-peak offsets)
  uint16_t* bpix = reinterpret_cast<uint16_t*>(dsm + static_cast<size_t>(HW) * 4);   // [HW] bond peak pixel indices
  uint8_t* bcnt = reinterpret_cast<uint8_t*>(bpix + HW);                       // [HW] survivors per bond peak
  __shared__ int warp_sums[33];
  __shared__ float wz[kDecWarps][64];

  const int n = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int per = (HW + kDecThreads - 1) / kDecThreads;
  const int p0 = tid * per, p1 = min(p0 + per, HW);

  // ------------------------------------------------------------------ atoms
  for (int i = tid; i < HW; i += kDecThreads) map[i] = centre_value(ldmap(p, 0, n, 0, i, 1), p.centre_prob);
  __syncthreads();
  int cnt = 0;
  for (int i = p0; i < p1; ++i) cnt += is_peak(map, i / p.W, i % p.W, p.H, p.W, p.thr) ? 1 : 0;
  int total_atoms;
  int idx = block_exscan(cnt, warp_sums, &total_atoms);
  if (cnt) {
    for (int i = p0; i < p1; ++i) {
      const int y = i / p.W, x = i % p.W;
      if (!is_peak(map, y, x, p.H, p.W, p.thr)) continue;
      if (idx < p.atom_cap) {
        AbcAtomRec r;
        r.x = static_cast<uint16_t>(y);          // reference naming: x = row, y = column (img2smiles.py:178)
        r.y = static_cast<uint16_t>(x);
        r.type = static_cast<uint8_t>(argmax_map(p, 1, n, 0, 1, p.c_type, p.c_type, i));
        r.charge = static_cast<uint8_t>(argmax_map(p, 2, n, 0, 1, p.c_charge, p.c_charge, i));
        r.hs = static_cast<uint8_t>(argmax_map(p, 3, n, 0, 1, p.c_hs, p.c_hs, i));
        r.pad = 0;
        p.atoms[static_cast<size_t>(n) * p.atom_cap + idx] = r;
      }
      ++idx;
    }
  }
  __syncthreads();

  // ------------------------------------------------------------------ bond peaks (ordered list in smem)
  for (int i = tid; i < HW; i += kDecThreads) map[i] = centre_value(ldmap(p, 4, n, 0, i, 1), p.centre_prob);
  __syncthreads();
  cnt = 0;
  for (int i = p0; i < p1; ++i) cnt += is_peak(map, i / p.W, i % p.W, p.H, p.W, p.thr) ? 1 : 0;
  int total_bpeaks;
  idx = block_exscan(cnt, warp_sums, &total_bpeaks);
  for (int i = p0; i < p1 && cnt; ++i)
    if (is_peak(map, i / p.W, i % p.W, p.H, p.W, p.thr)) bpix[idx++] = static_cast<uint16_t>(i);
  __syncthreads();

  // ------------------------------------------------------------------ pass A: survivors per bond peak
  for (int b = warp; b < total_bpeaks; b += kDecWarps) {
    const int pix = bpix[b];
    if (lane < p.n_omega) wz[warp][lane] = ldmap(p, 7, n, lane, pix, p.n_omega);
    if (lane + 32 < p.n_omega) wz[warp][lane + 32] = ldmap(p, 7, n, lane + 32, pix, p.n_omega);
    __syncwarp();
    uint32_t lo, hi;
    omega_survivors(wz[warp], p.n_omega, p.thr_omega, p.omega_mode, &lo, &hi);
    if (lane == 0) bcnt[b] = static_cast<uint8_t>(__popc(lo) + __popc(hi));
    __syncwarp();
  }
  __syncthreads();

  // ------------------------------------------------------------------ exclusive offsets over bond peaks
  int* boff = reinterpret_cast<int*>(map);      // the bond map is no longer needed
  const int perb = (total_bpeaks + kDecThreads - 1) / kDecThreads;
  const int b0 = min(tid * perb, total_bpeaks), b1 = min(b0 + perb, total_bpeaks);
  cnt = 0;
  for (int b = b0; b < b1; ++b) cnt += bcnt[b];
  int total_bonds;
  idx = block_exscan(cnt, warp_sums, &total_bonds);
  for (int b = b0; b < b1; ++b) {
    boff[b] = idx;
    idx += bcnt[b];
  }
  __syncthreads();

  // ------------------------------------------------------------------ pass B: emit bond records
  for (int b = warp; b < total_bpeaks; b += kDecWarps) {
    if (bcnt[b] == 0) continue;
    const int pix = bpix[b];
    if (lane < p.n_omega) wz[warp][lane] = ldmap(p, 7, n, lane, pix, p.n_omega);
    if (lane + 32 < p.n_omega) wz[warp][lane + 32] = ldmap(p, 7, n, lane + 32, pix, p.n_omega);
    __syncwarp();
    uint32_t lo, hi;
    omega_survivors(wz[warp], p.n_omega, p.thr_omega, p.omega_mode, &lo, &hi);
    const int base = boff[b];
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const uint32_t mine = k == 0 ? lo : hi;
      if ((mine >> lane) & 1u) {
        const int w = lane + 32 * k;
        const int rank = __popc(mine & ((1u << lane) - 1u)) + (k == 1 ? __popc(lo) : 0);
        const int o = base + rank;
        if (o < p.bond_cap) {
          AbcBondRec r;
          r.x = static_cast<uint16_t>(pix / p.W);
          r.y = static_cast<uint16_t>(pix % p.W);
          r.omega = static_cast<uint8_t>(w);
          r.type = static_cast<uint8_t>(argmax_map(p, 5, n, w, p.n_omega, p.n_btype, p.n_btype * p.n_omega, pix));
          r.pad = 0;
          r.rho = fabsf(ldmap(p, 6, n, w, pix, p.n_omega));
          p.bonds[static_cast<size_t>(n) * p.bond_cap + o] = r;
        }
      }
    }
    __syncwarp();
  }
  if (tid == 0) {
    p.counts[n * 4 + 0] = total_atoms;
    p.counts[n * 4 + 1] = total_bonds;
    p.counts[n * 4 + 2] = total_bpeaks;
    p.counts[n * 4 + 3] = 0;
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Split decoder (default): grid (N, 2) -- blockIdx.y = 0 decodes the atoms of image n, 1 its bonds; the two halves share
// nothing (img2smiles.py:134-171 vs :177-193), so splitting doubles the CTAs in flight and halves the dependent phases
// per CTA. 512 threads; the centre map (HW fp32, float4 loads) is the only large shared-memory object (~70 KB per CTA
// -> three CTAs per SM), peaks are kept as one 64-bit flag word per thread (<= 64 consecutive pixels each) instead of
// index lists, and bond peaks are handled by the warp that owns their pixel range, in row-major order, so record
// offsets only need 16-entry scans over warps.
constexpr int kDec2Threads = 512;
constexpr int kDec2Warps = kDec2Threads / 32;

__global__ void __launch_bounds__(kDec2Threads) decode_split_kernel(const DecParams p) {
  extern __shared__ __align__(16) uint8_t dsm[];
  float* map = reinterpret_cast<float*>(dsm);                                  // [HW]
  __shared__ int warp_cnt[kDec2Warps];
  __shared__ float wz[kDec2Warps][64];

  const int HW = p.H * p.W;
  const int n = blockIdx.x, bonds = blockIdx.y;
  const int k = bonds ? 4 : 0;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  // ------------------------------------------------------------------ centre map -> shared memory
  const float* src = p.maps[k] + static_cast<size_t>(n) * HW;
  if (!((p.p8f_mask >> k) & 1) && (HW & 3) == 0 && (reinterpret_cast<uintptr_t>(src) & 15) == 0) {
    const float4* s4 = reinterpret_cast<const float4*>(src);
    float4* m4 = reinterpret_cast<float4*>(map);
    const int n4 = HW >> 2;
    for (int i0 = tid; i0 < n4; i0 += 8 * kDec2Threads) {         // eight 16-byte loads in flight per thread (64 KB per CTA at once)
      float4 v[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int i = i0 + u * kDec2Threads;
        if (i < n4) v[u] = __ldg(s4 + i);
      }
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int i = i0 + u * kDec2Threads;
        if (i < n4) {
          v[u].x = centre_value(v[u].x, p.centre_prob);
          v[u].y = centre_value(v[u].y, p.centre_prob);
          v[u].z = centre_value(v[u].z, p.centre_prob);
          v[u].w = centre_value(v[u].w, p.centre_prob);
          m4[i] = v[u];
        }
      }
    }
  } else {
    for (int i = tid; i < HW; i += kDec2Threads) map[i] = centre_value(ldmap(p, k, n, 0, i, 1), p.centre_prob);
  }
  __syncthreads();

  // ------------------------------------------------------------------ peaks
  // Warp w owns the pixel range [w * per * 32, (w + 1) * per * 32), per = ceil(HW / 512) <= 64. In iteration j its lanes
  // test the 32 consecutive pixels of run j (consecutive lanes -> consecutive shared-memory words: conflict-free; one
  // thread per 32-pixel run put all lanes of a warp on the same bank) and the ballot becomes the flag word of run j, kept
  // by lane j % 32 (runs 0..31 in `lo`, runs 32..63 in `hi`). Row-major order = warp, then lo runs by lane, then hi runs.
  const int per = (HW + kDec2Threads - 1) / kDec2Threads;
  const int wbase = warp * per * 32;
  uint32_t lo = 0, hi = 0;
  for (int j = 0; j < per; ++j) {
    const int i = wbase + j * 32 + lane;
    bool pk = false;
    if (i < HW) {
      const int y = i / p.W;
      pk = is_peak(map, y, i - y * p.W, p.H, p.W, p.thr);
    }
    const uint32_t m = __ballot_sync(0xffffffffu, pk);
    if ((j & 31) == lane) {
      if (j < 32) lo = m;
      else hi = m;
    }
  }
  const int cnt_lo = __popc(lo), cnt_hi = __popc(hi);
  int inc_lo = cnt_lo, inc_hi = cnt_hi;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int a = __shfl_up_sync(0xffffffffu, inc_lo, o), b = __shfl_up_sync(0xffffffffu, inc_hi, o);
    if (lane >= o) {
      inc_lo += a;
      inc_hi += b;
    }
  }
  const int tot_lo = __shfl_sync(0xffffffffu, inc_lo, 31), tot_hi = __shfl_sync(0xffffffffu, inc_hi, 31);
  if (lane == 0) warp_cnt[warp] = tot_lo + tot_hi;
  __syncthreads();
  int warp_off = 0, total_peaks = 0;
  for (int w = 0; w < kDec2Warps; ++w) {
    const int c = warp_cnt[w];
    if (w < warp) warp_off += c;
    total_peaks += c;
  }
  __syncthreads();                                                   // warp_cnt is reused below

  if (p.mode == 1) {
    // ---------------------------------------------------------------- sparse heads, step 1: ordered peak lists only
    const int stride = p.slots.list_stride;
    int32_t* list = p.peak_pix + static_cast<size_t>(n * 2 + bonds) * stride;
#pragma unroll 1
    for (int h = 0; h < 2; ++h) {
      uint32_t fl = h ? hi : lo;
      int idx = warp_off + (h ? tot_lo + inc_hi - cnt_hi : inc_lo - cnt_lo);
      const int base = wbase + (lane + 32 * h) * 32;
      while (fl) {
        if (idx < stride) list[idx] = base + __ffs(fl) - 1;
        fl &= fl - 1;
        ++idx;
      }
    }
    if (tid == 0) p.peak_cnt[n * 2 + bonds] = total_peaks;
    return;
  }

  if (!bonds) {
    // ---------------------------------------------------------------- atoms: one record per peak, row-major order
#pragma unroll 1
    for (int h = 0; h < 2; ++h) {
      uint32_t fl = h ? hi : lo;
      int idx = warp_off + (h ? tot_lo + inc_hi - cnt_hi : inc_lo - cnt_lo);
      const int base = wbase + (lane + 32 * h) * 32;
      while (fl) {
        const int i = base + __ffs(fl) - 1;
        fl &= fl - 1;
        if (idx < p.atom_cap) {
          AbcAtomRec r;
          r.x = static_cast<uint16_t>(i / p.W);          // reference naming: x = row, y = column (img2smiles.py:178)
          r.y = static_cast<uint16_t>(i % p.W);
          r.type = static_cast<uint8_t>(argmax_map(p, 1, n, 0, 1, p.c_type, p.c_type, i));
          r.charge = static_cast<uint8_t>(argmax_map(p, 2, n, 0, 1, p.c_charge, p.c_charge, i));
          r.hs = static_cast<uint8_t>(argmax_map(p, 3, n, 0, 1, p.c_hs, p.c_hs, i));
          r.pad = 0;
          p.atoms[static_cast<size_t>(n) * p.atom_cap + idx] = r;
        }
        ++idx;
      }
    }
    if (tid == 0) p.counts[n * 4 + 0] = total_peaks;
    return;
  }

  // ------------------------------------------------------------------ bonds: each warp walks the peaks of its own pixel
  // range in order; pass 0 counts the surviving omega bins, pass 1 emits the records
  int off = 0, total_bonds = 0;
  for (int pass = 0; pass < 2; ++pass) {
    int wcount = 0;
    for (int run = 0; run < per; ++run) {
      uint32_t fl = __shfl_sync(0xffffffffu, run < 32 ? lo : hi, run & 31);
      const int base = wbase + run * 32;
      while (fl) {                                                           // warp-uniform
        const int pix = base + __ffs(fl) - 1;
        fl &= fl - 1;
        if (lane < p.n_omega) wz[warp][lane] = ldmap(p, 7, n, lane, pix, p.n_omega);
        if (lane + 32 < p.n_omega) wz[warp][lane + 32] = ldmap(p, 7, n, lane + 32, pix, p.n_omega);
        __syncwarp();
        uint32_t slo, shi;
        omega_survivors(wz[warp], p.n_omega, p.thr_omega, p.omega_mode, &slo, &shi);
        if (pass == 1) {
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const uint32_t mine = h == 0 ? slo : shi;
            if ((mine >> lane) & 1u) {
              const int w = lane + 32 * h;
              const int o = off + wcount + __popc(mine & ((1u << lane) - 1u)) + (h == 1 ? __popc(slo) : 0);
              if (o < p.bond_cap) {
                AbcBondRec r;
                r.x = static_cast<uint16_t>(pix / p.W);
                r.y = static_cast<uint16_t>(pix % p.W);
                r.omega = static_cast<uint8_t>(w);
                r.type = static_cast<uint8_t>(argmax_map(p, 5, n, w, p.n_omega, p.n_btype, p.n_btype * p.n_omega, pix));
                r.pad = 0;
                r.rho = fabsf(ldmap(p, 6, n, w, pix, p.n_omega));
                p.bonds[static_cast<size_t>(n) * p.bond_cap + o] = r;
              }
            }
          }
        }
        wcount += __popc(slo) + __popc(shi);
        __syncwarp();
      }
    }
    if (pass == 0) {
      if (lane == 0) warp_cnt[warp] = wcount;
      __syncthreads();
      for (int w = 0; w < kDec2Warps; ++w) {
        const int c = warp_cnt[w];
        if (w < warp) off += c;
        total_bonds += c;
      }
    }
  }
  if (tid == 0) {
    p.counts[n * 4 + 1] = total_bonds;
    p.counts[n * 4 + 2] = total_peaks;
    p.counts[n * 4 + 3] = 0;
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Sparse heads (SURVEY.md section 8f, N4): the class / offset heads are only read at peaks, so the fused inference + decode
// path evaluates them only there. Peak i (row-major order) of group g = n * 2 + which (which = 0 atoms, 1 bond centres) of
// image n owns slot slot_base(g) + i of the compact tensors (peak_slots.cuh: g * peak_cap, or a batch-wide pool through
// exclusive offsets). gather_patches_kernel writes, for every valid slot, the 3x3 neighbourhood of the trunk (zero outside
// the image = the conv padding) as one "pixel" of a compact P8 tensor [1][9 * planes][P / 8][8][8] whose plane order
// (64-channel chunk, tap, plane) is the K order of the dense 3x3 implicit GEMM: a 1x1 abc_conv_igemm over it with the SAME
// packed conv1 weights performs, per output element, the same MMA sequence as the dense layer -> identical bits. One warp
// per slot; in the pooled layout its group comes from a binary search over the offsets (2N + 1 ints, served from L1).
__global__ void __launch_bounds__(256) gather_patches_kernel(const uint4* __restrict__ trunk, int H, int W, int planes,
                                                            const int32_t* __restrict__ peak_pix, const int32_t* __restrict__ peak_cnt,
                                                            SlotLayout sl, int groups, uint4* __restrict__ out, int P) {
  const int slot = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (slot >= P) return;
  const int g = slot_group(sl, slot, groups), i = slot - slot_base(sl, g);
  if (i >= slot_count(sl, g, peak_cnt[g])) return;             // unused slot: keeps its (finite) old contents
  const int n = g >> 1;
  const int pix = peak_pix[static_cast<size_t>(g) * sl.list_stride + i];
  const int y = pix / W, x = pix - y * W;
  const int nq = 9 * planes;
  const size_t rows = static_cast<size_t>(P >> 3);
  for (int q = lane; q < nq; q += 32) {
    const int kc = q / 72, r = q - kc * 72;                     // 72 = 9 taps x 8 planes per 64-channel chunk
    const int t = r >> 3, pl = r & 7;
    const int yy = y + t / 3 - 1, xx = x + t % 3 - 1;
    uint4 v = make_uint4(0, 0, 0, 0);
    if (yy >= 0 && yy < H && xx >= 0 && xx < W)
      v = __ldg(trunk + ((static_cast<size_t>(n) * planes + kc * 8 + pl) * H + yy) * W + xx);
    out[(q * rows + (slot >> 3)) * 8 + (slot & 7)] = v;
  }
}

// Pooled layout: off[g] = exclusive prefix sum of the untruncated counts cnt[0 .. g), off[groups] = total. One CTA; thread t
// owns a run of consecutive groups, so the slot order is the group order whatever the launch (no atomics).
__global__ void __launch_bounds__(kDecThreads) peak_offsets_kernel(const int32_t* __restrict__ cnt, int groups, int32_t* __restrict__ off) {
  __shared__ int warp_sums[33];
  const int per = (groups + kDecThreads - 1) / kDecThreads;
  const int b0 = min(static_cast<int>(threadIdx.x) * per, groups), b1 = min(b0 + per, groups);
  int s = 0;
  for (int b = b0; b < b1; ++b) s += cnt[b];
  int total;
  const int base = block_exscan(s, warp_sums, &total);
  slot_offsets(cnt + b0, b1 - b0, base, off + b0);
  if (threadIdx.x == 0) off[groups] = total;
}

// Fixed layout: at most 1024 slots per group (the documented peak_cap limit).
constexpr int kMaxPeakCap = 1024;
// Bond-centre peaks per round of decode_finish_kernel; a group with more peaks (pooled layout) takes several rounds.
constexpr int kFinishChunk = 1024;

// Step 3: records from the peak lists and the COMPACT class / offset logits (maps[1..3, 5..7] are [1][C][P] or planar-8
// [1][ceil(C/8)][P][8] over the P compact slots; ldmap is called with n = 0, pix = slot). Same record logic as
// decode_split_kernel; grid (N, 2). Peaks without a slot (beyond peak_cap, or past the pool) are skipped; the counts stay
// the untruncated ones so that the caller can tell.
__global__ void __launch_bounds__(kDec2Threads) decode_finish_kernel(const DecParams p) {
  __shared__ int warp_cnt[kDec2Warps];
  __shared__ float wz[kDec2Warps][64];
  __shared__ uint8_t bcnt[kFinishChunk];
  __shared__ int boff[kFinishChunk];
  const int n = blockIdx.x, bonds = blockIdx.y, g = n * 2 + bonds;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int raw = p.peak_cnt[g];
  const int cnt = slot_count(p.slots, g, raw);
  const int slot0 = slot_base(p.slots, g);
  const int32_t* list = p.peak_pix + static_cast<size_t>(g) * p.slots.list_stride;
  if (!bonds) {
    for (int i = tid; i < cnt; i += kDec2Threads) {
      if (i >= p.atom_cap) break;
      const int pix = list[i], slot = slot0 + i;
      AbcAtomRec r;
      r.x = static_cast<uint16_t>(pix / p.W);
      r.y = static_cast<uint16_t>(pix % p.W);
      r.type = static_cast<uint8_t>(argmax_map(p, 1, 0, 0, 1, p.c_type, p.c_type, slot));
      r.charge = static_cast<uint8_t>(argmax_map(p, 2, 0, 0, 1, p.c_charge, p.c_charge, slot));
      r.hs = static_cast<uint8_t>(argmax_map(p, 3, 0, 0, 1, p.c_hs, p.c_hs, slot));
      r.pad = 0;
      p.atoms[static_cast<size_t>(n) * p.atom_cap + i] = r;
    }
    if (tid == 0) p.counts[n * 4 + 0] = raw;
    return;
  }
  int total_bonds = 0;                                           // records of the earlier rounds (block-uniform)
  for (int c0 = 0; c0 < cnt; c0 += kFinishChunk) {
    const int cc = min(cnt - c0, kFinishChunk);
    // pass A: surviving omega bins per bond-centre peak
    for (int b = warp; b < cc; b += kDec2Warps) {
      const int slot = slot0 + c0 + b;
      if (lane < p.n_omega) wz[warp][lane] = ldmap(p, 7, 0, lane, slot, p.n_omega);
      if (lane + 32 < p.n_omega) wz[warp][lane + 32] = ldmap(p, 7, 0, lane + 32, slot, p.n_omega);
      __syncwarp();
      uint32_t slo, shi;
      omega_survivors(wz[warp], p.n_omega, p.thr_omega, p.omega_mode, &slo, &shi);
      if (lane == 0) bcnt[b] = static_cast<uint8_t>(__popc(slo) + __popc(shi));
      __syncwarp();
    }
    __syncthreads();
    // exclusive offsets over the peaks of this round (each thread owns `per` consecutive peaks)
    const int per = (cc + kDec2Threads - 1) / kDec2Threads;
    const int b0 = min(tid * per, cc), b1 = min(b0 + per, cc);
    int c = 0;
    for (int b = b0; b < b1; ++b) c += bcnt[b];
    int inc = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, inc, o);
      if (lane >= o) inc += t;
    }
    if (lane == 31) warp_cnt[warp] = inc;
    __syncthreads();
    int woff = 0, round_bonds = 0;
    for (int w = 0; w < kDec2Warps; ++w) {
      const int v = warp_cnt[w];
      if (w < warp) woff += v;
      round_bonds += v;
    }
    int off = total_bonds + woff + inc - c;
    for (int b = b0; b < b1; ++b) {
      boff[b] = off;
      off += bcnt[b];
    }
    __syncthreads();
    // pass B: emit
    for (int b = warp; b < cc; b += kDec2Warps) {
      if (bcnt[b] == 0) continue;
      const int slot = slot0 + c0 + b, pix = list[c0 + b];
      if (lane < p.n_omega) wz[warp][lane] = ldmap(p, 7, 0, lane, slot, p.n_omega);
      if (lane + 32 < p.n_omega) wz[warp][lane + 32] = ldmap(p, 7, 0, lane + 32, slot, p.n_omega);
      __syncwarp();
      uint32_t slo, shi;
      omega_survivors(wz[warp], p.n_omega, p.thr_omega, p.omega_mode, &slo, &shi);
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const uint32_t mine = h == 0 ? slo : shi;
        if ((mine >> lane) & 1u) {
          const int w = lane + 32 * h;
          const int o = boff[b] + __popc(mine & ((1u << lane) - 1u)) + (h == 1 ? __popc(slo) : 0);
          if (o < p.bond_cap) {
            AbcBondRec r;
            r.x = static_cast<uint16_t>(pix / p.W);
            r.y = static_cast<uint16_t>(pix % p.W);
            r.omega = static_cast<uint8_t>(w);
            r.type = static_cast<uint8_t>(argmax_map(p, 5, 0, w, p.n_omega, p.n_btype, p.n_btype * p.n_omega, slot));
            r.pad = 0;
            r.rho = fabsf(ldmap(p, 6, 0, w, slot, p.n_omega));
            p.bonds[static_cast<size_t>(n) * p.bond_cap + o] = r;
          }
        }
      }
      __syncwarp();
    }
    total_bonds += round_bonds;
    __syncthreads();                                             // bcnt / boff / warp_cnt are rewritten by the next round
  }
  if (tid == 0) {
    p.counts[n * 4 + 1] = total_bonds;
    p.counts[n * 4 + 2] = raw;
    p.counts[n * 4 + 3] = 0;
  }
}

}  // namespace abc

namespace {
int gather_patches(const void* trunk, int N, int H, int W, int planes, const int32_t* peak_pix, const int32_t* peak_cnt,
                   const abc::SlotLayout& sl, long long P, void* out, void* stream, const char* what) {
  using namespace abc;
  ABC_REQUIRE(trunk && peak_pix && peak_cnt && out, "%s: null pointer", what);
  ABC_REQUIRE(N > 0 && H > 0 && W > 0 && planes > 0 && planes % 8 == 0, "%s: planes=%d must be a multiple of 8 (64-channel chunks)", what, planes);
  ABC_REQUIRE(P < (1LL << 30), "%s: too many slots", what);
  gather_patches_kernel<<<static_cast<int>((P + 7) / 8), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const uint4*>(trunk), H, W, planes, peak_pix, peak_cnt, sl, 2 * N, static_cast<uint4*>(out), static_cast<int>(P));
  return launch_check("gather_patches_kernel");
}
}  // namespace

extern "C" int abc_gather_patches(const void* trunk, int N, int H, int W, int planes, const int32_t* peak_pix, const int32_t* peak_cnt,
                                  int peak_cap, void* out, void* stream) {
  using namespace abc;
  if (int rc = device_check()) return rc;
  ABC_REQUIRE(peak_cap >= 64 && peak_cap % 64 == 0 && peak_cap <= kMaxPeakCap, "abc_gather_patches: peak_cap=%d (multiple of 64, <= %d)", peak_cap, kMaxPeakCap);
  const SlotLayout sl{nullptr, peak_cap, 0, peak_cap};
  return gather_patches(trunk, N, H, W, planes, peak_pix, peak_cnt, sl, 2LL * N * peak_cap, out, stream, "abc_gather_patches");
}

extern "C" int abc_gather_patches_pooled(const void* trunk, int N, int H, int W, int planes, const int32_t* peak_pix,
                                         const int32_t* peak_cnt, const int32_t* peak_off, int pool_slots, void* out, void* stream) {
  using namespace abc;
  if (int rc = device_check()) return rc;
  ABC_REQUIRE(peak_off != nullptr, "abc_gather_patches_pooled: null peak_off");
  ABC_REQUIRE(pool_slots >= 64 && pool_slots % 64 == 0, "abc_gather_patches_pooled: pool_slots=%d (positive multiple of 64)", pool_slots);
  ABC_REQUIRE(2LL * N * H * W < (1LL << 31), "abc_gather_patches_pooled: 2 * N * H * W peak-list entries exceed the int32 range");
  const SlotLayout sl{peak_off, 0, pool_slots, H * W};
  return gather_patches(trunk, N, H, W, planes, peak_pix, peak_cnt, sl, pool_slots, out, stream, "abc_gather_patches_pooled");
}

extern "C" int abc_decode_peaks(const AbcDecodeDesc* d, void* stream) {
  using namespace abc;
  if (int rc = device_check()) return rc;
  ABC_REQUIRE(d != nullptr, "abc_decode_peaks: null descriptor");
  const int mode = d->sparse_mode;
  ABC_REQUIRE(mode >= 0 && mode <= 2, "abc_decode_peaks: sparse_mode=%d", mode);
  for (int i = 0; i < 8; ++i) {
    const bool centre = i == 0 || i == 4;
    const bool needed = mode == 0 || (mode == 1 && centre) || (mode == 2 && !centre);
    ABC_REQUIRE(!needed || d->maps[i] != nullptr, "abc_decode_peaks: map %d is null", i);
  }
  ABC_REQUIRE(mode == 1 || (d->atoms && d->bonds && d->counts), "abc_decode_peaks: null output");
  const bool pooled = mode != 0 && d->pool_slots != 0;
  if (mode != 0 && !pooled)
    ABC_REQUIRE(d->peak_pix && d->peak_cnt && d->peak_cap >= 64 && d->peak_cap % 64 == 0 && d->peak_cap <= kMaxPeakCap,
                "abc_decode_peaks: sparse modes need peak_pix / peak_cnt and peak_cap (multiple of 64, <= %d)", kMaxPeakCap);
  if (pooled)
    ABC_REQUIRE(d->peak_pix && d->peak_cnt && d->peak_off && d->pool_slots >= 64 && d->pool_slots % 64 == 0 &&
                    d->pool_slots < (1 << 30) && 2LL * d->N * d->H * d->W < (1LL << 31),
                "abc_decode_peaks: the pooled layout needs peak_pix / peak_cnt / peak_off, pool_slots=%d (positive multiple of 64, "
                "< 2^30) and 2 * N * H * W < 2^31", d->pool_slots);
  ABC_REQUIRE(d->N > 0 && d->H > 0 && d->W > 0, "abc_decode_peaks: bad geometry");
  ABC_REQUIRE(static_cast<int64_t>(d->H) * d->W <= 32768 && d->H <= 65535 && d->W <= 65535,
              "abc_decode_peaks: H*W=%lld exceeds the 32768-pixel per-image limit of the shared-memory decoder",
              static_cast<long long>(d->H) * d->W);
  ABC_REQUIRE(d->n_omega >= 4 && d->n_omega <= 64 && d->n_omega % 2 == 0, "abc_decode_peaks: n_omega=%d (even, 4..64)", d->n_omega);
  ABC_REQUIRE(d->c_type >= 1 && d->c_type <= 255 && d->c_charge >= 1 && d->c_charge <= 255 && d->c_hs >= 1 &&
                  d->c_hs <= 255 && d->n_btype >= 1 && d->n_btype <= 255,
              "abc_decode_peaks: class counts out of range");
  ABC_REQUIRE(mode == 1 || (d->atom_cap > 0 && d->bond_cap > 0), "abc_decode_peaks: capacities must be positive");
  ABC_REQUIRE(d->omega_mode == 0 || d->omega_mode == 1, "abc_decode_peaks: omega_mode=%d", d->omega_mode);
  DecParams p;
  for (int i = 0; i < 8; ++i) p.maps[i] = d->maps[i];
  p.N = d->N; p.H = d->H; p.W = d->W;
  p.c_type = d->c_type; p.c_charge = d->c_charge; p.c_hs = d->c_hs; p.n_omega = d->n_omega; p.n_btype = d->n_btype;
  p.thr = d->thr; p.omega_mode = d->omega_mode;
  p.p8f_mask = d->p8f_mask & 0xff;
  p.centre_prob = d->centre_prob ? 1 : 0;
  p.thr_omega = p.centre_prob ? d->thr_omega : d->thr;
  p.atoms = d->atoms; p.atom_cap = d->atom_cap; p.bonds = d->bonds; p.bond_cap = d->bond_cap; p.counts = d->counts;
  p.peak_pix = d->peak_pix; p.peak_cnt = d->peak_cnt; p.mode = mode;
  p.slots = pooled ? SlotLayout{d->peak_off, 0, d->pool_slots, d->H * d->W} : SlotLayout{nullptr, d->peak_cap, 0, d->peak_cap};
  p.hw_gather = mode != 2 ? d->H * d->W : pooled ? d->pool_slots : 2 * d->N * d->peak_cap;
  if (mode == 2) {
    decode_finish_kernel<<<dim3(d->N, 2, 1), kDec2Threads, 0, static_cast<cudaStream_t>(stream)>>>(p);
    return launch_check("decode_finish_kernel");
  }
  static const bool v1 = getenv("ABCNET_DECODE_V1") != nullptr;     // the one-CTA-per-image kernel (kept for comparison)
  if (!v1 || mode == 1) {
    const size_t smem2 = static_cast<size_t>(d->H) * d->W * 4;
    static size_t smem2_set = 0;
    if (smem2 > 40 * 1024 && smem2 > smem2_set) {
      ABC_CUDA(cudaFuncSetAttribute(decode_split_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem2)));
      smem2_set = smem2;
    }
    decode_split_kernel<<<dim3(d->N, 2, 1), kDec2Threads, smem2, static_cast<cudaStream_t>(stream)>>>(p);
    if (int rc = launch_check("decode_split_kernel")) return rc;
    if (!pooled) return ABC_OK;
    peak_offsets_kernel<<<1, kDecThreads, 0, static_cast<cudaStream_t>(stream)>>>(d->peak_cnt, 2 * d->N, d->peak_off);
    return launch_check("peak_offsets_kernel");
  }
  const size_t smem = static_cast<size_t>(d->H) * d->W * 7;       // 4 B map + 2 B pixel list + 1 B survivor counts
  static size_t smem_set = 0;
  if (smem > 48 * 1024 && smem > smem_set) {
    ABC_CUDA(cudaFuncSetAttribute(decode_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    smem_set = smem;
  }
  decode_kernel<<<d->N, kDecThreads, smem, static_cast<cudaStream_t>(stream)>>>(p);
  return launch_check("decode_kernel");
}

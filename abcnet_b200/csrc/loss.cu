// Fused heat-map / class losses of ABC-Net: one pass for the 8 numerators + 8 denominators, one pass for dL/dlogits.
//
// Replaces the ~60 ATen element-wise / reduction kernels (and their autograd twins) of
// /root/reference/src/train.py:95-137 (= src/multi_gpu_train2.py:140-192 when type_weights == NULL):
//   clamp(sigmoid|softmax, 1e-5, 1-1e-5), the two centre focal losses, the three atom class losses, the bond-type
//   loss over view(-1, 6, n_omega, H, W), the rho L1 loss weighted by sum_type(target) and the omega focal loss
//   weighted per pixel by the sum of its omega targets. Numerators / denominators are accumulated in fp64
//   (the reference's rho / omega terms are fp64 because of the float64 targets, utils.py:91-92).
// Bandwidth class: every logit and target is read once per pass, every dlogit written once; one thread per pixel,
// consecutive threads = consecutive pixels of one NCHW channel plane (coalesced).
#include <cuda_bf16.h>

#include "common.cuh"
#include "det_slots.cuh"

namespace abc {

constexpr float kLo = 1e-5f, kHi = 1.f - 1e-5f;
constexpr int kLossThreads = 256;
constexpr int kMaxC = 16;       // max classes per soft-max group (14 atom types, 6 bond types)

struct LossParams {
  const float* z[8];
  const void* t[8];
  int tgt_f64;
  int N, HW;
  int c_type, c_charge, c_hs, n_omega, n_btype;
  const float* type_w;
  double* sums;
  const float* scale;
  float* dz[8];
};

__device__ __forceinline__ float sigmoidf(float z) { return 1.f / (1.f + expf(-z)); }
__device__ __forceinline__ float clampp(float p) { return fminf(fmaxf(p, kLo), kHi); }

// focal centre-style term (train.py:107-108): value and d/dz (without the global scale)
template <bool BWD>
__device__ __forceinline__ float focal_sigmoid(float z, float t, float* dzv) {
  const float ps = sigmoidf(z);
  const float p = clampp(ps);
  const float pos = (t == 1.f) ? 1.f : 0.f;
  const float omt = 1.f - t;
  const float w4 = omt * omt * omt * omt;
  const float lp = logf(p), l1p = logf(1.f - p);
  const float val = -pos * (1.f - p) * (1.f - p) * lp - w4 * p * p * l1p;
  if (BWD) {
    const float dldp = pos * (2.f * (1.f - p) * lp - (1.f - p) * (1.f - p) / p) + w4 * (-2.f * p * l1p + p * p / (1.f - p));
    const float pass = (ps >= kLo && ps <= kHi) ? 1.f : 0.f;
    *dzv = dldp * pass * ps * (1.f - ps);
  }
  return val;
}

// soft-max focal class loss (train.py:109-114,119) over C channels spaced by `cs` floats; returns numerator,
// accumulates sum of targets in *tsum; BWD: writes dz (scaled) in place.
template <bool BWD>
__device__ __forceinline__ float focal_softmax(const float* z, const float* t, int C, size_t cs, const float* cw,
                                               float* tsum, float scale, float* dz) {
  float zv[kMaxC], tv[kMaxC];
  float mx = -INFINITY;
  for (int c = 0; c < C; ++c) {
    zv[c] = z[c * cs];
    tv[c] = t[c * cs];
    mx = fmaxf(mx, zv[c]);
  }
  float den = 0.f;
  for (int c = 0; c < C; ++c) {
    zv[c] = expf(zv[c] - mx);
    den += zv[c];
  }
  const float inv = 1.f / den;
  float num = 0.f, ts = 0.f, gdot = 0.f;
  float g[kMaxC];
  for (int c = 0; c < C; ++c) {
    const float ps = zv[c] * inv;
    const float p = clampp(ps);
    const float w = cw ? cw[c] : 1.f;
    const float lp = logf(p);
    num += -w * tv[c] * (1.f - p) * (1.f - p) * lp;
    ts += tv[c];
    if (BWD) {
      const float pass = (ps >= kLo && ps <= kHi) ? 1.f : 0.f;
      g[c] = -w * tv[c] * (-2.f * (1.f - p) * lp + (1.f - p) * (1.f - p) / p) * pass;
      gdot += g[c] * ps;
      zv[c] = ps;
    }
  }
  if (BWD)
    for (int c = 0; c < C; ++c) dz[c * cs] = scale * zv[c] * (g[c] - gdot);
  *tsum = ts;
  return num;
}

__device__ __forceinline__ float ld_tgt(const void* base, size_t i, int f64) {
  return f64 ? static_cast<float>(static_cast<const double*>(base)[i]) : static_cast<const float*>(base)[i];
}

// DET: the block totals go to slot blockIdx.x of ws [blocks][16] (det_slots.cuh) instead of fp64 atomics.
template <bool BWD, bool SUMS, bool DET = false>
__global__ void __launch_bounds__(kLossThreads) loss_kernel(const LossParams p, double* __restrict__ ws) {
  const long long gid = static_cast<long long>(blockIdx.x) * kLossThreads + threadIdx.x;
  const long long total = static_cast<long long>(p.N) * p.HW;
  float acc[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) acc[i] = 0.f;
  if (gid < total) {
    const int n = static_cast<int>(gid / p.HW);
    const int pix = static_cast<int>(gid - static_cast<long long>(n) * p.HW);
    const size_t hw = static_cast<size_t>(p.HW);
    float sc[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) sc[k] = BWD ? (p.scale ? p.scale[k] : 1.f) : 0.f;
    float d;
    {   // atom / bond centre maps
      const size_t o = static_cast<size_t>(n) * hw + pix;
      const float ta = static_cast<const float*>(p.t[0])[o];
      acc[ABC_L_ATOM] = focal_sigmoid<BWD>(p.z[0][o], ta, &d);
      acc[8 + ABC_L_ATOM] = (ta == 1.f) ? 1.f : 0.f;
      if (BWD) p.dz[0][o] = sc[ABC_L_ATOM] * d;
      const float tb = static_cast<const float*>(p.t[4])[o];
      acc[ABC_L_BOND] = focal_sigmoid<BWD>(p.z[4][o], tb, &d);
      acc[8 + ABC_L_BOND] = (tb == 1.f) ? 1.f : 0.f;
      if (BWD) p.dz[4][o] = sc[ABC_L_BOND] * d;
    }
    {   // atom type / charge / H-count
      size_t o = (static_cast<size_t>(n) * p.c_type) * hw + pix;
      acc[ABC_L_TYPE] = focal_softmax<BWD>(p.z[1] + o, static_cast<const float*>(p.t[1]) + o, p.c_type, hw, p.type_w,
                                           &acc[8 + ABC_L_TYPE], sc[ABC_L_TYPE], BWD ? p.dz[1] + o : nullptr);
      o = (static_cast<size_t>(n) * p.c_charge) * hw + pix;
      acc[ABC_L_CHARGE] = focal_softmax<BWD>(p.z[2] + o, static_cast<const float*>(p.t[2]) + o, p.c_charge, hw, nullptr,
                                             &acc[8 + ABC_L_CHARGE], sc[ABC_L_CHARGE], BWD ? p.dz[2] + o : nullptr);
      o = (static_cast<size_t>(n) * p.c_hs) * hw + pix;
      acc[ABC_L_HS] = focal_softmax<BWD>(p.z[3] + o, static_cast<const float*>(p.t[3]) + o, p.c_hs, hw, nullptr,
                                         &acc[8 + ABC_L_HS], sc[ABC_L_HS], BWD ? p.dz[3] + o : nullptr);
    }
    // bond types / rho: per omega bin
    const size_t obt = (static_cast<size_t>(n) * p.n_btype * p.n_omega) * hw + pix;
    const size_t ow = (static_cast<size_t>(n) * p.n_omega) * hw + pix;
    float omega_tsum = 0.f;
    for (int w = 0; w < p.n_omega; ++w) omega_tsum += ld_tgt(p.t[7], ow + w * hw, p.tgt_f64);
    for (int w = 0; w < p.n_omega; ++w) {
      float tsum;
      acc[ABC_L_BTYPE] += focal_softmax<BWD>(p.z[5] + obt + w * hw, static_cast<const float*>(p.t[5]) + obt + w * hw,
                                             p.n_btype, hw * p.n_omega, nullptr, &tsum, sc[ABC_L_BTYPE],
                                             BWD ? p.dz[5] + obt + w * hw : nullptr);
      acc[8 + ABC_L_BTYPE] += tsum;
      const float zr = p.z[6][ow + w * hw];
      const float tr = ld_tgt(p.t[6], ow + w * hw, p.tgt_f64);
      const float diff = fabsf(zr) - tr;
      acc[ABC_L_RHO] += fabsf(diff) * tsum;
      if (BWD) {
        const float sd = diff > 0.f ? 1.f : (diff < 0.f ? -1.f : 0.f);
        const float sz = zr > 0.f ? 1.f : (zr < 0.f ? -1.f : 0.f);
        p.dz[6][ow + w * hw] = sc[ABC_L_RHO] * sd * sz * tsum;
      }
      const float tw = ld_tgt(p.t[7], ow + w * hw, p.tgt_f64);
      acc[ABC_L_OMEGA] += omega_tsum * focal_sigmoid<BWD>(p.z[7][ow + w * hw], tw, &d);
      if (BWD) p.dz[7][ow + w * hw] = sc[ABC_L_OMEGA] * omega_tsum * d;
    }
    acc[8 + ABC_L_RHO] = acc[8 + ABC_L_BTYPE];
    acc[8 + ABC_L_OMEGA] = omega_tsum;
  }
  if (SUMS) {
    __shared__ double red[16][kLossThreads / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      double v = static_cast<double>(acc[i]);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if (lane == 0) red[i][warp] = v;
    }
    __syncthreads();
    if (threadIdx.x < 16) {
      double v = 0.0;
      for (int w = 0; w < kLossThreads / 32; ++w) v += red[threadIdx.x][w];
      if constexpr (DET) ws[det_slot_index(blockIdx.x, 16, threadIdx.x)] = v;
      else if (v != 0.0) atomicAdd(p.sums + threadIdx.x, v);
    }
  }
}


// ------------------------------------------------------------------------------------------------------------------
// Specialised kernel for the v2 head list (14 atom types, 3 charges, 2 H-counts, 6 bond types; any n_omega).
// * 256 threads = 64 consecutive pixels x 4 omega groups: the 60-bin loops of one pixel are split over 4 threads and every
//   load / store is a 256-byte contiguous run per 64 threads;
// * compile-time class counts -> the soft-max vectors live in registers (the generic kernel keeps them in local memory);
// * every term except the two centre maps is multiplied by a target (or by a sum of targets) that is zero at ~99.9 % of the
//   positions (utils.py:94-228 rasterises 3x3 neighbourhoods): where all targets of a group are zero both the loss term and
//   its gradient are exactly zero whatever the logit, so the logits are not even read there. The pass is bound by reading
//   the dense targets once and (backward) writing the dense gradient once.
constexpr int kPx = 64;

// Core of the class loss for a compile-time class count: returns the numerator, *tsum = sum of the targets, and (BWD) the gradient
// scale * dL/dz of the C logits in dzv (registers; exactly zero when every target of the group is zero -- the logits are not read then).
template <int C, bool BWD>
__device__ __forceinline__ float focal_softmax_core(const float* __restrict__ z, const float* __restrict__ t, size_t cs,
                                                    const float* __restrict__ cw, float* tsum, float scale, float* dzv) {
  float tv[C];
  float ts = 0.f;
  bool any = false;
#pragma unroll
  for (int c = 0; c < C; ++c) {
    tv[c] = t[c * cs];
    ts += tv[c];
    any |= tv[c] != 0.f;
  }
  *tsum = ts;
  if (!any) {
    if (BWD) {
#pragma unroll
      for (int c = 0; c < C; ++c) dzv[c] = 0.f;
    }
    return 0.f;
  }
  float zv[C];
  float mx = -INFINITY;
#pragma unroll
  for (int c = 0; c < C; ++c) {
    zv[c] = z[c * cs];
    mx = fmaxf(mx, zv[c]);
  }
  float den = 0.f;
#pragma unroll
  for (int c = 0; c < C; ++c) {
    zv[c] = expf(zv[c] - mx);
    den += zv[c];
  }
  const float inv = 1.f / den;
  float num = 0.f, gdot = 0.f;
  float g[C];
#pragma unroll
  for (int c = 0; c < C; ++c) {
    const float ps = zv[c] * inv;
    const float p = clampp(ps);
    const float w = cw ? cw[c] : 1.f;
    const float lp = logf(p);
    num += -w * tv[c] * (1.f - p) * (1.f - p) * lp;
    if (BWD) {
      const float pass = (ps >= kLo && ps <= kHi) ? 1.f : 0.f;
      g[c] = -w * tv[c] * (-2.f * (1.f - p) * lp + (1.f - p) * (1.f - p) / p) * pass;
      gdot += g[c] * ps;
      zv[c] = ps;
    }
  }
  if (BWD) {
#pragma unroll
    for (int c = 0; c < C; ++c) dzv[c] = scale * zv[c] * (g[c] - gdot);
  }
  return num;
}

template <int C, bool BWD>
__device__ __forceinline__ float focal_softmax_c(const float* __restrict__ z, const float* __restrict__ t, size_t cs,
                                                 const float* __restrict__ cw, float* tsum, float scale, float* __restrict__ dz) {
  float dzv[C];
  const float num = focal_softmax_core<C, BWD>(z, t, cs, cw, tsum, scale, dzv);
  if (BWD) {
#pragma unroll
    for (int c = 0; c < C; ++c) dz[c * cs] = dzv[c];
  }
  return num;
}

template <bool BWD, bool SUMS, bool DET = false>
__global__ void __launch_bounds__(256) loss_kernel_v2(const LossParams p, double* __restrict__ ws) {
  constexpr int CT = 14, CC = 3, CH = 2, NB = 6;
  __shared__ float osum[4][kPx];
  __shared__ double red[16][8];
  const int px = threadIdx.x & (kPx - 1), wg = threadIdx.x >> 6;
  const long long total = static_cast<long long>(p.N) * p.HW;
  const size_t hw = static_cast<size_t>(p.HW);
  const int w0 = (wg * p.n_omega) >> 2, w1 = ((wg + 1) * p.n_omega) >> 2;
  float sc[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) sc[k] = BWD ? (p.scale ? p.scale[k] : 1.f) : 0.f;
  float acc[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) acc[i] = 0.f;
  const long long ntiles = (total + kPx - 1) / kPx;
  for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const long long gid = tile * kPx + px;
    const bool live = gid < total;
    int n = 0, pix = 0;
    if (live) {
      n = static_cast<int>(gid / p.HW);
      pix = static_cast<int>(gid - static_cast<long long>(n) * p.HW);
    }
    const size_t ow = (static_cast<size_t>(n) * p.n_omega) * hw + pix;
    // per-pixel sum of the omega targets (train.py:124): partial per omega group, combined through shared memory
    float part = 0.f;
    if (live)
      for (int w = w0; w < w1; ++w) part += ld_tgt(p.t[7], ow + w * hw, p.tgt_f64);
    osum[wg][px] = part;
    __syncthreads();
    const float omega_tsum = osum[0][px] + osum[1][px] + osum[2][px] + osum[3][px];
    __syncthreads();
    if (!live) continue;
    float d;
    if (wg == 0) {          // centre maps (dense terms)
      const size_t o = static_cast<size_t>(n) * hw + pix;
      const float ta = static_cast<const float*>(p.t[0])[o];
      acc[ABC_L_ATOM] += focal_sigmoid<BWD>(p.z[0][o], ta, &d);
      acc[8 + ABC_L_ATOM] += (ta == 1.f) ? 1.f : 0.f;
      if (BWD) p.dz[0][o] = sc[ABC_L_ATOM] * d;
      const float tb = static_cast<const float*>(p.t[4])[o];
      acc[ABC_L_BOND] += focal_sigmoid<BWD>(p.z[4][o], tb, &d);
      acc[8 + ABC_L_BOND] += (tb == 1.f) ? 1.f : 0.f;
      if (BWD) p.dz[4][o] = sc[ABC_L_BOND] * d;
      acc[8 + ABC_L_OMEGA] += omega_tsum;
    } else if (wg == 1) {   // atom types
      float ts;
      const size_t o = (static_cast<size_t>(n) * CT) * hw + pix;
      acc[ABC_L_TYPE] += focal_softmax_c<CT, BWD>(p.z[1] + o, static_cast<const float*>(p.t[1]) + o, hw, p.type_w, &ts,
                                                  sc[ABC_L_TYPE], BWD ? p.dz[1] + o : nullptr);
      acc[8 + ABC_L_TYPE] += ts;
    } else if (wg == 2) {   // charges, H counts
      float ts;
      size_t o = (static_cast<size_t>(n) * CC) * hw + pix;
      acc[ABC_L_CHARGE] += focal_softmax_c<CC, BWD>(p.z[2] + o, static_cast<const float*>(p.t[2]) + o, hw, nullptr, &ts,
                                                    sc[ABC_L_CHARGE], BWD ? p.dz[2] + o : nullptr);
      acc[8 + ABC_L_CHARGE] += ts;
      o = (static_cast<size_t>(n) * CH) * hw + pix;
      acc[ABC_L_HS] += focal_softmax_c<CH, BWD>(p.z[3] + o, static_cast<const float*>(p.t[3]) + o, hw, nullptr, &ts,
                                                sc[ABC_L_HS], BWD ? p.dz[3] + o : nullptr);
      acc[8 + ABC_L_HS] += ts;
    }
    const size_t obt = (static_cast<size_t>(n) * NB * p.n_omega) * hw + pix;
    for (int w = w0; w < w1; ++w) {
      float tsum;
      acc[ABC_L_BTYPE] += focal_softmax_c<NB, BWD>(p.z[5] + obt + w * hw, static_cast<const float*>(p.t[5]) + obt + w * hw,
                                                   hw * p.n_omega, nullptr, &tsum, sc[ABC_L_BTYPE],
                                                   BWD ? p.dz[5] + obt + w * hw : nullptr);
      acc[8 + ABC_L_BTYPE] += tsum;
      if (tsum != 0.f) {
        const float zr = p.z[6][ow + w * hw];
        const float tr = ld_tgt(p.t[6], ow + w * hw, p.tgt_f64);
        const float diff = fabsf(zr) - tr;
        acc[ABC_L_RHO] += fabsf(diff) * tsum;
        if (BWD) {
          const float sd = diff > 0.f ? 1.f : (diff < 0.f ? -1.f : 0.f);
          const float sz = zr > 0.f ? 1.f : (zr < 0.f ? -1.f : 0.f);
          p.dz[6][ow + w * hw] = sc[ABC_L_RHO] * sd * sz * tsum;
        }
      } else if (BWD) {
        p.dz[6][ow + w * hw] = 0.f;
      }
      if (omega_tsum != 0.f) {
        const float tw = ld_tgt(p.t[7], ow + w * hw, p.tgt_f64);
        acc[ABC_L_OMEGA] += omega_tsum * focal_sigmoid<BWD>(p.z[7][ow + w * hw], tw, &d);
        if (BWD) p.dz[7][ow + w * hw] = sc[ABC_L_OMEGA] * omega_tsum * d;
      } else if (BWD) {
        p.dz[7][ow + w * hw] = 0.f;
      }
    }
  }
  if (SUMS) {
    acc[8 + ABC_L_RHO] = acc[8 + ABC_L_BTYPE];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      double v = static_cast<double>(acc[i]);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if (lane == 0) red[i][warp] = v;
    }
    __syncthreads();
    if (threadIdx.x < 16) {
      double v = 0.0;
      for (int w = 0; w < 8; ++w) v += red[threadIdx.x][w];
      if constexpr (DET) ws[det_slot_index(blockIdx.x, 16, threadIdx.x)] = v;
      else if (v != 0.0) atomicAdd(p.sums + threadIdx.x, v);
    }
  }
}

// ------------------------------------------------------------------------------------------------------------------
// Same pass with the (unscaled) gradient written as the tensor-core operand of the head data- / weight-gradient GEMMs:
// bf16 P8 [N][planes_k][H*W][8] per head instead of fp32 NCHW, plus the per-channel sums of the fp32 gradient (the bias
// gradient of the 1x1 head convolutions, src/unet.py:70). Saves the fp32 round trip of the 501-channel gradient and the
// conversion pass (abc_nchw_to_p8_ex). A thread owns WHOLE half-planes: the omega bins are split over the four thread
// groups in chunks of 4 bins, and 4 consecutive channels (t * n_omega + w .. + 3, n_omega % 4 == 0) are one aligned 8-byte
// half of a P8 vector; channel padding and padding planes are written as zeros. Bias gradients: the two dense centre heads
// through the block reduction, every other head by fp64 atomics at its non-zero gradients only (~0.1 % of the positions).
struct LossP8Params {
  uint4* dz[8];
  int planes[8];
  double* dbias[8];
  double* ws;         // DET: per-block slots [blocks][loss_elems(true, n_omega)] (det_slots.cuh)
};

__device__ __forceinline__ uint2 pack4_bf16(const float* v) {
  const __nv_bfloat162 a = __floats2bfloat162_rn(v[0], v[1]), b = __floats2bfloat162_rn(v[2], v[3]);
  return make_uint2(*reinterpret_cast<const uint32_t*>(&a), *reinterpret_cast<const uint32_t*>(&b));
}

// C <= 16 gradient values of one pixel -> the head's P8 planes (zero channel padding, zero padding planes)
template <int C>
__device__ __forceinline__ void store_small_head(uint4* __restrict__ base, int planes, size_t n, size_t hw, size_t pix, const float* dzv,
                                                 double* __restrict__ dbias, bool atomics) {
  float v[16];
#pragma unroll
  for (int c = 0; c < 16; ++c) v[c] = c < C ? dzv[c] : 0.f;
  uint4* o = base + (n * planes) * hw + pix;
  uint4 q0, q1;
  {
    const uint2 a = pack4_bf16(v), b = pack4_bf16(v + 4), c = pack4_bf16(v + 8), d = pack4_bf16(v + 12);
    q0 = make_uint4(a.x, a.y, b.x, b.y);
    q1 = make_uint4(c.x, c.y, d.x, d.y);
  }
  o[0] = q0;
  if (planes > 1) o[hw] = q1;
  for (int pl = 2; pl < planes; ++pl) o[pl * hw] = make_uint4(0, 0, 0, 0);
  if (atomics) {
#pragma unroll
    for (int c = 0; c < C; ++c)
      if (dzv[c] != 0.f) atomicAdd(dbias + c, static_cast<double>(dzv[c]));
  }
}

// Deterministic form of the sparse bias-gradient atomics: the live lanes `lm` of a warp add their values of one channel in lane
// order (usually none is non-zero, one ballot), and lane 0 adds the total to the warp's own shared accumulator.
__device__ __forceinline__ void det_bias_add(double* acc, float v, unsigned lm) {
  unsigned nz = __ballot_sync(lm, v != 0.f);
  if (nz == 0u) return;
  double t = 0.0;
  while (nz) {
    const int b = __ffs(nz) - 1;
    nz &= nz - 1;
    t += static_cast<double>(__shfl_sync(lm, v, b));
  }
  if ((threadIdx.x & 31) == 0) *acc += t;
}

// Shared memory that only the instantiations which call this declare (the default kernels keep their shared-memory layout).
template <typename T, int N>
__device__ __forceinline__ T* shared_array() {
  __shared__ T a[N];
  return a;
}

// DET: the bias gradients of heads 1-3 and 5-7 are summed per warp in shared memory (a thread group = two warps sees every
// pixel of its channels), the block writes its slot of p.ws ([blocks][loss_elems(true, n_omega)], det_slots.cuh).
template <bool DET = false>
__global__ void __launch_bounds__(256) loss_kernel_v2_p8(const LossParams p, const LossP8Params o) {
  constexpr int CT = 14, CC = 3, CH = 2, NB = 6;
  constexpr int kBiasCh = 19 + 8 * kLossMaxOmegaDet;            // heads 1, 2, 3 (14 + 3 + 2), then 5, 6, 7 (8 n_omega)
  __shared__ float osum[4][kPx];
  __shared__ double red[18][8];
  double* bacc = nullptr;                                        // [2][kBiasCh]: one accumulator row per warp of a thread group
  if constexpr (DET) {
    bacc = shared_array<double, 2 * kBiasCh>();
    for (int i = threadIdx.x; i < 2 * kBiasCh; i += 256) bacc[i] = 0.0;
    __syncthreads();
  }
  double* wacc = bacc + ((threadIdx.x >> 5) & 1) * kBiasCh;
  const int b5 = 19, b6 = 19 + NB * p.n_omega, b7 = b6 + p.n_omega;
  const int px = threadIdx.x & (kPx - 1), wg = threadIdx.x >> 6;
  const long long total = static_cast<long long>(p.N) * p.HW;
  const size_t hw = static_cast<size_t>(p.HW);
  const int cpg = ((p.n_omega >> 2) + 3) >> 2;                           // 4-bin chunks per thread group
  const int w0 = min(wg * cpg * 4, p.n_omega), w1 = min(w0 + cpg * 4, p.n_omega);
  float acc[18];
#pragma unroll
  for (int i = 0; i < 18; ++i) acc[i] = 0.f;
  const long long ntiles = (total + kPx - 1) / kPx;
  for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const long long gid = tile * kPx + px;
    const bool live = gid < total;
    size_t n = 0, pix = 0;
    if (live) {
      n = static_cast<size_t>(gid / p.HW);
      pix = static_cast<size_t>(gid - static_cast<long long>(n) * p.HW);
    }
    const size_t ow = (n * p.n_omega) * hw + pix;
    float part = 0.f;
    if (live)
      for (int w = w0; w < w1; ++w) part += ld_tgt(p.t[7], ow + w * hw, p.tgt_f64);
    osum[wg][px] = part;
    __syncthreads();
    const float omega_tsum = osum[0][px] + osum[1][px] + osum[2][px] + osum[3][px];
    __syncthreads();
    const unsigned lm = DET ? __ballot_sync(0xffffffffu, live) : 0u;    // live lanes: a prefix of the warp
    if (!live) continue;
    float d;
    if (wg == 0) {          // centre maps (dense terms): bias gradients through the block reduction
      const size_t oc = n * hw + pix;
      const float ta = static_cast<const float*>(p.t[0])[oc];
      acc[ABC_L_ATOM] += focal_sigmoid<true>(p.z[0][oc], ta, &d);
      acc[8 + ABC_L_ATOM] += (ta == 1.f) ? 1.f : 0.f;
      acc[16] += d;
      store_small_head<1>(o.dz[0], o.planes[0], n, hw, pix, &d, nullptr, false);
      const float tb = static_cast<const float*>(p.t[4])[oc];
      acc[ABC_L_BOND] += focal_sigmoid<true>(p.z[4][oc], tb, &d);
      acc[8 + ABC_L_BOND] += (tb == 1.f) ? 1.f : 0.f;
      acc[17] += d;
      store_small_head<1>(o.dz[4], o.planes[4], n, hw, pix, &d, nullptr, false);
      acc[8 + ABC_L_OMEGA] += omega_tsum;
    } else if (wg == 1) {   // atom types
      float ts, dzv[CT];
      const size_t oc = (n * CT) * hw + pix;
      acc[ABC_L_TYPE] += focal_softmax_core<CT, true>(p.z[1] + oc, static_cast<const float*>(p.t[1]) + oc, hw, p.type_w, &ts, 1.f, dzv);
      acc[8 + ABC_L_TYPE] += ts;
      store_small_head<CT>(o.dz[1], o.planes[1], n, hw, pix, dzv, o.dbias[1], !DET);
      if constexpr (DET)
#pragma unroll
        for (int c = 0; c < CT; ++c) det_bias_add(wacc + c, dzv[c], lm);
    } else if (wg == 2) {   // charges, H counts
      float ts, dzc[CC], dzh[CH];
      size_t oc = (n * CC) * hw + pix;
      acc[ABC_L_CHARGE] += focal_softmax_core<CC, true>(p.z[2] + oc, static_cast<const float*>(p.t[2]) + oc, hw, nullptr, &ts, 1.f, dzc);
      acc[8 + ABC_L_CHARGE] += ts;
      store_small_head<CC>(o.dz[2], o.planes[2], n, hw, pix, dzc, o.dbias[2], !DET);
      oc = (n * CH) * hw + pix;
      acc[ABC_L_HS] += focal_softmax_core<CH, true>(p.z[3] + oc, static_cast<const float*>(p.t[3]) + oc, hw, nullptr, &ts, 1.f, dzh);
      acc[8 + ABC_L_HS] += ts;
      store_small_head<CH>(o.dz[3], o.planes[3], n, hw, pix, dzh, o.dbias[3], !DET);
      if constexpr (DET) {
#pragma unroll
        for (int c = 0; c < CC; ++c) det_bias_add(wacc + CT + c, dzc[c], lm);
#pragma unroll
        for (int c = 0; c < CH; ++c) det_bias_add(wacc + CT + CC + c, dzh[c], lm);
      }
    } else {                // the least loaded group writes the channel padding of the omega-indexed heads
      const uint2 zero2 = make_uint2(0, 0);
      for (int c0 = NB * p.n_omega; c0 < o.planes[5] * 8; c0 += 4)
        reinterpret_cast<uint2*>(o.dz[5] + (n * o.planes[5] + (c0 >> 3)) * hw + pix)[(c0 >> 2) & 1] = zero2;
      for (int c0 = p.n_omega; c0 < o.planes[6] * 8; c0 += 4)
        reinterpret_cast<uint2*>(o.dz[6] + (n * o.planes[6] + (c0 >> 3)) * hw + pix)[(c0 >> 2) & 1] = zero2;
      for (int c0 = p.n_omega; c0 < o.planes[7] * 8; c0 += 4)
        reinterpret_cast<uint2*>(o.dz[7] + (n * o.planes[7] + (c0 >> 3)) * hw + pix)[(c0 >> 2) & 1] = zero2;
    }
    const size_t obt = (n * NB * p.n_omega) * hw + pix;
    for (int w = w0; w < w1; w += 4) {
      float bt[NB][4], rr[4], oo[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const size_t wo = static_cast<size_t>(w + k) * hw;
        float tsum, dzv[NB];
        acc[ABC_L_BTYPE] += focal_softmax_core<NB, true>(p.z[5] + obt + wo, static_cast<const float*>(p.t[5]) + obt + wo,
                                                         hw * p.n_omega, nullptr, &tsum, 1.f, dzv);
        acc[8 + ABC_L_BTYPE] += tsum;
#pragma unroll
        for (int t = 0; t < NB; ++t) bt[t][k] = dzv[t];
        rr[k] = 0.f;
        if (tsum != 0.f) {
#pragma unroll
          for (int t = 0; t < NB; ++t)
            if (!DET && dzv[t] != 0.f) atomicAdd(o.dbias[5] + t * p.n_omega + w + k, static_cast<double>(dzv[t]));
          const float zr = p.z[6][ow + wo];
          const float tr = ld_tgt(p.t[6], ow + wo, p.tgt_f64);
          const float diff = fabsf(zr) - tr;
          acc[ABC_L_RHO] += fabsf(diff) * tsum;
          const float sd = diff > 0.f ? 1.f : (diff < 0.f ? -1.f : 0.f);
          const float sz = zr > 0.f ? 1.f : (zr < 0.f ? -1.f : 0.f);
          rr[k] = sd * sz * tsum;
          if (!DET && rr[k] != 0.f) atomicAdd(o.dbias[6] + w + k, static_cast<double>(rr[k]));
        }
        oo[k] = 0.f;
        if (omega_tsum != 0.f) {
          const float tw = ld_tgt(p.t[7], ow + wo, p.tgt_f64);
          acc[ABC_L_OMEGA] += omega_tsum * focal_sigmoid<true>(p.z[7][ow + wo], tw, &d);
          oo[k] = omega_tsum * d;
          if (!DET && oo[k] != 0.f) atomicAdd(o.dbias[7] + w + k, static_cast<double>(oo[k]));
        }
        if constexpr (DET) {              // outside the per-lane branches: every live lane of the warp takes part
#pragma unroll
          for (int t = 0; t < NB; ++t) det_bias_add(wacc + b5 + t * p.n_omega + w + k, bt[t][k], lm);
          det_bias_add(wacc + b6 + w + k, rr[k], lm);
          det_bias_add(wacc + b7 + w + k, oo[k], lm);
        }
      }
#pragma unroll
      for (int t = 0; t < NB; ++t) {
        const int c0 = t * p.n_omega + w;
        reinterpret_cast<uint2*>(o.dz[5] + (n * o.planes[5] + (c0 >> 3)) * hw + pix)[(c0 >> 2) & 1] = pack4_bf16(bt[t]);
      }
      reinterpret_cast<uint2*>(o.dz[6] + (n * o.planes[6] + (w >> 3)) * hw + pix)[(w >> 2) & 1] = pack4_bf16(rr);
      reinterpret_cast<uint2*>(o.dz[7] + (n * o.planes[7] + (w >> 3)) * hw + pix)[(w >> 2) & 1] = pack4_bf16(oo);
    }
  }
  acc[8 + ABC_L_RHO] = acc[8 + ABC_L_BTYPE];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int i = 0; i < 18; ++i) {
    double v = static_cast<double>(acc[i]);
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) v += __shfl_xor_sync(0xffffffffu, v, s);
    if (lane == 0) red[i][warp] = v;
  }
  __syncthreads();
  if constexpr (DET) {
    const int n = loss_elems(true, p.n_omega);
    if (threadIdx.x < 18) {
      double v = 0.0;
      for (int w = 0; w < 8; ++w) v += red[threadIdx.x][w];
      o.ws[det_slot_index(blockIdx.x, n, threadIdx.x)] = v;
    }
    for (int c = threadIdx.x; c < 19 + 8 * p.n_omega; c += 256) o.ws[det_slot_index(blockIdx.x, n, 18 + c)] = bacc[c] + bacc[kBiasCh + c];
    return;
  }
  if (threadIdx.x < 18) {
    double v = 0.0;
    for (int w = 0; w < 8; ++w) v += red[threadIdx.x][w];
    if (v != 0.0) atomicAdd(threadIdx.x < 16 ? p.sums + threadIdx.x : (threadIdx.x == 16 ? o.dbias[0] : o.dbias[4]), v);
  }
}

static bool is_v2(const LossParams& p) { return p.c_type == 14 && p.c_charge == 3 && p.c_hs == 2 && p.n_btype == 6 && p.n_omega >= 4; }

// blocks of the loss launches: the v2 kernels (and loss_kernel_v2_p8) stride over 64-pixel tiles, the generic one does not
static unsigned loss_blocks(const LossParams& p) {
  const long long total = static_cast<long long>(p.N) * p.HW;
  if (is_v2(p)) {
    const long long tiles = (total + kPx - 1) / kPx, cap = 148ll * 8 * 4;
    return static_cast<unsigned>(tiles < cap ? tiles : cap);
  }
  return static_cast<unsigned>((total + kLossThreads - 1) / kLossThreads);
}

template <bool BWD, bool SUMS, bool DET = false>
static int launch_loss(const LossParams& p, cudaStream_t st, double* ws = nullptr) {
  const unsigned blocks = loss_blocks(p);
  if (is_v2(p)) {
    loss_kernel_v2<BWD, SUMS, DET><<<blocks, 256, 0, st>>>(p, ws);
    return launch_check("loss_kernel_v2");
  }
  loss_kernel<BWD, SUMS, DET><<<blocks, kLossThreads, 0, st>>>(p, ws);
  return launch_check("loss_kernel");
}

static int fill(const AbcLossDesc* d, LossParams* p, bool bwd, bool sums) {
  ABC_REQUIRE(d != nullptr, "abc_loss: null descriptor");
  for (int i = 0; i < 8; ++i) {
    ABC_REQUIRE(d->logits[i] && d->targets[i], "abc_loss: logits / targets %d null", i);
    if (bwd) ABC_REQUIRE(d->dlogits[i] != nullptr, "abc_loss_backward: dlogits %d null", i);
    p->z[i] = d->logits[i];
    p->t[i] = d->targets[i];
    p->dz[i] = d->dlogits[i];
  }
  ABC_REQUIRE(d->N > 0 && d->H > 0 && d->W > 0, "abc_loss: bad geometry");
  ABC_REQUIRE(d->c_type <= kMaxC && d->c_charge <= kMaxC && d->c_hs <= kMaxC && d->n_btype <= kMaxC && d->c_type >= 1 &&
                  d->c_charge >= 1 && d->c_hs >= 1 && d->n_btype >= 1 && d->n_omega >= 1,
              "abc_loss: class counts must be in [1, %d]", kMaxC);
  if (sums) ABC_REQUIRE(d->sums != nullptr, "abc_loss: sums is null");
  if (bwd && !sums) ABC_REQUIRE(d->scale != nullptr, "abc_loss_backward: scale is null");
  p->tgt_f64 = d->tgt_f64;
  p->N = d->N;
  p->HW = d->H * d->W;
  p->c_type = d->c_type; p->c_charge = d->c_charge; p->c_hs = d->c_hs; p->n_omega = d->n_omega; p->n_btype = d->n_btype;
  p->type_w = d->type_weights;
  p->sums = d->sums;
  p->scale = d->scale;
  return ABC_OK;
}

}  // namespace abc

extern "C" int abc_loss_partials(const AbcLossDesc* d, void* stream) {
  using namespace abc;
  if (int rc = device_check()) return rc;
  LossParams p{};
  // fused mode: when every dlogits pointer is given, the same pass also writes the UNSCALED gradient (scale = 1, or
  // desc->scale if non-null); the caller applies u_k / denom_k afterwards (abc_nchw_to_p8_ex does it while converting).
  bool fused = d != nullptr;
  for (int i = 0; fused && i < 8; ++i) fused = d->dlogits[i] != nullptr;
  if (int rc = fill(d, &p, fused, true)) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (d->ws) {                   // deterministic: block totals to slots, summed in block order
    if (int rc = fused ? launch_loss<true, true, true>(p, st, d->ws) : launch_loss<false, true, true>(p, st, d->ws)) return rc;
    return det_reduce(d->ws, static_cast<int>(loss_blocks(p)), 16, det_out1(p.sums, 16), 0, st);
  }
  ABC_CUDA(cudaMemsetAsync(p.sums, 0, 16 * sizeof(double), st));
  return fused ? launch_loss<true, true>(p, st) : launch_loss<false, true>(p, st);
}

extern "C" int abc_loss_backward(const AbcLossDesc* d, void* stream) {
  using namespace abc;
  if (int rc = device_check()) return rc;
  LossParams p{};
  if (int rc = fill(d, &p, true, false)) return rc;
  return launch_loss<true, false>(p, static_cast<cudaStream_t>(stream));
}

extern "C" int abc_loss_partials_p8(const AbcLossDesc* d, const AbcLossP8Out* out, void* stream) {
  using namespace abc;
  if (int rc = device_check()) return rc;
  LossParams p{};
  if (int rc = fill(d, &p, false, true)) return rc;
  ABC_REQUIRE(out != nullptr, "abc_loss_partials_p8: null output descriptor");
  ABC_REQUIRE(p.c_type == 14 && p.c_charge == 3 && p.c_hs == 2 && p.n_btype == 6 && p.n_omega >= 4 && p.n_omega % 4 == 0,
              "abc_loss_partials_p8: only the v2 head list (14 / 3 / 2 / 6 classes, n_omega %% 4 == 0); use abc_loss_partials + abc_nchw_to_p8_ex");
  const int chans[8] = {1, p.c_type, p.c_charge, p.c_hs, 1, p.n_btype * p.n_omega, p.n_omega, p.n_omega};
  LossP8Params o{};
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  for (int k = 0; k < 8; ++k) {
    ABC_REQUIRE(out->dz[k] && out->dbias[k], "abc_loss_partials_p8: dz / dbias %d null", k);
    ABC_REQUIRE((reinterpret_cast<uintptr_t>(out->dz[k]) & 15) == 0, "abc_loss_partials_p8: dz %d must be 16-byte aligned", k);
    ABC_REQUIRE(out->planes[k] * 8 >= chans[k] && out->planes[k] <= 65535, "abc_loss_partials_p8: planes[%d] = %d too small for %d channels", k,
                out->planes[k], chans[k]);
    o.dz[k] = static_cast<uint4*>(out->dz[k]);
    o.planes[k] = out->planes[k];
    o.dbias[k] = out->dbias[k];
    if (!d->ws) ABC_CUDA(cudaMemsetAsync(out->dbias[k], 0, chans[k] * sizeof(double), st));
  }
  const unsigned blocks = loss_blocks(p);
  if (d->ws) {                   // deterministic: sums and bias gradients per block to slots, summed in block order
    ABC_REQUIRE(p.n_omega <= kLossMaxOmegaDet, "abc_loss_partials_p8: deterministic mode supports n_omega <= %d", kLossMaxOmegaDet);
    o.ws = d->ws;
    loss_kernel_v2_p8<true><<<blocks, 256, 0, st>>>(p, o);
    if (int rc = launch_check("loss_kernel_v2_p8")) return rc;
    DetOut r{};
    const int order[9] = {-1, 0, 4, 1, 2, 3, 5, 6, 7};            // the slot layout of loss_elems(true, n_omega)
    int end = 0;
    for (int i = 0; i < 9; ++i) {
      end += order[i] < 0 ? 16 : chans[order[i]];
      r.ptr[i] = order[i] < 0 ? static_cast<void*>(p.sums) : static_cast<void*>(o.dbias[order[i]]);
      r.end[i] = end;
    }
    r.count = 9;
    return det_reduce(d->ws, static_cast<int>(blocks), loss_elems(true, p.n_omega), r, 0, st);
  }
  ABC_CUDA(cudaMemsetAsync(p.sums, 0, 16 * sizeof(double), st));
  loss_kernel_v2_p8<<<blocks, 256, 0, st>>>(p, o);
  return launch_check("loss_kernel_v2_p8");
}

// Workspace of the deterministic loss passes (AbcLossDesc.ws): abc_loss_partials (p8 = 0) or abc_loss_partials_p8 (p8 = 1).
extern "C" size_t abc_loss_workspace_bytes(const AbcLossDesc* d, int p8) {
  using namespace abc;
  if (!d || d->N <= 0 || d->H <= 0 || d->W <= 0) return 0;
  LossParams p{};
  p.N = d->N; p.HW = d->H * d->W;
  p.c_type = d->c_type; p.c_charge = d->c_charge; p.c_hs = d->c_hs; p.n_omega = d->n_omega; p.n_btype = d->n_btype;
  return det_ws_bytes(loss_blocks(p), loss_elems(p8 != 0, d->n_omega), sizeof(double));
}

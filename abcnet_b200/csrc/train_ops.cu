// Training-mode companions of the convolution kernels (bandwidth class, P8 bf16 layout [N][planes][H][W][8]):
//   abc_bn_stats        per-channel sum / sum of squares of a conv output (batch statistics of nn.BatchNorm2d in
//                       train mode, /root/reference/src/unet.py:13,16,67), fp32 partials, fp64 accumulation
//   abc_bn_finalize     mean / biased var -> (scale, shift, mean, invstd); running-stat update (momentum 0.1, unbiased var)
//   abc_bn_act          a = act(z * scale + shift) [* dropout mask / (1-p)], optional fused MaxPool2d(2) output
//   abc_bn_act_bwd_*    backward of the same chain including max-pool routing (autograd of unet.py:11-18,30,66-69):
//                       reduce: s1 = sum g, s2 = sum g * xhat ; apply: dz = scale * (g - s1/M - xhat * s2/M)
//   abc_nchw_to_p8      fp32 NCHW -> bf16 P8 (zero padded channels), feeds dlogits to the tensor-core kernels
//   abc_channel_sum     per-channel sum of a P8 tensor (bias gradients of convs not followed by BatchNorm)
#include <cstdlib>
#include <cuda_bf16.h>

#include "bn_launch.cuh"
#include "common.cuh"
#include "p8_device.cuh"

namespace abc {

struct P8View {
  const uint4* ptr;   // base of the buffer
  int planes;         // planes in the buffer
  int plane_off;      // first plane of the channel range
};

__device__ __forceinline__ void unpack8(const uint4& u, float* v) {
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float2 f = __bfloat1622float2(h[i]);
    v[2 * i] = f.x;
    v[2 * i + 1] = f.y;
  }
}
__device__ __forceinline__ float bf16r(float x) { return __bfloat162float(__float2bfloat16_rn(x)); }

__device__ __forceinline__ float act_fwd(float x, int act) {
  if (act == 1) return fmaxf(x, 0.f);
  if (act == 2) return x > 0.f ? x : 0.01f * x;
  return x;
}

// ------------------------------------------------------------------------------------------- common pieces
// All BatchNorm-side kernels use the same decomposition: blockIdx.y = 8-channel plane, blockIdx.z = image, blockIdx.x
// strides over the pixels (or 2x2 pixel blocks) of that plane. Consecutive threads touch consecutive 16-byte vectors
// (512 contiguous bytes per warp and load), the per-channel constants are block-uniform, and no integer division is
// needed on the per-pixel path.
__device__ __forceinline__ void load8f(const float* __restrict__ src, float* dst) {
  const float4 a = reinterpret_cast<const float4*>(src)[0], b = reinterpret_cast<const float4*>(src)[1];
  dst[0] = a.x; dst[1] = a.y; dst[2] = a.z; dst[3] = a.w; dst[4] = b.x; dst[5] = b.y; dst[6] = b.z; dst[7] = b.w;
}

// Block-wide sums of K per-thread fp32 partials v(0) .. v(K-1): a warp shuffle tree in fp32, then the 8 warp totals in fp64
// in warp order. Thread i < K returns the block total of partial i. Every thread of the block calls it.
template <int K, typename F>
__device__ __forceinline__ double block_sum(F v, double (*red)[8]) {
  static_assert(kBnThreads == 8 * 32, "one red[][] slot per warp");
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int i = 0; i < K; ++i) {
    float x = v(i);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
    if (lane == 0) red[i][warp] = static_cast<double>(x);
  }
  __syncthreads();
  double t = 0.0;
  if (threadIdx.x < K)
#pragma unroll
    for (int w = 0; w < 8; ++w) t += red[threadIdx.x][w];
  return t;
}

// block-wide sum of 16 per-thread fp32 partials (8 channels x 2 statistics) -> fp64 atomics
__device__ __forceinline__ void block_reduce16(const float* a, const float* b, double* __restrict__ ga, double* __restrict__ gb,
                                               int c0, double (*red)[8]) {
  const double t = block_sum<16>([&](int i) { return i < 8 ? a[i] : b[i - 8]; }, red);
  if (threadIdx.x < 16) atomicAdd((threadIdx.x < 8 ? ga : gb) + c0 + (threadIdx.x & 7), t);
}

// ------------------------------------------------------------------------------------------- statistics
__global__ void __launch_bounds__(kBnThreads) bn_stats_kernel(P8View z, int HW, double* __restrict__ sum, double* __restrict__ sumsq) {
  const int plane = blockIdx.y, n = blockIdx.z;
  const uint4* __restrict__ zb = z.ptr + (static_cast<size_t>(n) * z.planes + z.plane_off + plane) * HW;
  float s[8], q[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) s[i] = q[i] = 0.f;
  const int stride = gridDim.x * kBnThreads;
  int e = blockIdx.x * kBnThreads + threadIdx.x;
  for (; e + stride < HW; e += 2 * stride) {          // two independent 16-byte loads in flight per thread
    const uint4 u0 = zb[e], u1 = zb[e + stride];
    float v[8], w[8];
    unpack8u(u0, v);
    unpack8u(u1, w);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      s[i] += v[i] + w[i];
      q[i] = fmaf(v[i], v[i], fmaf(w[i], w[i], q[i]));
    }
  }
  if (e < HW) {
    float v[8];
    unpack8u(zb[e], v);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      s[i] += v[i];
      q[i] = fmaf(v[i], v[i], q[i]);
    }
  }
  __shared__ double red[16][8];
  block_reduce16(s, q, sum, sumsq, plane * 8, red);
}

__global__ void bn_finalize_kernel(const double* __restrict__ sum, const double* __restrict__ sumsq, int C, double count,
                                   const float* __restrict__ gamma, const float* __restrict__ beta, float eps, float momentum,
                                   float* __restrict__ running_mean, float* __restrict__ running_var,
                                   float* __restrict__ scale, float* __restrict__ shift, float* __restrict__ mean_out,
                                   float* __restrict__ invstd_out) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const double m = sum[c] / count;
  double var = sumsq[c] / count - m * m;
  if (var < 0.0) var = 0.0;
  const float invstd = static_cast<float>(1.0 / sqrt(var + static_cast<double>(eps)));
  const float sc = gamma[c] * invstd;
  scale[c] = sc;
  shift[c] = beta[c] - static_cast<float>(m) * sc;
  mean_out[c] = static_cast<float>(m);
  invstd_out[c] = invstd;
  if (running_mean) {
    const double unbiased = count > 1.0 ? var * count / (count - 1.0) : var;
    running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * static_cast<float>(m);
    running_var[c] = (1.f - momentum) * running_var[c] + momentum * static_cast<float>(unbiased);
  }
}

// ------------------------------------------------------------------------------------------- forward normalise + act (+ pool)
struct BnActParams {
  P8View z;
  uint4* out;       // may be null
  int out_planes, out_plane_off;
  uint4* pool;      // may be null
  int pool_planes, pool_plane_off;
  int N, H, W, planes;   // planes = C / 8
  const float* scale;
  const float* shift;
  int act;
  float drop_p;
  unsigned long long seed;
  const unsigned long long* seed_dev;
  unsigned char* drop_mask;   // optional [N][planes][HW]: bit i of a byte = channel i of that P8 vector was kept
};

template <bool POOL>
__global__ void __launch_bounds__(kBnThreads) bn_act_kernel(const BnActParams p) {
  const int plane = blockIdx.y, n = blockIdx.z;
  const int HW = p.H * p.W;
  float sc[8], sh[8];
  load8f(p.scale + plane * 8, sc);
  load8f(p.shift + plane * 8, sh);
  const uint4* __restrict__ zb = p.z.ptr + (static_cast<size_t>(n) * p.z.planes + p.z.plane_off + plane) * HW;
  uint4* __restrict__ ob = p.out ? p.out + (static_cast<size_t>(n) * p.out_planes + p.out_plane_off + plane) * HW : nullptr;
  const int stride = gridDim.x * kBnThreads;
  if (!POOL) {
    const unsigned long long seed = p.seed + (p.seed_dev ? *p.seed_dev : 0ull);
    const unsigned long long vbase = (static_cast<unsigned long long>(n) * p.planes + plane) * HW;   // index of the plane's first vector
    for (int e = blockIdx.x * kBnThreads + threadIdx.x; e < HW; e += stride) {
      float v[8], dm[8];
      unpack8u(zb[e], v);
      if (p.drop_p > 0.f) {
        drop_scale8(seed, vbase + e, p.drop_p, dm);
        if (p.drop_mask != nullptr) {               // the backward passes then read 1 byte instead of hashing again
          unsigned bits = 0;
#pragma unroll
          for (int i = 0; i < 8; ++i) bits |= (dm[i] != 0.f ? 1u : 0u) << i;
          p.drop_mask[vbase + e] = static_cast<unsigned char>(bits);
        }
      }
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        float a = act_fwd(fmaf(v[i], sc[i], sh[i]), p.act);
        if (p.drop_p > 0.f) a *= dm[i];
        v[i] = a;
      }
      ob[e] = pack8(v);
    }
  } else {
    const int bw = p.W >> 1, hw2 = (p.H >> 1) * bw;
    uint4* __restrict__ pb = p.pool + (static_cast<size_t>(n) * p.pool_planes + p.pool_plane_off + plane) * hw2;
    for (int b = blockIdx.x * kBnThreads + threadIdx.x; b < hw2; b += stride) {
      const int by = b / bw, bx = b - by * bw;
      const int i00 = 2 * by * p.W + 2 * bx;
      const uint4 u[4] = {zb[i00], zb[i00 + 1], zb[i00 + p.W], zb[i00 + p.W + 1]};
      float mx[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) mx[i] = -INFINITY;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        float v[8];
        unpack8u(u[k], v);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          v[i] = bf16r(act_fwd(fmaf(v[i], sc[i], sh[i]), p.act));
          mx[i] = fmaxf(mx[i], v[i]);
        }
        if (ob) ob[i00 + (k >> 1) * p.W + (k & 1)] = pack8(v);
      }
      pb[b] = pack8(mx);
    }
  }
}

// ------------------------------------------------------------------------------------------- backward
struct BnActBwdParams {
  P8View z;                 // saved conv output
  P8View dA;                // gradient wrt the full-resolution activation (ptr may be null)
  P8View dP;                // gradient wrt the pooled activation (ptr may be null)
  int N, H, W, planes;
  const float* scale;
  const float* shift;
  const float* mean;
  const float* invstd;
  int act;
  float drop_p;
  unsigned long long seed;
  const unsigned long long* seed_dev;
  double* s1;               // [C] sum g          (reduce: out, apply: in)
  double* s2;               // [C] sum g * xhat
  uint4* dz;                // apply: output
  int dz_planes, dz_plane_off;
  double count;
  const float* gscale;      // [C] or null: per-channel factor on dA / dP (everything downstream is linear in g)
  const unsigned char* drop_mask;   // the mask bytes bn_act wrote (null: regenerate the mask from the counter-based hash)
};

// Gradient g wrt the BatchNorm output for one pixel (8 channels): g = dA * act'(pre) * dropout scale.
// mbits >= 0: the saved keep bits of this vector (AbcBnActDesc.drop_mask); < 0: regenerate them.
__device__ __forceinline__ void bwd_pixel(const BnActBwdParams& p, const float* v, const float* d, const float* sc, const float* sh,
                                          unsigned long long seed, unsigned long long vbase, int e, float* g, int mbits = -1) {
  float dm[8];
  if (p.drop_p > 0.f) {
    if (mbits >= 0) {
      const float keep = 1.f / (1.f - p.drop_p);
#pragma unroll
      for (int i = 0; i < 8; ++i) dm[i] = ((mbits >> i) & 1) ? keep : 0.f;
    } else {
      drop_scale8(seed, vbase + e, p.drop_p, dm);
    }
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const float pre = fmaf(v[i], sc[i], sh[i]);
    float m = act_grad(pre, p.act);
    if (p.drop_p > 0.f) m *= dm[i];
    g[i] = d[i] * m;
  }
}

// Same for a 2x2 block whose pooled gradient dp is routed to the first maximum of the (bf16) activation.
__device__ __forceinline__ void bwd_block4(const BnActBwdParams& p, const float (&v)[4][8], const float (&d)[4][8], const float* dp,
                                           const float* sc, const float* sh, float (&g)[4][8]) {
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    float pre[4], a[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      pre[k] = fmaf(v[k][i], sc[i], sh[i]);
      a[k] = bf16r(act_fwd(pre[k], p.act));
    }
    // first maximum in window order (torch max_pool2d): strict > when moving to a later element
    const bool b1 = a[1] > a[0];
    const float m01 = b1 ? a[1] : a[0];
    const bool b3 = a[3] > a[2];
    const float m23 = b3 ? a[3] : a[2];
    const bool hi = m23 > m01;
    const int best = hi ? (b3 ? 3 : 2) : (b1 ? 1 : 0);
#pragma unroll
    for (int k = 0; k < 4; ++k) g[k][i] = (d[k][i] + (best == k ? dp[i] : 0.f)) * act_grad(pre[k], p.act);
  }
}

// reduce: s1 = sum g, s2 = sum g * xhat (xhat = (z - mean) * invstd, accumulated as sum g*z and combined per block)
template <bool POOL, int MINB = 2>
__global__ void __launch_bounds__(kBnThreads, MINB) bn_act_bwd_reduce_kernel(const BnActBwdParams p) {
  const int plane = blockIdx.y, n = blockIdx.z;
  const int HW = p.H * p.W;
  float sc[8], sh[8];
  load8f(p.scale + plane * 8, sc);
  load8f(p.shift + plane * 8, sh);
  const uint4* __restrict__ zb = p.z.ptr + (static_cast<size_t>(n) * p.z.planes + p.z.plane_off + plane) * HW;
  const uint4* __restrict__ db = p.dA.ptr ? p.dA.ptr + (static_cast<size_t>(n) * p.dA.planes + p.dA.plane_off + plane) * HW : nullptr;
  float s1[8], t2[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) s1[i] = t2[i] = 0.f;
  const int stride = gridDim.x * kBnThreads;
  if (!POOL) {
    const unsigned long long seed = p.seed + (p.seed_dev ? *p.seed_dev : 0ull);
    const unsigned long long vbase = (static_cast<unsigned long long>(n) * p.planes + plane) * HW;
    const unsigned char* __restrict__ mk = (p.drop_p > 0.f && p.drop_mask != nullptr) ? p.drop_mask + vbase : nullptr;
    int e = blockIdx.x * kBnThreads + threadIdx.x;
    for (; e + stride < HW; e += 2 * stride) {            // four independent 16-byte loads in flight per thread
      const uint4 zu0 = zb[e], du0 = db[e], zu1 = zb[e + stride], du1 = db[e + stride];
      const int m0 = mk ? mk[e] : -1, m1 = mk ? mk[e + stride] : -1;
      float v[8], d[8], g[8], w[8], f[8], h[8];
      unpack8u(zu0, v);
      unpack8u(du0, d);
      unpack8u(zu1, w);
      unpack8u(du1, f);
      bwd_pixel(p, v, d, sc, sh, seed, vbase, e, g, m0);
      bwd_pixel(p, w, f, sc, sh, seed, vbase, e + stride, h, m1);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        s1[i] += g[i] + h[i];
        t2[i] = fmaf(g[i], v[i], fmaf(h[i], w[i], t2[i]));
      }
    }
    if (e < HW) {
      float v[8], d[8], g[8];
      const uint4 zu = zb[e], du = db[e];
      const int m0 = mk ? mk[e] : -1;
      unpack8u(zu, v);
      unpack8u(du, d);
      bwd_pixel(p, v, d, sc, sh, seed, vbase, e, g, m0);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        s1[i] += g[i];
        t2[i] = fmaf(g[i], v[i], t2[i]);
      }
    }
  } else {
    const int bw = p.W >> 1, hw2 = (p.H >> 1) * bw;
    const uint4* __restrict__ pb = p.dP.ptr + (static_cast<size_t>(n) * p.dP.planes + p.dP.plane_off + plane) * hw2;
    for (int b = blockIdx.x * kBnThreads + threadIdx.x; b < hw2; b += stride) {
      const int by = b / bw, bx = b - by * bw;
      const int i00 = 2 * by * p.W + 2 * bx;
      float v[4][8], d[4][8], g[4][8], dp[8];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int e = i00 + (k >> 1) * p.W + (k & 1);
        unpack8u(zb[e], v[k]);
        if (db) {
          unpack8u(db[e], d[k]);
        } else {
#pragma unroll
          for (int i = 0; i < 8; ++i) d[k][i] = 0.f;
        }
      }
      unpack8u(pb[b], dp);
      bwd_block4(p, v, d, dp, sc, sh, g);
#pragma unroll
      for (int k = 0; k < 4; ++k)
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          s1[i] += g[k][i];
          t2[i] = fmaf(g[k][i], v[k][i], t2[i]);
        }
    }
  }
  // sum g * xhat = invstd * (sum g*z - mean * sum g): linear, so every block adds its own share
  float mean[8], istd[8], s2[8];
  load8f(p.mean + plane * 8, mean);
  load8f(p.invstd + plane * 8, istd);
  if (p.gscale != nullptr) {                // g is linear in dA: the per-channel factor is applied to the sums
    float gs[8];
    load8f(p.gscale + plane * 8, gs);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      s1[i] *= gs[i];
      t2[i] *= gs[i];
    }
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) s2[i] = istd[i] * (t2[i] - mean[i] * s1[i]);
  __shared__ double red[16][8];
  block_reduce16(s1, s2, p.s1, p.s2, plane * 8, red);
}

// apply: dz = scale * (g - s1/M - xhat * s2/M) = scale * g + cb * z + ca  with per-channel constants ca, cb
template <bool POOL, int MINB = 2>
__global__ void __launch_bounds__(kBnThreads, MINB) bn_act_bwd_apply_kernel(const BnActBwdParams p) {
  const int plane = blockIdx.y, n = blockIdx.z;
  const int HW = p.H * p.W;
  __shared__ float cst[2][8];
  if (threadIdx.x < 8) {
    const int c = plane * 8 + threadIdx.x;
    const float m1 = static_cast<float>(p.s1[c] / p.count), m2 = static_cast<float>(p.s2[c] / p.count);
    const float sc = p.scale[c], is = p.invstd[c], mu = p.mean[c];
    cst[0][threadIdx.x] = sc * (m2 * is * mu - m1);
    cst[1][threadIdx.x] = -sc * m2 * is;
  }
  __syncthreads();
  float sc[8], sh[8], ca[8], cb[8], sg[8];
  load8f(p.scale + plane * 8, sc);
  load8f(p.shift + plane * 8, sh);
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    ca[i] = cst[0][i];
    cb[i] = cst[1][i];
    sg[i] = sc[i];
  }
  if (p.gscale != nullptr) {                // coefficient of g: BatchNorm scale x the per-channel factor on dA (s1, s2 already hold it)
    float gs[8];
    load8f(p.gscale + plane * 8, gs);
#pragma unroll
    for (int i = 0; i < 8; ++i) sg[i] *= gs[i];
  }
  const uint4* __restrict__ zb = p.z.ptr + (static_cast<size_t>(n) * p.z.planes + p.z.plane_off + plane) * HW;
  const uint4* __restrict__ db = p.dA.ptr ? p.dA.ptr + (static_cast<size_t>(n) * p.dA.planes + p.dA.plane_off + plane) * HW : nullptr;
  uint4* __restrict__ ob = p.dz + (static_cast<size_t>(n) * p.dz_planes + p.dz_plane_off + plane) * HW;
  const int stride = gridDim.x * kBnThreads;
  if (!POOL) {
    const unsigned long long seed = p.seed + (p.seed_dev ? *p.seed_dev : 0ull);
    const unsigned long long vbase = (static_cast<unsigned long long>(n) * p.planes + plane) * HW;
    const unsigned char* __restrict__ mk = (p.drop_p > 0.f && p.drop_mask != nullptr) ? p.drop_mask + vbase : nullptr;
    int e = blockIdx.x * kBnThreads + threadIdx.x;
    for (; e + stride < HW; e += 2 * stride) {            // four independent 16-byte loads in flight per thread
      const uint4 zu0 = zb[e], du0 = db[e], zu1 = zb[e + stride], du1 = db[e + stride];
      const int m0 = mk ? mk[e] : -1, m1 = mk ? mk[e + stride] : -1;
      float v[8], d[8], g[8], w[8], f[8], h[8];
      unpack8u(zu0, v);
      unpack8u(du0, d);
      unpack8u(zu1, w);
      unpack8u(du1, f);
      bwd_pixel(p, v, d, sc, sh, seed, vbase, e, g, m0);
      bwd_pixel(p, w, f, sc, sh, seed, vbase, e + stride, h, m1);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        g[i] = fmaf(g[i], sg[i], fmaf(v[i], cb[i], ca[i]));
        h[i] = fmaf(h[i], sg[i], fmaf(w[i], cb[i], ca[i]));
      }
      ob[e] = pack8(g);
      ob[e + stride] = pack8(h);
    }
    if (e < HW) {
      float v[8], d[8], g[8];
      const uint4 zu = zb[e], du = db[e];
      const int m0 = mk ? mk[e] : -1;
      unpack8u(zu, v);
      unpack8u(du, d);
      bwd_pixel(p, v, d, sc, sh, seed, vbase, e, g, m0);
#pragma unroll
      for (int i = 0; i < 8; ++i) g[i] = fmaf(g[i], sg[i], fmaf(v[i], cb[i], ca[i]));
      ob[e] = pack8(g);
    }
  } else {
    const int bw = p.W >> 1, hw2 = (p.H >> 1) * bw;
    const uint4* __restrict__ pb = p.dP.ptr + (static_cast<size_t>(n) * p.dP.planes + p.dP.plane_off + plane) * hw2;
    for (int b = blockIdx.x * kBnThreads + threadIdx.x; b < hw2; b += stride) {
      const int by = b / bw, bx = b - by * bw;
      const int i00 = 2 * by * p.W + 2 * bx;
      float v[4][8], d[4][8], g[4][8], dp[8];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int e = i00 + (k >> 1) * p.W + (k & 1);
        unpack8u(zb[e], v[k]);
        if (db) {
          unpack8u(db[e], d[k]);
        } else {
#pragma unroll
          for (int i = 0; i < 8; ++i) d[k][i] = 0.f;
        }
      }
      unpack8u(pb[b], dp);
      bwd_block4(p, v, d, dp, sc, sh, g);
#pragma unroll
      for (int k = 0; k < 4; ++k) {
#pragma unroll
        for (int i = 0; i < 8; ++i) g[k][i] = fmaf(g[k][i], sg[i], fmaf(v[k][i], cb[i], ca[i]));
        ob[i00 + (k >> 1) * p.W + (k & 1)] = pack8(g[k]);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------- layout / sums
__global__ void __launch_bounds__(256) nchw_to_p8_kernel(const float* __restrict__ src, uint4* __restrict__ dst, int N, int C,
                                                         int HW, int planes) {
  const long long total = static_cast<long long>(N) * planes * HW;
  const long long t = static_cast<long long>(blockIdx.x) * 256 + threadIdx.x;
  if (t >= total) return;
  const int pix = static_cast<int>(t % HW);
  const long long r = t / HW;
  const int plane = static_cast<int>(r % planes);
  const int n = static_cast<int>(r / planes);
  float v[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int c = plane * 8 + i;
    v[i] = c < C ? src[(static_cast<size_t>(n) * C + c) * HW + pix] : 0.f;
  }
  dst[t] = pack8(v);
}

// fp32 NCHW -> bf16 P8 with an optional device-side scale, zero-filled padding planes and per-channel sums of the scaled
// values (the bias gradient of the 1x1 head convolutions): one pass over the loss gradient instead of three.
__global__ void __launch_bounds__(kBnThreads) nchw_to_p8_ex_kernel(const float* __restrict__ src, uint4* __restrict__ dst, int C,
                                                                   int HW, int dst_planes, const float* __restrict__ scale,
                                                                   double* __restrict__ dbias) {
  const int plane = blockIdx.y, n = blockIdx.z;
  const float sc = scale ? *scale : 1.f;
  const float* __restrict__ sb = src + (static_cast<size_t>(n) * C + plane * 8) * HW;
  uint4* __restrict__ db = dst + (static_cast<size_t>(n) * dst_planes + plane) * HW;
  const int nvalid = min(8, max(0, C - plane * 8));
  float s[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) s[i] = 0.f;
  for (int e = blockIdx.x * kBnThreads + threadIdx.x; e < HW; e += gridDim.x * kBnThreads) {
    float v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      v[i] = i < nvalid ? sb[static_cast<size_t>(i) * HW + e] * sc : 0.f;
      s[i] += v[i];
    }
    db[e] = pack8(v);
  }
  if (dbias != nullptr && nvalid > 0) {      // block-uniform condition
    __shared__ double red[8][8];
    const double t = block_sum<8>([&](int i) { return s[i]; }, red);
    if (threadIdx.x < nvalid) atomicAdd(dbias + plane * 8 + threadIdx.x, t);
  }
}

// dW[16][9], db-free: gradient of the first 1 -> 16 convolution (no dgrad: the image needs no gradient)
// img_cstride: channels of the image tensor (1 for the binary stem); img points at the channel to differentiate.
// dw_costride: floats between consecutive output channels in dw ([16][cin][9]: cin * 9).
template <typename T>
__global__ void __launch_bounds__(256) conv_c1_wgrad_kernel(const T* __restrict__ img, P8View dz, int N, int H, int W,
                                                            float* __restrict__ dw, int img_cstride, int dw_costride) {
  __shared__ float acc[144];
  if (threadIdx.x < 144) acc[threadIdx.x] = 0.f;
  __syncthreads();
  float loc[144];
#pragma unroll
  for (int i = 0; i < 144; ++i) loc[i] = 0.f;
  const long long total = static_cast<long long>(N) * H * W;
  for (long long e = static_cast<long long>(blockIdx.x) * 256 + threadIdx.x; e < total; e += static_cast<long long>(gridDim.x) * 256) {
    const int n = static_cast<int>(e / (static_cast<long long>(H) * W));
    const int pix = static_cast<int>(e - static_cast<long long>(n) * H * W);
    const int y = pix / W, x = pix - y * W;
    float t[9];
#pragma unroll
    for (int dy = 0; dy < 3; ++dy)
#pragma unroll
      for (int dx = 0; dx < 3; ++dx) {
        const int yy = y + dy - 1, xx = x + dx - 1;
        t[dy * 3 + dx] = (yy >= 0 && yy < H && xx >= 0 && xx < W)
                             ? static_cast<float>(img[static_cast<size_t>(n) * img_cstride * H * W + static_cast<size_t>(yy) * W + xx]) : 0.f;
      }
    float g[16];
    unpack8(dz.ptr[(static_cast<size_t>(n) * dz.planes + dz.plane_off) * H * W + pix], g);
    unpack8(dz.ptr[(static_cast<size_t>(n) * dz.planes + dz.plane_off + 1) * H * W + pix], g + 8);
#pragma unroll
    for (int co = 0; co < 16; ++co)
#pragma unroll
      for (int k = 0; k < 9; ++k) loc[co * 9 + k] = fmaf(g[co], t[k], loc[co * 9 + k]);
  }
#pragma unroll
  for (int i = 0; i < 144; ++i) {
    float v = loc[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) atomicAdd(&acc[i], v);
  }
  __syncthreads();
  if (threadIdx.x < 144) atomicAdd(dw + (threadIdx.x / 9) * dw_costride + threadIdx.x % 9, acc[threadIdx.x]);
}

// Same gradient for sparse (binarised, ~5 % ink) images: dW[co][ky][kx] = sum over INK pixels q of img[q] * dz[q - (ky-1, kx-1)][co].
// A warp scans 32 consecutive pixels per step (one coalesced image load), ballots the non-zero ones and, for each of them, all
// 32 lanes together gather the 3 x 3 x 16 neighbourhood of dz: slot s = lane + 32 j -> (tap = s / 16, channel = s % 16), so 16
// consecutive lanes read the 32 contiguous bytes of one pixel. Work is proportional to the ink count (0.84 M of 16.8 M pixels
// per 64-image batch) instead of 144 FMAs for every pixel; a dense image degrades gracefully to the cost of the dense kernel.
template <typename T>
__global__ void __launch_bounds__(256) conv_c1_wgrad_sparse_kernel(const T* __restrict__ img, P8View dz, int N, int H, int W,
                                                                   float* __restrict__ dw) {
  __shared__ float acc[144];
  if (threadIdx.x < 144) acc[threadIdx.x] = 0.f;
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const long long HW = static_cast<long long>(H) * W, total = HW * N;
  const long long warp_global = static_cast<long long>(blockIdx.x) * 8 + (threadIdx.x >> 5);
  const long long n_warps = static_cast<long long>(gridDim.x) * 8;
  const __nv_bfloat16* __restrict__ dzh = reinterpret_cast<const __nv_bfloat16*>(dz.ptr);
  int sdy[5], sdx[5], sco[5];
  float loc[5];
#pragma unroll
  for (int j = 0; j < 5; ++j) {
    const int sl = lane + 32 * j, tap = sl >> 4;
    sdy[j] = tap / 3 - 1;
    sdx[j] = tap % 3 - 1;
    sco[j] = sl < 144 ? (sl & 15) : -1;
    loc[j] = 0.f;
  }
  for (long long base = warp_global * 32; base < total; base += n_warps * 32) {
    const long long e = base + lane;
    const float v = e < total ? static_cast<float>(img[e]) : 0.f;
    unsigned mask = __ballot_sync(0xffffffffu, v != 0.f);
    while (mask) {
      const int b = __ffs(mask) - 1;
      mask &= mask - 1;
      const float vq = __shfl_sync(0xffffffffu, v, b);
      const long long q = base + b;
      const int n = static_cast<int>(q / HW);
      const int pix = static_cast<int>(q - n * HW);
      const int y = pix / W, x = pix - y * W;
#pragma unroll
      for (int j = 0; j < 5; ++j) {
        const int py = y - sdy[j], px = x - sdx[j];
        if (sco[j] >= 0 && py >= 0 && py < H && px >= 0 && px < W) {
          const size_t off = (((static_cast<size_t>(n) * dz.planes + dz.plane_off + (sco[j] >> 3)) * H + py) * W + px) * 8 + (sco[j] & 7);
          loc[j] = fmaf(vq, __bfloat162float(dzh[off]), loc[j]);
        }
      }
    }
  }
#pragma unroll
  for (int j = 0; j < 5; ++j) {
    const int sl = lane + 32 * j;
    if (sl < 144) atomicAdd(&acc[(sl & 15) * 9 + (sl >> 4)], loc[j]);      // dw layout [co][tap]
  }
  __syncthreads();
  if (threadIdx.x < 144) atomicAdd(dw + threadIdx.x, acc[threadIdx.x]);
}

// P8 [N][planes][2H][2W][8] -> 4 phase tensors stacked on the plane axis: dst[N][4*cp][H][W][8], phase = 2*py + px
__global__ void __launch_bounds__(256) deinterleave2_kernel(P8View src, uint4* __restrict__ dst, int N, int cp, int H, int W) {
  const long long total = static_cast<long long>(N) * 4 * cp * H * W;
  const long long t = static_cast<long long>(blockIdx.x) * 256 + threadIdx.x;
  if (t >= total) return;
  const int x = static_cast<int>(t % W);
  long long r = t / W;
  const int y = static_cast<int>(r % H);
  r /= H;
  const int pl = static_cast<int>(r % (4 * cp));
  const int n = static_cast<int>(r / (4 * cp));
  const int phase = pl / cp, plane = pl - phase * cp;
  const int py = phase >> 1, px = phase & 1;
  dst[t] = src.ptr[((static_cast<size_t>(n) * src.planes + src.plane_off + plane) * (2 * H) + 2 * y + py) * (2 * W) + 2 * x + px];
}

}  // namespace abc

using namespace abc;

static int p8_check(const void* ptr, int planes, int plane_off, int cplanes, const char* what) {
  ABC_REQUIRE(ptr != nullptr && (reinterpret_cast<uintptr_t>(ptr) & 15) == 0, "%s: null or misaligned pointer", what);
  ABC_REQUIRE(plane_off >= 0 && cplanes >= 1 && plane_off + cplanes <= planes, "%s: plane range", what);
  return ABC_OK;
}

extern "C" int abc_bn_stats(const void* z, int N, int H, int W, int planes, int plane_off, int C, double* sum, double* sumsq,
                            void* stream) {
  if (int rc = device_check()) return rc;
  ABC_REQUIRE(C >= 8 && C % 8 == 0 && N > 0 && N <= 65535 && H > 0 && W > 0 && sum && sumsq, "abc_bn_stats: bad arguments");
  ABC_REQUIRE(static_cast<long long>(H) * W < (1ll << 30), "abc_bn_stats: image too large");
  if (int rc = p8_check(z, planes, plane_off, C / 8, "abc_bn_stats")) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  ABC_CUDA(cudaMemsetAsync(sum, 0, C * sizeof(double), st));
  ABC_CUDA(cudaMemsetAsync(sumsq, 0, C * sizeof(double), st));
  P8View v{static_cast<const uint4*>(z), planes, plane_off};
  const BnLaunch l = bn_launch_config(BnPass::kStats, N, C / 8, H, W);
  bn_stats_kernel<<<l.grid, l.block, 0, st>>>(v, H * W, sum, sumsq);
  return launch_check("bn_stats_kernel");
}

extern "C" int abc_bn_finalize(const double* sum, const double* sumsq, int C, double count, const float* gamma, const float* beta,
                               float eps, float momentum, float* running_mean, float* running_var, float* scale, float* shift,
                               float* mean, float* invstd, void* stream) {
  if (int rc = device_check()) return rc;
  ABC_REQUIRE(sum && sumsq && gamma && beta && scale && shift && mean && invstd && C > 0 && count > 0, "abc_bn_finalize: bad arguments");
  bn_finalize_kernel<<<(C + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(sum, sumsq, C, count, gamma, beta, eps, momentum,
                                                                                      running_mean, running_var, scale, shift, mean, invstd);
  return launch_check("bn_finalize_kernel");
}

extern "C" int abc_bn_act(const AbcBnActDesc* d, void* stream) {
  if (int rc = device_check()) return rc;
  ABC_REQUIRE(d && d->scale && d->shift, "abc_bn_act: null descriptor / scale / shift");
  ABC_REQUIRE(d->C >= 8 && d->C % 8 == 0 && d->N > 0 && d->H > 0 && d->W > 0, "abc_bn_act: bad geometry (C=%d H=%d W=%d)", d->C, d->H, d->W);
  ABC_REQUIRE(!d->pool || (d->H % 2 == 0 && d->W % 2 == 0), "abc_bn_act: fused max-pool needs even H, W");
  ABC_REQUIRE(d->out || d->pool, "abc_bn_act: no output");
  if (int rc = p8_check(d->z, d->z_planes, d->z_plane_off, d->C / 8, "abc_bn_act(z)")) return rc;
  if (d->out) if (int rc = p8_check(d->out, d->out_planes, d->out_plane_off, d->C / 8, "abc_bn_act(out)")) return rc;
  if (d->pool) if (int rc = p8_check(d->pool, d->pool_planes, d->pool_plane_off, d->C / 8, "abc_bn_act(pool)")) return rc;
  ABC_REQUIRE(d->N <= 65535 && static_cast<long long>(d->H) * d->W < (1ll << 30), "abc_bn_act: N or image too large");
  ABC_REQUIRE(!(d->pool && d->drop_p > 0.f), "abc_bn_act: dropout and fused max-pool are not combined");
  ABC_REQUIRE((reinterpret_cast<uintptr_t>(d->scale) & 15) == 0 && (reinterpret_cast<uintptr_t>(d->shift) & 15) == 0,
              "abc_bn_act: scale / shift must be 16-byte aligned");
  BnActParams p;
  p.z = P8View{static_cast<const uint4*>(d->z), d->z_planes, d->z_plane_off};
  p.out = static_cast<uint4*>(d->out); p.out_planes = d->out_planes; p.out_plane_off = d->out_plane_off;
  p.pool = static_cast<uint4*>(d->pool); p.pool_planes = d->pool_planes; p.pool_plane_off = d->pool_plane_off;
  p.N = d->N; p.H = d->H; p.W = d->W; p.planes = d->C / 8;
  p.scale = d->scale; p.shift = d->shift; p.act = d->act; p.drop_p = d->drop_p; p.seed = d->seed;
  p.seed_dev = reinterpret_cast<const unsigned long long*>(d->seed_dev);
  p.drop_mask = static_cast<unsigned char*>(d->drop_mask);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const BnLaunch l = bn_launch_config(d->pool ? BnPass::kPool : BnPass::kPixels, d->N, p.planes, d->H, d->W);
  if (d->pool) bn_act_kernel<true><<<l.grid, l.block, 0, st>>>(p);
  else bn_act_kernel<false><<<l.grid, l.block, 0, st>>>(p);
  return launch_check("bn_act_kernel");
}

extern "C" int abc_bn_act_backward(const AbcBnActBwdDesc* d, void* stream) {
  if (int rc = device_check()) return rc;
  ABC_REQUIRE(d && d->scale && d->shift && d->mean && d->invstd && d->s1 && d->s2 && d->dz, "abc_bn_act_backward: null argument");
  ABC_REQUIRE(d->C >= 8 && d->C % 8 == 0 && d->N > 0 && d->H > 0 && d->W > 0, "abc_bn_act_backward: bad geometry");
  ABC_REQUIRE(!d->dP || (d->H % 2 == 0 && d->W % 2 == 0), "abc_bn_act_backward: pooled gradient needs even H, W");
  ABC_REQUIRE(d->dA || d->dP, "abc_bn_act_backward: no incoming gradient");
  const int cp = d->C / 8;
  if (int rc = p8_check(d->z, d->z_planes, d->z_plane_off, cp, "abc_bn_act_backward(z)")) return rc;
  if (d->dA) if (int rc = p8_check(d->dA, d->dA_planes, d->dA_plane_off, cp, "abc_bn_act_backward(dA)")) return rc;
  if (d->dP) if (int rc = p8_check(d->dP, d->dP_planes, d->dP_plane_off, cp, "abc_bn_act_backward(dP)")) return rc;
  if (int rc = p8_check(d->dz, d->dz_planes, d->dz_plane_off, cp, "abc_bn_act_backward(dz)")) return rc;
  ABC_REQUIRE(d->N <= 65535 && static_cast<long long>(d->H) * d->W < (1ll << 30), "abc_bn_act_backward: N or image too large");
  ABC_REQUIRE(!(d->dP && d->drop_p > 0.f), "abc_bn_act_backward: dropout and max-pool routing are not combined");
  for (const float* q : {d->scale, d->shift, d->mean, d->invstd})
    ABC_REQUIRE((reinterpret_cast<uintptr_t>(q) & 15) == 0, "abc_bn_act_backward: per-channel vectors must be 16-byte aligned");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  BnActBwdParams p;
  p.z = P8View{static_cast<const uint4*>(d->z), d->z_planes, d->z_plane_off};
  p.dA = P8View{static_cast<const uint4*>(d->dA), d->dA_planes, d->dA_plane_off};
  p.dP = P8View{static_cast<const uint4*>(d->dP), d->dP_planes, d->dP_plane_off};
  p.N = d->N; p.H = d->H; p.W = d->W; p.planes = cp;
  p.scale = d->scale; p.shift = d->shift; p.mean = d->mean; p.invstd = d->invstd;
  p.act = d->act; p.drop_p = d->drop_p; p.seed = d->seed;
  p.seed_dev = reinterpret_cast<const unsigned long long*>(d->seed_dev);
  p.s1 = d->s1; p.s2 = d->s2;
  p.dz = static_cast<uint4*>(d->dz); p.dz_planes = d->dz_planes; p.dz_plane_off = d->dz_plane_off;
  p.count = static_cast<double>(d->N) * d->H * d->W;
  p.gscale = d->gscale;
  p.drop_mask = static_cast<const unsigned char*>(d->drop_mask);
  ABC_REQUIRE((reinterpret_cast<uintptr_t>(d->gscale) & 15) == 0, "abc_bn_act_backward: gscale must be 16-byte aligned");
  ABC_CUDA(cudaMemsetAsync(d->s1, 0, d->C * sizeof(double), st));
  ABC_CUDA(cudaMemsetAsync(d->s2, 0, d->C * sizeof(double), st));
  const BnLaunch l = bn_launch_config(d->dP ? BnPass::kPool : BnPass::kPixels, d->N, cp, d->H, d->W);
  if (d->dP) {
    bn_act_bwd_reduce_kernel<true><<<l.grid, l.block, 0, st>>>(p);
    if (int rc = launch_check("bn_act_bwd_reduce_kernel")) return rc;
    bn_act_bwd_apply_kernel<true><<<l.grid, l.block, 0, st>>>(p);
  } else {
    // resident blocks per SM (register cap) of the two passes: ABCNET_BN_MINB = <reduce digit><apply digit>, read once
    static const int minb = [] { const char* e = getenv("ABCNET_BN_MINB"); return e ? atoi(e) : 34; }();
    if (minb / 10 == 4) bn_act_bwd_reduce_kernel<false, 4><<<l.grid, l.block, 0, st>>>(p);
    else bn_act_bwd_reduce_kernel<false, 3><<<l.grid, l.block, 0, st>>>(p);
    if (int rc = launch_check("bn_act_bwd_reduce_kernel")) return rc;
    if (minb % 10 == 4) bn_act_bwd_apply_kernel<false, 4><<<l.grid, l.block, 0, st>>>(p);
    else if (minb % 10 == 3) bn_act_bwd_apply_kernel<false, 3><<<l.grid, l.block, 0, st>>>(p);
    else bn_act_bwd_apply_kernel<false, 2><<<l.grid, l.block, 0, st>>>(p);
  }
  return launch_check("bn_act_bwd_apply_kernel");
}

extern "C" int abc_nchw_to_p8(const float* src, void* dst, int N, int C, int H, int W, void* stream) {
  if (int rc = device_check()) return rc;
  ABC_REQUIRE(src && dst && N > 0 && C > 0 && H > 0 && W > 0, "abc_nchw_to_p8: bad arguments");
  const int planes = (C + 7) / 8;
  const long long total = static_cast<long long>(N) * planes * H * W;
  nchw_to_p8_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      src, static_cast<uint4*>(dst), N, C, H * W, planes);
  return launch_check("nchw_to_p8_kernel");
}

extern "C" int abc_nchw_to_p8_ex(const float* src, void* dst, int N, int C, int H, int W, int dst_planes, const float* scale,
                                 double* dbias, void* stream) {
  if (int rc = device_check()) return rc;
  ABC_REQUIRE(src && dst && N > 0 && N <= 65535 && C > 0 && H > 0 && W > 0, "abc_nchw_to_p8_ex: bad arguments");
  ABC_REQUIRE(dst_planes >= (C + 7) / 8 && dst_planes <= 65535, "abc_nchw_to_p8_ex: dst_planes=%d too small for C=%d", dst_planes, C);
  ABC_REQUIRE((reinterpret_cast<uintptr_t>(dst) & 15) == 0, "abc_nchw_to_p8_ex: dst must be 16-byte aligned");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (dbias) ABC_CUDA(cudaMemsetAsync(dbias, 0, C * sizeof(double), st));
  const BnLaunch l = bn_launch_config(BnPass::kPixels, N, dst_planes, H, W);
  nchw_to_p8_ex_kernel<<<l.grid, l.block, 0, st>>>(src, static_cast<uint4*>(dst), C, H * W, dst_planes, scale, dbias);
  return launch_check("nchw_to_p8_ex_kernel");
}

extern "C" int abc_channel_sum(const void* x, int N, int H, int W, int planes, int plane_off, int C, double* sum, double* sumsq_scratch,
                               void* stream) {
  return abc_bn_stats(x, N, H, W, planes, plane_off, C, sum, sumsq_scratch, stream);
}

extern "C" int abc_conv3x3_c1_wgrad(const void* img, int img_is_u8, const void* dz, int dz_planes, int dz_plane_off, int N, int H, int W,
                                    float* dw, void* stream) {
  if (int rc = device_check()) return rc;
  ABC_REQUIRE(img && dw && N > 0 && H > 0 && W > 0, "abc_conv3x3_c1_wgrad: bad arguments");
  if (int rc = p8_check(dz, dz_planes, dz_plane_off, 2, "abc_conv3x3_c1_wgrad(dz)")) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  ABC_CUDA(cudaMemsetAsync(dw, 0, 144 * sizeof(float), st));
  P8View v{static_cast<const uint4*>(dz), dz_planes, dz_plane_off};
  static const bool dense = getenv("ABCNET_C1_WGRAD_DENSE") != nullptr;      // the 144-FMA-per-pixel kernel (kept for comparison)
  if (!dense) {
    const int blocks = 148 * 8;
    if (img_is_u8)
      conv_c1_wgrad_sparse_kernel<uint8_t><<<blocks, 256, 0, st>>>(static_cast<const uint8_t*>(img), v, N, H, W, dw);
    else
      conv_c1_wgrad_sparse_kernel<float><<<blocks, 256, 0, st>>>(static_cast<const float*>(img), v, N, H, W, dw);
    return launch_check("conv_c1_wgrad_sparse_kernel");
  }
  const int blocks = 148 * 4;
  if (img_is_u8)
    conv_c1_wgrad_kernel<uint8_t><<<blocks, 256, 0, st>>>(static_cast<const uint8_t*>(img), v, N, H, W, dw, 1, 9);
  else
    conv_c1_wgrad_kernel<float><<<blocks, 256, 0, st>>>(static_cast<const float*>(img), v, N, H, W, dw, 1, 9);
  return launch_check("conv_c1_wgrad_kernel");
}

// Weight gradient of the general stem (abc_conv3x3_cn): dw fp32 [16][cin][9], one pass over dz per input channel.
extern "C" int abc_conv3x3_cn_wgrad(const float* img, int cin, const void* dz, int dz_planes, int dz_plane_off, int N, int H, int W,
                                    float* dw, void* stream) {
  if (int rc = device_check()) return rc;
  ABC_REQUIRE(img && dw && N > 0 && H > 0 && W > 0 && cin >= 1 && cin <= 8, "abc_conv3x3_cn_wgrad: bad arguments");
  if (int rc = p8_check(dz, dz_planes, dz_plane_off, 2, "abc_conv3x3_cn_wgrad(dz)")) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  ABC_CUDA(cudaMemsetAsync(dw, 0, static_cast<size_t>(144) * cin * sizeof(float), st));
  P8View v{static_cast<const uint4*>(dz), dz_planes, dz_plane_off};
  for (int ci = 0; ci < cin; ++ci) {
    conv_c1_wgrad_kernel<float><<<148 * 4, 256, 0, st>>>(img + static_cast<size_t>(ci) * H * W, v, N, H, W, dw + ci * 9, cin, cin * 9);
    if (int rc = launch_check("conv_c1_wgrad_kernel")) return rc;
  }
  return ABC_OK;
}

extern "C" int abc_deinterleave2(const void* src, int src_planes, int src_plane_off, int C, void* dst, int N, int H, int W, void* stream) {
  if (int rc = device_check()) return rc;
  ABC_REQUIRE(dst && C >= 8 && C % 8 == 0 && N > 0 && H > 0 && W > 0, "abc_deinterleave2: bad arguments");
  if (int rc = p8_check(src, src_planes, src_plane_off, C / 8, "abc_deinterleave2(src)")) return rc;
  P8View v{static_cast<const uint4*>(src), src_planes, src_plane_off};
  const long long total = static_cast<long long>(N) * 4 * (C / 8) * H * W;
  deinterleave2_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      v, static_cast<uint4*>(dst), N, C / 8, H, W);
  return launch_check("deinterleave2_kernel");
}

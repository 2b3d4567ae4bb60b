// Error state, device probing and launch accounting for the C-ABI.
#include "common.cuh"

namespace abc {

static thread_local char g_err[512] = "";
std::atomic<int64_t> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

static std::atomic<int> g_dev_ok[kMaxDevices];      // zero-initialised; 1 = sm_100 confirmed
static std::atomic<int> g_dev_sms[kMaxDevices];

int current_device() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) {
    cudaGetLastError();
    return -1;
  }
  return dev;
}

int device_check() {
  const int dev = current_device();
  if (dev < 0) {
    set_error("no CUDA device available (abcnet_b200 has no CPU fallback)");
    return ABC_ERR_NO_DEVICE;
  }
  if (dev < kMaxDevices && g_dev_ok[dev].load(std::memory_order_relaxed)) return ABC_OK;
  int major = 0;
  if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess || major != 10) {
    cudaGetLastError();
    set_error("device %d has compute capability major %d; the kernels are built for sm_100a only", dev, major);
    return ABC_ERR_NO_DEVICE;
  }
  if (dev < kMaxDevices) g_dev_ok[dev].store(1, std::memory_order_relaxed);
  return ABC_OK;
}

void* tensor_map_encode_fn() {
  static void* const fn = [] {                       // C++11 magic static: initialised exactly once, thread-safe
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      return ptr;
    cudaGetLastError();
    return static_cast<void*>(nullptr);
  }();
  return fn;
}

int sm_count() {
  const int dev = current_device();
  if (dev < 0) return 0;
  if (dev < kMaxDevices) {
    const int c = g_dev_sms[dev].load(std::memory_order_relaxed);
    if (c > 0) return c;
  }
  int n = 0;
  if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  if (dev < kMaxDevices) g_dev_sms[dev].store(n, std::memory_order_relaxed);
  return n;
}

// One block per 32 consecutive elements: lane = element, warp w sums the contiguous slot range [w S / 8, (w + 1) S / 8) in
// order, thread w == 0 then adds the 8 warp totals in warp order.
template <typename T>
__global__ void __launch_bounds__(256) det_reduce_kernel(const T* __restrict__ ws, int slots, int n, const DetOut out, int add) {
  __shared__ T part[8][32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int e = blockIdx.x * 32 + lane;
  const int s0 = static_cast<int>(static_cast<long long>(slots) * warp / 8), s1 = static_cast<int>(static_cast<long long>(slots) * (warp + 1) / 8);
  T t = 0;
  if (e < n)
    for (int s = s0; s < s1; ++s) t += ws[static_cast<size_t>(s) * n + e];
  part[warp][lane] = t;
  __syncthreads();
  if (warp != 0 || e >= n) return;
  T r = part[0][lane];
#pragma unroll
  for (int w = 1; w < 8; ++w) r += part[w][lane];
  int k = 0, start = 0;
  while (e >= out.end[k]) start = out.end[k++];
  T* dst = static_cast<T*>(out.ptr[k]) + (e - start);
  *dst = add ? *dst + r : r;
}

template <typename T>
static int det_reduce_t(const T* ws, int slots, int n, const DetOut& out, int add, cudaStream_t st) {
  ABC_REQUIRE(ws && slots > 0 && n > 0 && out.count >= 1 && out.count <= kDetMaxOut && out.end[out.count - 1] == n,
              "det_reduce: bad workspace / output segments");
  det_reduce_kernel<T><<<(n + 31) / 32, 256, 0, st>>>(ws, slots, n, out, add);
  return launch_check("det_reduce_kernel");
}
int det_reduce(const float* ws, int slots, int n, const DetOut& out, int add, cudaStream_t st) {
  return det_reduce_t(ws, slots, n, out, add, st);
}
int det_reduce(const double* ws, int slots, int n, const DetOut& out, int add, cudaStream_t st) {
  return det_reduce_t(ws, slots, n, out, add, st);
}

}  // namespace abc

extern "C" {
const char* abc_last_error(void) { return abc::g_err; }
int abc_version(void) { return 103; }
int abc_device_ok(void) { return abc::device_check() == ABC_OK ? 1 : 0; }
int abc_sm_count(void) {
  int n = abc::sm_count();
  return n > 0 ? n : ABC_ERR_NO_DEVICE;
}
int64_t abc_launch_count(void) { return abc::g_launches.load(); }
}

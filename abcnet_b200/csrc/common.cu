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

}  // namespace abc

extern "C" {
const char* abc_last_error(void) { return abc::g_err; }
int abc_version(void) { return 102; }
int abc_device_ok(void) { return abc::device_check() == ABC_OK ? 1 : 0; }
int abc_sm_count(void) {
  int n = abc::sm_count();
  return n > 0 ? n : ABC_ERR_NO_DEVICE;
}
int64_t abc_launch_count(void) { return abc::g_launches.load(); }
}

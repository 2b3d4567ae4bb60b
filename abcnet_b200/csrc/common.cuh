// Host-side helpers shared by the C-ABI translation units.
#pragma once
#include <atomic>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cuda_runtime.h>

#include "../../include/abcnet_b200.h"

namespace abc {

void set_error(const char* fmt, ...);
extern std::atomic<int64_t> g_launches;
int device_check();   // ABC_OK or ABC_ERR_NO_DEVICE (message set); the positive answer is cached per device
int sm_count();
int current_device();  // cudaGetDevice, -1 on failure
void* tensor_map_encode_fn();   // cuTensorMapEncodeTiled through the runtime's driver entry point (resolved once, thread-safe); nullptr if unavailable

constexpr int kMaxDevices = 64;

// Per-device one-time initialisation (cudaFuncSetAttribute is a per-device setting): thread-safe, no mutable global
// state beyond the immutable "done" flags (SURVEY.md section 8b threading contract).
struct PerDeviceOnce {
  std::atomic<int> done[kMaxDevices];
  PerDeviceOnce() { for (auto& d : done) d.store(0, std::memory_order_relaxed); }
  // runs fn() until it has succeeded once on the current device; fn is idempotent, so a race merely repeats it
  template <typename F>
  cudaError_t run(F&& fn) {
    const int dev = current_device();
    if (dev < 0 || dev >= kMaxDevices) return fn();
    if (done[dev].load(std::memory_order_acquire)) return cudaSuccess;
    const cudaError_t e = fn();
    if (e == cudaSuccess) done[dev].store(1, std::memory_order_release);
    return e;
  }
};

#define ABC_CUDA(expr)                                                                         \
  do {                                                                                         \
    cudaError_t _e = (expr);                                                                   \
    if (_e != cudaSuccess) {                                                                   \
      ::abc::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return ABC_ERR_CUDA;                                                                     \
    }                                                                                          \
  } while (0)

#define ABC_REQUIRE(cond, ...)        \
  do {                                \
    if (!(cond)) {                    \
      ::abc::set_error(__VA_ARGS__);  \
      return ABC_ERR_INVALID;         \
    }                                 \
  } while (0)

// Fixed-order reduction of the deterministic mode (det_slots.cuh): for e < n, r = sum over s < slots of ws[s * n + e], added in
// slot-index order (contiguous slot ranges per warp, then the warp totals in warp order -- fixed for given slots and n). The
// element range is cut into consecutive output segments (ends ascending, the last one == n): element e of segment k goes to
// out[k][e - start of k]; add != 0 adds r to the value there instead of overwriting it.
constexpr int kDetMaxOut = 10;
struct DetOut {
  void* ptr[kDetMaxOut];
  int end[kDetMaxOut];
  int count;
};
int det_reduce(const float* ws, int slots, int n, const DetOut& out, int add, cudaStream_t st);
int det_reduce(const double* ws, int slots, int n, const DetOut& out, int add, cudaStream_t st);
inline DetOut det_out1(void* a, int n) { DetOut o{}; o.ptr[0] = a; o.end[0] = n; o.count = 1; return o; }
inline DetOut det_out2(void* a, void* b, int n) { DetOut o{}; o.ptr[0] = a; o.end[0] = n; o.ptr[1] = b; o.end[1] = 2 * n; o.count = 2; return o; }

inline int launch_check(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error("launch of %s failed: %s", what, cudaGetErrorString(e));
    return ABC_ERR_CUDA;
  }
  g_launches.fetch_add(1, std::memory_order_relaxed);
  return ABC_OK;
}

}  // namespace abc

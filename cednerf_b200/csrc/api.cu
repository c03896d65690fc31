// Library-level entry points of libcednerf_b200.so: error reporting and build identification.
#include <stdarg.h>
#include <string.h>

#include "common.cuh"

#include <atomic>

static thread_local char g_last_error[512] = "";
static std::atomic<long long> g_launches{0};

void cednerf_count_launches(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

// number of kernels this library has launched in this process (every entry point counts its own)
CEDNERF_EXPORT int64_t cednerf_launch_count(void) { return (int64_t)g_launches.load(std::memory_order_relaxed); }

void cednerf_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_last_error, sizeof(g_last_error), fmt, ap);
  va_end(ap);
}

CEDNERF_EXPORT const char* cednerf_last_error(void) { return g_last_error; }

CEDNERF_EXPORT int cednerf_abi_version(void) { return 4; }

// 0 when the current device can run this library (compute capability 10.x), else a negative code.
CEDNERF_EXPORT int cednerf_check_device(void) {
  int dev = 0, major = 0, minor = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) {
    cednerf_set_error("cednerf_check_device: %s", cudaGetErrorString(e));
    return (int)e;
  }
  cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
  cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev);
  if (major != 10) {
    cednerf_set_error("cednerf_check_device: built for sm_100a, device is sm_%d%d", major, minor);
    return CEDNERF_ERR_UNSUPPORTED;
  }
  return 0;
}

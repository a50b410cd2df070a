// Host plumbing shared by every translation unit of the library: the error message behind dwmh_last_error, the CUDA
// error checks, the device guard of the entry points, the SM count and weight uploads.  common.cuh holds the device side.
#pragma once
#include <cuda_runtime.h>
#include <cstdarg>
#include <cstdio>
#include <string>
#include <vector>

#define CU_TRY(expr) do { cudaError_t e__ = (expr); if (e__ != cudaSuccess) \
  return dwmh::fail("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); } while (0)
#define DW_TRY(expr) do { int r__ = (expr); if (r__) return r__; } while (0)
#define DEV_GUARD(dev) dwmh::DevGuard dev_guard__(dev); if (!dev_guard__.ok) return dwmh::fail("cudaSetDevice(%d) failed", (int)(dev))

namespace dwmh {

// The calling thread's last error message (what dwmh_last_error returns).
inline thread_local std::string g_err;

// Sets g_err from a printf format; returns 1, the entry points' error code.
inline int fail(const char* fmt, ...) {
  char buf[1024];
  va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof buf, fmt, ap); va_end(ap);
  g_err = buf;
  return 1;
}

// Entry points run on `dev` and leave the caller's current device as they found it.
struct DevGuard {
  int prev = -1; bool ok = false;
  explicit DevGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
    ok = (prev == dev) || cudaSetDevice(dev) == cudaSuccess;
    if (prev == dev) prev = -1;
  }
  ~DevGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

// SMs of `device`, queried once per device; 148 (a B200) if the query fails.
inline int sm_count(int device) {
  static int sms[64] = {0};
  if (device < 0 || device >= 64) return 148;
  if (!sms[device]) cudaDeviceGetAttribute(&sms[device], cudaDevAttrMultiProcessorCount, device);
  return sms[device] > 0 ? sms[device] : 148;
}

// (Re)allocates *dst on the current device and copies `src` into it.
template <typename V>
int upload(V** dst, const std::vector<V>& src) {
  if (*dst) { cudaFree(*dst); *dst = nullptr; }
  CU_TRY(cudaMalloc((void**)dst, src.size() * sizeof(V)));
  CU_TRY(cudaMemcpy(*dst, src.data(), src.size() * sizeof(V), cudaMemcpyHostToDevice));
  return 0;
}

}  // namespace dwmh

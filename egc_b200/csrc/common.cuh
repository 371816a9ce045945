// Shared helpers for libegc_b200 (sm_100a).  Host-side error plumbing + small device utilities.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "egc_b200.h"

#define EGC_STR2(x) #x
#define EGC_STR(x) EGC_STR2(x)

namespace egc {

// thread-local "last error" message (api.cu)
void set_error(const char* fmt, ...);

inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

#define EGC_REQUIRE(cond, ...)                        \
  do {                                                \
    if (!(cond)) {                                    \
      ::egc::set_error(__VA_ARGS__);                  \
      return EGC_ERR_INVALID_ARGUMENT;                \
    }                                                 \
  } while (0)

#define EGC_CUDA(expr)                                                                        \
  do {                                                                                        \
    cudaError_t egc_e_ = (expr);                                                              \
    if (egc_e_ != cudaSuccess) {                                                              \
      ::egc::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(egc_e_), __FILE__,  \
                       __LINE__);                                                             \
      return EGC_ERR_CUDA;                                                                    \
    }                                                                                         \
  } while (0)

#define EGC_LAUNCH_CHECK(name)                                                                \
  do {                                                                                        \
    cudaError_t egc_e_ = cudaGetLastError();                                                  \
    if (egc_e_ != cudaSuccess) {                                                              \
      ::egc::set_error("launch of %s failed: %s", name, cudaGetErrorString(egc_e_));          \
      return EGC_ERR_CUDA;                                                                    \
    }                                                                                         \
  } while (0)

constexpr int kWarp = 32;
constexpr unsigned kFull = 0xffffffffu;

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
inline int ceil_div(int64_t a, int64_t b) { return static_cast<int>((a + b - 1) / b); }

// carve typed arrays out of a caller-provided workspace
struct Carver {
  char* base;
  size_t off = 0;
  explicit Carver(void* p) : base(static_cast<char*>(p)) {}
  template <typename T>
  T* take(size_t n) {
    off = align_up(off, 256);
    T* p = reinterpret_cast<T*>(base + off);
    off += n * sizeof(T);
    return p;
  }
  size_t used() const { return align_up(off, 256); }
};

// number of SMs of the current device (cached)
int sm_count();

// Raises cudaFuncAttributeMaxDynamicSharedMemorySize of `func` to `bytes` once per device: the attribute belongs to the
// function in the current device's context, so a process that launches on several devices sets it on each.  `done` holds
// the call site's per-device flags.
constexpr int kMaxDevices = 64;
inline cudaError_t max_dynamic_smem_once(const void* func, int bytes, bool (&done)[kMaxDevices]) {
  int dev = 0;
  if (cudaError_t e = cudaGetDevice(&dev)) return e;
  const bool cached = dev >= 0 && dev < kMaxDevices;
  if (cached && done[dev]) return cudaSuccess;
  const cudaError_t e = cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e == cudaSuccess && cached) done[dev] = true;
  return e;
}

// Every kernel launch goes through a LaunchScope: counts the launch and, when profiling is on,
// brackets it with CUDA events on the launching stream (api.cu).
struct LaunchScope {
  LaunchScope(const char* name, cudaStream_t st);
  ~LaunchScope();
  cudaStream_t st_;
  int slot_;
};

}  // namespace egc

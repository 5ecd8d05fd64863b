// Shared helpers for libunreal_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/unreal_b200.h"

#if defined(__CUDACC__)
#define UNREAL_HD __host__ __device__ __forceinline__
#else
#define UNREAL_HD inline
#endif

namespace unreal {

// thread-local error text behind unreal_last_error()
void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what);
// SM count of the current device (0 and the error text set when it cannot be queried)
int sm_count();
// Opts `kernel` into `bytes` (> 48 KB) of dynamic shared memory on the current device.  The attribute is per device, so
// the call is made once per (kernel, device); later calls cost a cudaGetDevice and a lookup.  Thread-safe.
int allow_dynamic_smem(const void* kernel, int bytes);

inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

#define UNREAL_REQUIRE(cond, ...)          \
  do {                                     \
    if (!(cond)) {                         \
      ::unreal::set_error(__VA_ARGS__);    \
      return UNREAL_EINVAL;                \
    }                                      \
  } while (0)

#define UNREAL_CUDA(call)                                        \
  do {                                                           \
    cudaError_t e__ = (call);                                    \
    if (e__ != cudaSuccess) return ::unreal::cuda_fail(e__, #call); \
  } while (0)

// every launch is followed by this: launch-configuration errors surface at the call site
#define UNREAL_LAUNCH_CHECK(name)                                     \
  do {                                                                \
    cudaError_t e__ = cudaGetLastError();                             \
    if (e__ != cudaSuccess) return ::unreal::cuda_fail(e__, name);    \
  } while (0)

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

int get_tunable(const char* name, int dflt);

// pixel_change84.cu: HBM-rate pixel change of 84x84x3 frames; -100 = not applicable
int pixel_change84(const void* p0, int64_t stride0, const void* p1, int64_t stride1, int dtype, float* pc,
                   int sequences, int l, cudaStream_t st);

}  // namespace unreal

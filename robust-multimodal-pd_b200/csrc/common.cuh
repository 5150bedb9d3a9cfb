// Shared helpers for libpdfusion_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#ifdef __CUDACC__
#include <curand_philox4x32_x.h>
#endif

#include "../../include/pdfusion_b200.h"

namespace pdf {

void set_error(const char* fmt, ...);
void count_launch(int n = 1);

inline cudaStream_t as_stream(pdf_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }

#define PDF_CHECK_CUDA(expr)                                                                  \
  do {                                                                                        \
    cudaError_t _e = (expr);                                                                  \
    if (_e != cudaSuccess) {                                                                  \
      pdf::set_error("%s:%d %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e));    \
      return PDF_ERR_CUDA;                                                                    \
    }                                                                                         \
  } while (0)

#define PDF_CHECK_LAUNCH()                                                                    \
  do {                                                                                        \
    pdf::count_launch();                                                                      \
    cudaError_t _e = cudaGetLastError();                                                      \
    if (_e != cudaSuccess) {                                                                  \
      pdf::set_error("%s:%d kernel launch -> %s", __FILE__, __LINE__, cudaGetErrorString(_e)); \
      return PDF_ERR_CUDA;                                                                    \
    }                                                                                         \
  } while (0)

#define PDF_REQUIRE(cond, ...)                                                                \
  do {                                                                                        \
    if (!(cond)) {                                                                            \
      pdf::set_error(__VA_ARGS__);                                                            \
      return PDF_ERR_ARG;                                                                     \
    }                                                                                         \
  } while (0)

// monotone float <-> uint key (for atomicMax/atomicMin on floats of either sign)
__host__ __device__ inline uint32_t float_to_ordered(float f) {
  uint32_t b;
#ifdef __CUDA_ARCH__
  b = __float_as_uint(f);
#else
  memcpy(&b, &f, 4);
#endif
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__host__ __device__ inline float ordered_to_float(uint32_t k) {
  uint32_t b = (k & 0x80000000u) ? (k & 0x7fffffffu) : ~k;
#ifdef __CUDA_ARCH__
  return __uint_as_float(b);
#else
  float f;
  memcpy(&f, &b, 4);
  return f;
#endif
}

inline int ceil_div(long long a, long long b) { return (int)((a + b - 1) / b); }

// Programmatic dependent launch: the kernel may be scheduled while its predecessor in the stream drains; its prologue
// (barrier init, TMEM allocation, tensor-map prefetch, weight loads) then overlaps the predecessor's tail, and pdl_wait()
// blocks until the predecessor has completed and its writes are visible.  Kernels launched this way MUST call pdl_wait()
// before their first access to memory the predecessor touches.
bool pdl_enabled();
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = pdl_enabled() ? 1 : 0;
  cfg.attrs = attr; cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// Philox4x32-10 (Salmon et al., SC'11; curand's constants and rounds): four 32-bit words, a pure function of (counter, key).  The
// device's stateless random streams: the bootstrap weights (metrics.cu, counters (unit, b, 0, 0)) and the Monte-Carlo dropout masks
// (uncertainty.cu, counters with the top bit of word 3 set), each from key = (seed low, seed high).
__device__ __forceinline__ uint4 philox4x32_10(uint4 counter, uint2 key) { return curand_Philox4x32_10(counter, key); }
#endif

int num_sms();

}  // namespace pdf

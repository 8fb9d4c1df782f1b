// Shared helpers for the tmc_b200 C-ABI library (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#define TMC_OK 0
#define TMC_ERR_ARG 1
#define TMC_ERR_CUDA 2
#define TMC_ERR_UNSUPPORTED 3

#define TMC_API extern "C" __attribute__((visibility("default")))

// CUDA caps gridDim.y and gridDim.z at 65535.  Entry points that put a caller's job / item / plane count there either
// split longer calls into slices of at most this many or reject them (include/tmc_b200.h says which).
constexpr int kMaxGridYZ = 65535;

// thread-local message for tmc_last_error()
void tmc_set_error(const char* fmt, ...);
// bookkeeping for bench.py: every kernel launch of this library is counted
void tmc_count_launch();
// optional per-kernel device timing (tmc_kernel_timing): CUDA events recorded on the launching stream right before and
// right after a launch; no-ops unless switched on
void tmc_timing_begin(cudaStream_t stream);
void tmc_timing_end(const char* kernel, cudaStream_t stream);
// launch statement bracketed by the timing events and counted
#define TMC_TIMED(name, stream, ...) \
  do {                               \
    tmc_timing_begin(stream);        \
    __VA_ARGS__;                     \
    tmc_timing_end(name, stream);    \
    tmc_count_launch();              \
  } while (0)

#define TMC_CHECK_ARG(cond, ...)          \
  do {                                    \
    if (!(cond)) {                        \
      tmc_set_error(__VA_ARGS__);         \
      return TMC_ERR_ARG;                 \
    }                                     \
  } while (0)

#define TMC_CHECK_LAUNCH(name)                                                   \
  do {                                                                           \
    cudaError_t e__ = cudaGetLastError();                                        \
    if (e__ != cudaSuccess) {                                                    \
      tmc_set_error("%s: CUDA launch failed: %s", name, cudaGetErrorString(e__)); \
      return TMC_ERR_CUDA;                                                       \
    }                                                                            \
  } while (0)

#define TMC_CUDA(call)                                                          \
  do {                                                                          \
    cudaError_t e__ = (call);                                                   \
    if (e__ != cudaSuccess) {                                                   \
      tmc_set_error("%s failed: %s", #call, cudaGetErrorString(e__));           \
      return TMC_ERR_CUDA;                                                      \
    }                                                                           \
  } while (0)

static inline int tmc_div_up(long a, long b) { return (int)((a + b - 1) / b); }

// ---- device helpers -------------------------------------------------------------------

__device__ __forceinline__ float2 cadd(float2 a, float2 b) { return make_float2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ float2 csub(float2 a, float2 b) { return make_float2(a.x - b.x, a.y - b.y); }
__device__ __forceinline__ float2 cmul(float2 a, float2 b) {
  return make_float2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x);
}
// conj(a) * b
__device__ __forceinline__ float2 cmul_conj(float2 a, float2 b) {
  return make_float2(a.x * b.x + a.y * b.y, a.x * b.y - a.y * b.x);
}

// torch.linspace(0, 1, n)[i] in fp32 (ATen computes the upper half from the end point)
__device__ __forceinline__ float linspace01(int i, int n) {
  if (n <= 1) return 0.0f;
  float step = __fdiv_rn(1.0f, (float)(n - 1));
  int half = n / 2;
  return (i < half) ? __fmul_rn(step, (float)i) : __fsub_rn(1.0f, __fmul_rn(step, (float)(n - 1 - i)));
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

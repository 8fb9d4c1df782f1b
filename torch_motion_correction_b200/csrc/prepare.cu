// Movie preparation ahead of the estimators: detector-native pixel types -> fp32, gain multiply, hot-pixel
// replacement, per-frame mean removal.
//
// Replaces the NumPy pre-processing of the reference's example workflow (examples/ttMotion.py:90-202: gain_correct,
// remove_hot_pixels, set_frames_mean_zero, `.to(torch.float32)` at :357) for movies that arrive from the host in their
// native type (uint8 / uint16 / int16 counts, float16): the PCIe copy moves 1-2 bytes per pixel instead of 4 and the
// conversion runs at HBM speed on the device, fused with the gain multiply and the per-frame moments.
#include "common.cuh"
#include <cuda_fp16.h>

namespace {

constexpr int kPrepThreads = 256;

template <typename T>
__device__ __forceinline__ float to_f32(T v) { return (float)v; }
template <>
__device__ __forceinline__ float to_f32<__half>(__half v) { return __half2float(v); }

// dst[f][i] = float(src[f][i]) * gain[i]; moments[f] += {sum, sum of squares} of the converted frame (double)
template <typename T>
__global__ void __launch_bounds__(kPrepThreads)
convert_stack_kernel(const T* __restrict__ src, long n, const float* __restrict__ gain, float* __restrict__ dst,
                     double* __restrict__ moments) {
  constexpr int VEC = 16 / sizeof(T);  // source elements per 16-byte load
  const int f = blockIdx.y;
  const T* s = src + (long)f * n;
  float* d = dst + (long)f * n;
  const bool aligned = ((reinterpret_cast<uintptr_t>(s) | reinterpret_cast<uintptr_t>(d)) & 15) == 0 &&
                       (gain == nullptr || (reinterpret_cast<uintptr_t>(gain) & 15) == 0);
  const long nvec = aligned ? n / VEC : 0;
  float fs = 0.f, fss = 0.f;
  double ds = 0.0, dss = 0.0;
  int folded = 0;
  for (long i = (long)blockIdx.x * kPrepThreads + threadIdx.x; i < nvec; i += (long)gridDim.x * kPrepThreads) {
    const uint4 raw = __ldg(reinterpret_cast<const uint4*>(s) + i);
    const T* e = reinterpret_cast<const T*>(&raw);
    float v[VEC];
#pragma unroll
    for (int k = 0; k < VEC; ++k) v[k] = to_f32<T>(e[k]);
    if (gain != nullptr) {
#pragma unroll
      for (int k = 0; k < VEC; k += 4) {
        const float4 g = __ldg(reinterpret_cast<const float4*>(gain + i * VEC + k));
        v[k] *= g.x;
        v[k + 1] *= g.y;
        v[k + 2] *= g.z;
        v[k + 3] *= g.w;
      }
    }
#pragma unroll
    for (int k = 0; k < VEC; k += 4) {
      reinterpret_cast<float4*>(d + i * VEC + k)[0] = make_float4(v[k], v[k + 1], v[k + 2], v[k + 3]);
      fs += (v[k] + v[k + 1]) + (v[k + 2] + v[k + 3]);
      fss += (v[k] * v[k] + v[k + 1] * v[k + 1]) + (v[k + 2] * v[k + 2] + v[k + 3] * v[k + 3]);
    }
    if (++folded == 16) {  // fp32 partials folded into double every 16 vectors: cheap inner loop, ~1e-7 error
      ds += (double)fs;
      dss += (double)fss;
      fs = fss = 0.f;
      folded = 0;
    }
  }
  for (long i = nvec * VEC + (long)blockIdx.x * kPrepThreads + threadIdx.x; i < n; i += (long)gridDim.x * kPrepThreads) {
    float v = to_f32<T>(s[i]);
    if (gain != nullptr) v *= __ldg(gain + i);
    d[i] = v;
    fs += v;
    fss += v * v;
  }
  ds += (double)fs;
  dss += (double)fss;
  if (moments != nullptr) {
    ds = warp_sum(ds);
    dss = warp_sum(dss);
    if ((threadIdx.x & 31) == 0) {
      atomicAdd(moments + 2 * f, ds);
      atomicAdd(moments + 2 * f + 1, dss);
    }
  }
}

// hot pixels of frame f: |v - mean_f| > threshold * std_f (population std, like np.std) -> list entries
// {flat index inside the stack, replacement value}; the replacement is one of the up to 8 neighbours of the ORIGINAL
// frame, picked by a hash of the pixel position (the reference draws it with np.random.choice: statistically the same,
// reproducible here)
struct HotPixel {
  long index;
  float value;
  int frame;
};

__device__ __forceinline__ unsigned hash3(unsigned a, unsigned b, unsigned c) {
  unsigned h = a * 0x9E3779B1u ^ (b + 0x7F4A7C15u) * 0x85EBCA77u ^ (c + 0x165667B1u) * 0xC2B2AE3Du;
  h ^= h >> 15;
  h *= 0x2C1B3C6Du;
  h ^= h >> 12;
  h *= 0x297A2D39u;
  h ^= h >> 15;
  return h;
}

__global__ void __launch_bounds__(kPrepThreads)
find_hot_pixels_kernel(const float* __restrict__ stack, int h, int w, const double* __restrict__ moments, float threshold,
                       HotPixel* __restrict__ list, int capacity, int* __restrict__ count) {
  const int f = blockIdx.y;
  const long n = (long)h * w;
  const double mean_d = moments[2 * f] / (double)n;
  const double var = moments[2 * f + 1] / (double)n - mean_d * mean_d;
  const float mean = (float)mean_d, limit = threshold * (float)sqrt(var > 0.0 ? var : 0.0);
  const float* frame = stack + (long)f * n;
  for (long i = (long)blockIdx.x * kPrepThreads + threadIdx.x; i < n; i += (long)gridDim.x * kPrepThreads) {
    const float v = __ldg(frame + i);
    if (v > mean + limit || v < mean - limit) {
      const int y = (int)(i / w), x = (int)(i - (long)y * w);
      const int y0 = max(0, y - 1), y1 = min(h - 1, y + 1), x0 = max(0, x - 1), x1 = min(w - 1, x + 1);
      const int cols = x1 - x0 + 1, cells = (y1 - y0 + 1) * cols;  // neighbourhood incl. the pixel itself
      if (cells > 1) {
        int pick = (int)(hash3((unsigned)f, (unsigned)y, (unsigned)x) % (unsigned)(cells - 1));
        const int self = (y - y0) * cols + (x - x0);
        if (pick >= self) ++pick;  // skip the hot pixel itself
        const float rep = __ldg(frame + (long)(y0 + pick / cols) * w + x0 + pick % cols);
        const int slot = atomicAdd(count, 1);
        if (slot < capacity) {
          HotPixel hp;
          hp.index = (long)f * n + i;
          hp.value = rep;
          hp.frame = f;
          list[slot] = hp;
        }
      }
    }
  }
}

// stack[index] = value for every list entry; moments[frame].sum follows the replacement (for the mean removal)
__global__ void apply_hot_pixels_kernel(float* __restrict__ stack, const HotPixel* __restrict__ list, int capacity,
                                        const int* __restrict__ count, double* __restrict__ moments) {
  const int n = min(*count, capacity);
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const HotPixel hp = list[i];
    const float old = stack[hp.index];
    stack[hp.index] = hp.value;
    atomicAdd(moments + 2 * hp.frame, (double)hp.value - (double)old);
  }
}

// frame -= mean(frame)  (set_frames_mean_zero), means from the moments
__global__ void __launch_bounds__(kPrepThreads)
subtract_frame_means_kernel(float* __restrict__ stack, long n, const double* __restrict__ moments) {
  const int f = blockIdx.y;
  const float mean = (float)(moments[2 * f] / (double)n);
  float* frame = stack + (long)f * n;
  if (((reinterpret_cast<uintptr_t>(frame)) & 15) == 0 && n % 4 == 0) {
    float4* p = reinterpret_cast<float4*>(frame);
    for (long i = (long)blockIdx.x * kPrepThreads + threadIdx.x; i < n / 4; i += (long)gridDim.x * kPrepThreads) {
      float4 v = p[i];
      v.x -= mean;
      v.y -= mean;
      v.z -= mean;
      v.w -= mean;
      p[i] = v;
    }
  } else {
    for (long i = (long)blockIdx.x * kPrepThreads + threadIdx.x; i < n; i += (long)gridDim.x * kPrepThreads) frame[i] -= mean;
  }
}

// frames whose loads one thread keeps in flight before it adds them (16 B each on the vector path)
constexpr int kGroupUnroll = 4;

__device__ __forceinline__ float4 add_rn(float4 a, float4 b) {
  return make_float4(__fadd_rn(a.x, b.x), __fadd_rn(a.y, b.y), __fadd_rn(a.z, b.z), __fadd_rn(a.w, b.w));
}
__device__ __forceinline__ float add_rn(float a, float b) { return __fadd_rn(a, b); }

// dst[g][i] = src[first_g][i] + src[first_g + 1][i] + ... (left to right, one rounding per add): group g holds frames
// g * group_size .. and the last group also takes the t % group_size leftovers.  One thread owns one element (a float4
// on the vector path) of one group; it issues kGroupUnroll frames' loads before adding them in ascending order.
template <typename V>
__global__ void __launch_bounds__(kPrepThreads)
group_frames_kernel(const V* __restrict__ src, long n, int t, int group_size, int n_groups, V* __restrict__ dst) {
  const int g = blockIdx.y;
  const long i = (long)blockIdx.x * kPrepThreads + threadIdx.x;
  if (i >= n) return;
  const int first = g * group_size;
  const int count = (g == n_groups - 1) ? t - first : group_size;
  const V* p = src + (long)first * n + i;
  V acc = __ldg(p);
  int f = 1;
  for (; f + kGroupUnroll <= count; f += kGroupUnroll) {
    V v[kGroupUnroll];
#pragma unroll
    for (int k = 0; k < kGroupUnroll; ++k) v[k] = __ldg(p + (long)(f + k) * n);
#pragma unroll
    for (int k = 0; k < kGroupUnroll; ++k) acc = add_rn(acc, v[k]);
  }
  for (; f < count; ++f) acc = add_rn(acc, __ldg(p + (long)f * n));
  dst[(long)g * n + i] = acc;
}

int blocks_per_frame(int t) {
  int b = (148 * 8 + t - 1) / t;
  return b < 1 ? 1 : b;
}

}  // namespace

// src (t, n) in its native type (dtype 0 uint8, 1 uint16, 2 int16, 3 float16, 4 float32, 5 int8) -> dst (t, n) fp32, times
// gain (n) when given; moments (t, 2) double = per-frame {sum, sum of squares} of the result (nullable; zeroed here)
TMC_API int tmc_convert_stack(const void* src, int dtype, int t, long n, const float* gain, float* dst, double* moments,
                              cudaStream_t stream) {
  TMC_CHECK_ARG(src && dst && t >= 1 && n >= 1, "convert_stack: bad arguments");
  TMC_CHECK_ARG(t <= kMaxGridYZ, "convert_stack: at most %d frames per call, got %d", kMaxGridYZ, t);
  TMC_CHECK_ARG(dtype >= 0 && dtype <= 5,
                "convert_stack: dtype must be 0 (uint8), 1 (uint16), 2 (int16), 3 (float16), 4 (float32) or 5 (int8)");
  if (moments) TMC_CUDA(cudaMemsetAsync(moments, 0, sizeof(double) * 2 * (size_t)t, stream));
  dim3 grid(blocks_per_frame(t), t);
  switch (dtype) {
    case 0: TMC_TIMED("convert_stack_kernel", stream, convert_stack_kernel<unsigned char><<<grid, kPrepThreads, 0, stream>>>((const unsigned char*)src, n, gain, dst, moments)); break;
    case 1: TMC_TIMED("convert_stack_kernel", stream, convert_stack_kernel<unsigned short><<<grid, kPrepThreads, 0, stream>>>((const unsigned short*)src, n, gain, dst, moments)); break;
    case 2: TMC_TIMED("convert_stack_kernel", stream, convert_stack_kernel<short><<<grid, kPrepThreads, 0, stream>>>((const short*)src, n, gain, dst, moments)); break;
    case 3: TMC_TIMED("convert_stack_kernel", stream, convert_stack_kernel<__half><<<grid, kPrepThreads, 0, stream>>>((const __half*)src, n, gain, dst, moments)); break;
    case 5: TMC_TIMED("convert_stack_kernel", stream, convert_stack_kernel<signed char><<<grid, kPrepThreads, 0, stream>>>((const signed char*)src, n, gain, dst, moments)); break;
    default: TMC_TIMED("convert_stack_kernel", stream, convert_stack_kernel<float><<<grid, kPrepThreads, 0, stream>>>((const float*)src, n, gain, dst, moments)); break;
  }
  TMC_CHECK_LAUNCH("tmc_convert_stack");
  return TMC_OK;
}

// bytes of the hot-pixel list for `capacity` entries (+ the counter)
TMC_API long tmc_hot_pixel_workspace_bytes(int capacity) { return (long)capacity * (long)sizeof(HotPixel) + 16; }

// remove_hot_pixels (examples/ttMotion.py:125-178): stack (t, h, w) fp32 in place; moments (t, 2) double of the stack
// (tmc_convert_stack) on entry, kept consistent with the replacements on exit; pixels further than threshold population
// standard deviations from their frame's mean are replaced by one of their neighbours.  hot_count (device int, nullable
// -> inside workspace) receives the number found; at most `capacity` are replaced.
TMC_API int tmc_remove_hot_pixels(float* stack, int t, int h, int w, double* moments, float threshold, int capacity,
                                  void* workspace, int* hot_count, cudaStream_t stream) {
  TMC_CHECK_ARG(stack && moments && workspace && t >= 1 && h >= 1 && w >= 1 && capacity >= 1 && threshold > 0.f,
                "remove_hot_pixels: bad arguments");
  TMC_CHECK_ARG(t <= kMaxGridYZ, "remove_hot_pixels: at most %d frames per call, got %d", kMaxGridYZ, t);
  int* count = reinterpret_cast<int*>(workspace);
  HotPixel* list = reinterpret_cast<HotPixel*>(reinterpret_cast<char*>(workspace) + 16);
  TMC_CUDA(cudaMemsetAsync(count, 0, sizeof(int), stream));
  dim3 grid(blocks_per_frame(t), t);
  TMC_TIMED("find_hot_pixels_kernel", stream, find_hot_pixels_kernel<<<grid, kPrepThreads, 0, stream>>>(stack, h, w, moments, threshold, list, capacity, count));
  TMC_TIMED("apply_hot_pixels_kernel", stream, apply_hot_pixels_kernel<<<64, 256, 0, stream>>>(stack, list, capacity, count, moments));
  if (hot_count) TMC_CUDA(cudaMemcpyAsync(hot_count, count, sizeof(int), cudaMemcpyDeviceToDevice, stream));
  TMC_CHECK_LAUNCH("tmc_remove_hot_pixels");
  return TMC_OK;
}

// set_frames_mean_zero (examples/ttMotion.py:180-202): every frame minus its own mean (moments[f].sum / n), in place
TMC_API int tmc_subtract_frame_means(float* stack, int t, long n, const double* moments, cudaStream_t stream) {
  TMC_CHECK_ARG(stack && moments && t >= 1 && n >= 1, "subtract_frame_means: bad arguments");
  TMC_CHECK_ARG(t <= kMaxGridYZ, "subtract_frame_means: at most %d frames per call, got %d", kMaxGridYZ, t);
  dim3 grid(blocks_per_frame(t), t);
  TMC_TIMED("subtract_frame_means_kernel", stream, subtract_frame_means_kernel<<<grid, kPrepThreads, 0, stream>>>(stack, n, moments));
  TMC_CHECK_LAUNCH("tmc_subtract_frame_means");
  return TMC_OK;
}

// frame grouping: movie (t, h, w) -> groups (t / frame_group, h, w), sums of frame_group consecutive frames, the last
// group also taking the t % frame_group leftover frames.  Each sum is x[first], then x[f] added in ascending order with
// one fp32 rounding per add.  float4 loads when both pointers are 16-byte aligned and h * w % 4 == 0, scalar otherwise.
TMC_API int tmc_group_frames(const float* movie, int t, int h, int w, int frame_group, float* groups, cudaStream_t stream) {
  TMC_CHECK_ARG(movie && groups, "group_frames: null pointer");
  TMC_CHECK_ARG(t >= 1 && h >= 1 && w >= 1, "group_frames: bad movie shape (%d, %d, %d)", t, h, w);
  TMC_CHECK_ARG(frame_group >= 1, "group_frames: frame_group must be >= 1, got %d", frame_group);
  const int n_groups = t / frame_group;
  TMC_CHECK_ARG(n_groups >= 2 && n_groups <= 65535,
                "group_frames: %d frames in groups of %d give %d groups, need 2 .. 65535", t, frame_group, n_groups);
  const long n = (long)h * w;
  const bool vec = n % 4 == 0 && ((reinterpret_cast<uintptr_t>(movie) | reinterpret_cast<uintptr_t>(groups)) & 15) == 0;
  if (vec) {
    dim3 grid(tmc_div_up(n / 4, kPrepThreads), n_groups);
    TMC_TIMED("group_frames_kernel", stream, group_frames_kernel<float4><<<grid, kPrepThreads, 0, stream>>>(
        reinterpret_cast<const float4*>(movie), n / 4, t, frame_group, n_groups, reinterpret_cast<float4*>(groups)));
  } else {
    dim3 grid(tmc_div_up(n, kPrepThreads), n_groups);
    TMC_TIMED("group_frames_kernel", stream, group_frames_kernel<float><<<grid, kPrepThreads, 0, stream>>>(
        movie, n, t, frame_group, n_groups, groups));
  }
  TMC_CHECK_LAUNCH("tmc_group_frames");
  return TMC_OK;
}

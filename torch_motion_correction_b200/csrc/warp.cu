// Deformation-field warp of a movie stack: per-pixel bicubic lookup of the per-frame shift
// lattice (reflection padding) followed by a bicubic gather of the frame (border-clamped
// taps, zero outside), either written as a (t,h,w) stack or accumulated over frames into one
// (h,w) sum without materialising the warped stack, or accumulated into several frame-weighted (h,w) sums at once
// (tmc_warp_lattice_sums: half-set and low-rank dose-weighted sums).
//
// Replaces the reference's correct_motion.py:81-185 (`_correct_frame`, `get_pixel_shifts`) and
// torch_image_interpolation.sample_image_2d / F.grid_sample(bicubic, align_corners=True)
// underneath it (SURVEY.md Appendix A.2, quirk Q17).  The fp32 coordinate round trip
// pixel -> [-1,1] -> pixel of grid_sample is reproduced operation by operation (no FMA
// contraction on that chain) because it alone costs ~3.5e-5 relative L2 otherwise.
#include "common.cuh"
#include <stdlib.h>

namespace {

constexpr float kA = -0.75f;  // Keys cubic convolution parameter used by ATen's bicubic

// ATen get_cubic_upsample_coefficients
__device__ __forceinline__ void cubic_weights(float t, float (&w)[4]) {
  // ((A x - 5A) x + 8A) x - 4A   and   ((A + 2) x - (A + 3)) x x + 1, three FMAs each
  float x = t + 1.0f;
  w[0] = fmaf(fmaf(fmaf(kA, x, -5.0f * kA), x, 8.0f * kA), x, -4.0f * kA);
  x = t;
  w[1] = fmaf(fmaf(kA + 2.0f, x, -(kA + 3.0f)) * x, x, 1.0f);
  x = 1.0f - t;
  w[2] = fmaf(fmaf(kA + 2.0f, x, -(kA + 3.0f)) * x, x, 1.0f);
  x = 2.0f - t;
  w[3] = fmaf(fmaf(fmaf(kA, x, -5.0f * kA), x, 8.0f * kA), x, -4.0f * kA);
}

// c / d for a divisor known per launch: q0 = c * (1/d), one Newton step on the residual.  Correctly
// rounded for all but vanishingly rare operands -- a third of the instructions of __fdiv_rn.
struct Divisor {
  float d, rcp;
};
__device__ __forceinline__ Divisor make_divisor(float d) {
  Divisor v;
  v.d = d;
  v.rcp = __frcp_rn(d);
  return v;
}
__device__ __forceinline__ float div_by(float c, const Divisor& v) {
  const float q0 = __fmul_rn(c, v.rcp);
  const float r = fmaf(-q0, v.d, c);
  return fmaf(r, v.rcp, q0);
}

// grid_round_trip with the divisor prepared once per thread
struct RoundTrip {
  Divisor denom;  // 0.5 n - 0.5
  float scale;    // n - 1
};
__device__ __forceinline__ RoundTrip make_round_trip(int n) {
  RoundTrip r;
  r.denom = make_divisor(__fsub_rn(__fmul_rn(0.5f, (float)n), 0.5f));
  r.scale = (float)(n - 1);
  return r;
}
__device__ __forceinline__ float round_trip(float c, const RoundTrip& r) {
  const float g = __fsub_rn(div_by(c, r.denom), 1.0f);
  return __fmul_rn(__fmul_rn(__fadd_rn(g, 1.0f), 0.5f), r.scale);
}

// array coordinate -> grid_sample [-1,1] -> unnormalised source coordinate, as fp32 ops:
//   g = c / (0.5*n - 0.5) - 1          (array_to_grid_sample, align_corners=True)
//   u = ((g + 1) / 2) * (n - 1)        (grid_sampler_unnormalize)
__device__ __forceinline__ float grid_round_trip(float c, int n) {
  float denom = __fsub_rn(__fmul_rn(0.5f, (float)n), 0.5f);
  float g = __fsub_rn(__fdiv_rn(c, denom), 1.0f);
  return __fmul_rn(__fmul_rn(__fadd_rn(g, 1.0f), 0.5f), (float)(n - 1));
}

// ATen reflect_coordinates(align_corners=True) + clip, on an integer index
__device__ __forceinline__ int reflect_index(int i, int n) {
  if (n <= 1) return 0;
  int span = n - 1;
  int a = i < 0 ? -i : i;
  int flips = a / span;
  int extra = a - flips * span;
  int r = (flips & 1) ? span - extra : extra;
  return min(max(r, 0), n - 1);
}

struct LatticeAxis {
  int j[4];    // reflected tap indices
  float w[4];  // cubic weights
  int i0;      // floor index (for "same taps" tests)
};

// lattice lookup coordinate of pixel index p along an axis of image length n, lattice length L
// (correct_motion.py:162-172): q = (p / (n-1)) * (L-1), then the grid_sample round trip.
__device__ __forceinline__ LatticeAxis lattice_axis(int p, int n, int L) {
  LatticeAxis a;
  float q = __fmul_rn(__fdiv_rn((float)p, (float)(n - 1)), (float)(L - 1));
  float u = grid_round_trip(q, L);
  float f = floorf(u);
  cubic_weights(__fsub_rn(u, f), a.w);
  a.i0 = (int)f;
#pragma unroll
  for (int k = 0; k < 4; ++k) a.j[k] = reflect_index(a.i0 - 1 + k, L);
  return a;
}

struct ImageAxis {
  int j[4];
  float w[4];
  bool inside;
};

// sampling coordinate c = p + shift along an axis of length n (sample_image_2d semantics)
__device__ __forceinline__ ImageAxis image_axis(float c, int n) {
  ImageAxis a;
  a.inside = (c >= 0.0f) && (c <= (float)(n - 1));
  float u = grid_round_trip(c, n);
  float f = floorf(u);
  cubic_weights(__fsub_rn(u, f), a.w);
  // clamp in float first: a wild shift must not overflow the int conversion
  int i0 = (int)fminf(fmaxf(f, -4.0f), (float)(n + 4));
#pragma unroll
  for (int k = 0; k < 4; ++k) a.j[k] = min(max(i0 - 1 + k, 0), n - 1);
  return a;
}

__device__ __forceinline__ float gather_bicubic(const float* __restrict__ frame, int w, const ImageAxis& ay, const ImageAxis& ax) {
  float acc = 0.f;
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const float* row = frame + (long)ay.j[r] * w;
    float v = ax.w[0] * __ldg(row + ax.j[0]) + ax.w[1] * __ldg(row + ax.j[1]) + ax.w[2] * __ldg(row + ax.j[2]) +
              ax.w[3] * __ldg(row + ax.j[3]);
    acc += ay.w[r] * v;
  }
  return acc;
}

constexpr int kTileX = 128;      // threads along x
constexpr int kTileYGroups = 2;  // thread rows per CTA
constexpr int kRows = 4;         // vertically adjacent output pixels per thread
constexpr int kMinBlocks = 2;    // CTAs per SM that warp_lattice_kernel's register budget must allow

// Stage 1: interpolate every lattice row along x once per (frame, channel, lattice row, image
// column): RX[f][ch][a][x] = sum_b wx_b(x) * L[f][ch][a][jx_b(x)].  Same x-then-y order as ATen.
// pad == 1: every frame gets lh + 3 rows of (channel y, channel x) row pairs, row p holding lattice row reflect(p - 1) --
// the reflection padding of the y taps materialised, so that the 4 taps of a pixel are always 4 consecutive rows
// (i0 .. i0 + 3): layout (T, lh + 3, 2, W).
constexpr int kRxPad = 3;
__global__ void lattice_xinterp_kernel(const float* __restrict__ lattice, int T, int lh, int lw, int W, float* __restrict__ rx,
                                       int pad) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  if (x >= W) return;
  const LatticeAxis lx = lattice_axis(x, W, lw);
  const int lhp = lh + kRxPad * pad;
  const long rows = (long)T * 2 * lhp;
  for (long r = blockIdx.y; r < rows; r += gridDim.y) {
    // pad == 0: rows ordered (frame, channel, lattice row); pad == 1: (frame, padded lattice row, channel)
    long plane;
    int a;
    if (pad) {
      const long fr = r / (2 * lhp);
      const int rem = (int)(r - fr * 2 * lhp);
      plane = fr * 2 + (rem & 1);
      a = reflect_index((rem >> 1) - 1, lh);
    } else {
      plane = r / lhp;
      a = (int)(r - plane * lhp);
    }
    const float* p = lattice + (plane * lh + a) * lw;
    rx[r * W + x] = lx.w[0] * __ldg(p + lx.j[0]) + lx.w[1] * __ldg(p + lx.j[1]) + lx.w[2] * __ldg(p + lx.j[2]) +
                    lx.w[3] * __ldg(p + lx.j[3]);
  }
}

__device__ __forceinline__ float2 f2(float a, float b) { return make_float2(a, b); }
__device__ __forceinline__ float2 dup(float a) { return make_float2(a, a); }

// ATen get_cubic_upsample_coefficients on two fractions at once (.x = y axis, .y = x axis), same FMA chains
__device__ __forceinline__ void cubic_weights2(float2 t, float2 (&w)[4]) {
  const float2 A = dup(kA), m5A = dup(-5.0f * kA), p8A = dup(8.0f * kA), m4A = dup(-4.0f * kA);
  const float2 A2 = dup(kA + 2.0f), mA3 = dup(-(kA + 3.0f)), one = dup(1.0f);
  float2 x = __fadd2_rn(t, one);
  w[0] = __ffma2_rn(__ffma2_rn(__ffma2_rn(A, x, m5A), x, p8A), x, m4A);
  w[1] = __ffma2_rn(__fmul2_rn(__ffma2_rn(A2, t, mA3), t), t, one);
  x = __ffma2_rn(t, dup(-1.0f), one);  // 1 - t, one rounding
  w[2] = __ffma2_rn(__fmul2_rn(__ffma2_rn(A2, x, mA3), x), x, one);
  x = __ffma2_rn(t, dup(-1.0f), dup(2.0f));  // 2 - t
  w[3] = __ffma2_rn(__ffma2_rn(__ffma2_rn(A, x, m5A), x, p8A), x, m4A);
}

// border / outside pixels (grid_sample padding_mode="border" taps, zero outside): the generic scalar path
__device__ __noinline__ float gather_border(const float* __restrict__ frame, int H, int W, float cy, float cx) {
  if (!(cy >= 0.0f && cy <= (float)(H - 1) && cx >= 0.0f && cx <= (float)(W - 1))) return 0.f;
  const ImageAxis ay = image_axis(cy, H), ax = image_axis(cx, W);
  return gather_bicubic(frame, W, ay, ax);
}

// One output pixel over all frames on the generic scalar path (threads whose rows straddle a lattice cell)
template <bool WRITE_STACK, bool NORMALISE>
__device__ __noinline__ float warp_pixel_generic(const float* __restrict__ image, int T, int H, int W, const float* __restrict__ rx,
                                                 int lh, float inv_px, float mean, float inv_std, float* __restrict__ out_stack,
                                                 int x, int y) {
  const LatticeAxis a = lattice_axis(y, H, lh);
  const size_t rx_plane = (size_t)(lh + kRxPad) * W;  // (T, lh + 3, 2, W): lattice row j lives in padded row j + 1
  float acc = 0.f;
  for (int f = 0; f < T; ++f) {
    const float* Ry = rx + (size_t)f * 2 * rx_plane + x + 2 * W;
    const float* Rx = Ry + W;
    float sy = a.w[0] * __ldg(Ry + (size_t)a.j[0] * 2 * W), sx = a.w[0] * __ldg(Rx + (size_t)a.j[0] * 2 * W);
#pragma unroll
    for (int k = 1; k < 4; ++k) {
      sy = fmaf(a.w[k], __ldg(Ry + (size_t)a.j[k] * 2 * W), sy);
      sx = fmaf(a.w[k], __ldg(Rx + (size_t)a.j[k] * 2 * W), sx);
    }
    const float cy = __fadd_rn((float)y, __fmul_rn(sy, inv_px));
    const float cx = __fadd_rn((float)x, __fmul_rn(sx, inv_px));
    float v = gather_border(image + (size_t)f * H * W, H, W, cy, cx);
    if (NORMALISE) v = (v - mean) * inv_std;
    if (WRITE_STACK) out_stack[((size_t)f * H + y) * W + x] = v;
    acc += v;
  }
  return acc;
}

// ---- frame-weighted sums: out_sums[s] = sum_f weights[s][f] * warped frame f --------------------------------------------
// Per sum, a thread keeps the accumulators of its kRows (= 4) pixels as one float4 in thread-private shared memory
// (acc[s * stride]): up to kMaxSums of them would not fit the 128-register budget of the warp kernels.  With a weight of
// exactly 1, fmaf(1, v, a) == a + v, so an all-ones row reproduces the plain frame sum bit for bit.
constexpr int kMaxSums = 19;  // per launch (tmc_warp_lattice_sums); the caller splits larger requests into passes

__device__ __forceinline__ void zero_sums(float4* acc, int stride, int n_sums) {
  for (int s = 0; s < n_sums; ++s) acc[s * stride] = make_float4(0.f, 0.f, 0.f, 0.f);
}
__device__ __forceinline__ void accumulate_sums(float4* acc, int stride, const float* __restrict__ weights, int T, int f,
                                                int n_sums, const float (&v)[4]) {
  const float* wf = weights + f;
  for (int s = 0; s < n_sums; ++s, wf += T, acc += stride) {
    const float ws = __ldg(wf);
    float4 a = *acc;
    a.x = fmaf(ws, v[0], a.x);
    a.y = fmaf(ws, v[1], a.y);
    a.z = fmaf(ws, v[2], a.z);
    a.w = fmaf(ws, v[3], a.w);
    *acc = a;
  }
}
__device__ __forceinline__ void store_sums(const float4* acc, int stride, int n_sums, float* __restrict__ out, int H, int W,
                                           int x, int y_base, int y_end) {
  for (int s = 0; s < n_sums; ++s) {
    const float4 a = acc[s * stride];
    const float v[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
    for (int r = 0; r < 4; ++r)
      if (y_base + r < y_end) out[((size_t)s * H + y_base + r) * W + x] = v[r];
  }
}

// warp_pixel_generic for the weighted sums: acc points at the pixel's component of the thread's float4 of sum 0
__device__ __noinline__ void warp_pixel_generic_sums(const float* __restrict__ image, int T, int H, int W,
                                                     const float* __restrict__ rx, int lh, float inv_px,
                                                     const float* __restrict__ weights, int n_sums, float* acc, int stride,
                                                     int x, int y) {
  const LatticeAxis a = lattice_axis(y, H, lh);
  const size_t rx_plane = (size_t)(lh + kRxPad) * W;
  for (int f = 0; f < T; ++f) {
    const float* Ry = rx + (size_t)f * 2 * rx_plane + x + 2 * W;
    const float* Rx = Ry + W;
    float sy = a.w[0] * __ldg(Ry + (size_t)a.j[0] * 2 * W), sx = a.w[0] * __ldg(Rx + (size_t)a.j[0] * 2 * W);
#pragma unroll
    for (int k = 1; k < 4; ++k) {
      sy = fmaf(a.w[k], __ldg(Ry + (size_t)a.j[k] * 2 * W), sy);
      sx = fmaf(a.w[k], __ldg(Rx + (size_t)a.j[k] * 2 * W), sx);
    }
    const float cy = __fadd_rn((float)y, __fmul_rn(sy, inv_px));
    const float cx = __fadd_rn((float)x, __fmul_rn(sx, inv_px));
    const float v = gather_border(image + (size_t)f * H * W, H, W, cy, cx);
    for (int s = 0; s < n_sums; ++s) acc[s * stride] = fmaf(__ldg(weights + (size_t)s * T + f), v, acc[s * stride]);
  }
}

// Stage 2: one thread = kRows vertically adjacent output pixels of one column; the coordinate chain of a pixel
// (Angstrom -> px, grid_sample round trip, cubic weights) runs on both axes at once as packed fp32x2 arithmetic
// and the 8 lattice taps of a frame are shared by the thread's pixels.
// measured alternatives on B200 (C2, fused sum): 4 rows per thread at 128 registers (2 CTAs per SM) 4.3 ms (4.1 ms with
// the shared tap rows); capped at 80 registers (3 CTAs per SM) 5.4 ms (4.9 ms with shared tap rows); 2 rows per thread 4.6-4.8 ms; uncapped registers (1 CTA per SM) 6.2 ms;
// prefetch.global.L2 of the next frame's rows +2 %
// (the weighted sums keep no sum in registers but load the weights: at 2 CTAs per SM they would spill, so 1)
template <bool WRITE_STACK, bool WRITE_SUM, bool NORMALISE, bool WEIGHTED = false>
__global__ void __launch_bounds__(kTileX* kTileYGroups, WEIGHTED ? 1 : kMinBlocks)
warp_lattice_kernel(const float* __restrict__ image, int T, int H, int W, const float* __restrict__ rx, int lh,
                    float pixel_spacing, const float* __restrict__ mean_std, float* __restrict__ out_stack,
                    float* __restrict__ out_sum, int accumulate_sum, int x_begin, int x_end, int y_begin, int y_end,
                    const float* __restrict__ weights, int n_sums, float* __restrict__ out_sums) {
  // the launch covers the output rectangle [x_begin, x_end) x [y_begin, y_end)
  const int x = x_begin + blockIdx.x * kTileX + threadIdx.x;
  const int y_base = y_begin + (blockIdx.y * kTileYGroups + threadIdx.y) * kRows;
  if (x >= x_end || y_base >= y_end) return;
  const int y_last = y_end - 1;
  // WEIGHTED: n_sums float4 accumulators per thread (dynamic shared memory, stride = threads per CTA)
  static_assert(!WEIGHTED || (kRows == 4 && !WRITE_STACK && !WRITE_SUM && !NORMALISE), "weighted sums: 4 rows, no other output");
  extern __shared__ float4 sums_smem[];
  constexpr int kSumStride = kTileX * kTileYGroups;
  float4* const sums_acc = sums_smem + threadIdx.y * kTileX + threadIdx.x;
  if constexpr (WEIGHTED) zero_sums(sums_acc, kSumStride, n_sums);

  // lattice taps along y: rows of RX (offsets in floats) and duplicated weights per pixel
  int jy[4];
  float2 wy[kRows][4];
  bool same_cell = true;
  {
    const LatticeAxis a0 = lattice_axis(y_base, H, lh);
#pragma unroll
    for (int k = 0; k < 4; ++k) jy[k] = (a0.j[k] + 1) * 2 * W;  // (T, lh + 3, 2, W): lattice row j lives in padded row j + 1
#pragma unroll
    for (int r = 0; r < kRows; ++r) {
      const LatticeAxis a = lattice_axis(min(y_base + r, y_last), H, lh);
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        wy[r][k] = dup(a.w[k]);
        same_cell = same_cell && (a.j[k] == a0.j[k]);
      }
    }
  }
  float mean = 0.f, inv_std = 1.f;
  if (NORMALISE) {
    mean = __ldg(mean_std);
    inv_std = 1.0f / __ldg(mean_std + 1);
  }
  float acc[kRows];
#pragma unroll
  for (int r = 0; r < kRows; ++r) acc[r] = 0.f;
  if (!same_cell) {
    // the rows of this thread straddle a lattice cell (warp-uniform, ~kRows in every H / lh rows)
    if constexpr (WEIGHTED) {
      for (int r = 0; r < kRows && y_base + r < y_end; ++r)
        warp_pixel_generic_sums(image, T, H, W, rx, lh, 1.0f / pixel_spacing, weights, n_sums,
                                reinterpret_cast<float*>(sums_acc) + r, 4 * kSumStride, x, y_base + r);
      store_sums(sums_acc, kSumStride, n_sums, out_sums, H, W, x, y_base, y_end);
      return;
    }
    for (int r = 0; r < kRows; ++r) {
      const int y = y_base + r;
      if (y >= y_end) break;
      const float a = warp_pixel_generic<WRITE_STACK, NORMALISE>(image, T, H, W, rx, lh, 1.0f / pixel_spacing, mean, inv_std,
                                                                   out_stack, x, y);
      if (WRITE_SUM) {
        float* o = out_sum + (long)y * W + x;
        *o = accumulate_sum ? (*o + a) : a;
      }
    }
    return;
  }

  // grid_sample round trip constants, .x = y axis (H), .y = x axis (W)
  const float dy = __fsub_rn(__fmul_rn(0.5f, (float)H), 0.5f), dx = __fsub_rn(__fmul_rn(0.5f, (float)W), 0.5f);
  const float2 nden = f2(-dy, -dx), rcp = f2(__frcp_rn(dy), __frcp_rn(dx));
  const float2 scale = f2((float)(H - 1), (float)(W - 1));
  const float2 inv_px = dup(1.0f / pixel_spacing);
  const float xf = (float)x;
  // all loads are (CTA-uniform 64-bit base) + (32-bit offset): no per-thread 64-bit pointer arithmetic
  const unsigned rx_plane = (unsigned)(lh + kRxPad) * (unsigned)W;
  unsigned jo[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) jo[k] = (unsigned)jy[k] + (unsigned)x;
  const float* rx_frame = rx;
  const float* frame = image;
  float2 Rn[4];  // (y shift, x shift) lattice rows at this column, loaded one frame ahead
#pragma unroll
  for (int k = 0; k < 4; ++k) Rn[k] = f2(__ldg(rx_frame + jo[k]), __ldg(rx_frame + W + jo[k]));
  for (int f = 0; f < T; ++f, frame += (size_t)H * W) {
    float2 R[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) R[k] = Rn[k];
    if (f + 1 < T) {
      rx_frame += 2 * (size_t)rx_plane;
#pragma unroll
      for (int k = 0; k < 4; ++k) Rn[k] = f2(__ldg(rx_frame + jo[k]), __ldg(rx_frame + W + jo[k]));
    }
    // stage A: sampling coordinates of the thread's pixels -> tap pointers and fractions
    float2 c[kRows], frac[kRows];
    const float* p[kRows];
    bool all_interior = true;
#pragma unroll
    for (int r = 0; r < kRows; ++r) {
      float2 s = __fmul2_rn(wy[r][0], R[0]);
      s = __ffma2_rn(wy[r][1], R[1], s);
      s = __ffma2_rn(wy[r][2], R[2], s);
      s = __ffma2_rn(wy[r][3], R[3], s);
      // Angstrom -> px, then pixel_grid + pixel_shifts (two roundings, like the reference)
      c[r] = __fadd2_rn(f2((float)min(y_base + r, y_last), xf), __fmul2_rn(s, inv_px));
      // grid_sample round trip: g = c / (0.5 n - 0.5) - 1 ; u = ((g + 1) / 2) (n - 1); the division as
      // q0 = c * rcp, one Newton step on the residual (Divisor above)
      const float2 q0 = __fmul2_rn(c[r], rcp);
      const float2 q = __ffma2_rn(__ffma2_rn(q0, nden, c[r]), rcp, q0);
      const float2 g = __fadd2_rn(q, dup(-1.0f));
      const float2 u = __fmul2_rn(__fmul2_rn(__fadd2_rn(g, dup(1.0f)), dup(0.5f)), scale);
      const float2 fl = f2(floorf(u.x), floorf(u.y));
      frac[r] = __ffma2_rn(fl, dup(-1.0f), u);
      const int iy = (int)fl.x, ix = (int)fl.y;
      // interior (implies 0 <= c <= n - 1): all 16 taps at immediate offsets of one pointer
      const bool interior = (unsigned)(iy - 1) <= (unsigned)(H - 4) && (unsigned)(ix - 1) <= (unsigned)(W - 4);
      all_interior = all_interior && interior;
      p[r] = frame + (interior ? (unsigned)((iy - 1) * W + (ix - 1)) : 0u);
    }
    float v[kRows];
    // vertically adjacent pixels whose sampling points are vertically adjacent too (same column of taps, consecutive
    // rows: the shifts differ by ~1e-3 px per row, so almost always) share their tap rows: kRows + 3 rows of 4 taps
    bool stacked = all_interior;
#pragma unroll
    for (int r = 1; r < kRows; ++r) stacked = stacked && (p[r] == p[0] + r * W);
    if (stacked) {
      float row[kRows + 3][4];
      {
        const float* q = p[0];
#pragma unroll
        for (int a = 0; a < kRows + 3; ++a, q += W)
#pragma unroll
          for (int b = 0; b < 4; ++b) row[a][b] = __ldg(q + b);
      }
#pragma unroll
      for (int r = 0; r < kRows; ++r) {
        float2 w[4];  // .x = weight along y, .y = weight along x
        cubic_weights2(frac[r], w);
        float2 r01 = __fmul2_rn(dup(w[0].y), f2(row[r][0], row[r + 1][0]));
        float2 r23 = __fmul2_rn(dup(w[0].y), f2(row[r + 2][0], row[r + 3][0]));
#pragma unroll
        for (int b = 1; b < 4; ++b) {
          r01 = __ffma2_rn(dup(w[b].y), f2(row[r][b], row[r + 1][b]), r01);
          r23 = __ffma2_rn(dup(w[b].y), f2(row[r + 2][b], row[r + 3][b]), r23);
        }
        const float2 t2 = __ffma2_rn(f2(w[2].x, w[3].x), r23, __fmul2_rn(f2(w[0].x, w[1].x), r01));
        v[r] = t2.x + t2.y;
      }
    } else if (all_interior) {
      // stage B: every tap of every pixel in flight at once; stage C: weights (while the loads fly) and the sums
      float tap[kRows][4][4];
#pragma unroll
      for (int r = 0; r < kRows; ++r) {
        const float* row = p[r];
#pragma unroll
        for (int a = 0; a < 4; ++a, row += W)
#pragma unroll
          for (int b = 0; b < 4; ++b) tap[r][a][b] = __ldg(row + b);
      }
#pragma unroll
      for (int r = 0; r < kRows; ++r) {
        float2 w[4];  // .x = weight along y, .y = weight along x
        cubic_weights2(frac[r], w);
        // rows (0,1) and (2,3) as packed pairs
        float2 r01 = __fmul2_rn(dup(w[0].y), f2(tap[r][0][0], tap[r][1][0]));
        float2 r23 = __fmul2_rn(dup(w[0].y), f2(tap[r][2][0], tap[r][3][0]));
#pragma unroll
        for (int b = 1; b < 4; ++b) {
          r01 = __ffma2_rn(dup(w[b].y), f2(tap[r][0][b], tap[r][1][b]), r01);
          r23 = __ffma2_rn(dup(w[b].y), f2(tap[r][2][b], tap[r][3][b]), r23);
        }
        const float2 t2 = __ffma2_rn(f2(w[2].x, w[3].x), r23, __fmul2_rn(f2(w[0].x, w[1].x), r01));
        v[r] = t2.x + t2.y;
      }
    } else {
      // image border in reach: border-clamped taps / zero outside on the generic scalar path
#pragma unroll
      for (int r = 0; r < kRows; ++r) v[r] = gather_border(frame, H, W, c[r].x, c[r].y);
    }
#pragma unroll
    for (int r = 0; r < kRows; ++r) {
      const int y = y_base + r;
      if (y < y_end) {
        float o = v[r];
        if (NORMALISE) o = (o - mean) * inv_std;
        if (WRITE_STACK) out_stack[((size_t)f * H + y) * W + x] = o;
        if (WRITE_SUM) acc[r] += o;
      }
    }
    if constexpr (WEIGHTED) accumulate_sums(sums_acc, kSumStride, weights, T, f, n_sums, v);
  }
  if constexpr (WEIGHTED) store_sums(sums_acc, kSumStride, n_sums, out_sums, H, W, x, y_base, y_end);
  if (WRITE_SUM) {
#pragma unroll
    for (int r = 0; r < kRows; ++r) {
      const int y = y_base + r;
      if (y < y_end) {
        float* o = out_sum + (long)y * W + x;
        *o = accumulate_sum ? (*o + acc[r]) : acc[r];
      }
    }
  }
}

#include "warp_tma.cuh"

// ---- backward of the warp w.r.t. the shift lattice (correct_motion_two_grids, grad=True) ------------------
// d out / d shift = (1 / px) * sum_ab w'_a(t_y) w_b(t_x) tap_ab   (ATen grid_sampler_2d_backward, bicubic:
// gradient flows through the cubic coefficients only; clamped taps and the outside-zero mask carry none)

__device__ __forceinline__ void cubic_weights_grad(float t, float (&w)[4]) {
  // true derivatives d w_k / d t of cubic_weights (ATen's get_cubic_coefficients_grad stores the negatives
  // and subtracts them)
  float x = t + 1.0f;
  w[0] = (3.0f * kA * x - 10.0f * kA) * x + 8.0f * kA;
  x = t;
  w[1] = (3.0f * (kA + 2.0f) * x - 2.0f * (kA + 3.0f)) * x;
  x = 1.0f - t;
  w[2] = -(3.0f * (kA + 2.0f) * x - 2.0f * (kA + 3.0f)) * x;
  x = 2.0f - t;
  w[3] = -((3.0f * kA * x - 10.0f * kA) * x + 8.0f * kA);
}

// grad_rx[f][c][a][x] += grad_out[f][y][x] * d out / d s_c * wy_k(y)   for the 4 lattice rows a = jy_k(y)
__global__ void warp_lattice_backward_kernel(const float* __restrict__ image, int T, int H, int W, const float* __restrict__ rx,
                                             int lh, float pixel_spacing, const float* __restrict__ grad_out,
                                             float* __restrict__ grad_rx) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y;
  if (x >= W) return;
  const LatticeAxis ly = lattice_axis(y, H, lh);
  const RoundTrip rty = make_round_trip(H), rtx = make_round_trip(W);
  const float inv_px = 1.0f / pixel_spacing;
  const size_t rx_plane = (size_t)lh * W;
  for (int f = 0; f < T; ++f) {
    const float go = grad_out[((size_t)f * H + y) * W + x];
    if (go == 0.f) continue;
    const float* Ry = rx + (size_t)f * 2 * rx_plane + x;
    const float* Rx = Ry + rx_plane;
    float sy = 0.f, sx = 0.f;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      sy = fmaf(ly.w[k], __ldg(Ry + (size_t)ly.j[k] * W), sy);
      sx = fmaf(ly.w[k], __ldg(Rx + (size_t)ly.j[k] * W), sx);
    }
    const float cy = __fadd_rn((float)y, __fmul_rn(sy, inv_px));
    const float cx = __fadd_rn((float)x, __fmul_rn(sx, inv_px));
    if (!(cy >= 0.0f && cy <= (float)(H - 1) && cx >= 0.0f && cx <= (float)(W - 1))) continue;
    const float uy = round_trip(cy, rty), ux = round_trip(cx, rtx);
    const float fy = floorf(uy), fx = floorf(ux);
    float ay[4], ax[4], day[4], dax[4];
    cubic_weights(uy - fy, ay);
    cubic_weights(ux - fx, ax);
    cubic_weights_grad(uy - fy, day);
    cubic_weights_grad(ux - fx, dax);
    const int iy = (int)fy, ix = (int)fx;
    const float* frame = image + (size_t)f * H * W;
    float dvy = 0.f, dvx = 0.f;
#pragma unroll
    for (int a = 0; a < 4; ++a) {
      const float* p = frame + (size_t)min(max(iy - 1 + a, 0), H - 1) * W;
      float row = 0.f, drow = 0.f;
#pragma unroll
      for (int b = 0; b < 4; ++b) {
        const float tap = __ldg(p + min(max(ix - 1 + b, 0), W - 1));
        row = fmaf(ax[b], tap, row);
        drow = fmaf(dax[b], tap, drow);
      }
      dvy = fmaf(day[a], row, dvy);
      dvx = fmaf(ay[a], drow, dvx);
    }
    const float gy = go * dvy * inv_px, gx = go * dvx * inv_px;
    float* Gy = grad_rx + (size_t)f * 2 * rx_plane + x;
    float* Gx = Gy + rx_plane;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      atomicAdd(Gy + (size_t)ly.j[k] * W, gy * ly.w[k]);
      atomicAdd(Gx + (size_t)ly.j[k] * W, gx * ly.w[k]);
    }
  }
}

// grad_lattice[r][jx_b(x)] += wx_b(x) * grad_rx[r][x]   (transpose of lattice_xinterp_kernel)
__global__ void lattice_xinterp_backward_kernel(const float* __restrict__ grad_rx, long rows, int lw, int W,
                                                float* __restrict__ grad_lattice) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  if (x >= W) return;
  const LatticeAxis lx = lattice_axis(x, W, lw);
  for (long r = blockIdx.y; r < rows; r += gridDim.y) {
    const float g = grad_rx[r * W + x];
    if (g == 0.f) continue;
#pragma unroll
    for (int b = 0; b < 4; ++b) atomicAdd(grad_lattice + r * lw + lx.j[b], g * lx.w[b]);
  }
}

// (t, y, x) in [0,1]^3 of every lattice node, (T, lh, lw, 3), matching spline_lattice_kernel
__global__ void lattice_tyx_kernel(int T, int frame_offset, int total_frames, int lh, int lw, float* __restrict__ tyx) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long)T * lh * lw) return;
  const int ix = i % lw;
  const long r = i / lw;
  const int iy = r % lh;
  const int f = r / lh;
  tyx[3 * i] = linspace01(f + frame_offset, total_frames);
  tyx[3 * i + 1] = linspace01(iy, lh);
  tyx[3 * i + 2] = linspace01(ix, lw);
}

// get_pixel_shifts (correct_motion.py:132-185): (h, w, 2) px shifts of one lattice (2, lh, lw)
__global__ void pixel_shifts_kernel(const float* __restrict__ lattice, int lh, int lw, int H, int W, float pixel_spacing,
                                    float* __restrict__ out) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y;
  if (x >= W) return;
  const LatticeAxis lx = lattice_axis(x, W, lw);
  const LatticeAxis ly = lattice_axis(y, H, lh);
  const long plane = (long)lh * lw;
  float s[2];
#pragma unroll
  for (int ch = 0; ch < 2; ++ch) {
    float acc = 0.f;
#pragma unroll
    for (int a = 0; a < 4; ++a) {
      const float* p = lattice + ch * plane + (long)ly.j[a] * lw;
      float v = lx.w[0] * __ldg(p + lx.j[0]) + lx.w[1] * __ldg(p + lx.j[1]) + lx.w[2] * __ldg(p + lx.j[2]) +
                lx.w[3] * __ldg(p + lx.j[3]);
      acc += ly.w[a] * v;
    }
    s[ch] = __fdiv_rn(acc, pixel_spacing);
  }
  float2* o = reinterpret_cast<float2*>(out) + (long)y * W + x;
  *o = make_float2(s[0], s[1]);
}

// correct_motion_slow (correct_motion.py:371-427) given per-pixel shifts computed elsewhere:
// out[f](y,x) = bicubic(frame_f; y + shift_y, x + shift_x) with shifts (t, h, w, 2) in px
__global__ void warp_dense_shifts_kernel(const float* __restrict__ image, int T, int H, int W, const float* __restrict__ shifts,
                                         float* __restrict__ out_stack) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y;
  const int f = blockIdx.z;
  if (x >= W) return;
  const long i = ((long)f * H + y) * W + x;
  const float2 s = reinterpret_cast<const float2*>(shifts)[i];
  ImageAxis ay = image_axis(__fadd_rn((float)y, s.x), H);
  ImageAxis ax = image_axis(__fadd_rn((float)x, s.y), W);
  float v = 0.f;
  if (ay.inside && ax.inside) v = gather_bicubic(image + (long)f * H * W, W, ay, ax);
  out_stack[i] = v;
}

// normalised (t, y, x) coordinates of every pixel of frame f (correct_motion.py:401-409)
__global__ void pixel_tyx_kernel(int H, int W, int T, int frame_offset, int total_frames, float* __restrict__ tyx) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y;
  const int f = blockIdx.z;
  if (x >= W) return;
  float* o = tyx + (((long)f * H + y) * W + x) * 3;
  o[0] = linspace01(f + frame_offset, total_frames);
  o[1] = __fdiv_rn((float)y, (float)(H - 1));
  o[2] = __fdiv_rn((float)x, (float)(W - 1));
}

}  // namespace

TMC_API long tmc_warp_workspace_floats(int t, int w, int lh) { return (long)t * 2 * (lh + kRxPad) * w; }

// image (t,h,w); lattice (t,2,lh,lw) in Angstrom; mean_std nullable device float[2] (input affine
// (v - mean) / std applied to the warped value, zero outside); out_stack (t,h,w) nullable;
// out_sum (h,w) nullable; accumulate_sum != 0 adds to out_sum; workspace:
// tmc_warp_workspace_floats(t, w, lh) floats.
// shared by tmc_warp_lattice and tmc_warp_lattice_sums (weights != nullptr: the weighted sums, arguments validated)
static int warp_lattice_launch(const float* image, int t, int h, int w, const float* lattice, int lh, int lw,
                               float pixel_spacing, const float* mean_std, float* out_stack, float* out_sum,
                               int accumulate_sum, const float* weights, int n_sums, float* out_sums, float* workspace,
                               cudaStream_t stream) {
  {
    // every thread sets up its column's taps once (two divisions) and then walks over rows: few, long-lived CTAs
    long rows = (long)t * 2 * (lh + kRxPad);
    const int col_blocks = tmc_div_up(w, 128);
    long row_blocks = (148l * 8 + col_blocks - 1) / col_blocks;
    if (row_blocks > rows) row_blocks = rows;
    dim3 g1(col_blocks, (unsigned)row_blocks);
    TMC_TIMED("lattice_xinterp_kernel", stream, lattice_xinterp_kernel<<<g1, 128, 0, stream>>>(lattice, t, lh, lw, w, workspace, 1));
  }
  const bool s = out_stack != nullptr, a = out_sum != nullptr, n = mean_std != nullptr;
  if (tma::supported(image, workspace, t, h, w, lh)) {
    // frame tiles staged by TMA, one persistent CTA per SM
    CUtensorMap img_map, rx_map;
    const bool ok = tma::make_map_3d(&img_map, image, (uint64_t)w, (uint64_t)h, (uint64_t)t, tma::kBoxW, tma::kBoxH, 1) &&
                    tma::make_map_3d(&rx_map, workspace, (uint64_t)w, 2, (uint64_t)t * (lh + kRxPad), tma::kTX, 2,
                                     (uint32_t)tma::staged_lattice_rows(h, lh));
    if (ok && (!weights || (tma::kMaxSmemBytes - 128 - n_sums * tma::kConsumers * (int)sizeof(float4)) /
                                   tma::stage_bytes_for(tma::staged_lattice_rows(h, lh)) >= 2)) {
      tma::SumsParams prm;  // passed as tma::Params to all but the weighted instantiation
      prm.image = image;
      prm.T = t;
      prm.H = h;
      prm.W = w;
      prm.rx = workspace;
      prm.lh = lh;
      prm.rx_rows = tma::staged_lattice_rows(h, lh);
      prm.stage_bytes = tma::stage_bytes_for(prm.rx_rows);
      prm.n_stages = tma::stages_for(prm.rx_rows);
      prm.weights = weights;
      prm.n_sums = n_sums;
      prm.out_sums = out_sums;
      prm.acc_bytes = weights ? n_sums * tma::kConsumers * (int)sizeof(float4) : 0;
      if (weights) {  // the accumulators take shared memory from the ring
        const int n = (tma::kMaxSmemBytes - 128 - prm.acc_bytes) / prm.stage_bytes;
        if (n < prm.n_stages) prm.n_stages = n;
      }
      const size_t smem_bytes = (size_t)prm.acc_bytes + (size_t)prm.n_stages * prm.stage_bytes + 128;  // + alignment slack
      prm.pixel_spacing = pixel_spacing;
      prm.mean_std = mean_std;
      prm.out_stack = out_stack;
      prm.out_sum = out_sum;
      prm.accumulate_sum = accumulate_sum;
      prm.tiles_x = tmc_div_up(w, tma::kTX);
      prm.n_tiles = prm.tiles_x * tmc_div_up(h, tma::kTY);
      tma::fill_constants(prm);
      int dev_id = 0, sms = 148;
      TMC_CUDA(cudaGetDevice(&dev_id));
      TMC_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev_id));
      const int grid = prm.n_tiles < sms ? prm.n_tiles : sms;
#define LAUNCH_TMA(S, A, N)                                                                                                  \
  {                                                                                                                          \
    TMC_CUDA(cudaFuncSetAttribute(tma::warp_tma_kernel<S, A, N>, cudaFuncAttributeMaxDynamicSharedMemorySize,                 \
                                  tma::kMaxSmemBytes));                                                                      \
    tmc_timing_begin(stream);                                                                                                \
    tma::warp_tma_kernel<S, A, N><<<grid, tma::kThreads, smem_bytes, stream>>>(img_map, rx_map, prm);                         \
    tmc_timing_end("warp_tma_kernel", stream);                                                                               \
  }
      if (weights) {
        TMC_CUDA(cudaFuncSetAttribute(tma::warp_tma_kernel<false, false, false, true>,
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, tma::kMaxSmemBytes));
        tmc_timing_begin(stream);
        tma::warp_tma_kernel<false, false, false, true><<<grid, tma::kThreads, smem_bytes, stream>>>(img_map, rx_map, prm);
        tmc_timing_end("warp_tma_kernel_sums", stream);
      } else if (s && a && n) LAUNCH_TMA(true, true, true)
      else if (s && a) LAUNCH_TMA(true, true, false)
      else if (s && n) LAUNCH_TMA(true, false, true)
      else if (s) LAUNCH_TMA(true, false, false)
      else if (n) LAUNCH_TMA(false, true, true)
      else LAUNCH_TMA(false, true, false)
#undef LAUNCH_TMA
      tmc_count_launch();
      TMC_CHECK_LAUNCH("tmc_warp_lattice(tma)");
      return TMC_OK;
    }
  }
  {
    dim3 block(kTileX, kTileYGroups);
    dim3 grid(tmc_div_up(w, kTileX), tmc_div_up(h, kTileYGroups * kRows));
    if (weights) {
      const int smem = n_sums * kTileX * kTileYGroups * (int)sizeof(float4);
      TMC_CUDA(cudaFuncSetAttribute(warp_lattice_kernel<false, false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    smem));
      TMC_TIMED("warp_lattice_kernel_sums", stream,
                warp_lattice_kernel<false, false, false, true><<<grid, block, smem, stream>>>(
                    image, t, h, w, workspace, lh, pixel_spacing, nullptr, nullptr, nullptr, 0, 0, w, 0, h, weights, n_sums,
                    out_sums));
      TMC_CHECK_LAUNCH("tmc_warp_lattice_sums");
      return TMC_OK;
    }
    tmc_timing_begin(stream);
#define LAUNCH(S, A, N)                                                                                          \
  warp_lattice_kernel<S, A, N><<<grid, block, 0, stream>>>(image, t, h, w, workspace, lh, pixel_spacing, mean_std, \
                                                           out_stack, out_sum, accumulate_sum, 0, w, 0, h, nullptr, 0, nullptr)
    if (s && a && n) LAUNCH(true, true, true);
    else if (s && a) LAUNCH(true, true, false);
    else if (s && n) LAUNCH(true, false, true);
    else if (s) LAUNCH(true, false, false);
    else if (n) LAUNCH(false, true, true);
    else LAUNCH(false, true, false);
#undef LAUNCH
    tmc_timing_end("warp_lattice_kernel", stream);
    tmc_count_launch();
  }
  TMC_CHECK_LAUNCH("tmc_warp_lattice");
  return TMC_OK;
}

TMC_API int tmc_warp_lattice(const float* image, int t, int h, int w, const float* lattice, int lh, int lw,
                             float pixel_spacing, const float* mean_std, float* out_stack, float* out_sum,
                             int accumulate_sum, float* workspace, cudaStream_t stream) {
  TMC_CHECK_ARG(image && lattice && workspace, "warp_lattice: null pointer");
  TMC_CHECK_ARG(out_stack || out_sum, "warp_lattice: need out_stack and/or out_sum");
  TMC_CHECK_ARG(t >= 1 && h >= 2 && w >= 2 && lh >= 1 && lw >= 1, "warp_lattice: bad shape t=%d h=%d w=%d lattice=%dx%d", t,
                h, w, lh, lw);
  TMC_CHECK_ARG(pixel_spacing > 0.f, "warp_lattice: pixel_spacing must be > 0");
  TMC_CHECK_ARG((long)(lh + kRxPad) * w < (1l << 31), "warp_lattice: lattice rows x width overflows int");
  return warp_lattice_launch(image, t, h, w, lattice, lh, lw, pixel_spacing, mean_std, out_stack, out_sum, accumulate_sum,
                             nullptr, 0, nullptr, workspace, stream);
}

// out_sums (n_sums, h, w) = sum_f frame_weights[s][f] * (frame f warped as by tmc_warp_lattice); frame_weights (n_sums, t)
// f32 device; 1 <= n_sums <= 19 (kMaxSums); workspace: tmc_warp_workspace_floats(t, w, lh) floats.
TMC_API int tmc_warp_lattice_sums(const float* image, int t, int h, int w, const float* lattice, int lh, int lw,
                                  float pixel_spacing, const float* frame_weights, int n_sums, float* out_sums,
                                  float* workspace, cudaStream_t stream) {
  TMC_CHECK_ARG(image && lattice && frame_weights && out_sums && workspace, "warp_lattice_sums: null pointer");
  TMC_CHECK_ARG(n_sums >= 1 && n_sums <= kMaxSums, "warp_lattice_sums: n_sums=%d outside [1, %d] (split into passes)", n_sums,
                kMaxSums);
  TMC_CHECK_ARG(t >= 1 && h >= 2 && w >= 2 && lh >= 1 && lw >= 1, "warp_lattice_sums: bad shape t=%d h=%d w=%d lattice=%dx%d",
                t, h, w, lh, lw);
  TMC_CHECK_ARG(pixel_spacing > 0.f, "warp_lattice_sums: pixel_spacing must be > 0");
  TMC_CHECK_ARG((long)(lh + kRxPad) * w < (1l << 31), "warp_lattice_sums: lattice rows x width overflows int");
  return warp_lattice_launch(image, t, h, w, lattice, lh, lw, pixel_spacing, nullptr, nullptr, nullptr, 0, frame_weights,
                             n_sums, out_sums, workspace, stream);
}

TMC_API int tmc_pixel_shifts(const float* lattice, int lh, int lw, int h, int w, float pixel_spacing, float* out,
                             cudaStream_t stream) {
  TMC_CHECK_ARG(lattice && out && lh >= 1 && lw >= 1 && h >= 2 && w >= 2 && pixel_spacing > 0.f, "pixel_shifts: bad arguments");
  TMC_CHECK_ARG(h <= kMaxGridYZ, "pixel_shifts: at most %d rows, got %d", kMaxGridYZ, h);
  dim3 grid(tmc_div_up(w, 128), h);
  TMC_TIMED("pixel_shifts_kernel", stream, pixel_shifts_kernel<<<grid, 128, 0, stream>>>(lattice, lh, lw, h, w, pixel_spacing, out));
  TMC_CHECK_LAUNCH("tmc_pixel_shifts");
  return TMC_OK;
}

TMC_API int tmc_warp_dense_shifts(const float* image, int t, int h, int w, const float* shifts, float* out_stack,
                                  cudaStream_t stream) {
  TMC_CHECK_ARG(image && shifts && out_stack && t >= 1 && h >= 2 && w >= 2, "warp_dense_shifts: bad arguments");
  TMC_CHECK_ARG(t <= kMaxGridYZ && h <= kMaxGridYZ, "warp_dense_shifts: at most %d frames and rows, got (%d, %d)", kMaxGridYZ, t, h);
  dim3 grid(tmc_div_up(w, 128), h, t);
  TMC_TIMED("warp_dense_shifts_kernel", stream, warp_dense_shifts_kernel<<<grid, 128, 0, stream>>>(image, t, h, w, shifts, out_stack));
  TMC_CHECK_LAUNCH("tmc_warp_dense_shifts");
  return TMC_OK;
}

TMC_API int tmc_pixel_tyx(int h, int w, int t, int frame_offset, int total_frames, float* tyx, cudaStream_t stream) {
  TMC_CHECK_ARG(tyx && t >= 1 && h >= 2 && w >= 2 && total_frames >= t + frame_offset, "pixel_tyx: bad arguments");
  TMC_CHECK_ARG(t <= kMaxGridYZ && h <= kMaxGridYZ, "pixel_tyx: at most %d frames and rows, got (%d, %d)", kMaxGridYZ, t, h);
  dim3 grid(tmc_div_up(w, 128), h, t);
  TMC_TIMED("pixel_tyx_kernel", stream, pixel_tyx_kernel<<<grid, 128, 0, stream>>>(h, w, t, frame_offset, total_frames, tyx));
  TMC_CHECK_LAUNCH("tmc_pixel_tyx");
  return TMC_OK;
}

// Backward of tmc_warp_lattice w.r.t. the lattice: grad_out (t,h,w) -> grad_lattice (t,2,lh,lw) (zeroed here).
// workspace: 2 * tmc_warp_workspace_floats(t, w, lh) floats.
TMC_API int tmc_warp_lattice_backward(const float* image, int t, int h, int w, const float* lattice, int lh, int lw,
                                      float pixel_spacing, const float* grad_out, float* grad_lattice, float* workspace,
                                      cudaStream_t stream) {
  TMC_CHECK_ARG(image && lattice && grad_out && grad_lattice && workspace, "warp_lattice_backward: null pointer");
  TMC_CHECK_ARG(t >= 1 && h >= 2 && w >= 2 && lh >= 1 && lw >= 1 && pixel_spacing > 0.f, "warp_lattice_backward: bad arguments");
  TMC_CHECK_ARG(h <= kMaxGridYZ, "warp_lattice_backward: at most %d rows, got %d", kMaxGridYZ, h);
  const long rows = (long)t * 2 * lh;
  float* rx = workspace;
  float* grad_rx = workspace + rows * w;
  dim3 g1(tmc_div_up(w, 128), (unsigned)(rows < 4096 ? rows : 4096));
  TMC_TIMED("lattice_xinterp_kernel", stream, lattice_xinterp_kernel<<<g1, 128, 0, stream>>>(lattice, t, lh, lw, w, rx, 0));
  TMC_CUDA(cudaMemsetAsync(grad_rx, 0, sizeof(float) * (size_t)rows * w, stream));
  TMC_CUDA(cudaMemsetAsync(grad_lattice, 0, sizeof(float) * (size_t)rows * lw, stream));
  dim3 g2(tmc_div_up(w, 128), h);
  TMC_TIMED("warp_lattice_backward_kernel", stream, warp_lattice_backward_kernel<<<g2, 128, 0, stream>>>(image, t, h, w, rx, lh, pixel_spacing, grad_out, grad_rx));
  TMC_TIMED("lattice_xinterp_backward_kernel", stream, lattice_xinterp_backward_kernel<<<g1, 128, 0, stream>>>(grad_rx, rows, lw, w, grad_lattice));
  TMC_CHECK_LAUNCH("tmc_warp_lattice_backward");
  return TMC_OK;
}

// normalised (t, y, x) of every node of the (t, lh, lw) lattice: tyx (t, lh, lw, 3)
TMC_API int tmc_lattice_tyx(int t, int frame_offset, int total_frames, int lh, int lw, float* tyx, cudaStream_t stream) {
  TMC_CHECK_ARG(tyx && t >= 1 && lh >= 1 && lw >= 1 && frame_offset >= 0 && frame_offset + t <= total_frames,
                "lattice_tyx: bad arguments");
  const long n = (long)t * lh * lw;
  TMC_TIMED("lattice_tyx_kernel", stream, lattice_tyx_kernel<<<tmc_div_up(n, 128), 128, 0, stream>>>(t, frame_offset, total_frames, lh, lw, tyx));
  TMC_CHECK_LAUNCH("tmc_lattice_tyx");
  return TMC_OK;
}

// Band-limited 1024-point row transforms as four polyphase 256-point FFTs that live entirely inside one warp
// (included by fourier.cu inside its anonymous namespace; same contracts as rows_forward_p2<1024, MODE> and
// rows_inverse_argmax_p2<1024>).
//
// Only |k| < KX <= 128 of the 1024 row frequencies are ever needed (the band-pass keeps <= 128 / 1024 bins at the
// reference's default 10 Angstrom cut-off for pixel sizes up to 1.25 Angstrom).  With n = 4 m + q:
//   forward:  Z[k]     = sum_q W_1024^{q k} Y_q[k mod 256],   Y_q = DFT_256(z[4 m + q])
//   inverse:  x[4m+q]  = IDFT_256( Z[k] W_1024^{-q k} )[m]    (k <-> k mod 256 is one-to-one for |k| < 128)
// A 256-point DFT is 16 x 16: a thread owns 16 values, does a radix-16 butterfly in registers, the half-warp
// transposes through 16 x 17 complex words of shared memory (__syncwarp only) and a second radix-16 butterfly
// follows.  One warp = one row (pair): lane = (qh, j), the thread owns the sub-sequences q = 2 qh and 2 qh + 1
// (adjacent pixels: one 8-byte load per pair).  No block-wide barrier in the row loop, two shared-memory
// passes instead of six, and 15 % fewer flops than the 1024-point transform.
#pragma once

namespace poly {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr int kBuf = 16 * 17;              // transpose buffer of one half-warp (complex words)
constexpr int kWarpWords = 2 * kBuf + 256;  // + the row's Z[k] staging: [0, 128) k >= 0, [128, 256) k = -(i - 128)
// twiddle tables laid out so that the 16 lanes of a half-warp read consecutive words (no bank conflicts):
//   tw_step[k2][j] = W_256^{j k2} (between the two radix-16 steps), tw_comb[q - 1][kk] = W_1024^{q k}, k = kk or kk - 256
constexpr int kTableWords = 256 + 3 * 256;
constexpr size_t smem_bytes = (size_t)(kTableWords + kWarps * kWarpWords) * sizeof(float2);

// 256-point forward DFT over a half-warp: lane j holds v[r] = y[j + 16 r]; on return Y[j + 16 k1] = v[bitrev(k1)]
__device__ __forceinline__ void fft256_halfwarp(float2 (&v)[16], int j, float2* __restrict__ buf, const float2* __restrict__ tw_step) {
  tmcfft::fft_reg<16>(v);
#pragma unroll
  for (int k2 = 0; k2 < 16; ++k2) {
    float2 u = v[tmcfft::bitrev<16>(k2)];
    if (k2 > 0) u = cmul(u, tw_step[k2 * 16 + j]);
    buf[k2 * 17 + j] = u;
  }
  __syncwarp();
#pragma unroll
  for (int m1 = 0; m1 < 16; ++m1) v[m1] = buf[j * 17 + m1];
  __syncwarp();
  tmcfft::fft_reg<16>(v);
}

__device__ __forceinline__ void load_tables(float2* tw_step, float2* tw_comb, const float2* __restrict__ tw) {
  for (int i = threadIdx.x; i < 256; i += kThreads) tw_step[i] = __ldg(tw + 4 * (((i & 15) * (i >> 4)) & 255));
  for (int i = threadIdx.x; i < 3 * 256; i += kThreads) {
    const int q = i / 256 + 1, kk = i & 255;
    const int k = kk < 128 ? kk : kk - 256;
    tw_comb[i] = __ldg(tw + ((q * k) & 1023));
  }
}

// ---- forward rows: image window * mask^e (two real signals packed) -> tmp[plane][y][kx < KX] --------
// MODE 1: frame_b == frame_a with mask powers (1, 2); MODE 2: two frames (or one, frame_b < 0), power 1 each.
// 3 CTAs per SM (80 registers) pay off for MODE 1 and the inverse (measured -0.3 ms per movie); MODE 2 holds a second
// image row pair and would spill (+1.2 ms), it stays at 2 CTAs per SM
template <int MODE>
__global__ void __launch_bounds__(kThreads, MODE == 1 ? 3 : 2)
rows_forward_poly(const float* __restrict__ image, int H, int W, const float* __restrict__ mean_std,
                  const float* __restrict__ mask, const int* __restrict__ jobs, const int* __restrict__ frame_shifts,
                  int x_margin, int ylo, int yhi, int NY, int KX, const float2* __restrict__ tw, float2* __restrict__ tmp,
                  int rows_per_cta) {
  constexpr int N = 1024;
  extern __shared__ float2 smem[];
  float2* tw_step = smem;
  float2* tw_comb = smem + 256;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int qh = lane >> 4, j = lane & 15;
  float2* buf = smem + kTableWords + warp * kWarpWords + qh * kBuf;
  float2* zrow = smem + kTableWords + warp * kWarpWords + 2 * kBuf;
  load_tables(tw_step, tw_comb, tw);
  const int job = blockIdx.y;
  const int fa = jobs[job * 6 + 0], fb = jobs[job * 6 + 2];
  const int y0 = jobs[job * 6 + 4], x0 = jobs[job * 6 + 5];
  float mean = 0.f, inv_std = 1.f;
  if (mean_std != nullptr) {
    mean = __ldg(mean_std);
    inv_std = 1.0f / __ldg(mean_std + 1);
  }
  const Window wa = make_window(image, fa, y0, x0, frame_shifts, H, W, ylo, yhi, N, x_margin);
  const Window wb = make_window(image, fb >= 0 ? fb : fa, y0, x0, frame_shifts, H, W, ylo, yhi, N, x_margin);
  const float* img_a = wa.fast_base(W);
  const bool has_b = fb >= 0;
  const bool separate_b = MODE == 2 && has_b;
  const float* img_b = wb.fast_base(W);
  const int row_begin = ylo + blockIdx.x * rows_per_cta;
  const int row_end = min(yhi, row_begin + rows_per_cta);
  float2* plane_a = tmp + (long)(2 * job) * NY * KX;
  float2* plane_b = plane_a + (long)NY * KX;
  const int q0 = 2 * qh;  // this thread owns the sub-sequences q0 and q0 + 1: pixels x = 4 (j + 16 r) + q0 (+ 1)
  __syncthreads();        // twiddle tables
  for (int y = row_begin + warp; y < row_end; y += kWarps) {
    float2 va[16], vb[16];
    {
      const float* ra = img_a + (long)y * W + 4 * j + q0;
      const float* rb = separate_b ? img_b + (long)y * W + 4 * j + q0 : nullptr;
      const float* rm = mask ? mask + (long)y * N + 4 * j + q0 : nullptr;
      const bool vec_a = (reinterpret_cast<uintptr_t>(ra) & 7) == 0;
      const bool vec_b = (reinterpret_cast<uintptr_t>(rb) & 7) == 0;
      // two batches of 8 element pairs: enough loads in flight without holding all staging values in registers
#pragma unroll
      for (int h0 = 0; h0 < 16; h0 += 8) {
        float2 pa[8], pb[8], pm[8];
        if (wa.wrap) {  // CTA-uniform: the window leaves the frame where the mask is not zero
#pragma unroll
          for (int r = 0; r < 8; ++r) {
            const int x = 4 * j + q0 + 64 * (h0 + r);
            pa[r] = make_float2(__ldg(wa.wrapped(y, x, H, W)), __ldg(wa.wrapped(y, x + 1, H, W)));
          }
        } else if (vec_a) {
#pragma unroll
          for (int r = 0; r < 8; ++r) pa[r] = __ldg(reinterpret_cast<const float2*>(ra + 64 * (h0 + r)));
        } else {
#pragma unroll
          for (int r = 0; r < 8; ++r) pa[r] = make_float2(__ldg(ra + 64 * (h0 + r)), __ldg(ra + 64 * (h0 + r) + 1));
        }
        if (separate_b) {
          if (wb.wrap) {
#pragma unroll
            for (int r = 0; r < 8; ++r) {
              const int x = 4 * j + q0 + 64 * (h0 + r);
              pb[r] = make_float2(__ldg(wb.wrapped(y, x, H, W)), __ldg(wb.wrapped(y, x + 1, H, W)));
            }
          } else if (vec_b) {
#pragma unroll
            for (int r = 0; r < 8; ++r) pb[r] = __ldg(reinterpret_cast<const float2*>(rb + 64 * (h0 + r)));
          } else {
#pragma unroll
            for (int r = 0; r < 8; ++r) pb[r] = make_float2(__ldg(rb + 64 * (h0 + r)), __ldg(rb + 64 * (h0 + r) + 1));
          }
        }
#pragma unroll
        for (int r = 0; r < 8; ++r)
          pm[r] = rm ? __ldg(reinterpret_cast<const float2*>(rm + 64 * (h0 + r))) : make_float2(1.f, 1.f);
#pragma unroll
        for (int r = 0; r < 8; ++r) {
          const float a0 = (pa[r].x - mean) * inv_std, a1 = (pa[r].y - mean) * inv_std;
          float2 z0, z1;
          z0.x = a0 * pm[r].x;
          z1.x = a1 * pm[r].y;
          if (MODE == 1) {
            z0.y = z0.x * pm[r].x;
            z1.y = z1.x * pm[r].y;
          } else {
            z0.y = separate_b ? (pb[r].x - mean) * inv_std * pm[r].x : 0.f;
            z1.y = separate_b ? (pb[r].y - mean) * inv_std * pm[r].y : 0.f;
          }
          va[h0 + r] = z0;
          vb[h0 + r] = z1;
        }
      }
    }
    fft256_halfwarp(va, j, buf, tw_step);
    fft256_halfwarp(vb, j, buf, tw_step);
    // Z[k] = sum_q W^{q k} Y_q[k mod 256] for the needed k; lanes j and j + 16 hold the two halves of the sum
#pragma unroll
    for (int k1 = 0; k1 < 16; ++k1) {
      if (16 * k1 < KX || 16 * k1 + 15 > 256 - KX) {  // warp-uniform: some lane of this register slot is in the band
        const int kk = j + 16 * k1;
        const bool pos = kk < KX, neg = kk > 256 - KX;
        float2 ya = va[tmcfft::bitrev<16>(k1)];
        const float2 yb = vb[tmcfft::bitrev<16>(k1)];
        if (qh) ya = cmul(ya, tw_comb[256 + kk]);  // q = 2
        float2 p = cadd(ya, cmul(yb, tw_comb[q0 * 256 + kk]));  // q = q0 + 1
        p.x += __shfl_xor_sync(0xffffffffu, p.x, 16);
        p.y += __shfl_xor_sync(0xffffffffu, p.y, 16);
        if (qh == 0 && pos) zrow[kk] = p;
        if (qh == 1 && neg) zrow[128 + 256 - kk] = p;
      }
    }
    __syncwarp();
    for (int k = lane; k < KX; k += 32) {
      const float2 zk = zrow[k];
      const float2 zn = k == 0 ? zk : zrow[128 + k];
      plane_a[(long)y * KX + k] = make_float2(0.5f * (zk.x + zn.x), 0.5f * (zk.y - zn.y));
      if (has_b) plane_b[(long)y * KX + k] = make_float2(0.5f * (zk.y + zn.y), -0.5f * (zk.x - zn.x));
    }
    __syncwarp();
  }
}

// ---- inverse rows + argmax: tmp[item][y][kx] -> partial[item][cta] ------------------------------------
// CTA = kRowsPerCta rows (row pairs, two per warp); same partial layout as rows_inverse_argmax_p2<1024>.
constexpr int kRowsPerCta = 32;

__global__ void __launch_bounds__(kThreads, 3)
rows_inverse_argmax_poly(const float2* __restrict__ tmp, int NY, int KX, const float2* __restrict__ tw,
                         PeakCandidate* __restrict__ partial) {
  constexpr int N = 1024;
  extern __shared__ float2 smem[];
  float2* tw_step = smem;
  float2* tw_comb = smem + 256;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int qh = lane >> 4, j = lane & 15;
  float2* buf = smem + kTableWords + warp * kWarpWords + qh * kBuf;
  load_tables(tw_step, tw_comb, tw);
  const long item = blockIdx.y;
  const float2* src = tmp + item * NY * KX;
  const int q0 = 2 * qh;
  float best = -INFINITY;
  int best_idx = 0x7fffffff;
  __syncthreads();
  for (int pair = warp; pair < kRowsPerCta / 2; pair += kWarps) {
    const int ya = blockIdx.x * kRowsPerCta + 2 * pair;
    if (ya >= NY) break;
    const bool has_b = ya + 1 < NY;
    const float2* rowa = src + (long)ya * KX;
    float2 va[16], vb[16];
#pragma unroll
    for (int r = 0; r < 16; ++r) {
      float2 z0 = make_float2(0.f, 0.f), z1 = z0;
      if (16 * r < KX || 16 * r + 15 > 256 - KX) {
        const int kk = j + 16 * r;
        const bool pos = kk < KX, neg = kk > 256 - KX;
        if (pos || neg) {
          const int ka = pos ? kk : 256 - kk;  // |k|
          const float2 ca = __ldg(rowa + ka);
          const float2 cb = has_b ? __ldg(rowa + KX + ka) : make_float2(0.f, 0.f);
          // packed spectrum entry of (row ya -> real part, row ya + 1 -> imaginary part), stored (im, re): the forward
          // transforms below then act as the inverse; multiplying the swapped value by W^{+q k} equals swapping
          // Z[k] W^{-q k}
          const float2 z = c2r_pack<N>(ca, cb, pos ? kk : N - ka, KX);
          z0 = qh ? cmul(z, tw_comb[256 + kk]) : z;
          z1 = cmul(z, tw_comb[q0 * 256 + kk]);
        }
      }
      va[r] = z0;
      vb[r] = z1;
    }
    fft256_halfwarp(va, j, buf, tw_step);
    fft256_halfwarp(vb, j, buf, tw_step);
    // the thread visits its samples in increasing index order (row ya left to right, then row ya + 1; pairs ascend), so
    // "strictly greater" keeps the first of equal maxima: one compare and two selects per sample
    const int ia0 = ya * N + 4 * j + q0;
#pragma unroll
    for (int k1 = 0; k1 < 16; ++k1) {
      const float2 a = va[tmcfft::bitrev<16>(k1)], b = vb[tmcfft::bitrev<16>(k1)];  // swapped: .y = row ya, .x = row ya + 1
      if (a.y > best) {
        best = a.y;
        best_idx = ia0 + 64 * k1;
      }
      if (b.y > best) {
        best = b.y;
        best_idx = ia0 + 64 * k1 + 1;
      }
    }
    if (has_b) {
#pragma unroll
      for (int k1 = 0; k1 < 16; ++k1) {
        const float2 a = va[tmcfft::bitrev<16>(k1)], b = vb[tmcfft::bitrev<16>(k1)];
        if (a.x > best) {
          best = a.x;
          best_idx = ia0 + N + 64 * k1;
        }
        if (b.x > best) {
          best = b.x;
          best_idx = ia0 + N + 64 * k1 + 1;
        }
      }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, best, o);
    const int oi = __shfl_xor_sync(0xffffffffu, best_idx, o);
    if (better(ov, oi, best, best_idx)) {
      best = ov;
      best_idx = oi;
    }
  }
  __shared__ float sval[kWarps];
  __shared__ int sidx[kWarps];
  if (lane == 0) {
    sval[warp] = best;
    sidx[warp] = best_idx;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int i = 1; i < kWarps; ++i)
      if (better(sval[i], sidx[i], best, best_idx)) {
        best = sval[i];
        best_idx = sidx[i];
      }
    PeakCandidate c;
    c.val = best;
    c.idx = best_idx;
    partial[item * gridDim.x + blockIdx.x] = c;
  }
}

}  // namespace poly

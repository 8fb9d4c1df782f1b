// Band-limited 2-D real DFTs of masked image patches / whole frames, cross-correlation
// products, inverse transforms with fused peak search, Fourier-shift of whole frames.
//
// Replaces, for the hot path, what the reference does with torch.fft.rfftn / irfftn and
// elementwise complex passes at estimate_motion_xc.py:77-123,338-369, correct_motion.py:484-496
// and estimate_motion_optimizer.py:371-372.  Design notes (DESIGN.md §FFT):
//  * a 2-D transform is a row pass and a column pass, each a batch of 1-D shared-memory FFTs
//    (fft_core.cuh); only the kx / ky bins inside the band-pass box are ever written, so the
//    intermediate is KX/(N/2+1) of a full spectrum and the outputs are band-limited;
//  * two real rows are packed into one complex transform (the patch under two different mask
//    powers -- quirk Q1 -- or two frames / two output rows);
//  * rows outside the mask support are skipped; the inverse row pass feeds a block-wide argmax
//    instead of storing the correlation surface.
#include "common.cuh"
#include <stdlib.h>
#include "fft_core.cuh"
#include "fft_core2.cuh"

namespace {

using tmcfft::pad_idx;
using tmcfft::padded_len;

constexpr int kThreads = 256;

__host__ __device__ constexpr int batch_for(int n) { return n >= 4096 ? 1 : (4096 / n > 16 ? 16 : 4096 / n); }

template <int N>
constexpr size_t fft_smem_bytes() {
  return 2ull * batch_for(N) * padded_len(N) * sizeof(float2);
}

// ---- transform plans ----------------------------------------------------------------------
// A plan buffer (device, complex64) for a length-n DFT is  twiddles W_M^m [M] | chirp [n] | bhat [M]
// with M == n for supported powers of two (no chirp / bhat) and otherwise M = next_pow2(2n - 1):
// arbitrary lengths run as Bluestein chirp-z convolutions on the same shared-memory FFT core.

inline bool pow2_n(int n) { return n >= 16 && n <= 8192 && (n & (n - 1)) == 0; }
inline int fft_size_for(int n) {  // 0: unsupported
  if (pow2_n(n)) return n;
  if (n < 2) return 0;
  int m = 16;
  while (m < 2 * n - 1) m <<= 1;
  return m <= 8192 ? m : 0;
}

// Axes longer than the shared-memory transforms reach (n > 4096 and not a power of two <= 8192: K3 frames are
// 5760 x 4092, super-resolution 11520 x 8184) are decimated: n = R n' with n' supported, and with j = R m + r
//   forward:  X[k] = sum_r W_n^{r k} Y_r[k mod n'],   Y_r = DFT_n'(x[R m + r])
//   inverse:  x[R m + r] = IDFT_n'( Z_r )[m],   Z_r[j] = sum_q X[j + q n'] W_n^{-r (j + q n')}
// (a band that spans <= n' bins aliases without collisions: one term per j).  The generic kernels below loop over r;
// R == 1 is the plain transform.
inline int decimation_for(int n) {  // 0: unsupported
  if (fft_size_for(n) > 0) return 1;
  // sub-sequences of exactly 8192 points leave no shared memory for the accumulators of a full spectrum: take them last
  for (int r = 2; r <= 8; ++r)
    if (n % r == 0 && fft_size_for(n / r) > 0 && n / r != 8192) return r;
  for (int r = 2; r <= 8; ++r)
    if (n % r == 0 && fft_size_for(n / r) > 0) return r;
  return 0;
}

struct AxisPlan {
  const float2* tw;     // W_M^m
  const float2* chirp;  // exp(-i pi j^2 / n), j < n   (Bluestein only)
  const float2* bhat;   // FFT_M of the wrapped conjugate chirp (Bluestein only)
  int n;                // length of the shared-memory transforms (n_total / R)
  int R;                // decimation factor
  int n_total;          // length of the axis
};

inline AxisPlan make_axis_plan(const void* buf, int n_total) {
  const int R = decimation_for(n_total) > 0 ? decimation_for(n_total) : 1;
  const int n = n_total / R;
  const int m = fft_size_for(n);
  AxisPlan p;
  p.tw = (const float2*)buf;
  p.chirp = p.tw + m;
  p.bhat = p.chirp + n;
  p.n = n;
  p.R = R;
  p.n_total = n_total;
  return p;
}

// W_N^{e} = exp(-2 pi i e / N) for any integer e (reduced exactly before the fp32 sincospi)
__device__ __forceinline__ float2 twiddle_n(long e, int N) {
  long m = e % N;
  if (m < 0) m += N;
  float s, c;
  sincospif(-2.0f * (float)m / (float)N, &s, &c);
  return make_float2(c, s);
}

__global__ void twiddle_kernel(int n, float2* __restrict__ tw) {
  int m = blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= n) return;
  double s, c;
  sincospi(-2.0 * (double)m / (double)n, &s, &c);
  tw[m] = make_float2((float)c, (float)s);
}

// chirp[j] = exp(-i pi j^2 / n) ; b[j] = conj(chirp[|j|]) wrapped into length m, zero elsewhere
__global__ void chirp_kernel(int n, int m, float2* __restrict__ chirp, float2* __restrict__ b) {
  int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= m) return;
  float2 bv = make_float2(0.f, 0.f);
  auto w = [&](int q) {  // exp(-i pi q^2 / n), q^2 reduced mod 2n exactly
    long r = ((long)q * q) % (2l * n);
    double s, c;
    sincospi(-(double)r / (double)n, &s, &c);
    return make_float2((float)c, (float)s);
  };
  if (j < n) {
    float2 v = w(j);
    chirp[j] = v;
    bv = make_float2(v.x, -v.y);
  } else if (m - j < n) {
    float2 v = w(m - j);
    bv = make_float2(v.x, -v.y);
  }
  b[j] = bv;
}

// Length-n DFT of B sequences held (padded) in `a` (entries [0, n) valid); `b` is scratch.
// BLU == false: n == M, plain FFT.  BLU == true: Bluestein with FFT size M >= 2n - 1.
// The caller syncs after filling `a`; the result (natural order, entries [0, n)) is in the
// returned buffer and a __syncthreads() has been issued.
template <int M, bool BLU>
__device__ __forceinline__ float2* dft_smem(float2* a, float2* b, const AxisPlan& plan) {
  constexpr int B = batch_for(M);
  if constexpr (!BLU) {
    return tmcfft::fft_forward<M, B, kThreads>(a, b, plan.tw);
  } else {
    constexpr int STRIDE = padded_len(M);
    const int n = plan.n;
    for (int idx = threadIdx.x; idx < B * M; idx += kThreads) {
      const int s = idx / M, j = idx % M;
      float2* p = a + s * STRIDE + pad_idx(j);
      *p = j < n ? cmul(*p, __ldg(plan.chirp + j)) : make_float2(0.f, 0.f);
    }
    __syncthreads();
    float2* r = tmcfft::fft_forward<M, B, kThreads>(a, b, plan.tw);
    float2* other = (r == a) ? b : a;
    for (int idx = threadIdx.x; idx < B * M; idx += kThreads) {
      const int s = idx / M, j = idx % M;
      float2* p = r + s * STRIDE + pad_idx(j);
      const float2 v = cmul(*p, __ldg(plan.bhat + j));
      *p = make_float2(v.y, v.x);  // swapped: the next forward FFT acts as the inverse
    }
    __syncthreads();
    float2* c = tmcfft::fft_forward<M, B, kThreads>(r, other, plan.tw);
    const float inv_m = 1.0f / (float)M;
    for (int idx = threadIdx.x; idx < B * n; idx += kThreads) {
      const int s = idx / n, k = idx % n;
      float2* p = c + s * STRIDE + pad_idx(k);
      const float2 v = make_float2(p->y * inv_m, p->x * inv_m);
      *p = cmul(v, __ldg(plan.chirp + k));
    }
    __syncthreads();
    return c;
  }
}

// plain batched complex rows (plan construction, tests): out[r] = DFT_n(in[r])
template <int M, bool BLU>
__global__ void __launch_bounds__(kThreads)
c2c_rows_kernel(const float2* __restrict__ in, int rows, AxisPlan plan, float2* __restrict__ out) {
  constexpr int B = batch_for(M);
  constexpr int STRIDE = padded_len(M);
  extern __shared__ float2 smem[];
  float2* a = smem;
  float2* b = smem + B * STRIDE;
  const int n = BLU ? plan.n : M;
  const int row0 = blockIdx.x * B;
  for (int idx = threadIdx.x; idx < B * n; idx += kThreads) {
    const int s = idx / n, j = idx % n;
    a[s * STRIDE + pad_idx(j)] = row0 + s < rows ? in[(long)(row0 + s) * n + j] : make_float2(0.f, 0.f);
  }
  __syncthreads();
  const float2* r = dft_smem<M, BLU>(a, b, plan);
  for (int idx = threadIdx.x; idx < B * n; idx += kThreads) {
    const int s = idx / n, j = idx % n;
    if (row0 + s < rows) out[(long)(row0 + s) * n + j] = r[s * STRIDE + pad_idx(j)];
  }
}

// ---- forward: row pass ---------------------------------------------------------------------

struct RowJob {  // one packed pair of real rows-sets: a -> real part, b -> imaginary part
  int frame_a, exp_a, frame_b, exp_b, y0, x0;
};

// The window a job reads from one frame.  frame_shifts (nullable, (T, 2) int32 = (dy, dx)) moves the window of every
// frame by a whole number of pixels: reading the window at origin + shift is what the reference gets by first rolling
// the frame (an integer-pixel Fourier shift, correct_motion.py:484-496) and then extracting the patch at the origin.
// The roll is circular, so a window that leaves the frame wraps around -- unless it only leaves it where the mask is
// zero anyway (the first / last x_margin columns and the rows outside [ylo, yhi)): then the plain reads stay inside the
// movie buffer, hit the neighbouring rows' finite pixels and are multiplied by zero like the wrapped ones.
struct Window {
  const float* frame;  // first pixel of the frame
  int oy, ox;          // window origin inside the frame (may lie outside it)
  bool wrap;           // reads have to be wrapped around the frame edges (slow path)
  __device__ __forceinline__ const float* fast_base(int W) const { return frame + (long)oy * W + ox; }
  __device__ __forceinline__ const float* wrapped(int y, int x, int H, int W) const {
    int ry = (oy + y) % H, cx = (ox + x) % W;
    if (ry < 0) ry += H;
    if (cx < 0) cx += W;
    return frame + (long)ry * W + cx;
  }
};

__device__ __forceinline__ Window make_window(const float* image, int frame, int y0, int x0, const int* __restrict__ frame_shifts,
                                              int H, int W, int ylo, int yhi, int NX, int x_margin) {
  Window w;
  w.frame = image + (long)frame * H * W;
  w.oy = y0;
  w.ox = x0;
  if (frame_shifts != nullptr) {
    w.oy += __ldg(frame_shifts + 2 * frame);
    w.ox += __ldg(frame_shifts + 2 * frame + 1);
  }
  const bool rows_inside = w.oy + ylo >= 0 && w.oy + yhi <= H;
  const bool cols_inside = w.ox >= 0 && w.ox + NX <= W;
  const bool cols_masked = w.ox >= -x_margin && w.ox + NX <= W + x_margin;
  // plain reads of the first / last frame row with columns beyond the row would leave the movie buffer
  const bool buffer_end = (w.oy + ylo == 0 && w.ox < 0) || (w.oy + yhi == H && w.ox + NX > W);
  w.wrap = !(rows_inside && (cols_inside || (cols_masked && !buffer_end)));
  return w;
}

template <int MX, bool BLU>
__global__ void __launch_bounds__(kThreads)
rows_forward_kernel(const float* __restrict__ image, int H, int W, const float* __restrict__ mean_std,
                    const float* __restrict__ mask, const int* __restrict__ jobs, const int* __restrict__ frame_shifts,
                    int x_margin, int ylo, int yhi, int NY, int KX, AxisPlan plan, float2* __restrict__ tmp) {
  constexpr int B = batch_for(MX);
  constexpr int STRIDE = padded_len(MX);
  const int NS = BLU ? plan.n : MX;             // length of the shared-memory transforms
  const int R = plan.R, NX = plan.n_total;      // decimation factor, window width
  extern __shared__ float2 smem[];
  float2* a = smem;
  float2* b = smem + B * STRIDE;
  float2* acc_pos = smem + 2 * B * STRIDE;      // R > 1 only: Z[k], Z[-k] accumulated over the sub-sequences
  float2* acc_neg = acc_pos + B * KX;
  const int job = blockIdx.y;
  const int fa = jobs[job * 6 + 0], ea = jobs[job * 6 + 1], fb = jobs[job * 6 + 2], eb = jobs[job * 6 + 3];
  const int y0 = jobs[job * 6 + 4], x0 = jobs[job * 6 + 5];
  const int row0 = ylo + blockIdx.x * B;
  float mean = 0.f, stdv = 1.f;
  const bool norm = mean_std != nullptr;
  if (norm) {
    mean = __ldg(mean_std);
    stdv = __ldg(mean_std + 1);
  }
  const Window wa = make_window(image, fa, y0, x0, frame_shifts, H, W, ylo, yhi, NX, x_margin);
  const Window wb = make_window(image, fb >= 0 ? fb : fa, y0, x0, frame_shifts, H, W, ylo, yhi, NX, x_margin);
  for (int r = 0; r < R; ++r) {
    for (int idx = threadIdx.x; idx < B * NS; idx += kThreads) {
      const int s = idx / NS, m_ = idx % NS;
      const int x = R * m_ + r;
      const int y = row0 + s;
      float2 z = make_float2(0.f, 0.f);
      if (y < yhi) {
        const float m = mask ? __ldg(mask + (long)y * NX + x) : 1.0f;
        float va = __ldg(wa.wrap ? wa.wrapped(y, x, H, W) : wa.fast_base(W) + (long)y * W + x);
        if (norm) va = __fdiv_rn(__fsub_rn(va, mean), stdv);
        for (int e = 0; e < ea; ++e) va = __fmul_rn(va, m);
        z.x = va;
        if (fb >= 0) {
          float vb = __ldg(wb.wrap ? wb.wrapped(y, x, H, W) : wb.fast_base(W) + (long)y * W + x);
          if (norm) vb = __fdiv_rn(__fsub_rn(vb, mean), stdv);
          for (int e = 0; e < eb; ++e) vb = __fmul_rn(vb, m);
          z.y = vb;
        }
      }
      a[s * STRIDE + pad_idx(m_)] = z;
    }
    __syncthreads();
    const float2* res = dft_smem<MX, BLU>(a, b, plan);
    for (int idx = threadIdx.x; idx < B * KX; idx += kThreads) {
      const int s = idx / KX, k = idx % KX;
      const int y = row0 + s;
      if (y >= yhi) continue;
      const int kp = k % NS;
      float2 zk = res[s * STRIDE + pad_idx(kp)];
      float2 zn = res[s * STRIDE + pad_idx(kp == 0 ? 0 : NS - kp)];
      if (R > 1) {
        const float2 tw = twiddle_n((long)r * k, NX);
        zk = cmul(zk, tw);
        zn = cmul(zn, make_float2(tw.x, -tw.y));
        if (r > 0) {
          zk = cadd(zk, acc_pos[idx]);
          zn = cadd(zn, acc_neg[idx]);
        }
        acc_pos[idx] = zk;
        acc_neg[idx] = zn;
        if (r + 1 < R) continue;
      }
      // Z = A + iB with A, B Hermitian:  A = (Z[k] + conj Z[-k]) / 2,  B = (Z[k] - conj Z[-k]) / 2i
      tmp[((long)(2 * job) * NY + y) * KX + k] = make_float2(0.5f * (zk.x + zn.x), 0.5f * (zk.y - zn.y));
      if (fb >= 0) tmp[((long)(2 * job + 1) * NY + y) * KX + k] = make_float2(0.5f * (zk.y + zn.y), -0.5f * (zk.x - zn.x));
    }
    __syncthreads();  // the transform buffers are refilled by the next sub-sequence
  }
}

// ---- forward: column pass --------------------------------------------------------------------

// plane p of tmp [NY][KX] -> out[p][KY][KX], ky = ky_start + kyb (wrapped), times weight[kyb][kx]
template <int MY, bool BLU>
__global__ void __launch_bounds__(kThreads)
cols_forward_kernel(const float2* __restrict__ tmp, int ylo, int yhi, int KX, int KY, int ky_start,
                    const float* __restrict__ weight, AxisPlan plan, float2* __restrict__ out) {
  constexpr int B = batch_for(MY);
  constexpr int STRIDE = padded_len(MY);
  const int NS = BLU ? plan.n : MY;
  const int R = plan.R, NY = plan.n_total;
  extern __shared__ float2 smem[];
  float2* a = smem;
  float2* b = smem + B * STRIDE;
  float2* acc = smem + 2 * B * STRIDE;  // R > 1 only
  const long plane = blockIdx.y;
  const int kx0 = blockIdx.x * B;
  const float2* src = tmp + plane * NY * KX;
  float2* dst = out + plane * KY * KX;
  for (int r = 0; r < R; ++r) {
    for (int idx = threadIdx.x; idx < B * NS; idx += kThreads) {
      const int s = idx % B, m_ = idx / B;
      const int y = R * m_ + r;
      float2 z = make_float2(0.f, 0.f);
      if (y >= ylo && y < yhi && kx0 + s < KX) z = src[(long)y * KX + kx0 + s];
      a[s * STRIDE + pad_idx(m_)] = z;
    }
    __syncthreads();
    const float2* res = dft_smem<MY, BLU>(a, b, plan);
    for (int idx = threadIdx.x; idx < B * KY; idx += kThreads) {
      const int s = idx % B, kyb = idx / B;
      if (kx0 + s >= KX) continue;
      const int ky = ky_start + kyb;
      const int pos = ((ky % NS) + NS) % NS;
      float2 v = res[s * STRIDE + pad_idx(pos)];
      if (R > 1) {
        v = cmul(v, twiddle_n((long)r * ky, NY));
        if (r > 0) v = cadd(v, acc[idx]);
        acc[idx] = v;
        if (r + 1 < R) continue;
      }
      if (weight) {
        const float wgt = __ldg(weight + (long)kyb * KX + kx0 + s);
        v.x *= wgt;
        v.y *= wgt;
      }
      dst[(long)kyb * KX + kx0 + s] = v;
    }
    __syncthreads();
  }
}

// ---- cross-correlation products ------------------------------------------------------------

// out[i] = conj(spec[ref_plane[i]]) * spec[cur_plane[i]]   (estimate_motion_xc.py:112,349)
__global__ void xc_pair_product_kernel(const float2* __restrict__ spec, const int* __restrict__ ref_plane,
                                       const int* __restrict__ cur_plane, long plane_elems, float2* __restrict__ out) {
  const long i = blockIdx.y;
  const float2* r = spec + (long)ref_plane[i] * plane_elems;
  const float2* c = spec + (long)cur_plane[i] * plane_elems;
  float2* o = out + i * plane_elems;
  for (long e = (long)blockIdx.x * blockDim.x + threadIdx.x; e < plane_elems; e += (long)gridDim.x * blockDim.x)
    o[e] = cmul_conj(r[e], c[e]);
}

// Leave-one-out reference with the reference's cache aliasing (quirk Q1).  Planes are laid out
// [frame j][patch g][part] with part 0 = rfft2(mask P_j) W and part 1 = rfft2(mask^2 P_j) W.
// Frame k's reference spectrum is  ( sum_{j != k} (c_kj ? part1_j : part0_j) ) / (T - 1)  where
// c_kj in {0,1} says whether frame j had already been masked in place when frame k was processed.
// c is given as per-k delta lists relative to k-1 (delta = +-(j+1)); T <= 50 gives c_kj = [j < k].
__global__ void xc_leave_one_out_kernel(const float2* __restrict__ spec, int T, int G, long plane_elems,
                                        const int* __restrict__ delta_offsets, const int* __restrict__ deltas,
                                        int k_begin, int k_count, float2* __restrict__ out) {
  const int g = blockIdx.y;
  const long e = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= plane_elems) return;
  auto part = [&](int j, int p) { return spec[((long)(j * G + g) * 2 + p) * plane_elems + e]; };
  float2 total = make_float2(0.f, 0.f);
  for (int j = 0; j < T; ++j) total = cadd(total, part(j, 0));
  float2 extra = make_float2(0.f, 0.f);  // sum_j c_kj (part1_j - part0_j)
  const float cnt = (float)(T - 1);
  for (int k = 0; k < T; ++k) {
    for (int d = delta_offsets[k]; d < delta_offsets[k + 1]; ++d) {
      const int v = deltas[d];
      const int j = (v > 0 ? v : -v) - 1;
      const float2 diff = csub(part(j, 1), part(j, 0));
      extra = v > 0 ? cadd(extra, diff) : csub(extra, diff);
    }
    if (k < k_begin || k >= k_begin + k_count) continue;  // frame-split movies: only the local frames
    const float2 cur = part(k, 0);
    float2 ref = cadd(csub(total, cur), extra);
    ref.x = __fdiv_rn(ref.x, cnt);
    ref.y = __fdiv_rn(ref.y, cnt);
    out[((long)(k - k_begin) * G + g) * plane_elems + e] = cmul_conj(ref, cur);
  }
}

// ---- inverse: column pass --------------------------------------------------------------------

// in[item][KY][KX] (ky = ky_start + kyb) -> tmp[item][NY][KX] = unnormalised inverse DFT along y
template <int MY, bool BLU>
__global__ void __launch_bounds__(kThreads)
cols_inverse_kernel(const float2* __restrict__ in, int KX, int KY, int ky_start, AxisPlan plan,
                    float2* __restrict__ tmp) {
  constexpr int B = batch_for(MY);
  constexpr int STRIDE = padded_len(MY);
  const int NS = BLU ? plan.n : MY;
  const int R = plan.R, NY = plan.n_total;
  extern __shared__ float2 smem[];
  float2* a = smem;
  float2* b = smem + B * STRIDE;
  const long item = blockIdx.y;
  const int kx0 = blockIdx.x * B;
  const float2* src = in + item * KY * KX;
  float2* dst = tmp + item * NY * KX;
  for (int r = 0; r < R; ++r) {
    // position j of the sub-sequence's spectrum gathers every band row ky = j (mod n'): one row for a band of <= n'
    // rows, R rows for a full spectrum
    for (int idx = threadIdx.x; idx < B * NS; idx += kThreads) {
      const int s = idx % B, pos = idx / B;
      float2 z = make_float2(0.f, 0.f);
      if (kx0 + s < KX) {
        int kyb = (pos - ky_start) % NS;
        if (kyb < 0) kyb += NS;
        for (; kyb < KY; kyb += NS) {
          float2 v = src[(long)kyb * KX + kx0 + s];
          if (R > 1) v = cmul(v, twiddle_n(-(long)r * (ky_start + kyb), NY));
          z = cadd(z, v);
        }
      }
      a[s * STRIDE + pad_idx(pos)] = make_float2(z.y, z.x);  // re/im swap: inverse via forward
    }
    __syncthreads();
    const float2* res = dft_smem<MY, BLU>(a, b, plan);
    for (int idx = threadIdx.x; idx < B * NS; idx += kThreads) {
      const int s = idx % B, m_ = idx / B;
      if (kx0 + s >= KX) continue;
      const float2 v = res[s * STRIDE + pad_idx(m_)];
      dst[(long)(R * m_ + r) * KX + kx0 + s] = make_float2(v.y, v.x);
    }
    __syncthreads();
  }
}

// ---- inverse: row pass (complex-to-real, two rows per transform) ------------------------------

// entry k in [0, NX) of the packed spectrum Z = Ca + i Cb of rows ya (real part) and yb (imaginary part), times the
// sub-sequence twiddle W_NX^{-r k}; Ca, Cb are given on [0, KX) and Hermitian beyond
__device__ __forceinline__ float2 c2r_entry(const float2* __restrict__ rowa, const float2* __restrict__ rowb, int KX, int NX,
                                            int R, int r, int k) {
  const bool neg = 2 * k > NX;
  const int kk = neg ? NX - k : k;
  if (kk >= KX) return make_float2(0.f, 0.f);
  const float2 ca = rowa[kk];
  const float2 cb = rowb ? rowb[kk] : make_float2(0.f, 0.f);
  if (kk == 0 || 2 * kk == NX) {  // c2r ignores the imaginary part of the DC / Nyquist bins
    const float sgn = (kk != 0 && (r & 1)) ? -1.f : 1.f;  // W^{-r N/2} = (-1)^r
    return make_float2(sgn * ca.x, sgn * cb.x);
  }
  // Z[k] = Ca + i Cb ; Z[N-k] = conj(Ca) + i conj(Cb)
  float2 z = neg ? make_float2(ca.x + cb.y, cb.x - ca.y) : make_float2(ca.x - cb.y, ca.y + cb.x);
  if (R > 1) {
    const float2 tw = twiddle_n(-(long)r * kk, NX);
    z = cmul(z, neg ? make_float2(tw.x, -tw.y) : tw);
  }
  return z;
}

// builds the packed spectrum of rows ya (real part) and yb (imaginary part) in `a_seq` (zeroed by the caller unless
// `gather`), re/im swapped; for a decimated axis (R > 1) the spectrum of sub-sequence r: entries times W^{-/+ r k},
// aliased onto k mod NS.  gather: the band may alias onto itself (2 KX - 1 > NS), every position sums its R sources.
__device__ __forceinline__ void load_c2r_pair(const float2* __restrict__ rowa, const float2* __restrict__ rowb, int KX,
                                              int NX, int NS, int R, int r, bool gather, float2* __restrict__ a_seq) {
  if (gather) {
    for (int j = threadIdx.x; j < NS; j += kThreads) {
      float2 z = make_float2(0.f, 0.f);
      for (int q = 0; q < R; ++q) z = cadd(z, c2r_entry(rowa, rowb, KX, NX, R, r, j + q * NS));
      a_seq[pad_idx(j)] = make_float2(z.y, z.x);
    }
    return;
  }
  for (int k = threadIdx.x; k < KX; k += kThreads) {
    const float2 zp = c2r_entry(rowa, rowb, KX, NX, R, r, k);
    const int kp = k % NS;
    a_seq[pad_idx(kp)] = make_float2(zp.y, zp.x);
    if (k != 0 && 2 * k != NX) {
      const float2 zn = c2r_entry(rowa, rowb, KX, NX, R, r, NX - k);
      a_seq[pad_idx(kp == 0 ? 0 : NS - kp)] = make_float2(zn.y, zn.x);
    }
  }
}

struct PeakCandidate {
  float val;
  int idx;
};

__device__ __forceinline__ bool better(float v, int i, float bv, int bi) { return v > bv || (v == bv && i < bi); }

// tmp[item][NY][KX] -> per-CTA maximum of the real correlation surface: partial[item][blockIdx.x]
template <int MX, bool BLU>
__global__ void __launch_bounds__(kThreads)
rows_inverse_argmax_kernel(const float2* __restrict__ tmp, int NY, int KX, AxisPlan plan,
                           PeakCandidate* __restrict__ partial) {
  constexpr int B = batch_for(MX);
  constexpr int STRIDE = padded_len(MX);
  const int NS = BLU ? plan.n : MX;
  const int R = plan.R, NX = plan.n_total;
  extern __shared__ float2 smem[];
  float2* a = smem;
  float2* b = smem + B * STRIDE;
  const long item = blockIdx.y;
  const int row0 = blockIdx.x * 2 * B;
  const float2* src = tmp + item * NY * KX;
  float best = -INFINITY;
  int best_idx = 0x7fffffff;
  const bool gather = R > 1 && 2 * KX - 1 > NS;  // the band aliases onto itself: full spectrum of a decimated axis
  for (int r = 0; r < R; ++r) {
    for (int idx = threadIdx.x; idx < B * STRIDE; idx += kThreads) a[idx] = make_float2(0.f, 0.f);
    __syncthreads();
    for (int s = 0; s < B; ++s) {
      const int ya = row0 + 2 * s, yb = ya + 1;
      if (ya < NY)
        load_c2r_pair(src + (long)ya * KX, yb < NY ? src + (long)yb * KX : nullptr, KX, NX, NS, R, r, gather, a + s * STRIDE);
    }
    __syncthreads();
    const float2* res = dft_smem<MX, BLU>(a, b, plan);
    for (int idx = threadIdx.x; idx < B * NS; idx += kThreads) {
      const int s = idx / NS, m_ = idx % NS;
      const int ya = row0 + 2 * s;
      if (ya >= NY) continue;
      const float2 v = res[s * STRIDE + pad_idx(m_)];  // swapped: v.y = row ya, v.x = row ya+1
      const int ia = ya * NX + R * m_ + r;
      if (better(v.y, ia, best, best_idx)) {
        best = v.y;
        best_idx = ia;
      }
      if (ya + 1 < NY && better(v.x, ia + NX, best, best_idx)) {
        best = v.x;
        best_idx = ia + NX;
      }
    }
    __syncthreads();
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
  __shared__ float sval[kThreads / 32];
  __shared__ int sidx[kThreads / 32];
  if ((threadIdx.x & 31) == 0) {
    sval[threadIdx.x >> 5] = best;
    sidx[threadIdx.x >> 5] = best_idx;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int i = 1; i < kThreads / 32; ++i)
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

// tmp[item][NY][KX] -> out[item][NY][NX] real, scaled (irfftn "backward" normalisation)
template <int MX, bool BLU>
__global__ void __launch_bounds__(kThreads)
rows_inverse_store_kernel(const float2* __restrict__ tmp, int NY, int KX, AxisPlan plan, float scale,
                          float* __restrict__ out) {
  constexpr int B = batch_for(MX);
  constexpr int STRIDE = padded_len(MX);
  const int NS = BLU ? plan.n : MX;
  const int R = plan.R, NX = plan.n_total;
  extern __shared__ float2 smem[];
  float2* a = smem;
  float2* b = smem + B * STRIDE;
  const long item = blockIdx.y;
  const int row0 = blockIdx.x * 2 * B;
  const float2* src = tmp + item * NY * KX;
  float* dst = out + item * NY * NX;
  const bool gather = R > 1 && 2 * KX - 1 > NS;  // the band aliases onto itself: full spectrum of a decimated axis
  for (int r = 0; r < R; ++r) {
    for (int idx = threadIdx.x; idx < B * STRIDE; idx += kThreads) a[idx] = make_float2(0.f, 0.f);
    __syncthreads();
    for (int s = 0; s < B; ++s) {
      const int ya = row0 + 2 * s, yb = ya + 1;
      if (ya < NY)
        load_c2r_pair(src + (long)ya * KX, yb < NY ? src + (long)yb * KX : nullptr, KX, NX, NS, R, r, gather, a + s * STRIDE);
    }
    __syncthreads();
    const float2* res = dft_smem<MX, BLU>(a, b, plan);
    for (int idx = threadIdx.x; idx < B * NS; idx += kThreads) {
      const int s = idx / NS, m_ = idx % NS;
      const int ya = row0 + 2 * s;
      if (ya >= NY) continue;
      const float2 v = res[s * STRIDE + pad_idx(m_)];
      const int x = R * m_ + r;
      dst[(long)ya * NX + x] = v.y * scale;
      if (ya + 1 < NY) dst[(long)(ya + 1) * NX + x] = v.x * scale;
    }
    __syncthreads();
  }
}

#include "fourier_p2.cuh"
#include "fourier_poly.cuh"

// TMC_FFT_POLY=0 selects the 1024-point block-level row kernels instead of the polyphase ones (A/B testing)
inline bool use_poly() {
  static const bool on = [] {
    const char* e = getenv("TMC_FFT_POLY");
    return !(e && e[0] == '0');
  }();
  return on;
}

// rows of two frames as half-length transforms of pixel pairs (rows_forward_real2n) for 8192- and 4096-point rows;
// TMC_FFT_REAL2N=0 selects the full-length kernels (A/B testing; read per call: tests toggle it).  Measured, 40 frames:
// 8192^2 12.4 -> 4.7 ms, 4096^2 1.28 -> 1.20 ms.
inline bool use_real2n(int) {
  const char* e = getenv("TMC_FFT_REAL2N");
  return !(e && e[0] == '0');
}

// TMC_FFT_COL_QUADS=0 selects the one-column-per-CTA kernel for 4096-point whole-frame columns (A/B testing)
inline bool use_col_quads() {
  const char* e = getenv("TMC_FFT_COL_QUADS");
  return !(e && e[0] == '0');
}

template <int M, bool BLU>
constexpr bool use_fast_path() {
  return !BLU && M >= 256;
}

// ---- peak finalisation: argmax over CTAs, 3-point parabola, wrap ---------------------------

// value of the real surface at (y, x) from the column-transformed rows (direct KX-term sum)
__device__ __forceinline__ float direct_value(const float2* __restrict__ row, int KX, int NX, int x) {
  float acc = 0.f;
  for (int k = threadIdx.x; k < KX; k += blockDim.x) {
    const float2 c = row[k];
    if (k == 0 || 2 * k == NX) {
      const float sgn = (k != 0 && (x & 1)) ? -1.f : 1.f;
      acc += sgn * c.x;
    } else {
      float s, co;
      const int m = (int)(((long)k * x) % NX);
      sincospif(2.0f * (float)m / (float)NX, &s, &co);
      acc += 2.0f * (c.x * co - c.y * s);
    }
  }
  return acc;
}

__device__ __forceinline__ float block_sum_128(float v, float* sh) {
  v = warp_sum(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
  __syncthreads();
  return sh[0] + sh[1] + sh[2] + sh[3];
}

// shifts[item] = (sy, sx) in px: estimate_motion_xc.py:354-369,414-483 (quirks Q6, Q7)
__global__ void __launch_bounds__(128)
peak_finalize_kernel(const float2* __restrict__ tmp, const PeakCandidate* __restrict__ partial, int nparts, int NY, int NX,
                     int KX, int sub_pixel, float* __restrict__ shifts) {
  __shared__ float sh[4];
  __shared__ int s_idx;
  const long item = blockIdx.x;
  if (threadIdx.x == 0) {
    float best = -INFINITY;
    int bi = 0x7fffffff;
    for (int i = 0; i < nparts; ++i) {
      const PeakCandidate c = partial[item * nparts + i];
      if (better(c.val, c.idx, best, bi)) {
        best = c.val;
        bi = c.idx;
      }
    }
    s_idx = bi;
  }
  __syncthreads();
  const int y = s_idx / NX, x = s_idx % NX;
  float py = (float)y, px = (float)x;
  if (sub_pixel && y >= 1 && y < NY - 1 && x >= 1 && x < NX - 1) {
    const float2* rows = tmp + item * NY * KX;
    const float v0 = block_sum_128(direct_value(rows + (long)y * KX, KX, NX, x), sh);
    const float vym = block_sum_128(direct_value(rows + (long)(y - 1) * KX, KX, NX, x), sh);
    const float vyp = block_sum_128(direct_value(rows + (long)(y + 1) * KX, KX, NX, x), sh);
    const float vxm = block_sum_128(direct_value(rows + (long)y * KX, KX, NX, x - 1), sh);
    const float vxp = block_sum_128(direct_value(rows + (long)y * KX, KX, NX, x + 1), sh);
    if (vyp != vym) py += 0.5f * (vym - vyp) / (vym - 2.0f * v0 + vyp);
    if (vxp != vxm) px += 0.5f * (vxm - vxp) / (vxm - 2.0f * v0 + vxp);
  }
  if (threadIdx.x == 0) {
    shifts[item * 2 + 0] = (py <= (float)(NY / 2)) ? py : py - (float)NY;
    shifts[item * 2 + 1] = (px <= (float)(NX / 2)) ? px : px - (float)NX;
  }
}

// ---- whole-frame Fourier shift (correct_motion_fast) -----------------------------------------

// spec[f][NY][KX] *= exp(-2 pi i (fy sy + fx sx)), shifts = sign * field[(c, f)] (field (2, T, 1, 1))
__global__ void fourier_shift_kernel(float2* __restrict__ spec, int T, int NY, int NX, int KX, const float* __restrict__ field,
                                     float sign) {
  const int f = blockIdx.z, ky = blockIdx.y;
  const int kx = blockIdx.x * blockDim.x + threadIdx.x;
  if (kx >= KX) return;
  const float sy = sign * __ldg(field + f), sx = sign * __ldg(field + T + f);
  // torch.fft.fftfreq: integer index times fp32(1/n)
  const float fy = __fmul_rn((float)(ky < (NY + 1) / 2 ? ky : ky - NY), (float)(1.0 / (double)NY));
  const float fx = __fmul_rn((float)kx, (float)(1.0 / (double)NX));
  const float c = -6.283185307179586f;  // fp32(-2 pi)
  const float ang = __fadd_rn(__fmul_rn(__fmul_rn(c, fy), sy), __fmul_rn(__fmul_rn(c, fx), sx));
  float s, co;
  sincosf(ang, &s, &co);
  float2* p = spec + ((long)f * NY + ky) * KX + kx;
  *p = cmul(*p, make_float2(co, s));
}

// ---- dispatch helpers ------------------------------------------------------------------------

#define TMC_FOR_EACH_M(X) X(16) X(32) X(64) X(128) X(256) X(512) X(1024) X(2048) X(4096) X(8192)

// timing label of a size-templated kernel (the two sizes of the benchmark get their own rows)
template <int MM>
constexpr const char* sized_label(const char* l4096, const char* l1024, const char* other) {
  return MM == 4096 ? l4096 : (MM == 1024 ? l1024 : other);
}

template <int V>
struct IntC {
  static constexpr int value = V;
};
template <bool V>
struct BoolC {
  static constexpr bool value = V;
};

// calls f(IntC<M>{}, BoolC<BLU>{}) for the FFT size / algorithm that serves a length-n transform
template <typename F>
int dispatch_fft(int n_total, const char* who, F&& f) {
  const int R = decimation_for(n_total);
  const int n = R > 0 ? n_total / R : n_total;
  const int m = R > 0 ? fft_size_for(n) : 0;
  const bool blu = m != n;
  switch (m) {
#define CASE(MM) \
  case MM:       \
    return blu ? f(IntC<MM>{}, BoolC<true>{}) : f(IntC<MM>{}, BoolC<false>{});
    TMC_FOR_EACH_M(CASE)
#undef CASE
    default:
      break;
  }
  tmc_set_error("%s: transform length %d is not supported (powers of two up to 8192, any length up to 4096, and "
                "multiples by 2..8 of those for band-limited transforms)", who, n_total);
  return TMC_ERR_UNSUPPORTED;
}

template <typename K>
int enable_smem(K kernel, size_t bytes) {
  if (bytes > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e != cudaSuccess) {
      tmc_set_error("cudaFuncSetAttribute(%zu bytes) failed: %s", bytes, cudaGetErrorString(e));
      return TMC_ERR_CUDA;
    }
  }
  return TMC_OK;
}

constexpr size_t kMaxSmem = 227 * 1024;

// shared memory of the generic kernels' transform buffers for FFT size m (runtime twin of fft_smem_bytes)
inline size_t fft_smem_runtime(int m) { return 2ull * batch_for(m) * padded_len(m) * sizeof(float2); }

// a decimated axis of length n: do the accumulators of a FULL spectrum (row pass: n/2+1 bins twice, column pass: n bins)
// fit beside the transform buffers?
inline bool decimated_full_fits(int n) {
  const int R = decimation_for(n);
  if (R <= 1) return R == 1;
  const int m = fft_size_for(n / R), b = batch_for(m);
  return fft_smem_runtime(m) + 2ull * b * (n / 2 + 1) * sizeof(float2) <= kMaxSmem &&
         fft_smem_runtime(m) + 1ull * b * n * sizeof(float2) <= kMaxSmem;
}

// row pass of tmc_rfft2_band: tmp[2 job + {0, 1}][y][kx] = row DFTs of the jobs' windows, kx < kx_count
int rfft2_rows(const float* image, int h, int w, const float* mean_std, const float* mask, int ny, int nx, const int* jobs,
               int njobs, int job_mode, const int* frame_shifts, int x_margin, int ylo, int yhi, int kx_count,
               const AxisPlan& px, void* tmp, cudaStream_t stream) {
  return dispatch_fft(nx, "rfft2_band", [&](auto M, auto BLU) {
    constexpr int MM = decltype(M)::value;
    constexpr bool BB = decltype(BLU)::value;
    if constexpr (MM == 1024 && !BB) {
      // polyphase path: four 256-point warp-level FFTs per row, only the band is ever formed
      if (yhi > ylo && kx_count <= 128 && job_mode != 0 && use_poly() && px.R == 1) {
        int rows_per_cta = 32;  // measured on C2: 64 .. 256 rows per CTA change the row kernels by less than 2 %
        while (rows_per_cta > 8 && (long)tmc_div_up(yhi - ylo, rows_per_cta) * njobs < 148 * 6) rows_per_cta -= 8;
        dim3 grid(tmc_div_up(yhi - ylo, rows_per_cta), njobs);
        if (job_mode == 1) {
          if (int e = enable_smem(poly::rows_forward_poly<1>, poly::smem_bytes)) return e;
          TMC_TIMED("rows_forward_poly<1>", stream,
                    poly::rows_forward_poly<1><<<grid, poly::kThreads, poly::smem_bytes, stream>>>(
                        image, h, w, mean_std, mask, jobs, frame_shifts, x_margin, ylo, yhi, ny, kx_count, px.tw, (float2*)tmp,
                        rows_per_cta));
        } else {
          if (int e = enable_smem(poly::rows_forward_poly<2>, poly::smem_bytes)) return e;
          TMC_TIMED("rows_forward_poly<2>", stream,
                    poly::rows_forward_poly<2><<<grid, poly::kThreads, poly::smem_bytes, stream>>>(
                        image, h, w, mean_std, mask, jobs, frame_shifts, x_margin, ylo, yhi, ny, kx_count, px.tw, (float2*)tmp,
                        rows_per_cta));
        }
        return TMC_OK;
      }
    }
    if constexpr ((MM == 8192 || MM == 4096) && !BB) {
      // rows of two frames as two half-length complex transforms of pixel pairs instead of one full-length transform
      // of a packed pair (the 8192-point kernel is confined to one 8-warp CTA per SM)
      if (yhi > ylo && job_mode == 2 && px.R == 1 && kx_count <= MM / 2 && use_real2n(MM)) {
        constexpr int NH = MM / 2;
        constexpr int B = fft2::Cfg<NH>::B;
        int rows_per_cta = B * 4;
        while (rows_per_cta > B && (long)tmc_div_up(yhi - ylo, rows_per_cta) * njobs < 148 * 8) rows_per_cta -= B;
        dim3 grid(tmc_div_up(yhi - ylo, rows_per_cta), njobs);
        constexpr size_t smem = rows_forward_real2n_smem_bytes<NH>();
        if (int e = enable_smem(rows_forward_real2n<NH>, smem)) return e;
        TMC_TIMED(MM == 8192 ? "rows_forward_real2n<4096>" : "rows_forward_real2n<2048>", stream,
                  rows_forward_real2n<NH><<<grid, fft2::kThreads, smem, stream>>>(image, h, w, mean_std, mask, jobs, frame_shifts, x_margin,
                                                                                   ylo, yhi, ny, kx_count, px.tw, (float2*)tmp,
                                                                                   rows_per_cta));
        return TMC_OK;
      }
    }
    if constexpr (use_fast_path<MM, BB>()) if (px.R == 1) {
      if (yhi > ylo) {
        constexpr int B = fft2::Cfg<MM>::B;
        // enough CTAs to fill the chip a few times over, each amortising its twiddle-table load
        int rows_per_cta = B * 4;
        while (rows_per_cta > B && (long)tmc_div_up(yhi - ylo, rows_per_cta) * njobs < 148 * 8) rows_per_cta -= B;
        dim3 grid(tmc_div_up(yhi - ylo, rows_per_cta), njobs);
        constexpr size_t smem = rows_forward_smem_bytes<MM>();
#define TMC_ROWS_FWD(MODE)                                                                                      \
  {                                                                                                             \
    if (int e = enable_smem(rows_forward_p2<MM, MODE>, smem)) return e;                                         \
    tmc_timing_begin(stream);                                                                                   \
    rows_forward_p2<MM, MODE><<<grid, fft2::kThreads, smem, stream>>>(image, h, w, mean_std, mask, jobs, frame_shifts, \
                                                                     x_margin, ylo, yhi, ny, kx_count, px.tw,          \
                                                                     (float2*)tmp, rows_per_cta);                      \
    tmc_timing_end(MM == 4096 ? "rows_forward_p2<4096>" : "rows_forward_p2", stream);                            \
  }
        if (job_mode == 1) TMC_ROWS_FWD(1) else if (job_mode == 2) TMC_ROWS_FWD(2) else TMC_ROWS_FWD(0)
#undef TMC_ROWS_FWD
        tmc_count_launch();
      }
      return TMC_OK;
    }
    // generic kernel (Bluestein lengths, small transforms, decimated long axes); the accumulators of a decimated axis
    // follow the two transform buffers
    const size_t smem = fft_smem_bytes<MM>() + (px.R > 1 ? 2ull * batch_for(MM) * kx_count * sizeof(float2) : 0);
    if (smem > kMaxSmem) {
      tmc_set_error("rfft2_band: band of %d bins too wide for the decimated row transform of length %d", kx_count, nx);
      return TMC_ERR_UNSUPPORTED;
    }
    if (int e = enable_smem(rows_forward_kernel<MM, BB>, smem)) return e;
    dim3 grid(tmc_div_up(yhi - ylo, batch_for(MM)), njobs);
    if (yhi > ylo) {
      TMC_TIMED("rows_forward_kernel", stream, rows_forward_kernel<MM, BB><<<grid, kThreads, smem, stream>>>(
          image, h, w, mean_std, mask, jobs, frame_shifts, x_margin, ylo, yhi, ny, kx_count, px, (float2*)tmp));
    }
    return TMC_OK;
  });
}

}  // namespace

// ---- C ABI ---------------------------------------------------------------------------------------

// 1: full transforms of this length are supported (a power of two up to 8192, any length up to 4096, or 2..8 times
//    such a length while the accumulators of the full spectrum fit in shared memory: up to 12158, and 12288, 16384);
// 2: band-limited transforms only (longer decimated axes, up to 32768);
// 0: unsupported
TMC_API int tmc_fft_supported_length(int n) {
  if (fft_size_for(n) > 0) return 1;
  const int R = decimation_for(n);
  if (R == 0) return 0;
  return decimated_full_fits(n) ? 1 : 2;
}

// complex64 elements of the plan buffer for a length-n transform (0: unsupported length)
TMC_API long tmc_fft_plan_elems(int n_total) {
  const int R = decimation_for(n_total);
  if (R == 0) return 0;
  const int n = n_total / R;
  const int m = fft_size_for(n);
  return m == n ? (long)m : 2l * m + n;
}

// fills `plan` (tmc_fft_plan_elems(n) complex64): twiddles [+ Bluestein chirp and filter spectrum]
TMC_API int tmc_fft_plan_init(int n_total, void* plan, cudaStream_t stream) {
  TMC_CHECK_ARG(plan, "fft_plan_init: null pointer");
  const int R = decimation_for(n_total);
  if (R == 0) {
    tmc_set_error("fft_plan_init: transform length %d is not supported", n_total);
    return TMC_ERR_UNSUPPORTED;
  }
  const int n = n_total / R;  // the plan serves the shared-memory transforms of the decimated axis
  const int m = fft_size_for(n);
  float2* tw = (float2*)plan;
  TMC_TIMED("twiddle_kernel", stream, twiddle_kernel<<<tmc_div_up(m, 128), 128, 0, stream>>>(m, tw));
  if (m != n) {
    float2* chirp = tw + m;
    float2* bhat = chirp + n;
    TMC_TIMED("chirp_kernel", stream, chirp_kernel<<<tmc_div_up(m, 128), 128, 0, stream>>>(n, m, chirp, bhat));
    // bhat <- FFT_m(bhat) in place (one row, plain power-of-two transform)
    AxisPlan p;
    p.tw = tw;
    p.chirp = nullptr;
    p.bhat = nullptr;
    p.n = m;
    p.R = 1;
    p.n_total = m;
    int rc = dispatch_fft(m, "fft_plan_init", [&](auto M, auto) {
      constexpr int MM = decltype(M)::value;
      if (int e = enable_smem(c2c_rows_kernel<MM, false>, fft_smem_bytes<MM>())) return e;
      TMC_TIMED("c2c_rows_kernel", stream, c2c_rows_kernel<MM, false><<<1, kThreads, fft_smem_bytes<MM>(), stream>>>(bhat, 1, p, bhat));
      return TMC_OK;
    });
    if (rc) return rc;
  }
  TMC_CHECK_LAUNCH("tmc_fft_plan_init");
  return TMC_OK;
}

// out[r] = DFT_n(in[r]) (inverse != 0: unnormalised inverse) for `rows` complex64 rows; in may equal out
TMC_API int tmc_fft_c2c_rows(const void* in, int rows, int n, const void* plan, void* out, cudaStream_t stream) {
  TMC_CHECK_ARG(in && out && plan && rows >= 1, "fft_c2c_rows: bad arguments");
  TMC_CHECK_ARG(fft_size_for(n) > 0, "fft_c2c_rows: full transforms need lengths up to 4096 or powers of two up to 8192, got %d", n);
  AxisPlan p = make_axis_plan(plan, n);
  int rc = dispatch_fft(n, "fft_c2c_rows", [&](auto M, auto BLU) {
    constexpr int MM = decltype(M)::value;
    constexpr bool BB = decltype(BLU)::value;
    if (int e = enable_smem(c2c_rows_kernel<MM, BB>, fft_smem_bytes<MM>())) return e;
    TMC_TIMED("c2c_rows_kernel", stream, c2c_rows_kernel<MM, BB><<<tmc_div_up(rows, batch_for(MM)), kThreads, fft_smem_bytes<MM>(), stream>>>(
        (const float2*)in, rows, p, (float2*)out));
    return TMC_OK;
  });
  if (rc) return rc;
  TMC_CHECK_LAUNCH("tmc_fft_c2c_rows");
  return TMC_OK;
}

// Band-limited forward 2-D real DFT of masked image windows.
//  image (T,H,W) f32; mean_std nullable device float[2]; mask (ny,nx) f32 nullable;
//  jobs (njobs,6) int32 device = {frame_a, exp_a, frame_b (-1: none), exp_b, y0, x0}; job_mode promises a
//  structure shared by ALL jobs (1: frame_b == frame_a, powers (1,2); 2: powers (1,1)) or 0 for generic;
//  frame_shifts nullable (t,2) int32 device = whole-pixel (dy, dx) added to the window origin of every frame (the
//  window wraps around the frame edges: identical to rolling the frame by an integer Fourier shift first, which is
//  what the reference's rigid pre-correction does, estimate_motion_xc.py:232-241); x_margin: the first and last
//  x_margin columns of the mask are all zero (0 if unknown);
//  rows [ylo,yhi) are the only non-zero rows of the mask; kx in [0,KX), ky in [ky_start, ky_start+KY);
//  weight (KY,KX) f32 nullable; plan_x/plan_y: tmc_fft_plan_init buffers for nx/ny;
//  tmp: 2*njobs*ny*KX complex64; out: (2*njobs, KY, KX) complex64, plane 2*job+0 = a, 2*job+1 = b.
TMC_API int tmc_rfft2_band(const float* image, int t, int h, int w, const float* mean_std, const float* mask, int ny, int nx,
                           const int* jobs, int njobs, int job_mode, const int* frame_shifts, int x_margin, int ylo, int yhi,
                           int kx_count, int ky_count, int ky_start, const float* weight, const void* plan_x,
                           const void* plan_y, void* tmp, void* out, cudaStream_t stream) {
  TMC_CHECK_ARG(image && jobs && plan_x && plan_y && tmp && out, "rfft2_band: null pointer");
  TMC_CHECK_ARG(job_mode >= 0 && job_mode <= 2, "rfft2_band: job_mode must be 0 (generic), 1 (mask powers 1,2 of one frame) or 2 (two frames)");
  TMC_CHECK_ARG(njobs >= 0 && t >= 1 && h >= ny && w >= nx, "rfft2_band: window (%d,%d) larger than image (%d,%d)", ny, nx, h, w);
  TMC_CHECK_ARG(0 <= ylo && ylo <= yhi && yhi <= ny, "rfft2_band: bad row support [%d,%d)", ylo, yhi);
  TMC_CHECK_ARG(x_margin >= 0 && 2 * x_margin <= nx, "rfft2_band: bad x_margin %d", x_margin);
  TMC_CHECK_ARG(kx_count >= 1 && kx_count <= nx / 2 + 1 && ky_count >= 1 && ky_count <= ny, "rfft2_band: bad band box");
  if (njobs == 0) return TMC_OK;
  constexpr int kMaxJobs = kMaxGridYZ / 2;  // the column pass puts 2 njobs planes on grid y
  if (njobs > kMaxJobs) {  // slices in stream order: each reuses tmp from the start
    for (int j0 = 0; j0 < njobs; j0 += kMaxJobs) {
      const int n = njobs - j0 < kMaxJobs ? njobs - j0 : kMaxJobs;
      if (int rc = tmc_rfft2_band(image, t, h, w, mean_std, mask, ny, nx, jobs + 6l * j0, n, job_mode, frame_shifts, x_margin,
                                  ylo, yhi, kx_count, ky_count, ky_start, weight, plan_x, plan_y, tmp,
                                  (float2*)out + 2l * j0 * ky_count * kx_count, stream))
        return rc;
    }
    return TMC_OK;
  }
  const AxisPlan px = make_axis_plan(plan_x, nx), py = make_axis_plan(plan_y, ny);
  int rc = rfft2_rows(image, h, w, mean_std, mask, ny, nx, jobs, njobs, job_mode, frame_shifts, x_margin, ylo, yhi, kx_count,
                      px, tmp, stream);
  if (rc) return rc;
  TMC_CHECK_LAUNCH("tmc_rfft2_band(rows)");
  rc = dispatch_fft(ny, "rfft2_band", [&](auto M, auto BLU) {
    constexpr int MM = decltype(M)::value;
    constexpr bool BB = decltype(BLU)::value;
    if constexpr (use_fast_path<MM, BB>()) if (py.R == 1) {
      if (int e = enable_smem(cols_forward_p2<MM>, fft2::Cfg<MM>::smem_bytes)) return e;
      dim3 grid(tmc_div_up(kx_count, fft2::Cfg<MM>::B), 2 * njobs);
      TMC_TIMED(sized_label<MM>("cols_forward_p2<4096>", "cols_forward_p2<1024>", "cols_forward_p2"), stream, cols_forward_p2<MM><<<grid, fft2::kThreads, fft2::Cfg<MM>::smem_bytes, stream>>>(
          (const float2*)tmp, ylo, yhi, kx_count, ky_count, ky_start, weight, py.tw, (float2*)out));
      return TMC_OK;
    }
    const size_t smem = fft_smem_bytes<MM>() + (py.R > 1 ? 1ull * batch_for(MM) * ky_count * sizeof(float2) : 0);
    if (smem > kMaxSmem) {
      tmc_set_error("rfft2_band: band of %d bins too wide for the decimated column transform of length %d", ky_count, ny);
      return TMC_ERR_UNSUPPORTED;
    }
    if (int e = enable_smem(cols_forward_kernel<MM, BB>, smem)) return e;
    dim3 grid(tmc_div_up(kx_count, batch_for(MM)), 2 * njobs);
    TMC_TIMED("cols_forward_kernel", stream, cols_forward_kernel<MM, BB><<<grid, kThreads, smem, stream>>>(
                  (const float2*)tmp, ylo, yhi, kx_count, ky_count, ky_start, weight, py, (float2*)out));
    return TMC_OK;
  });
  if (rc) return rc;
  TMC_CHECK_LAUNCH("tmc_rfft2_band(cols)");
  return TMC_OK;
}

// shifts[f] = (rint(scale * field[0][f]), rint(scale * field[1][f])) for a (2, t) field; *not_integer is set to 1 when
// some scaled value is further than 1e-4 from a whole number (the caller zeroes it first)
__global__ void integer_shifts_kernel(const float* __restrict__ field, int t, float scale, int* __restrict__ shifts,
                                      int* __restrict__ not_integer) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= t) return;
  const float sy = scale * field[f], sx = scale * field[t + f];
  const float ry = rintf(sy), rx = rintf(sx);
  shifts[2 * f] = (int)ry;
  shifts[2 * f + 1] = (int)rx;
  if (!(fabsf(sy - ry) <= 1e-4f && fabsf(sx - rx) <= 1e-4f && fabsf(ry) < 1e6f && fabsf(rx) < 1e6f)) *not_integer = 1;
}

// Whole-pixel window shifts for tmc_rfft2_band(frame_shifts) from a rigid (2, t, 1, 1) field: shifts (t, 2) int32,
// not_integer (device int, set to 0 / 1).  Replaces the rigid pre-correction pass of estimate_motion_xc.py:232-241 for
// fields that are whole pixels (the integer estimate of estimate_global_motion, quirk Q5).
TMC_API int tmc_integer_shifts(const float* field, int t, float scale, int* shifts, int* not_integer, cudaStream_t stream) {
  TMC_CHECK_ARG(field && shifts && not_integer && t >= 1, "integer_shifts: bad arguments");
  TMC_CUDA(cudaMemsetAsync(not_integer, 0, sizeof(int), stream));
  TMC_TIMED("integer_shifts_kernel", stream, integer_shifts_kernel<<<tmc_div_up(t, 128), 128, 0, stream>>>(field, t, scale, shifts, not_integer));
  TMC_CHECK_LAUNCH("tmc_integer_shifts");
  return TMC_OK;
}

// out[i] = conj(spec[ref_plane[i]]) * spec[cur_plane[i]], planes of plane_elems complex64
TMC_API int tmc_xc_pair_products(const void* spec, const int* ref_plane, const int* cur_plane, int nitems, long plane_elems,
                                 void* out, cudaStream_t stream) {
  TMC_CHECK_ARG(spec && ref_plane && cur_plane && out && nitems >= 0 && plane_elems >= 1, "xc_pair_products: bad arguments");
  if (nitems == 0) return TMC_OK;
  if (nitems > kMaxGridYZ) {
    for (int i0 = 0; i0 < nitems; i0 += kMaxGridYZ) {
      const int n = nitems - i0 < kMaxGridYZ ? nitems - i0 : kMaxGridYZ;
      if (int rc = tmc_xc_pair_products(spec, ref_plane + i0, cur_plane + i0, n, plane_elems, (float2*)out + i0 * plane_elems,
                                        stream))
        return rc;
    }
    return TMC_OK;
  }
  dim3 grid((unsigned)(tmc_div_up(plane_elems, 256) < 64 ? tmc_div_up(plane_elems, 256) : 64), nitems);
  TMC_TIMED("xc_pair_product_kernel", stream, xc_pair_product_kernel<<<grid, 256, 0, stream>>>((const float2*)spec, ref_plane, cur_plane, plane_elems, (float2*)out));
  TMC_CHECK_LAUNCH("tmc_xc_pair_products");
  return TMC_OK;
}

// spec planes [T][G][2]; out items [k_count][G] for frames k_begin .. k_begin + k_count - 1;
// delta lists: offsets (T+1) and signed (j+1) entries
TMC_API int tmc_xc_leave_one_out_products(const void* spec, int t, int g, long plane_elems, const int* delta_offsets,
                                          const int* deltas, int k_begin, int k_count, void* out, cudaStream_t stream) {
  TMC_CHECK_ARG(spec && delta_offsets && deltas && out && t >= 2 && g >= 1 && plane_elems >= 1,
                "xc_leave_one_out_products: bad arguments (need t >= 2)");
  TMC_CHECK_ARG(k_begin >= 0 && k_count >= 0 && k_begin + k_count <= t, "xc_leave_one_out_products: bad frame range");
  TMC_CHECK_ARG(g <= kMaxGridYZ, "xc_leave_one_out_products: at most %d patches per frame, got %d", kMaxGridYZ, g);
  if (k_count == 0) return TMC_OK;
  dim3 grid(tmc_div_up(plane_elems, 128), g);
  TMC_TIMED("xc_leave_one_out_kernel", stream, xc_leave_one_out_kernel<<<grid, 128, 0, stream>>>((const float2*)spec, t, g, plane_elems, delta_offsets, deltas,
                                                    k_begin, k_count, (float2*)out));
  TMC_CHECK_LAUNCH("tmc_xc_leave_one_out_products");
  return TMC_OK;
}

TMC_API int tmc_xc_peak_partials(int ny, int nx) {
  const int R = decimation_for(nx);
  if (R == 0) return -1;
  const int m = fft_size_for(nx / R);
  if (R == 1 && m == nx && m >= 256) {  // power-of-two fast path: several row-pair batches per CTA
    const int b = 256 / (m / 16) > 0 ? 256 / (m / 16) : 1;
    if (m == 8192 || m == 4096) {  // may run as half-length transforms, one row each (rows_inverse_argmax_real2n): more CTAs
      const int bh = 256 / (m / 32) > 0 ? 256 / (m / 32) : 1;
      return tmc_div_up(ny, bh * kRowIters);
    }
    return tmc_div_up(ny, 2 * b * kRowIters);
  }
  return tmc_div_up(ny, 2 * batch_for(m));
}

// Inverse 2-D transform of band-limited products + argmax (+ parabola) + wrap.
//  prod (nitems, KY, KX) complex64; tmp: nitems*ny*KX complex64; partial: nitems*tmc_xc_peak_partials(ny,nx)*8 bytes;
//  shifts (nitems, 2) f32 = (dy, dx) px.
TMC_API int tmc_xc_peaks(const void* prod, int nitems, int ny, int nx, int kx_count, int ky_count, int ky_start,
                         int sub_pixel, const void* plan_x, const void* plan_y, void* tmp, void* partial, float* shifts,
                         cudaStream_t stream) {
  TMC_CHECK_ARG(prod && plan_x && plan_y && tmp && partial && shifts, "xc_peaks: null pointer");
  TMC_CHECK_ARG(kx_count >= 1 && kx_count <= nx / 2 + 1 && ky_count >= 1 && ky_count <= ny, "xc_peaks: bad band box");
  if (nitems == 0) return TMC_OK;
  if (nitems > kMaxGridYZ) {  // slices in stream order: each reuses tmp and partial from the start
    for (int i0 = 0; i0 < nitems; i0 += kMaxGridYZ) {
      const int n = nitems - i0 < kMaxGridYZ ? nitems - i0 : kMaxGridYZ;
      if (int rc = tmc_xc_peaks((const float2*)prod + (long)i0 * ky_count * kx_count, n, ny, nx, kx_count, ky_count, ky_start,
                                sub_pixel, plan_x, plan_y, tmp, partial, shifts + 2l * i0, stream))
        return rc;
    }
    return TMC_OK;
  }
  const AxisPlan px = make_axis_plan(plan_x, nx), py = make_axis_plan(plan_y, ny);
  int rc = dispatch_fft(ny, "xc_peaks", [&](auto M, auto BLU) {
    constexpr int MM = decltype(M)::value;
    constexpr bool BB = decltype(BLU)::value;
    if constexpr (use_fast_path<MM, BB>()) if (py.R == 1) {
      if (int e = enable_smem(cols_inverse_p2<MM>, fft2::Cfg<MM>::smem_bytes)) return e;
      dim3 grid(tmc_div_up(kx_count, fft2::Cfg<MM>::B), nitems);
      TMC_TIMED(sized_label<MM>("cols_inverse_p2<4096>", "cols_inverse_p2<1024>", "cols_inverse_p2"), stream, cols_inverse_p2<MM><<<grid, fft2::kThreads, fft2::Cfg<MM>::smem_bytes, stream>>>(
          (const float2*)prod, kx_count, ky_count, ky_start, py.tw, (float2*)tmp));
      return TMC_OK;
    }
    if (int e = enable_smem(cols_inverse_kernel<MM, BB>, fft_smem_bytes<MM>())) return e;
    dim3 grid(tmc_div_up(kx_count, batch_for(MM)), nitems);
    TMC_TIMED("cols_inverse_kernel", stream, cols_inverse_kernel<MM, BB><<<grid, kThreads, fft_smem_bytes<MM>(), stream>>>((const float2*)prod, kx_count, ky_count, ky_start,
                                                                                 py, (float2*)tmp));
    return TMC_OK;
  });
  if (rc) return rc;
  TMC_CHECK_LAUNCH("tmc_xc_peaks(cols)");
  int nparts = tmc_xc_peak_partials(ny, nx);  // size of the caller's buffer per item; the kernel chosen may use fewer
  rc = dispatch_fft(nx, "xc_peaks", [&](auto M, auto BLU) {
    constexpr int MM = decltype(M)::value;
    constexpr bool BB = decltype(BLU)::value;
    if constexpr ((MM == 8192 || MM == 4096) && !BB) {
      // one row per half-length transform instead of two rows per full-length transform (see rows_forward_real2n)
      if (px.R == 1 && kx_count <= MM / 4 && use_real2n(MM)) {
        constexpr int NH = MM / 2;
        if (int e = enable_smem(rows_inverse_argmax_real2n<NH>, rows_inverse_real2n_smem_bytes<NH>())) return e;
        nparts = tmc_div_up(ny, rows_per_cta_inverse_real2n<NH>());
        dim3 grid(nparts, nitems);
        TMC_TIMED(MM == 8192 ? "rows_inverse_argmax_real2n<4096>" : "rows_inverse_argmax_real2n<2048>", stream,
                  rows_inverse_argmax_real2n<NH><<<grid, fft2::kThreads, rows_inverse_real2n_smem_bytes<NH>(), stream>>>(
                      (const float2*)tmp, ny, kx_count, px.tw, (PeakCandidate*)partial));
        return TMC_OK;
      }
      // the full-length p2 kernel below; a decimated axis (R > 1) runs the generic kernel, two rows per CTA
      if (px.R == 1) nparts = tmc_div_up(ny, rows_per_cta_inverse<MM>());
    }
    if constexpr (MM == 1024 && !BB) {
      if (kx_count <= 128 && use_poly() && px.R == 1) {
        if (int e = enable_smem(poly::rows_inverse_argmax_poly, poly::smem_bytes)) return e;
        dim3 grid(nparts, nitems);
        TMC_TIMED("rows_inverse_argmax_poly", stream, poly::rows_inverse_argmax_poly<<<grid, poly::kThreads, poly::smem_bytes, stream>>>((const float2*)tmp, ny, kx_count, px.tw,
                                                                                         (PeakCandidate*)partial));
        return TMC_OK;
      }
    }
    if constexpr (use_fast_path<MM, BB>()) if (px.R == 1) {
      if (int e = enable_smem(rows_inverse_argmax_p2<MM>, rows_inverse_smem_bytes<MM>())) return e;
      dim3 grid(nparts, nitems);
      TMC_TIMED(sized_label<MM>("rows_inverse_argmax_p2<4096>", "rows_inverse_argmax_p2<1024>", "rows_inverse_argmax_p2"), stream, rows_inverse_argmax_p2<MM><<<grid, fft2::kThreads, rows_inverse_smem_bytes<MM>(), stream>>>(
          (const float2*)tmp, ny, kx_count, px.tw, (PeakCandidate*)partial));
      return TMC_OK;
    }
    if (int e = enable_smem(rows_inverse_argmax_kernel<MM, BB>, fft_smem_bytes<MM>())) return e;
    dim3 grid(nparts, nitems);
    TMC_TIMED("rows_inverse_argmax_kernel", stream, rows_inverse_argmax_kernel<MM, BB><<<grid, kThreads, fft_smem_bytes<MM>(), stream>>>((const float2*)tmp, ny, kx_count, px,
                                                                                        (PeakCandidate*)partial));
    return TMC_OK;
  });
  if (rc) return rc;
  TMC_CHECK_LAUNCH("tmc_xc_peaks(rows)");
  TMC_TIMED("peak_finalize_kernel", stream, peak_finalize_kernel<<<nitems, 128, 0, stream>>>((const float2*)tmp, (const PeakCandidate*)partial, nparts, ny, nx,
                                                   kx_count, sub_pixel, shifts));
  TMC_CHECK_LAUNCH("tmc_xc_peaks(finalize)");
  return TMC_OK;
}

namespace {

// inverse column pass of a (nitems, KY, KX) box (ky = ky_start + kyb, the box spans every ky of length ny) -> tmp
// (nitems, ny, KX); entries beyond the box are zero
int irfft2_cols(const void* spec, int nitems, int ny, int KX, int KY, int ky_start, const AxisPlan& py, void* tmp,
                cudaStream_t stream, const char* who) {
  return dispatch_fft(ny, who, [&](auto M, auto BLU) {
    constexpr int MM = decltype(M)::value;
    constexpr bool BB = decltype(BLU)::value;
    if constexpr (use_fast_path<MM, BB>()) if (py.R == 1) {
      if (int e = enable_smem(cols_inverse_p2<MM>, fft2::Cfg<MM>::smem_bytes)) return e;
      dim3 grid(tmc_div_up(KX, fft2::Cfg<MM>::B), nitems);
      TMC_TIMED(sized_label<MM>("cols_inverse_p2<4096>", "cols_inverse_p2<1024>", "cols_inverse_p2"), stream, cols_inverse_p2<MM><<<grid, fft2::kThreads, fft2::Cfg<MM>::smem_bytes, stream>>>((const float2*)spec, KX, KY, ky_start, py.tw,
                                                                                      (float2*)tmp));
      return TMC_OK;
    }
    if (int e = enable_smem(cols_inverse_kernel<MM, BB>, fft_smem_bytes<MM>())) return e;
    dim3 grid(tmc_div_up(KX, batch_for(MM)), nitems);
    TMC_TIMED("cols_inverse_kernel", stream, cols_inverse_kernel<MM, BB><<<grid, kThreads, fft_smem_bytes<MM>(), stream>>>((const float2*)spec, KX, KY, ky_start, py, (float2*)tmp));
    return TMC_OK;
  });
}

// c2r row pass: tmp (nitems, ny, KX) -> out (nitems, ny, nx) f32 times `scale`.  Keeps only the real part of the
// kx = 0 and kx = nx/2 entries, as c2r does.
int irfft2_rows(const void* tmp, int nitems, int ny, int nx, int KX, const AxisPlan& px, float scale, float* out,
                cudaStream_t stream, const char* who) {
  return dispatch_fft(nx, who, [&](auto M, auto BLU) {
    constexpr int MM = decltype(M)::value;
    constexpr bool BB = decltype(BLU)::value;
    if constexpr (use_fast_path<MM, BB>()) if (px.R == 1) {
      if (int e = enable_smem(rows_inverse_store_p2<MM>, rows_inverse_smem_bytes<MM>())) return e;
      dim3 grid(tmc_div_up(ny, rows_per_cta_inverse<MM>()), nitems);
      TMC_TIMED(sized_label<MM>("rows_inverse_store_p2<4096>", "rows_inverse_store_p2<1024>", "rows_inverse_store_p2"), stream, rows_inverse_store_p2<MM><<<grid, fft2::kThreads, rows_inverse_smem_bytes<MM>(), stream>>>(
          (const float2*)tmp, ny, KX, px.tw, scale, out));
      return TMC_OK;
    }
    if (int e = enable_smem(rows_inverse_store_kernel<MM, BB>, fft_smem_bytes<MM>())) return e;
    dim3 grid(tmc_div_up(ny, 2 * batch_for(MM)), nitems);
    TMC_TIMED("rows_inverse_store_kernel", stream, rows_inverse_store_kernel<MM, BB><<<grid, kThreads, fft_smem_bytes<MM>(), stream>>>((const float2*)tmp, ny, KX, px,
                                                                                       scale, out));
    return TMC_OK;
  });
}

}  // namespace

// Full inverse: spec (nitems, ny, nx/2+1) complex64 -> out (nitems, ny, nx) f32 (irfftn, backward norm)
TMC_API int tmc_irfft2_full(const void* spec, int nitems, int ny, int nx, const void* plan_x, const void* plan_y, void* tmp,
                            float* out, cudaStream_t stream) {
  TMC_CHECK_ARG(spec && plan_x && plan_y && tmp && out, "irfft2_full: null pointer");
  if (nitems == 0) return TMC_OK;
  if (nitems > kMaxGridYZ) {  // slices in stream order: each reuses tmp from the start
    for (int i0 = 0; i0 < nitems; i0 += kMaxGridYZ) {
      const int n = nitems - i0 < kMaxGridYZ ? nitems - i0 : kMaxGridYZ;
      if (int rc = tmc_irfft2_full((const float2*)spec + (long)i0 * ny * (nx / 2 + 1), n, ny, nx, plan_x, plan_y, tmp,
                                   out + (long)i0 * ny * nx, stream))
        return rc;
    }
    return TMC_OK;
  }
  const AxisPlan px = make_axis_plan(plan_x, nx), py = make_axis_plan(plan_y, ny);
  if (int rc = irfft2_cols(spec, nitems, ny, nx / 2 + 1, ny, 0, py, tmp, stream, "irfft2_full")) return rc;
  if (int rc = irfft2_rows(tmp, nitems, ny, nx, nx / 2 + 1, px, 1.0f / ((float)nx * (float)ny), out, stream, "irfft2_full"))
    return rc;
  TMC_CHECK_LAUNCH("tmc_irfft2_full");
  return TMC_OK;
}

// Fourier crop ("binning") of whole frames: bytes of the workspace tmc_fourier_crop needs for t frames
TMC_API long tmc_fourier_crop_workspace_bytes(int t, int h, int w, int out_h, int out_w) {
  if (t < 1 || h < 1 || w < 1 || out_h < 1 || out_w < 2) return -1;
  const long planes = 2l * ((t + 1) / 2);
  return planes * ((long)h + out_h) * (out_w / 2 + 1) * (long)sizeof(float2);
}

namespace {

// TMC_FFT_CROP_FUSED=0 selects the composed column passes of tmc_fourier_crop where the fused kernel would run (A/B
// testing; read per call: tests toggle it)
inline bool use_crop_fused() {
  const char* e = getenv("TMC_FFT_CROP_FUSED");
  return !(e && e[0] == '0');
}

// calls f(IntC<N>{}, IntC<M>{}) when cols_crop_p2<N, M> serves a crop of h rows to out_h rows (powers of two, out_h h/2
// or h/4 and >= 256); returns -1 without calling f otherwise
template <typename F>
int dispatch_crop_cols(int h, int out_h, F&& f) {
#define TMC_CROP_CASE(NN, MM) \
  if (h == NN && out_h == MM) return f(IntC<NN>{}, IntC<MM>{});
  TMC_CROP_CASE(512, 256) TMC_CROP_CASE(1024, 512) TMC_CROP_CASE(1024, 256) TMC_CROP_CASE(2048, 1024)
  TMC_CROP_CASE(2048, 512) TMC_CROP_CASE(4096, 2048) TMC_CROP_CASE(4096, 1024) TMC_CROP_CASE(8192, 4096)
  TMC_CROP_CASE(8192, 2048)
#undef TMC_CROP_CASE
  return -1;
}

}  // namespace

// image (t, h, w) f32 -> out (t, out_h, out_w) f32: rfft2, keep ky in [-out_h/2, out_h/2) and kx in [0, out_w/2], irfft2 at
// (out_h, out_w), times out_h out_w / (h w) (the mean pixel value is kept).  Passes: rows r2c keeping kx <= out_w/2
// (tmc_rfft2_band's row pass); the columns, fused (cols_crop_p2: forward at h, keep the ky box, inverse at out_h, in one
// kernel) for the power-of-two crops dispatch_crop_cols lists, otherwise forward at h into the ky box and inverse at
// out_h as two passes; rows c2r at out_w.
// The box is not Hermitian on its self-paired columns kx = 0 and kx = out_w/2 (and ky = -out_h/2 has no partner); the
// c2r row pass keeps only the real part of those columns' inverse, which is the inverse of their Hermitian part, as
// numpy's and torch's irfft2 do.
// jobs: frame-pair jobs (tmc_rfft2_band format, job_mode 2) covering the t frames in order (plane index == frame index
// relative to out); workspace: tmc_fourier_crop_workspace_bytes(t, ...); plan_*: tmc_fft_plan_init buffers for w, h,
// out_w, out_h.
TMC_API int tmc_fourier_crop(const float* image, int t, int h, int w, int out_h, int out_w, const int* jobs, int njobs,
                             const void* plan_x, const void* plan_y, const void* plan_x_out, const void* plan_y_out,
                             void* workspace, float* out, cudaStream_t stream) {
  TMC_CHECK_ARG(image && jobs && plan_x && plan_y && plan_x_out && plan_y_out && workspace && out,
                "fourier_crop: null pointer");
  TMC_CHECK_ARG(t >= 1 && 2 * njobs >= t && njobs <= (t + 1) / 2, "fourier_crop: jobs do not cover the frames");
  TMC_CHECK_ARG(h >= 2 && w >= 2 && h % 2 == 0 && w % 2 == 0 && out_h >= 2 && out_w >= 2 && out_h % 2 == 0 &&
                    out_w % 2 == 0,
                "fourier_crop: sides must be even, got (%d, %d) -> (%d, %d)", h, w, out_h, out_w);
  TMC_CHECK_ARG(out_h <= h && out_w <= w, "fourier_crop: output (%d, %d) larger than the input (%d, %d)", out_h, out_w, h, w);
  TMC_CHECK_ARG(t <= kMaxGridYZ, "fourier_crop: at most %d frames per call, got %d", kMaxGridYZ, t);
  for (int n : {h, w, out_h, out_w})
    if (tmc_fft_supported_length(n) != 1) {
      tmc_set_error("fourier_crop: transform length %d is not supported for full-spectrum transforms", n);
      return TMC_ERR_UNSUPPORTED;
    }
  const int KX = out_w / 2 + 1;
  float2* rows = (float2*)workspace;                       // (2 njobs, h, KX), then (t, out_h, KX)
  float2* box = rows + 2l * njobs * h * KX;                // (2 njobs, out_h, KX)
  const AxisPlan px_in = make_axis_plan(plan_x, w), py_in = make_axis_plan(plan_y, h);
  const AxisPlan px = make_axis_plan(plan_x_out, out_w), py = make_axis_plan(plan_y_out, out_h);
  const float scale = 1.0f / ((float)h * (float)w);
  int rc = use_crop_fused() ? dispatch_crop_cols(h, out_h, [&](auto N, auto M) { return 0; }) : -1;
  if (rc == 0) {
    if ((rc = rfft2_rows(image, h, w, nullptr, nullptr, h, w, jobs, njobs, 2, nullptr, 0, 0, h, KX, px_in, rows, stream)))
      return rc;
    rc = dispatch_crop_cols(h, out_h, [&](auto N, auto M) {
      constexpr int NN = decltype(N)::value, MM = decltype(M)::value;
      constexpr size_t smem = cols_crop_smem_bytes<NN, MM>();
      if (int e = enable_smem(cols_crop_p2<NN, MM>, smem)) return e;
      dim3 grid(tmc_div_up(KX, fft2::Cfg<MM>::B), t);
      TMC_TIMED("cols_crop_p2", stream, cols_crop_p2<NN, MM><<<grid, fft2::kThreads, smem, stream>>>(
          (const float2*)rows, KX, py_in.tw, py.tw, box));
      return TMC_OK;
    });
    if (rc) return rc;
    rc = irfft2_rows(box, t, out_h, out_w, KX, px, scale, out, stream, "fourier_crop");
  } else {
    if ((rc = tmc_rfft2_band(image, t, h, w, nullptr, nullptr, h, w, jobs, njobs, 2, nullptr, 0, 0, h, KX, out_h,
                             -(out_h / 2), nullptr, plan_x, plan_y, rows, box, stream)))
      return rc;
    if ((rc = irfft2_cols(box, t, out_h, KX, out_h, -(out_h / 2), py, rows, stream, "fourier_crop"))) return rc;
    rc = irfft2_rows(rows, t, out_h, out_w, KX, px, scale, out, stream, "fourier_crop");
  }
  if (rc) return rc;
  TMC_CHECK_LAUNCH("tmc_fourier_crop");
  return TMC_OK;
}

// spec (t, ny, nx/2+1) *= exp(-2 pi i (fy sy + fx sx)); (sy, sx) = sign * field (2, t) (device)
TMC_API int tmc_fourier_shift(void* spec, int t, int ny, int nx, const float* field, float sign, cudaStream_t stream) {
  TMC_CHECK_ARG(spec && field && t >= 1 && ny >= 1 && nx >= 2, "fourier_shift: bad arguments");
  TMC_CHECK_ARG(t <= kMaxGridYZ && ny <= kMaxGridYZ, "fourier_shift: at most %d frames and rows, got (%d, %d)", kMaxGridYZ, t, ny);
  const int kx = nx / 2 + 1;
  dim3 grid(tmc_div_up(kx, 128), ny, t);
  TMC_TIMED("fourier_shift_kernel", stream, fourier_shift_kernel<<<grid, 128, 0, stream>>>((float2*)spec, t, ny, nx, kx, field, sign));
  TMC_CHECK_LAUNCH("tmc_fourier_shift");
  return TMC_OK;
}

// 1 when tmc_fourier_shift_frames has a fused implementation for (ny, nx) (power-of-two fast path)
TMC_API int tmc_fourier_shift_frames_supported(int ny, int nx) {
  return (fft_size_for(ny) == ny && ny >= 256 && fft_size_for(nx) == nx && nx >= 256) ? 1 : 0;
}

// correct_motion_fast in three passes: rows r2c -> columns (FFT, phase, inverse FFT) -> rows c2r.
//  image (t, ny, nx) f32 (normalised on load with mean_std, nullable); field (2, t) px shifts, applied as
//  sign * field; jobs: frame-pair jobs (tmc_rfft2_band format, job_mode 2) covering the t frames in order;
//  tmp: 2 * njobs * ny * (nx/2+1) complex64; phase: t * ny complex64; out (t, ny, nx) f32.
TMC_API int tmc_fourier_shift_frames(const float* image, int t, int ny, int nx, const float* mean_std, const int* jobs,
                                     int njobs, const float* field, float sign, const void* plan_x, const void* plan_y,
                                     void* tmp, void* phase, float* out, cudaStream_t stream) {
  TMC_CHECK_ARG(image && jobs && field && plan_x && plan_y && tmp && phase && out, "fourier_shift_frames: null pointer");
  TMC_CHECK_ARG(t >= 1 && 2 * njobs >= t, "fourier_shift_frames: jobs do not cover the frames");
  TMC_CHECK_ARG(t <= kMaxGridYZ && njobs <= kMaxGridYZ, "fourier_shift_frames: at most %d frames per call, got %d", kMaxGridYZ, t);
  if (!tmc_fourier_shift_frames_supported(ny, nx)) {
    tmc_set_error("fourier_shift_frames: fused path needs power-of-two frame sides >= 256, got (%d, %d)", ny, nx);
    return TMC_ERR_UNSUPPORTED;
  }
  const int kx = nx / 2 + 1;
  const AxisPlan px = make_axis_plan(plan_x, nx), py = make_axis_plan(plan_y, ny);
  int rc = dispatch_fft(nx, "fourier_shift_frames", [&](auto M, auto BLU) {
    constexpr int MM = decltype(M)::value;
    if constexpr (use_fast_path<MM, decltype(BLU)::value>()) {
      constexpr int B = fft2::Cfg<MM>::B;
      int rows_per_cta = B * 4;
      while (rows_per_cta > B && (long)tmc_div_up(ny, rows_per_cta) * njobs < 148 * 8) rows_per_cta -= B;
      constexpr size_t smem = rows_forward_smem_bytes<MM>();
      if (int e = enable_smem(rows_forward_p2<MM, 2>, smem)) return e;
      dim3 grid(tmc_div_up(ny, rows_per_cta), njobs);
      TMC_TIMED("rows_forward_p2", stream, rows_forward_p2<MM, 2><<<grid, fft2::kThreads, smem, stream>>>(image, ny, nx, mean_std, nullptr, jobs, nullptr, 0, 0, ny, ny,
                                                                    kx, px.tw, (float2*)tmp, rows_per_cta));
    }
    return TMC_OK;
  });
  if (rc) return rc;
  {
    dim3 grid(tmc_div_up(ny, 128), t);
    TMC_TIMED("shift_phase_y_kernel", stream, shift_phase_y_kernel<<<grid, 128, 0, stream>>>(field, t, ny, sign, (float2*)phase));
  }
  rc = dispatch_fft(ny, "fourier_shift_frames", [&](auto M, auto BLU) {
    constexpr int MM = decltype(M)::value;
    if constexpr (MM == 4096 && !decltype(BLU)::value) {
      if (use_col_quads()) {
        constexpr size_t smem = (size_t)(4 * fft2::Cfg<MM>::STRIDE + 64 + fft2::Cfg<MM>::TW_HI) * sizeof(float2);
        if (int e = enable_smem(cols_shift_quad_p2<MM>, smem)) return e;
        dim3 grid(tmc_div_up(kx, 4), t);
        TMC_TIMED("cols_shift_quad_p2", stream,
                  cols_shift_quad_p2<MM><<<grid, 512, smem, stream>>>((float2*)tmp, kx, nx, (const float2*)phase, field, t, sign, py.tw));
        return TMC_OK;
      }
    }
    if constexpr (use_fast_path<MM, decltype(BLU)::value>()) {
      if (int e = enable_smem(cols_shift_p2<MM>, fft2::Cfg<MM>::smem_bytes)) return e;
      dim3 grid(tmc_div_up(kx, fft2::Cfg<MM>::B), t);
      TMC_TIMED(sized_label<MM>("cols_shift_p2<4096>", "cols_shift_p2<1024>", "cols_shift_p2"), stream, cols_shift_p2<MM><<<grid, fft2::kThreads, fft2::Cfg<MM>::smem_bytes, stream>>>((float2*)tmp, kx, nx, (const float2*)phase,
                                                                                    field, t, sign, py.tw));
    }
    return TMC_OK;
  });
  if (rc) return rc;
  rc = dispatch_fft(nx, "fourier_shift_frames", [&](auto M, auto BLU) {
    constexpr int MM = decltype(M)::value;
    if constexpr (use_fast_path<MM, decltype(BLU)::value>()) {
      if (int e = enable_smem(rows_inverse_store_p2<MM>, rows_inverse_smem_bytes<MM>())) return e;
      dim3 grid(tmc_div_up(ny, rows_per_cta_inverse<MM>()), t);
      TMC_TIMED(sized_label<MM>("rows_inverse_store_p2<4096>", "rows_inverse_store_p2<1024>", "rows_inverse_store_p2"), stream, rows_inverse_store_p2<MM><<<grid, fft2::kThreads, rows_inverse_smem_bytes<MM>(), stream>>>(
          (const float2*)tmp, ny, kx, px.tw, 1.0f / ((float)nx * (float)ny), out));
    }
    return TMC_OK;
  });
  if (rc) return rc;
  TMC_CHECK_LAUNCH("tmc_fourier_shift_frames");
  return TMC_OK;
}

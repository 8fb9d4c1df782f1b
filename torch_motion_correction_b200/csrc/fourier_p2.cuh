// Power-of-two fast-path kernels on fft_core2.cuh (included by fourier.cu inside its anonymous
// namespace).  Same contracts as the generic kernels of the same name without the _p2 suffix.
#pragma once

// ---- forward rows: image window * mask^e (two real signals packed) -> tmp[plane][y][kx < KX] --------
//
// MODE 0: generic jobs {frame_a, power_a, frame_b, power_b}; 1: frame_b == frame_a with powers (1, 2)
// (the leave-one-out pair of quirk Q1); 2: two frames (or one, frame_b < 0), power 1 each.
// The pixels / mask values of the NEXT batch of rows are prefetched with cp.async into per-thread
// shared-memory slots while the current batch is being transformed (global-load latency was the
// dominant stall of the first version: profiles/r01_*).

__device__ __forceinline__ void cp_async_f32(float* smem_dst, const float* gmem_src) {
  const unsigned dst = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(dst), "l"(gmem_src));
}
__device__ __forceinline__ void cp_async_commit_and_wait() {
  asm volatile("cp.async.commit_group;\n" ::);
  asm volatile("cp.async.wait_group 0;\n" ::: "memory");
}

template <int N>
constexpr size_t rows_forward_smem_bytes() {
  return fft2::Cfg<N>::smem_bytes + 3ull * fft2::Cfg<N>::B * N * sizeof(float);
}

// 4096-point rows: uncapped the kernel takes 217 registers (1 CTA per SM, 12 % occupancy); at 128 registers two CTAs are
// resident and the whole-frame estimate is 0.4 ms faster (measured, C2)
template <int N, int MODE>
__global__ void __launch_bounds__(fft2::kThreads, N == 4096 ? 2 : 1)
rows_forward_p2(const float* __restrict__ image, int H, int W, const float* __restrict__ mean_std,
                const float* __restrict__ mask, const int* __restrict__ jobs, const int* __restrict__ frame_shifts,
                int x_margin, int ylo, int yhi, int NY, int KX, const float2* __restrict__ tw, float2* __restrict__ tmp,
                int rows_per_cta) {
  using C = fft2::Cfg<N>;
  using P = fft2::Plan<N>;
  extern __shared__ float2 smem[];
  const fft2::Smem<N> sm(smem);
  fft2::load_twiddles<N>(sm, tw);
  const int seq = threadIdx.x / C::TPS, j = threadIdx.x % C::TPS;
  float2* myseq = sm.data + seq * C::STRIDE;
  // per-thread staging slots: element e of this thread lives at stage_x[e * kThreads + threadIdx.x]
  float* stage_a = reinterpret_cast<float*>(smem + C::B * C::STRIDE + 64 + C::TW_HI);
  float* stage_b = stage_a + C::B * N;
  float* stage_m = stage_b + C::B * N;
  const int job = blockIdx.y;
  const int fa = jobs[job * 6 + 0], ea = jobs[job * 6 + 1], fb = jobs[job * 6 + 2], eb = jobs[job * 6 + 3];
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
  const bool separate_b = has_b && (MODE == 2 || (MODE == 0 && fb != fa));
  const float* img_b = wb.fast_base(W);
  const int row_begin = ylo + blockIdx.x * rows_per_cta;
  const int row_end = min(yhi, row_begin + rows_per_cta);
  float2* plane_a = tmp + (long)(2 * job) * NY * KX;
  float2* plane_b = plane_a + (long)NY * KX;

  auto prefetch = [&](int row0) {
    const int y = row0 + seq;
    if (y < row_end) {
#pragma unroll
      for (int e = 0; e < C::VPT; ++e) {
        const int x = P::First::in_index(j, e / P::First::R, e % P::First::R);
        const int slot = e * fft2::kThreads + threadIdx.x;
        cp_async_f32(stage_a + slot, wa.wrap ? wa.wrapped(y, x, H, W) : img_a + (long)y * W + x);
        if (separate_b) cp_async_f32(stage_b + slot, wb.wrap ? wb.wrapped(y, x, H, W) : img_b + (long)y * W + x);
        if (mask) cp_async_f32(stage_m + slot, mask + (long)y * N + x);
      }
    }
  };
  prefetch(row_begin);
  __syncthreads();  // twiddle tables
  for (int row0 = row_begin; row0 < row_end; row0 += C::B) {
    const int y = row0 + seq;
    const bool active = y < row_end;
    cp_async_commit_and_wait();
    float2 v[C::VPT];
#pragma unroll
    for (int e = 0; e < C::VPT; ++e) {
      float2 z = make_float2(0.f, 0.f);
      if (active) {
        const int slot = e * fft2::kThreads + threadIdx.x;
        const float m = mask ? stage_m[slot] : 1.0f;
        const float pa = (stage_a[slot] - mean) * inv_std;
        if (MODE == 1) {
          z.x = pa * m;
          z.y = z.x * m;
        } else if (MODE == 2) {
          z.x = pa * m;
          if (has_b) z.y = (stage_b[slot] - mean) * inv_std * m;
        } else {
          float va = pa;
          for (int k = 0; k < ea; ++k) va *= m;
          z.x = va;
          if (has_b) {
            float vb = separate_b ? (stage_b[slot] - mean) * inv_std : pa;
            for (int k = 0; k < eb; ++k) vb *= m;
            z.y = vb;
          }
        }
      }
      v[e] = z;
    }
    if (row0 + C::B < row_end) prefetch(row0 + C::B);  // overlaps with the transform below
    fft2::fft_regs_to_regs<N>(sm, myseq, j, v);
    __syncthreads();
    P::Last::store(myseq, j, v);
    __syncthreads();
    if (active) {
      for (int k = j; k < KX; k += C::TPS) {
        const float2 zk = myseq[fft2::pad_idx(k)];
        const float2 zn = myseq[fft2::pad_idx(k == 0 ? 0 : N - k)];
        plane_a[(long)y * KX + k] = make_float2(0.5f * (zk.x + zn.x), 0.5f * (zk.y - zn.y));
        if (has_b) plane_b[(long)y * KX + k] = make_float2(0.5f * (zk.y + zn.y), -0.5f * (zk.x - zn.x));
      }
    }
    __syncthreads();
  }
}

// ---- forward rows of length 2N as N-point complex transforms (one real row per transform) -------------------------
//
// x[0 .. 2N) real, z[m] = x[2m] + i x[2m+1], Z = DFT_N(z):  X[k] = E[k] + W_2N^k O[k] with
// E[k] = (Z[k] + conj Z[N-k]) / 2 (spectrum of the even samples), O[k] = (Z[k] - conj Z[N-k]) / 2i (odd samples).
// Same job format and output as rows_forward_p2<2N, 2> (two frames per job, mask power 1), but the two frames are two
// N-point transforms instead of one 2N-point transform of a packed pair: the 8192-point kernel holds 32 values per thread
// and 168 KB of shared memory (one 8-warp CTA per SM); this one runs in the 4096-point configuration (two CTAs per SM)
// and reads pixel PAIRS (8-byte loads).  tw2n: the W_2N^m table of the 2N-point plan; needs KX <= N.
__device__ __forceinline__ void cp_async_f32x2_any(float2* smem_dst, const float2* gmem_src) {
  const unsigned dst = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(dst), "l"(gmem_src));
}

template <int N>
constexpr size_t rows_forward_real2n_smem_bytes() {
  return fft2::Cfg<N>::smem_bytes + 2ull * fft2::Cfg<N>::B * N * sizeof(float2);
}

template <int N>
__global__ void __launch_bounds__(fft2::kThreads, N >= 2048 ? 2 : 1)
rows_forward_real2n(const float* __restrict__ image, int H, int W, const float* __restrict__ mean_std,
                    const float* __restrict__ mask, const int* __restrict__ jobs, const int* __restrict__ frame_shifts,
                    int x_margin, int ylo, int yhi, int NY, int KX, const float2* __restrict__ tw2n,
                    float2* __restrict__ tmp, int rows_per_cta) {
  using C = fft2::Cfg<N>;
  using P = fft2::Plan<N>;
  extern __shared__ float2 smem[];
  const fft2::Smem<N> sm(smem);
  fft2::load_twiddles<N>(sm, tw2n, 2);  // W_N^m = W_2N^{2m}: the tables of the N-point transform from the 2N-point plan
  const int seq = threadIdx.x / C::TPS, j = threadIdx.x % C::TPS;
  float2* myseq = sm.data + seq * C::STRIDE;
  float2* stage_p = smem + C::B * C::STRIDE + 64 + C::TW_HI;  // pixel pairs, slot e * kThreads + threadIdx.x
  float2* stage_m = stage_p + C::B * N;                        // mask pairs of the same row
  const int job = blockIdx.y;
  const int fa = jobs[job * 6 + 0], fb = jobs[job * 6 + 2];
  const int y0 = jobs[job * 6 + 4], x0 = jobs[job * 6 + 5];
  float mean = 0.f, inv_std = 1.f;
  if (mean_std != nullptr) {
    mean = __ldg(mean_std);
    inv_std = 1.0f / __ldg(mean_std + 1);
  }
  const Window wa = make_window(image, fa, y0, x0, frame_shifts, H, W, ylo, yhi, 2 * N, x_margin);
  const Window wb = make_window(image, fb >= 0 ? fb : fa, y0, x0, frame_shifts, H, W, ylo, yhi, 2 * N, x_margin);
  const int halves = fb >= 0 ? 2 : 1;
  const int row_begin = ylo + blockIdx.x * rows_per_cta;
  const int row_end = min(yhi, row_begin + rows_per_cta);
  const int nunits = row_end > row_begin ? ((row_end - row_begin + C::B - 1) / C::B) * halves : 0;
  float2* plane_a = tmp + (long)(2 * job) * NY * KX;

  auto prefetch = [&](int u) {
    const int y = row_begin + (u / halves) * C::B + seq;
    if (y >= row_end) return;
    const bool second = (u % halves) == 1;
    const Window& wd = second ? wb : wa;
    const float* row = wd.fast_base(W) + (long)y * W;
    const bool pair_ok = !wd.wrap && (reinterpret_cast<uintptr_t>(row) & 7) == 0;
#pragma unroll
    for (int e = 0; e < C::VPT; ++e) {
      const int x = 2 * P::First::in_index(j, e / P::First::R, e % P::First::R);
      const int slot = e * fft2::kThreads + threadIdx.x;
      if (pair_ok) {
        cp_async_f32x2_any(stage_p + slot, reinterpret_cast<const float2*>(row + x));
      } else {
        float* dst = reinterpret_cast<float*>(stage_p + slot);
        cp_async_f32(dst, wd.wrap ? wd.wrapped(y, x, H, W) : row + x);
        cp_async_f32(dst + 1, wd.wrap ? wd.wrapped(y, x + 1, H, W) : row + x + 1);
      }
      // the mask row serves both frames: staged with the first one
      if (mask && !second) cp_async_f32x2_any(stage_m + slot, reinterpret_cast<const float2*>(mask + (long)y * (2 * N) + x));
    }
  };
  if (nunits > 0) prefetch(0);
  __syncthreads();  // twiddle tables
  for (int u = 0; u < nunits; ++u) {
    const int y = row_begin + (u / halves) * C::B + seq;
    const bool active = y < row_end;
    const bool second = (u % halves) == 1;
    cp_async_commit_and_wait();
    float2 v[C::VPT];
#pragma unroll
    for (int e = 0; e < C::VPT; ++e) {
      float2 z = make_float2(0.f, 0.f);
      if (active) {
        const int slot = e * fft2::kThreads + threadIdx.x;
        const float2 px = stage_p[slot];
        const float2 m = mask ? stage_m[slot] : make_float2(1.f, 1.f);
        z.x = (px.x - mean) * inv_std * m.x;
        z.y = (px.y - mean) * inv_std * m.y;
      }
      v[e] = z;
    }
    if (u + 1 < nunits) prefetch(u + 1);  // overlaps with the transform below
    fft2::fft_regs_to_regs<N>(sm, myseq, j, v);
    __syncthreads();
    P::Last::store(myseq, j, v);
    __syncthreads();
    if (active) {
      float2* plane = plane_a + (second ? (long)NY * KX : 0l);
      for (int k = j; k < KX; k += C::TPS) {
        const float2 zk = myseq[fft2::pad_idx(k)];
        const float2 zn = myseq[fft2::pad_idx(k == 0 ? 0 : N - k)];
        const float2 ev = make_float2(0.5f * (zk.x + zn.x), 0.5f * (zk.y - zn.y));
        const float2 od = make_float2(0.5f * (zk.y + zn.y), -0.5f * (zk.x - zn.x));
        plane[(long)y * KX + k] = cadd(ev, cmul(__ldg(tw2n + k), od));
      }
    }
    __syncthreads();
  }
}

// ---- forward columns: tmp[plane][y][kx] -> out[plane][kyb][kx] * weight --------------------------------
template <int N>
__global__ void __launch_bounds__(fft2::kThreads)
cols_forward_p2(const float2* __restrict__ tmp, int ylo, int yhi, int KX, int KY, int ky_start,
                const float* __restrict__ weight, const float2* __restrict__ tw, float2* __restrict__ out) {
  using C = fft2::Cfg<N>;
  using P = fft2::Plan<N>;
  extern __shared__ float2 smem[];
  const fft2::Smem<N> sm(smem);
  fft2::load_twiddles<N>(sm, tw);
  const int seq = threadIdx.x % C::B, j = threadIdx.x / C::B;  // neighbouring threads -> neighbouring kx
  float2* myseq = sm.data + seq * C::STRIDE;
  const long plane = blockIdx.y;
  const int kx = blockIdx.x * C::B + seq;
  const bool active = kx < KX;
  const float2* src = tmp + plane * N * KX + kx;
  float2 v[C::VPT];
#pragma unroll
  for (int g = 0; g < P::First::G; ++g)
#pragma unroll
    for (int r = 0; r < P::First::R; ++r) {
      const int y = P::First::in_index(j, g, r);
      v[g * P::First::R + r] = (active && y >= ylo && y < yhi) ? src[(long)y * KX] : make_float2(0.f, 0.f);
    }
  __syncthreads();
  fft2::fft_regs_to_regs<N>(sm, myseq, j, v);
  if (!active) return;
  float2* dst = out + plane * KY * KX + kx;
#pragma unroll
  for (int g = 0; g < P::Last::G; ++g)
#pragma unroll
    for (int r = 0; r < P::Last::R; ++r) {
      const int ky = P::Last::out_index(j, g, r);
      const int kyb = (ky - ky_start) & (N - 1);
      if (kyb < KY) {
        float2 val = P::Last::result(v, g, r);
        if (weight) {
          const float wgt = __ldg(weight + (long)kyb * KX + kx);
          val.x *= wgt;
          val.y *= wgt;
        }
        dst[(long)kyb * KX] = val;
      }
    }
}

// ---- inverse columns: in[item][kyb][kx] -> tmp[item][y][kx] (unnormalised inverse along y) ------------
template <int N>
__global__ void __launch_bounds__(fft2::kThreads)
cols_inverse_p2(const float2* __restrict__ in, int KX, int KY, int ky_start, const float2* __restrict__ tw,
                float2* __restrict__ tmp) {
  using C = fft2::Cfg<N>;
  using P = fft2::Plan<N>;
  extern __shared__ float2 smem[];
  const fft2::Smem<N> sm(smem);
  fft2::load_twiddles<N>(sm, tw);
  const int seq = threadIdx.x % C::B, j = threadIdx.x / C::B;
  float2* myseq = sm.data + seq * C::STRIDE;
  const long item = blockIdx.y;
  const int kx = blockIdx.x * C::B + seq;
  const bool active = kx < KX;
  const float2* src = in + item * KY * KX + kx;
  float2 v[C::VPT];
#pragma unroll
  for (int g = 0; g < P::First::G; ++g)
#pragma unroll
    for (int r = 0; r < P::First::R; ++r) {
      const int y = P::First::in_index(j, g, r);
      const int kyb = (y - ky_start) & (N - 1);
      float2 z = make_float2(0.f, 0.f);
      if (active && kyb < KY) {
        const float2 c = src[(long)kyb * KX];
        z = make_float2(c.y, c.x);  // re/im swap: inverse via forward
      }
      v[g * P::First::R + r] = z;
    }
  __syncthreads();
  fft2::fft_regs_to_regs<N>(sm, myseq, j, v);
  if (!active) return;
  float2* dst = tmp + item * N * KX + kx;
#pragma unroll
  for (int g = 0; g < P::Last::G; ++g)
#pragma unroll
    for (int r = 0; r < P::Last::R; ++r) {
      const float2 val = P::Last::result(v, g, r);
      dst[(long)P::Last::out_index(j, g, r) * KX] = make_float2(val.y, val.x);
    }
}

// ---- inverse rows (complex-to-real, two rows per transform) ------------------------------------------------
//
// Entry i of the packed spectrum of rows (ya -> real part, yb -> imaginary part) is built from
// Ca = rowa[k], Cb = rowb[k] with k = i (i < KX) or k = N - i (mirrored, conjugated); everything else is
// zero.  The (Ca, Cb) pairs of the NEXT batch of row pairs are prefetched with cp.async into per-thread
// shared-memory slots while the current batch is transformed.

__device__ __forceinline__ void cp_async_f32x2(float2* smem_dst, const float2* gmem_src) {
  const unsigned dst = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(dst), "l"(gmem_src));
}

constexpr int kRowIters = 4;  // row-pair batches per CTA in the inverse row kernels

template <int N>
__host__ __device__ constexpr int rows_per_cta_inverse() {
  return 2 * fft2::Cfg<N>::B * kRowIters;
}

template <int N>
__host__ __device__ constexpr size_t rows_inverse_smem_bytes() {
  return fft2::Cfg<N>::smem_bytes + 2ull * fft2::Cfg<N>::B * N * sizeof(float2);
}

// k index (into the band-limited rows) feeding packed entry i, or -1 if the entry is zero
template <int N>
__device__ __forceinline__ int c2r_source_index(int i, int KX) {
  if (i < KX) return i;
  const int k = N - i;
  return (k < KX && 2 * k != N) ? k : -1;
}

template <int N>
__device__ __forceinline__ float2 c2r_pack(float2 ca, float2 cb, int i, int KX) {
  if (i < KX) {
    if (i == 0 || 2 * i == N) return make_float2(cb.x, ca.x);  // c2r ignores Im of the DC / Nyquist bins
    return make_float2(ca.y + cb.x, ca.x - cb.y);              // Z[k] = Ca + i Cb, stored (im, re)
  }
  return make_float2(cb.x - ca.y, ca.x + cb.y);                // Z[N-k] = conj(Ca) + i conj(Cb), stored (im, re)
}

struct NoCoeff {
  __device__ void operator()(int, float2, float2) const {}
};

// Shared driver of the inverse row kernels: calls consume(ya, has_b, v) with the last-pass outputs of
// every row pair of row block blk (rows_per_cta_inverse<N>() rows; v swapped: .y = row ya, .x = row ya + 1), and before
// that on_coeff(i, Ca, Cb) with the coefficients of every packed entry i the calling thread builds.  tw: the W_N^m table,
// or the table of a transform tw_stride times longer.
template <int N, typename Consume, typename OnCoeff = NoCoeff>
__device__ __forceinline__ void rows_inverse_driver(const float2* __restrict__ src, int NY, int KX, int blk,
                                                    const float2* __restrict__ tw, int tw_stride, float2* smem,
                                                    Consume&& consume, OnCoeff&& on_coeff = OnCoeff{}) {
  using C = fft2::Cfg<N>;
  using P = fft2::Plan<N>;
  const fft2::Smem<N> sm(smem);
  fft2::load_twiddles<N>(sm, tw, tw_stride);
  const int seq = threadIdx.x / C::TPS, j = threadIdx.x % C::TPS;
  float2* myseq = sm.data + seq * C::STRIDE;
  float2* stage_a = smem + C::B * C::STRIDE + 64 + C::TW_HI;
  float2* stage_b = stage_a + C::B * N;
  auto row_of = [&](int it) { return blk * rows_per_cta_inverse<N>() + (it * C::B + seq) * 2; };
  auto prefetch = [&](int it) {
    const int ya = row_of(it);
    if (ya >= NY) return;
    const float2* rowa = src + (long)ya * KX;
    const bool has_b = ya + 1 < NY;
#pragma unroll
    for (int e = 0; e < C::VPT; ++e) {
      constexpr int R = P::First::R;
      // whole blocks of entries are zero for a band-limited spectrum: warp-uniform skip
      const int lo = (e / R) * C::TPS + (e % R) * P::First::NBR;
      if (lo >= KX && lo + C::TPS <= N - KX + 1) continue;
      const int k = c2r_source_index<N>(P::First::in_index(j, e / R, e % R), KX);
      if (k >= 0) {
        const int slot = e * fft2::kThreads + threadIdx.x;
        cp_async_f32x2(stage_a + slot, rowa + k);
        if (has_b) cp_async_f32x2(stage_b + slot, rowa + KX + k);
      }
    }
  };
  prefetch(0);
  __syncthreads();
  for (int it = 0; it < kRowIters; ++it) {
    const int ya = row_of(it);
    const bool active = ya < NY;
    const bool has_b = ya + 1 < NY;
    cp_async_commit_and_wait();
    float2 v[C::VPT];
#pragma unroll
    for (int e = 0; e < C::VPT; ++e) {
      constexpr int R = P::First::R;
      float2 z = make_float2(0.f, 0.f);
      const int lo = (e / R) * C::TPS + (e % R) * P::First::NBR;
      if (active && !(lo >= KX && lo + C::TPS <= N - KX + 1)) {
        const int i = P::First::in_index(j, e / R, e % R);
        if (c2r_source_index<N>(i, KX) >= 0) {
          const int slot = e * fft2::kThreads + threadIdx.x;
          const float2 ca = stage_a[slot], cb = has_b ? stage_b[slot] : make_float2(0.f, 0.f);
          on_coeff(i, ca, cb);
          z = c2r_pack<N>(ca, cb, i, KX);
        }
      }
      v[e] = z;
    }
    if (it + 1 < kRowIters) prefetch(it + 1);
    fft2::fft_regs_to_regs<N>(sm, myseq, j, v);
    if (active) consume(ya, has_b, j, v);
    __syncthreads();
  }
}

// ---- inverse rows + argmax: tmp[item][y][kx] -> partial[item][cta] ------------------------------------
template <int N>
__global__ void __launch_bounds__(fft2::kThreads, N == 4096 ? 3 : 1)
rows_inverse_argmax_p2(const float2* __restrict__ tmp, int NY, int KX, const float2* __restrict__ tw,
                       PeakCandidate* __restrict__ partial) {
  using P = fft2::Plan<N>;
  extern __shared__ float2 smem[];
  const long item = blockIdx.y;
  float best = -INFINITY;
  int best_idx = 0x7fffffff;
  rows_inverse_driver<N>(tmp + item * NY * KX, NY, KX, blockIdx.x, tw, 1, smem, [&](int ya, bool has_b, int j, const float2* v) {
    // the thread visits its samples in increasing index order (out_index = j + g TPS + r NS with G TPS == NS: r outer,
    // g inner; row ya, then row ya + 1; later calls have larger ya), so "strictly greater" keeps the first of equal
    // maxima: one compare and two selects per sample
#pragma unroll
    for (int r = 0; r < P::Last::R; ++r)
#pragma unroll
      for (int g = 0; g < P::Last::G; ++g) {
        const float val = P::Last::result(v, g, r).y;  // swapped: .y = row ya, .x = row ya + 1
        if (val > best) {
          best = val;
          best_idx = ya * N + P::Last::out_index(j, g, r);
        }
      }
    if (has_b) {
#pragma unroll
      for (int r = 0; r < P::Last::R; ++r)
#pragma unroll
        for (int g = 0; g < P::Last::G; ++g) {
          const float val = P::Last::result(v, g, r).x;
          if (val > best) {
            best = val;
            best_idx = (ya + 1) * N + P::Last::out_index(j, g, r);
          }
        }
    }
  });
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, best, o);
    const int oi = __shfl_xor_sync(0xffffffffu, best_idx, o);
    if (better(ov, oi, best, best_idx)) {
      best = ov;
      best_idx = oi;
    }
  }
  __shared__ float sval[fft2::kThreads / 32];
  __shared__ int sidx[fft2::kThreads / 32];
  if ((threadIdx.x & 31) == 0) {
    sval[threadIdx.x >> 5] = best;
    sidx[threadIdx.x >> 5] = best_idx;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int i = 1; i < fft2::kThreads / 32; ++i)
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

// The row blocks (CTA-sized groups of rows, one partial result each) an argmax row kernel visits: its whole grid
// (blockIdx.x = block, blockIdx.y = item) or, after the coarse bound (rows_coarse_bound_p2), only the live (item, block)
// pairs of `list`, which the CTAs of a one-dimensional grid share round-robin.
struct RowBlocks {
  const int2* list;  // nullptr: the whole grid
  const int* count;  // entries of list
  int per_item;      // blocks (partial slots) per item
};

template <typename F>
__device__ __forceinline__ void for_each_row_block(const RowBlocks& blocks, F&& f) {
  if (blocks.list == nullptr) {
    f((long)blockIdx.y, (int)blockIdx.x);
    return;
  }
  const int n = *blocks.count;
  for (int w = blockIdx.x; w < n; w += gridDim.x) {
    const int2 u = blocks.list[w];
    f((long)u.x, u.y);
  }
}

// ---- inverse rows of length 2N as N-point complex transforms + argmax ------------------------------------------------
//
// x[0 .. 2N) real with spectrum X[k], k < KX <= N / 2:  z[m] = x[2m] + i x[2m+1] = IDFT_N(Z),
// Z[k] = X[k] + i Y[k], Z[N-k] = conj X[k] + i conj Y[k], Y[k] = X[k] W_2N^{-k} -- the packed spectrum of the "two rows"
// Ca = X (even samples) and Cb = Y (odd samples) of the kernel above, with Cb formed on the fly: ONE row per N-point
// transform instead of two rows per 2N-point transform (the 8192-point kernel holds 32 values per thread and is
// confined to one CTA per SM).  tw2n: the W_2N^m table of the 2N-point plan.
template <int N>
__host__ __device__ constexpr int rows_per_cta_inverse_real2n() {
  return fft2::Cfg<N>::B * kRowIters;
}
template <int N>
constexpr size_t rows_inverse_real2n_smem_bytes() {
  return fft2::Cfg<N>::smem_bytes + 1ull * fft2::Cfg<N>::B * N * sizeof(float2);
}

template <int N>
__global__ void __launch_bounds__(fft2::kThreads, N >= 2048 ? 3 : 1)
rows_inverse_argmax_real2n(const float2* __restrict__ tmp, int NY, int KX, const float2* __restrict__ tw2n,
                           PeakCandidate* __restrict__ partial, RowBlocks blocks) {
  using C = fft2::Cfg<N>;
  using P = fft2::Plan<N>;
  extern __shared__ float2 smem[];
  const fft2::Smem<N> sm(smem);
  fft2::load_twiddles<N>(sm, tw2n, 2);  // W_N^m = W_2N^{2m}
  const int seq = threadIdx.x / C::TPS, j = threadIdx.x % C::TPS;
  float2* myseq = sm.data + seq * C::STRIDE;
  float2* stage_a = smem + C::B * C::STRIDE + 64 + C::TW_HI;
  __shared__ float sval[fft2::kThreads / 32];
  __shared__ int sidx[fft2::kThreads / 32];
  for_each_row_block(blocks, [&](long item, int blk) {
    const float2* src = tmp + item * NY * KX;
    auto row_of = [&](int it) { return blk * rows_per_cta_inverse_real2n<N>() + it * C::B + seq; };
    auto prefetch = [&](int it) {
      const int y = row_of(it);
      if (y >= NY) return;
      const float2* row = src + (long)y * KX;
#pragma unroll
      for (int e = 0; e < C::VPT; ++e) {
        constexpr int R = P::First::R;
        // whole blocks of entries are zero for a band-limited spectrum: warp-uniform skip
        const int lo = (e / R) * C::TPS + (e % R) * P::First::NBR;
        if (lo >= KX && lo + C::TPS <= N - KX + 1) continue;
        const int k = c2r_source_index<N>(P::First::in_index(j, e / R, e % R), KX);
        if (k >= 0) cp_async_f32x2(stage_a + e * fft2::kThreads + threadIdx.x, row + k);
      }
    };
    float best = -INFINITY;
    int best_idx = 0x7fffffff;
    prefetch(0);
    __syncthreads();
    for (int it = 0; it < kRowIters; ++it) {
      const int y = row_of(it);
      const bool active = y < NY;
      cp_async_commit_and_wait();
      float2 v[C::VPT];
#pragma unroll
      for (int e = 0; e < C::VPT; ++e) {
        constexpr int R = P::First::R;
        float2 z = make_float2(0.f, 0.f);
        const int lo = (e / R) * C::TPS + (e % R) * P::First::NBR;
        if (active && !(lo >= KX && lo + C::TPS <= N - KX + 1)) {
          const int i = P::First::in_index(j, e / R, e % R);
          const int k = c2r_source_index<N>(i, KX);
          if (k >= 0) {
            const float2 ca = stage_a[e * fft2::kThreads + threadIdx.x];
            const float2 w = __ldg(tw2n + k);  // W_2N^k; Y[k] = X[k] conj(W_2N^k)
            const float2 cb = make_float2(ca.x * w.x + ca.y * w.y, ca.y * w.x - ca.x * w.y);
            z = c2r_pack<N>(ca, cb, i, KX);
          }
        }
        v[e] = z;
      }
      if (it + 1 < kRowIters) prefetch(it + 1);
      fft2::fft_regs_to_regs<N>(sm, myseq, j, v);
      if (active) {
        // samples in increasing index order (m = out_index ascends with r outer, g inner; 2m before 2m + 1; later rows
        // later): a strictly-greater compare keeps the first of equal maxima
        const int base = y * (2 * N);
#pragma unroll
        for (int r = 0; r < P::Last::R; ++r)
#pragma unroll
          for (int g = 0; g < P::Last::G; ++g) {
            const float2 val = P::Last::result(v, g, r);  // swapped: .y = x[2m], .x = x[2m + 1]
            const int idx = base + 2 * P::Last::out_index(j, g, r);
            if (val.y > best) {
              best = val.y;
              best_idx = idx;
            }
            if (val.x > best) {
              best = val.x;
              best_idx = idx + 1;
            }
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
    if ((threadIdx.x & 31) == 0) {
      sval[threadIdx.x >> 5] = best;
      sidx[threadIdx.x >> 5] = best_idx;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      for (int i = 1; i < fft2::kThreads / 32; ++i)
        if (better(sval[i], sidx[i], best, best_idx)) {
          best = sval[i];
          best_idx = sidx[i];
        }
      PeakCandidate c;
      c.val = best;
      c.idx = best_idx;
      partial[item * blocks.per_item + blk] = c;
    }
  });
}

// ---- coarse bound of the peak search: the row blocks that can hold the maximum --------------------------------------
//
// After the column pass, row y of a correlation surface of N-point rows is the real trigonometric polynomial
//   r(x) = Re c_0 + 2 sum_{0 < k < KX} Re(c_k e^{2 pi i k x / N}),   |r''| <= M2_y = 2 sum_k (2 pi k / N)^2 |c_k|.
// With 2 KX - 1 <= M = N / 4, k -> k mod M is one-to-one on the band, so the M-point c2r transform of the same KX
// coefficients is r at x = 4m.  On a cell of width 4 between two such samples (the last cell ends at x = N = 0),
// r <= max(end samples) + (4^2 / 8) M2_y, so no sample of the row exceeds max_m r(4m) + 2 M2_y.
// eps_y bounds the fp32 error of the coarse and the fine transform of a row together: the elementwise error of a
// power-of-two FFT is a few eps32 per level of butterflies times the L1 norm of its (packed) input, so with
//   L1_y = |Re c_0| + 2 sum_{k>0} |c_k|,   eps_y = 32 eps32 (log2 N + 8) 2 max(L1_ya, L1_ya+1) + 1e-35
// (ya even: the row pair packed in one transform; the half-length kernels pack a row with its twisted copy) each of
// the two transforms is within half of eps_y.  Every fine value of row y is then at most
//   hi_y = max_m C_y(m) + 2 M2_y + eps_y,
// and the fine value at the row's largest coarse sample C_y is at least lo_y = max_m C_y(m) - eps_y.  The sums take
// |c_k| from above (abs_ru) and round upward, the subtraction downward, so both bounds hold as computed.  A row block whose largest hi_y is below
// T = max_y lo_y over the surface can neither hold the fine maximum nor tie with it (rows_select_live drops it); the
// row with the largest lo_y always stays.  Rows whose L1 norm passes 1e36 (or is not finite) get hi = NaN, which
// keeps every block of their surface live.
//
// Most rows cannot hold the maximum by a margin that needs no transform to see: |r(x)| <= L1_y, so every fine value of
// row y is at most hi0_y = L1_y + eps_y.  rows_l1_bound writes the largest hi0_y of every fine block as its hi.  The
// coarse bound then runs on one group per surface only (a group: the rows of one rows_coarse_bound_p2 row block), the
// seed, which holds the row with the largest L1 norm: it replaces the hi of the seed's blocks and writes the seed's lo,
// T0 = max lo_y over the seed; the other groups' lo slots hold the lowest finite float.  rows_select_live then drops a
// block whose hi is below T0, so it can neither hold the maximum nor tie with it.  Every slot is finite unless a row norm
// passes 1e36 (hi0 = NaN) or a coarse bound is NaN, and then every block of the surface stays live, as above.  Sampling
// the other groups as well was measured slower on C2 products: their hi0 already leaves almost only the blocks that
// the coarse bound leaves (DESIGN.md 8.3).

// maximum that propagates NaN from either side
__device__ __forceinline__ float max_nan(float a, float b) { return (a > b || a != a) ? a : b; }

// An upper bound of |c| without a square root (a directed-rounding square root costs more than the coarse transform):
// sqrt(M^2 + m^2) with M = max(|Re c|, |Im c|), m = min(...) is convex in m, so it lies below its chord
// M + (sqrt 2 - 1) m, at most 8 % above |c|.  NaN stays NaN.
__device__ __forceinline__ float abs_ru(float2 c) {
  const float ax = fabsf(c.x), ay = fabsf(c.y);
  return (ax != ax || ay != ay) ? NAN : __fmaf_ru(0.41421357f, fminf(ax, ay), fmaxf(ax, ay));  // 0.41421357f >= sqrt 2 - 1
}

// adds coefficient c_k (k < KX) of a row to its sums L1 and sum k^2 |c_k|, rounded upward
__device__ __forceinline__ void add_coeff(int k, float2 c, float& l1, float& k2) {
  const float a = k == 0 ? fabsf(c.x) : abs_ru(c);
  l1 = __fadd_ru(l1, k == 0 ? a : 2.f * a);
  k2 = __fadd_ru(k2, __fmul_ru((float)(k * k), a));
}

// hi_y and lo_y of the rows of a pair (ya, ya + 1) from each row's largest coarse sample, L1 and sum k^2 |c_k|
__device__ __forceinline__ void pair_bounds(const float (&cmax)[2], const float (&l1)[2], const float (&k2)[2], float eps_rel,
                                            float curv, float (&hi)[2], float (&lo)[2]) {
  const bool ok = l1[0] <= 1e36f && l1[1] <= 1e36f;  // false for NaN
  const float eps = __fadd_ru(__fmul_ru(eps_rel, fmaxf(l1[0], l1[1])), 1e-35f);
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    hi[h] = ok ? __fadd_ru(__fadd_ru(cmax[h], 2.f * __fmul_ru(curv, k2[h])), eps) : NAN;
    lo[h] = __fsub_rd(cmax[h], eps);
  }
}

// Bounds s_hi / s_lo of group blk's rows [row0, row0 + ROWS) -> hi[item][fine block] (largest hi_y of the block's
// fine_rows rows; fine_rows divides ROWS) and lo[item][blk] (largest lo_y).  Every thread calls it after a barrier.
__device__ __forceinline__ void store_block_bounds(const float* s_hi, const float* s_lo, int ROWS, int blk, int NY,
                                                   int fine_rows, long item, float* __restrict__ hi, float* __restrict__ lo) {
  const int row0 = blk * ROWS;
  const int rows = min(ROWS, NY - row0);
  const int nfine = (NY + fine_rows - 1) / fine_rows;
  const int ngroups = (NY + ROWS - 1) / ROWS;
  const int fb0 = row0 / fine_rows;
  for (int b = threadIdx.x; b < ROWS / fine_rows && fb0 + b < nfine; b += blockDim.x) {
    float h = -INFINITY;
    for (int r = b * fine_rows; r < (b + 1) * fine_rows && r < rows; ++r) h = max_nan(h, s_hi[r]);
    hi[item * nfine + fb0 + b] = h;
  }
  if (threadIdx.x < 32) {
    const int lane = threadIdx.x;
    float l = -INFINITY;
    for (int r = lane; r < rows; r += 32) l = max_nan(l, s_lo[r]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) l = max_nan(l, __shfl_xor_sync(0xffffffffu, l, o));
    if (lane == 0) lo[item * ngroups + blk] = l;
  }
}

// tmp[item][y][kx] of N = 4M point rows -> hi[item][fine block] (largest hi_y of the block's fine_rows rows) and
// lo[item][group] (largest lo_y of the group's rows) for the coarse groups of `groups` (rows_per_cta_inverse<M>() rows
// each).  tw: the W_N^m table of the N-point plan.  eps_rel: the factor of max(L1) in eps_y, curv: 2 (2 pi / N)^2, both
// rounded upward.  Smem: rows_inverse_smem_bytes<M>().
template <int M>
__global__ void __launch_bounds__(fft2::kThreads, 2)
rows_coarse_bound_p2(const float2* __restrict__ tmp, int NY, int KX, const float2* __restrict__ tw, int fine_rows,
                     float eps_rel, float curv, float* __restrict__ hi, float* __restrict__ lo, RowBlocks groups) {
  using C = fft2::Cfg<M>;
  using P = fft2::Plan<M>;
  constexpr int ROWS = rows_per_cta_inverse<M>();
  constexpr int W = C::TPS < 32 ? C::TPS : 32;  // lanes of one sequence in a warp
  constexpr int NW = C::TPS / W;                // warps of one sequence
  extern __shared__ float2 smem[];
  // per row and warp of its sequence: largest coarse sample, L1 and sum k^2 |c_k| of the warp's coefficients
  __shared__ float s_max[ROWS * NW], s_l1[ROWS * NW], s_k2[ROWS * NW];
  __shared__ float s_hi[ROWS], s_lo[ROWS];
  const int lane = threadIdx.x & 31;
  const unsigned seq_lanes = W == 32 ? 0xffffffffu : ((1u << W) - 1) << (lane & ~(W - 1));
  // the driver's first barrier keeps the next group's writes behind every thread's store_block_bounds
  for_each_row_block(groups, [&](long item, int blk) {
    const int row0 = blk * ROWS;
    float l1a = 0.f, l1b = 0.f, k2a = 0.f, k2b = 0.f;  // this thread's share of the current row pair's sums
    auto on_coeff = [&](int i, float2 ca, float2 cb) {
      if (i >= KX) return;  // entries i < KX hold every k = i of the band once
      add_coeff(i, ca, l1a, k2a);
      add_coeff(i, cb, l1b, k2b);
    };
    rows_inverse_driver<M>(tmp + item * NY * KX, NY, KX, blk, tw, 4, smem, [&](int ya, bool has_b, int j, const float2* v) {
      float ma = -INFINITY, mb = -INFINITY;
#pragma unroll
      for (int r = 0; r < P::Last::R; ++r)
#pragma unroll
        for (int g = 0; g < P::Last::G; ++g) {
          const float2 val = P::Last::result(v, g, r);  // swapped: .y = row ya, .x = row ya + 1
          ma = max_nan(ma, val.y);
          mb = max_nan(mb, val.x);
        }
#pragma unroll
      for (int o = W / 2; o > 0; o >>= 1) {
        ma = max_nan(ma, __shfl_xor_sync(seq_lanes, ma, o));
        mb = max_nan(mb, __shfl_xor_sync(seq_lanes, mb, o));
        l1a = __fadd_ru(l1a, __shfl_xor_sync(seq_lanes, l1a, o));
        l1b = __fadd_ru(l1b, __shfl_xor_sync(seq_lanes, l1b, o));
        k2a = __fadd_ru(k2a, __shfl_xor_sync(seq_lanes, k2a, o));
        k2b = __fadd_ru(k2b, __shfl_xor_sync(seq_lanes, k2b, o));
      }
      if (j % W == 0) {
        const int at = (ya - row0) * NW + j / W;
        s_max[at] = ma;
        s_l1[at] = l1a;
        s_k2[at] = k2a;
        if (has_b) {
          s_max[at + NW] = mb;
          s_l1[at + NW] = l1b;
          s_k2[at + NW] = k2b;
        }
      }
      l1a = l1b = k2a = k2b = 0.f;
    }, on_coeff);  // ends with a barrier
    if (threadIdx.x < ROWS / 2 && row0 + 2 * (int)threadIdx.x < NY) {
      const int r0 = 2 * threadIdx.x;
      float cmax[2], l1[2] = {0.f, 0.f}, k2[2] = {0.f, 0.f}, bhi[2], blo[2];
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        cmax[h] = -INFINITY;
        if (row0 + r0 + h < NY)
          for (int w = 0; w < NW; ++w) {
            const int at = (r0 + h) * NW + w;
            cmax[h] = max_nan(cmax[h], s_max[at]);
            l1[h] = __fadd_ru(l1[h], s_l1[at]);
            k2[h] = __fadd_ru(k2[h], s_k2[at]);
          }
      }
      pair_bounds(cmax, l1, k2, eps_rel, curv, bhi, blo);
      for (int h = 0; h < 2 && row0 + r0 + h < NY; ++h) {
        s_hi[r0 + h] = bhi[h];
        s_lo[r0 + h] = blo[h];
      }
    }
    __syncthreads();
    store_block_bounds(s_hi, s_lo, ROWS, blk, NY, fine_rows, item, hi, lo);
  });
}

// hi0 of a fine block from the largest L1 norm of its rows: L1 + eps (eps_y of that norm, rounded upward), NaN where
// the norm passes 1e36 or is not finite
__device__ __forceinline__ float l1_block_bound(float l1, float eps_rel) {
  return l1 <= 1e36f ? __fadd_ru(l1, __fadd_ru(__fmul_ru(eps_rel, l1), 1e-35f)) : NAN;
}

// tmp[item][y][kx] -> hi[item][fine block] = the block's largest hi0_y (one warp per block of fine_rows rows, one row
// per warp step; fine_rows is even, so both rows of every packed pair fall in one block).  Streams the column-pass
// output once: grid (ceil(nfine / 8), items) of 256 threads.  (A row pair per warp step measured slower on the 1024-point
// patch rows: 0.28 against 0.23 ms at C2.)
__global__ void __launch_bounds__(256)
rows_l1_bound(const float2* __restrict__ tmp, int NY, int KX, int fine_rows, float eps_rel, float* __restrict__ hi) {
  const int nfine = (NY + fine_rows - 1) / fine_rows;
  const int fb = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (fb >= nfine) return;
  const long item = blockIdx.y;
  const int y1 = min(NY, (fb + 1) * fine_rows);
  float best = 0.f;
  for (int y = fb * fine_rows; y < y1; ++y) {
    const float2* row = tmp + (item * NY + y) * KX;
    float l1 = 0.f, k2 = 0.f;  // k2 unused
#pragma unroll 4
    for (int k = lane; k < KX; k += 32) add_coeff(k, __ldg(row + k), l1, k2);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) l1 = __fadd_ru(l1, __shfl_xor_sync(0xffffffffu, l1, o));
    best = max_nan(best, l1);
  }
  if (lane == 0) hi[item * nfine + fb] = l1_block_bound(best, eps_rel);
}

// ---- inverse rows + store: tmp[item][y][kx] -> out[item][y][x] real ------------------------------------
template <int N>
__global__ void __launch_bounds__(fft2::kThreads)
rows_inverse_store_p2(const float2* __restrict__ tmp, int NY, int KX, const float2* __restrict__ tw, float scale,
                      float* __restrict__ out) {
  using P = fft2::Plan<N>;
  extern __shared__ float2 smem[];
  const long item = blockIdx.y;
  float* dst = out + item * NY * N;
  rows_inverse_driver<N>(tmp + item * NY * KX, NY, KX, blockIdx.x, tw, 1, smem, [&](int ya, bool has_b, int j, const float2* v) {
#pragma unroll
    for (int g = 0; g < P::Last::G; ++g)
#pragma unroll
      for (int r = 0; r < P::Last::R; ++r) {
        const float2 val = P::Last::result(v, g, r);
        const int x = P::Last::out_index(j, g, r);
        dst[(long)ya * N + x] = val.y * scale;
        if (has_b) dst[(long)(ya + 1) * N + x] = val.x * scale;
      }
  });
}

// ---- whole-frame Fourier shift, column pass: FFT along y, phase multiply, inverse FFT along y ----------
// tmp[plane = frame][y][kx] in place.  Fuses what would otherwise be three kernels and three round trips
// of the (t, ny, nx/2+1) spectrum through HBM (correct_motion.py:484-496).
// phase_y[f][ky] = exp(i * fp32(-2 pi) * fftfreq(ny)[ky] * s_y[f]) is precomputed; the x factor is one sincosf
// per thread.  exp(i(a+b)) = exp(ia) exp(ib): differs from the reference's cos/sin of the summed angle by
// fp32 rounding only.
template <int N>
__global__ void __launch_bounds__(fft2::kThreads, N <= 4096 ? 3 : 1)
cols_shift_p2(float2* __restrict__ tmp, int KX, int NX, const float2* __restrict__ phase_y, const float* __restrict__ field,
              int T, float sign, const float2* __restrict__ tw) {
  using C = fft2::Cfg<N>;
  using P = fft2::Plan<N>;
  extern __shared__ float2 smem[];
  const fft2::Smem<N> sm(smem);
  fft2::load_twiddles<N>(sm, tw);
  const int seq = threadIdx.x % C::B, j = threadIdx.x / C::B;
  float2* myseq = sm.data + seq * C::STRIDE;
  const int f = blockIdx.y;
  const int kx = blockIdx.x * C::B + seq;
  const bool active = kx < KX;
  float2* col = tmp + (long)f * N * KX + kx;
  float2 v[C::VPT];
#pragma unroll
  for (int g = 0; g < P::First::G; ++g)
#pragma unroll
    for (int r = 0; r < P::First::R; ++r)
      v[g * P::First::R + r] = active ? col[(long)P::First::in_index(j, g, r) * KX] : make_float2(0.f, 0.f);
  float2 ex;
  {
    const float sx = sign * __ldg(field + T + f);
    const float fx = __fmul_rn((float)kx, (float)(1.0 / (double)NX));
    float s, c;
    sincosf(__fmul_rn(__fmul_rn(-6.283185307179586f, fx), sx), &s, &c);
    ex = make_float2(c, s);
  }
  __syncthreads();
  fft2::fft_regs_to_regs<N>(sm, myseq, j, v);
  __syncthreads();  // every thread has taken its last-pass inputs out of shared memory
  const float2* py = phase_y + (long)f * N;
#pragma unroll
  for (int g = 0; g < P::Last::G; ++g)
#pragma unroll
    for (int r = 0; r < P::Last::R; ++r) {
      const int ky = P::Last::out_index(j, g, r);
      const float2 val = cmul(P::Last::result(v, g, r), cmul(__ldg(py + ky), ex));
      myseq[fft2::pad_idx(ky)] = make_float2(val.y, val.x);  // swapped: the next forward FFT is the inverse
    }
  __syncthreads();
  P::First::load(myseq, j, v);
  __syncthreads();
  fft2::fft_regs_to_regs<N>(sm, myseq, j, v);
  if (!active) return;
#pragma unroll
  for (int g = 0; g < P::Last::G; ++g)
#pragma unroll
    for (int r = 0; r < P::Last::R; ++r) {
      const float2 val = P::Last::result(v, g, r);
      col[(long)P::Last::out_index(j, g, r) * KX] = make_float2(val.y, val.x);
    }
}

// ---- Fourier crop, column pass: FFT along y at N, keep ky in [-M/2, M/2), inverse FFT at M ----------------------
// tmp[plane][y][kx] (N rows) -> out[plane][y'][kx] (M rows, unnormalised): the forward and inverse column passes of
// tmc_fourier_crop in one kernel, so the cropped spectrum never goes through HBM.  A CTA takes Cfg<M>::B columns; their
// N-point transforms run in groups of Cfg<N>::B, each group leaving its M kept bins (re/im swapped: the next forward FFT
// is the inverse) in the M-point buffers.  The M-point transform reads its inputs in the order cols_inverse_p2 reads
// them from HBM, so both crop paths compute the same values.
template <int N, int M>
constexpr size_t cols_crop_smem_bytes() {
  using CN = fft2::Cfg<N>;
  using CM = fft2::Cfg<M>;
  return (size_t)(CN::B * CN::STRIDE + CM::B * CM::STRIDE + 64 + CN::TW_HI + 64 + CM::TW_HI) * sizeof(float2);
}

template <int N, int M>
__global__ void __launch_bounds__(fft2::kThreads)
cols_crop_p2(const float2* __restrict__ tmp, int KX, const float2* __restrict__ tw_n, const float2* __restrict__ tw_m,
             float2* __restrict__ out) {
  using CN = fft2::Cfg<N>;
  using CM = fft2::Cfg<M>;
  using PN = fft2::Plan<N>;
  using PM = fft2::Plan<M>;
  static_assert(M < N && CM::B % CN::B == 0, "a CTA's M-point columns split into whole groups of N-point columns");
  extern __shared__ float2 smem[];
  float2* data_m = smem + CN::B * CN::STRIDE;
  float2* tables = data_m + CM::B * CM::STRIDE;
  fft2::Smem<N> sn(smem);
  sn.tw_lo = tables;
  sn.tw_hi = tables + 64;
  fft2::Smem<M> sm(data_m);
  sm.tw_lo = tables + 64 + CN::TW_HI;
  sm.tw_hi = sm.tw_lo + 64;
  fft2::load_twiddles<N>(sn, tw_n);
  fft2::load_twiddles<M>(sm, tw_m);
  const long plane = blockIdx.y;
  const int kx0 = blockIdx.x * CM::B;
  const float2* src = tmp + plane * N * KX;
  {
    const int seq = threadIdx.x % CN::B, j = threadIdx.x / CN::B;
    float2* myseq = smem + seq * CN::STRIDE;
#pragma unroll 1
    for (int grp = 0; grp < CM::B / CN::B; ++grp) {
      const int slot = grp * CN::B + seq;
      const bool active = kx0 + slot < KX;
      float2 v[CN::VPT];
#pragma unroll
      for (int g = 0; g < PN::First::G; ++g)
#pragma unroll
        for (int r = 0; r < PN::First::R; ++r)
          v[g * PN::First::R + r] = active ? src[(long)PN::First::in_index(j, g, r) * KX + kx0 + slot] : make_float2(0.f, 0.f);
      __syncthreads();  // tables loaded; the previous group has taken its last-pass inputs out of the N-point buffers
      fft2::fft_regs_to_regs<N>(sn, myseq, j, v);
      float2* mseq = data_m + slot * CM::STRIDE;
#pragma unroll
      for (int g = 0; g < PN::Last::G; ++g)
#pragma unroll
        for (int r = 0; r < PN::Last::R; ++r) {
          const int ky = PN::Last::out_index(j, g, r);
          const int pos = ky < M / 2 ? ky : (ky >= N - M / 2 ? ky - (N - M) : -1);
          if (pos >= 0) {
            const float2 val = PN::Last::result(v, g, r);
            mseq[fft2::pad_idx(pos)] = make_float2(val.y, val.x);
          }
        }
    }
  }
  __syncthreads();
  const int seq = threadIdx.x % CM::B, j = threadIdx.x / CM::B;
  float2* mseq = data_m + seq * CM::STRIDE;
  float2 u[CM::VPT];
  PM::First::load(mseq, j, u);
  __syncthreads();
  fft2::fft_regs_to_regs<M>(sm, mseq, j, u);
  const int kx = kx0 + seq;
  if (kx >= KX) return;
  float2* dst = out + plane * M * KX + kx;
#pragma unroll
  for (int g = 0; g < PM::Last::G; ++g)
#pragma unroll
    for (int r = 0; r < PM::Last::R; ++r) {
      const float2 val = PM::Last::result(u, g, r);
      dst[(long)PM::Last::out_index(j, g, r) * KX] = make_float2(val.y, val.x);
    }
}

// Four adjacent columns per CTA for the lengths whose FFT occupies a whole 256-thread group (Cfg<N>::B == 1, N = 4096):
// with one column per CTA every 8-byte element of the (ny, nx/2+1) spectrum costs its own 32-byte sector on the way in
// and on the way out (ncu r01g: 6.5x the algorithmic L2 traffic, the kernel's limiter).  Here a 512-thread CTA stages a
// 4-column strip (lane = (row, column): a warp request covers 8 rows x 32 contiguous bytes) in shared memory, two
// 256-thread groups transform two columns each in place, and the strip is written back the same way.
template <int N>
__global__ void __launch_bounds__(512, 1)
cols_shift_quad_p2(float2* __restrict__ tmp, int KX, int NX, const float2* __restrict__ phase_y, const float* __restrict__ field,
                   int T, float sign, const float2* __restrict__ tw) {
  using C = fft2::Cfg<N>;
  using P = fft2::Plan<N>;
  static_assert(C::B == 1 && C::TPS == 256, "one sequence per 256-thread group");
  extern __shared__ float2 smem[];
  fft2::Smem<N> sm(smem);          // data = 4 sequences, the twiddle tables follow them
  sm.tw_lo = smem + 4 * C::STRIDE;
  sm.tw_hi = sm.tw_lo + 64;
  for (int i = threadIdx.x; i < 64 + C::TW_HI; i += 512) sm.tw_lo[i] = i < 64 ? __ldg(tw + i) : __ldg(tw + (i - 64) * 64);
  const int f = blockIdx.y;
  const int kx0 = blockIdx.x * 4;
  float2* strip = tmp + (long)f * N * KX + kx0;
  // load: thread = (row slot, column)
  {
    const int c = threadIdx.x & 3, r0 = threadIdx.x >> 2;
    const bool live = kx0 + c < KX;
    float2* seq = smem + c * C::STRIDE;
#pragma unroll 8
    for (int y = r0; y < N; y += 128) seq[fft2::pad_idx(y)] = live ? strip[(long)y * KX + c] : make_float2(0.f, 0.f);
  }
  const int group = threadIdx.x >> 8, j = threadIdx.x & 255;
  const float2* py = phase_y + (long)f * N;
  const float sx = sign * __ldg(field + T + f);
  const float inv_nx = (float)(1.0 / (double)NX);
  __syncthreads();
#pragma unroll 1
  for (int cc = 0; cc < 2; ++cc) {
    const int c = group + 2 * cc;
    float2* myseq = smem + c * C::STRIDE;
    float2 ex;
    {
      float s, co;
      sincosf(__fmul_rn(__fmul_rn(-6.283185307179586f, __fmul_rn((float)(kx0 + c), inv_nx)), sx), &s, &co);
      ex = make_float2(co, s);
    }
    float2 v[C::VPT];
    P::First::load(myseq, j, v);
    __syncthreads();
    fft2::fft_regs_to_regs<N>(sm, myseq, j, v);
    __syncthreads();  // every thread has taken its last-pass inputs out of shared memory
#pragma unroll
    for (int g = 0; g < P::Last::G; ++g)
#pragma unroll
      for (int r = 0; r < P::Last::R; ++r) {
        const int ky = P::Last::out_index(j, g, r);
        const float2 val = cmul(P::Last::result(v, g, r), cmul(__ldg(py + ky), ex));
        myseq[fft2::pad_idx(ky)] = make_float2(val.y, val.x);  // swapped: the next forward FFT is the inverse
      }
    __syncthreads();
    P::First::load(myseq, j, v);
    __syncthreads();
    fft2::fft_regs_to_regs<N>(sm, myseq, j, v);
    __syncthreads();
#pragma unroll
    for (int g = 0; g < P::Last::G; ++g)
#pragma unroll
      for (int r = 0; r < P::Last::R; ++r) {
        const float2 val = P::Last::result(v, g, r);
        myseq[fft2::pad_idx(P::Last::out_index(j, g, r))] = make_float2(val.y, val.x);
      }
    __syncthreads();
  }
  {
    const int c = threadIdx.x & 3, r0 = threadIdx.x >> 2;
    if (kx0 + c < KX) {
      const float2* seq = smem + c * C::STRIDE;
#pragma unroll 8
      for (int y = r0; y < N; y += 128) strip[(long)y * KX + c] = seq[fft2::pad_idx(y)];
    }
  }
}

// phase_y[f][ky] for all frames (tiny)
__global__ void shift_phase_y_kernel(const float* __restrict__ field, int T, int NY, float sign, float2* __restrict__ phase_y) {
  const int ky = blockIdx.x * blockDim.x + threadIdx.x;
  const int f = blockIdx.y;
  if (ky >= NY) return;
  const float sy = sign * __ldg(field + f);
  const float fy = __fmul_rn((float)(ky < (NY + 1) / 2 ? ky : ky - NY), (float)(1.0 / (double)NY));
  float s, c;
  sincosf(__fmul_rn(__fmul_rn(-6.283185307179586f, fy), sy), &s, &c);
  phase_y[(long)f * NY + ky] = make_float2(c, s);
}

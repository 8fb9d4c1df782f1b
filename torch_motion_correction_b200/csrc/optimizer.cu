// Loss and analytic gradient of the spline-coefficient optimisation (estimate_local_motion).
//
// Replaces, per optimiser iteration, the reference's autograd graph through fourier_shift_dft_2d,
// the Fourier filters, the leave-one-out reference and _compute_loss
// (estimate_motion_optimizer.py:371-407,442-510,611-671; closed form: SURVEY.md Appendix E).
//
// Per patch g the inputs are the band-limited, filtered spectra FW_t = rfft2(mask P_t) * band * env
// (computed ONCE, not every iteration as the reference does, quirk Q19) and the per-frame shifts
// s_t (px).  With S_t = FW_t exp(i theta_t), theta_t = -2 pi (f_y s_y + f_x s_x), Sigma = sum_t S_t:
//   A_t = sum_f w |S_t|^2 (shift independent),  p_t = sum_f w Re(S_t conj Sigma),  q = sum_f w |Sigma|^2
// determine all three losses (w = 1 on the half spectrum for "mse", quirk Q13; Hermitian weights
// 1/2 for the real-space "cc" / "ncc"):
//   mse_g = a^2 (sum_t A_t - q / T),  a = T/(T-1)
//   cc_t  = (p_t - A_t) / (P (T-1)),  P = ph pw
//   ncc_t = cc_t / sqrt((A_t / P + eps)(B_t + eps)),  B_t = (q - 2 p_t + A_t) / (P (T-1)^2)
// and dL/ds_{t,y} = sum_f w (-c f_y) Im(S_t conj Z_t),  Z_t = (alpha_t + 2 beta) Sigma + sum_u alpha_u S_u,
// alpha_t = dL/dp_t, beta = dL/dq, c f_y = fp32(-2 pi) f_y as the reference forms it.
//
// Self-paired columns ("cc" / "ncc" only).  The reference takes the real-space patches with irfftn, whose c2r step keeps
// only the real part of the kx = 0 and (nx even) kx = nx/2 columns after the transform along y.  For a shift that is not
// a whole number of pixels S_t is not Hermitian-consistent there (the Nyquist column, and the ky = -ny/2 bin of the DC
// column when ny is even), so on those two columns the losses see H_t(ky) = (S_t(ky) + conj S_t(-ky mod ny)) / 2
// instead of S_t: Sigma, p_t, q and A_t are formed from H_t, which makes A_t shift dependent there (the kernels add
// A_t(H) - A_t(S) to the shift-independent norms every evaluation).  Because H_t(-ky) = conj H_t(ky), the gradient keeps
// the form above with the raw S_t and Z_t built from H_t, plus 2 gamma_t H_t (gamma_t = dL/dA_t) on those columns.
// The band box is symmetric in ky, so both bins of a pair lie in the same column of the box.  "mse" compares the
// half spectra directly and uses S_t everywhere.
#include "common.cuh"

namespace {

constexpr int kOptThreads = 128;

struct BandGeom {
  int ny, nx, KY, KX, ky_start;
};

// fp32(-2 pi) * f  with f = index * fp32(1/n)   (torch_fourier_shift on torch.fft.fftfreq grids)
__device__ __forceinline__ void bin_freqs(const BandGeom& g, int bin, float& cfy, float& cfx, float& herm) {
  const int kyb = bin / g.KX, kx = bin % g.KX;
  int ky = g.ky_start + kyb;
  ky = ((ky % g.ny) + g.ny) % g.ny;
  if (ky >= (g.ny + 1) / 2) ky -= g.ny;
  const float c = -6.283185307179586f;
  cfy = __fmul_rn(c, __fmul_rn((float)ky, (float)(1.0 / (double)g.ny)));
  cfx = __fmul_rn(c, __fmul_rn((float)kx, (float)(1.0 / (double)g.nx)));
  herm = (kx == 0 || 2 * kx == g.nx) ? 1.0f : 2.0f;
}

// box row of the bin (-ky mod ny, kx) that irfftn pairs with bin `bin` on a self-paired column (kx = 0, or kx = nx/2 with
// nx even), -1 on every other column; the ky = -ny/2 bin (ny even) is its own partner
__device__ __forceinline__ int partner_row(const BandGeom& g, int bin) {
  const int kyb = bin / g.KX, kx = bin % g.KX;
  if (kx != 0 && 2 * kx != g.nx) return -1;
  int ky = g.ky_start + kyb;
  ky = ((ky % g.ny) + g.ny) % g.ny;
  if (ky >= (g.ny + 1) / 2) ky -= g.ny;
  return 2 * ky == -g.ny ? kyb : -ky - g.ky_start;
}

// (S + conj S') / 2
__device__ __forceinline__ float2 hermitian_part(float2 s, float2 s_partner) {
  return make_float2(0.5f * (s.x + s_partner.x), 0.5f * (s.y - s_partner.y));
}

__device__ __forceinline__ float2 shifted(float2 fw, float cfy, float cfx, float sy, float sx) {
  const float ang = __fadd_rn(__fmul_rn(cfy, sy), __fmul_rn(cfx, sx));
  float s, c;
  sincosf(ang, &s, &c);
  return cmul(fw, make_float2(c, s));
}

__device__ __forceinline__ void block_accumulate(double v, double* target, double* sh) {
  v = warp_sum(v);
  if ((threadIdx.x & 31) == 0) atomicAdd(target, v);
  (void)sh;
}

// A[g][t] = sum_f w |FW_t|^2 for both weightings: norms[(g*T + t)*2 + {0: w=1, 1: hermitian}]
// (the shift-independent part: on the self-paired columns the "cc" / "ncc" kernels add A_t(H) - A_t(S) every
// evaluation, see the header; the tiled kernel, which runs only when those columns carry no pass-band weight beyond
// the Hermitian-consistent DC column, uses these norms as they are)
__global__ void __launch_bounds__(kOptThreads)
spectra_norms_kernel(const float2* __restrict__ spec, int T, int Tp, BandGeom geom, int frame_major,
                     double* __restrict__ norms) {
  const int g = blockIdx.y, G = gridDim.y;
  const int bins = geom.KY * geom.KX;
  const int bin = blockIdx.x * kOptThreads + threadIdx.x;
  float cfy, cfx, herm = 0.f;
  const bool live = bin < bins;
  if (live) bin_freqs(geom, bin, cfy, cfx, herm);
  for (int t = 0; t < T; ++t) {
    double v = 0.0;
    if (live) {
      // plane of (patch g, frame t): patch-major g * Tp + t, or frame-pair-major ((t / 2) G + g) 2 + t % 2
      const long plane = frame_major ? ((long)(t >> 1) * G + g) * 2 + (t & 1) : (long)g * Tp + t;
      const float2 z = spec[plane * bins + bin];
      v = (double)z.x * z.x + (double)z.y * z.y;
    }
    double v1 = warp_sum(v), v2 = warp_sum(v * herm);
    if ((threadIdx.x & 31) == 0 && (v1 != 0.0 || v2 != 0.0)) {
      atomicAdd(norms + ((long)g * T + t) * 2, v1);
      atomicAdd(norms + ((long)g * T + t) * 2 + 1, v2);
    }
  }
}

// per-bin state of the generic kernels: the bin's frequency factors and weight, and (hermitian weighting, self-paired
// column) the partner bin's offset and frequency factor, see the header
struct BinState {
  float cfy, cfx, w, pcfy;
  int partner;  // bin index of the partner, -1: S_t is used as it is
};

__device__ __forceinline__ BinState bin_state(const BandGeom& geom, int bin, bool live, int hermitian) {
  BinState b{0.f, 0.f, 0.f, 0.f, -1};
  if (!live) return b;
  float herm, pcfx;
  bin_freqs(geom, bin, b.cfy, b.cfx, herm);
  b.w = hermitian ? herm : 1.0f;
  const int pr = hermitian ? partner_row(geom, bin) : -1;
  if (pr >= 0) {
    b.partner = pr * geom.KX + bin % geom.KX;
    bin_freqs(geom, b.partner, b.pcfy, pcfx, herm);
  }
  return b;
}

// the spectrum the loss sees at frame t: S_t, or H_t on a self-paired column (s: the raw S_t)
__device__ __forceinline__ float2 loss_spectrum(const float2* __restrict__ sp_t, int bin, const BinState& b, float2 s, float sy,
                                                float sx) {
  if (b.partner < 0) return s;
  return hermitian_part(s, shifted(sp_t[b.partner - bin], b.pcfy, b.cfx, sy, sx));
}

// Sigma[g][bin], q[g], p[g][t] and (self-paired columns) dA[g][t] = A_t(H) - A_t(S)
__global__ void __launch_bounds__(kOptThreads)
loss_forward_kernel(const float2* __restrict__ spec, const float* __restrict__ shifts, int T, int Tp, BandGeom geom,
                    int hermitian, float2* __restrict__ sigma, double* __restrict__ q, double* __restrict__ p,
                    double* __restrict__ dA) {
  const int g = blockIdx.y;
  const int bins = geom.KY * geom.KX;
  const int bin = blockIdx.x * kOptThreads + threadIdx.x;
  const bool live = bin < bins;
  const BinState b = bin_state(geom, bin, live, hermitian);
  const float2* sp = spec + (long)g * Tp * bins + bin;
  const float* sh = shifts + (long)g * T * 2;
  float2 sum = make_float2(0.f, 0.f);
  if (live)
    for (int t = 0; t < T; ++t) {
      const float sy = __ldg(sh + 2 * t), sx = __ldg(sh + 2 * t + 1);
      sum = cadd(sum, loss_spectrum(sp + (long)t * bins, bin, b, shifted(sp[(long)t * bins], b.cfy, b.cfx, sy, sx), sy, sx));
    }
  if (live) sigma[(long)g * bins + bin] = sum;
  {
    double v = live ? (double)b.w * ((double)sum.x * sum.x + (double)sum.y * sum.y) : 0.0;
    v = warp_sum(v);
    if ((threadIdx.x & 31) == 0) atomicAdd(q + g, v);
  }
  const bool paired = __any_sync(0xffffffffu, b.partner >= 0);
  for (int t = 0; t < T; ++t) {
    double v = 0.0, d = 0.0;
    if (live) {
      const float sy = __ldg(sh + 2 * t), sx = __ldg(sh + 2 * t + 1);
      const float2 s = shifted(sp[(long)t * bins], b.cfy, b.cfx, sy, sx);
      const float2 h = loss_spectrum(sp + (long)t * bins, bin, b, s, sy, sx);
      v = (double)b.w * ((double)h.x * sum.x + (double)h.y * sum.y);  // Re(H conj Sigma)
      if (b.partner >= 0)
        d = (double)b.w * (((double)h.x * h.x + (double)h.y * h.y) - ((double)s.x * s.x + (double)s.y * s.y));
    }
    v = warp_sum(v);
    if ((threadIdx.x & 31) == 0) atomicAdd(p + (long)g * T + t, v);
    if (paired) {
      d = warp_sum(d);
      if ((threadIdx.x & 31) == 0 && d != 0.0) atomicAdd(dA + (long)g * T + t, d);
    }
  }
}

// loss_type: 0 mse, 1 cc, 2 ncc.  scale[g]: per-patch weight of the (mean-reduced) mini-batch loss.
// A_t = norms + dA (hermitian weighting).  Writes loss (+=), alpha[g][t], beta[g], gamma[g][t] = dL/dA_t.
// One thread per (g, t) pair is plenty.
__global__ void loss_scalars_kernel(const double* __restrict__ norms, const double* __restrict__ q, const double* __restrict__ p,
                                    const double* __restrict__ dA, const float* __restrict__ scale, int G, int T, int ph, int pw,
                                    int loss_type, float* __restrict__ alpha, float* __restrict__ beta, float* __restrict__ gamma,
                                    double* __restrict__ loss) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= G) return;
  const double sc = (double)scale[g];
  const double P = (double)ph * (double)pw;
  double l = 0.0, b = 0.0;
  for (int t = 0; t < T; ++t) gamma[(long)g * T + t] = 0.f;
  if (T < 2 || sc == 0.0) {
    for (int t = 0; t < T; ++t) alpha[(long)g * T + t] = 0.f;
    beta[g] = 0.f;
    return;
  }
  if (loss_type == 0) {
    const double a = (double)T / (double)(T - 1);
    double sumA = 0.0;
    for (int t = 0; t < T; ++t) {
      sumA += norms[((long)g * T + t) * 2 + 0];
      alpha[(long)g * T + t] = 0.f;
    }
    l = sc * a * a * (sumA - q[g] / T);
    b = -sc * a * a / T;
  } else if (loss_type == 1) {
    const double k = 1.0 / (P * (T - 1));
    for (int t = 0; t < T; ++t) {
      const double A = norms[((long)g * T + t) * 2 + 1] + dA[(long)g * T + t];
      l += -sc * k * (p[(long)g * T + t] - A);
      alpha[(long)g * T + t] = (float)(-sc * k);
      gamma[(long)g * T + t] = (float)(sc * k);
    }
  } else {
    const double eps = 1e-8;
    const double k = 1.0 / (P * (T - 1));
    const double kb = 1.0 / (P * (double)(T - 1) * (double)(T - 1));
    for (int t = 0; t < T; ++t) {
      const double A = norms[((long)g * T + t) * 2 + 1] + dA[(long)g * T + t];
      const double pt = p[(long)g * T + t];
      const double cc = k * (pt - A);
      const double X = A / P + eps;
      const double B = kb * (q[g] - 2.0 * pt + A) + eps;
      const double den = sqrt(X * B);
      const double ncc = cc / den;
      l += -sc * ncc;
      // d ncc / d p_t = k / den - cc / (2 den B) * dB/dp_t, dB/dp_t = -2 kb ; d ncc / d q = -cc / (2 den B) * kb
      const double dB = -0.5 * ncc / B;
      alpha[(long)g * T + t] = (float)(-sc * (k / den + dB * (-2.0 * kb)));
      b += -sc * dB * kb;
      // d ncc / d A_t = -k / den - ncc / (2 X) / P - ncc / (2 B) * kb
      gamma[(long)g * T + t] = (float)(-sc * (-k / den - 0.5 * ncc / (X * P) + dB * kb));
    }
  }
  beta[g] = (float)b;
  atomicAdd(loss, l);
}

// grad[g][t][2] += sum_f w (-c f) Im(S_t conj Z_t)
__global__ void __launch_bounds__(kOptThreads)
loss_backward_kernel(const float2* __restrict__ spec, const float* __restrict__ shifts, const float2* __restrict__ sigma,
                     const float* __restrict__ alpha, const float* __restrict__ beta, const float* __restrict__ gamma, int T,
                     int Tp, BandGeom geom, int hermitian, int has_alpha, float* __restrict__ grad) {
  const int g = blockIdx.y;
  const int bins = geom.KY * geom.KX;
  const int bin = blockIdx.x * kOptThreads + threadIdx.x;
  const bool live = bin < bins;
  const BinState b = bin_state(geom, bin, live, hermitian);
  const float w = b.w, cfy = b.cfy, cfx = b.cfx;
  const float2* sp = spec + (long)g * Tp * bins + bin;
  const float* sh = shifts + (long)g * T * 2;
  const float* al = alpha + (long)g * T;
  const float* ga = gamma + (long)g * T;
  const float be2 = 2.0f * __ldg(beta + g);
  float2 sum = make_float2(0.f, 0.f), wsum = make_float2(0.f, 0.f);
  if (live) {
    sum = sigma[(long)g * bins + bin];
    if (has_alpha)
      for (int t = 0; t < T; ++t) {
        const float sy = __ldg(sh + 2 * t), sx = __ldg(sh + 2 * t + 1);
        const float2 s = loss_spectrum(sp + (long)t * bins, bin, b, shifted(sp[(long)t * bins], cfy, cfx, sy, sx), sy, sx);
        const float a = __ldg(al + t);
        wsum.x += a * s.x;
        wsum.y += a * s.y;
      }
  }
  for (int t = 0; t < T; ++t) {
    float gy = 0.f, gx = 0.f;
    if (live) {
      const float sy = __ldg(sh + 2 * t), sx = __ldg(sh + 2 * t + 1);
      const float2 s = shifted(sp[(long)t * bins], cfy, cfx, sy, sx);
      const float a = (has_alpha ? __ldg(al + t) : 0.f) + be2;
      float2 z = make_float2(a * sum.x + wsum.x, a * sum.y + wsum.y);
      if (b.partner >= 0) {  // + 2 gamma_t H_t: A_t depends on the shift on this column
        const float2 h = loss_spectrum(sp + (long)t * bins, bin, b, s, sy, sx);
        const float g2 = 2.0f * __ldg(ga + t);
        z.x += g2 * h.x;
        z.y += g2 * h.y;
      }
      const float im = s.y * z.x - s.x * z.y;  // Im(S conj Z)
      gy = -w * cfy * im;
      gx = -w * cfx * im;
    }
    gy = warp_sum(gy);
    gx = warp_sum(gx);
    if ((threadIdx.x & 31) == 0 && (gy != 0.f || gx != 0.f)) {
      atomicAdd(grad + ((long)g * T + t) * 2, gy);
      atomicAdd(grad + ((long)g * T + t) * 2 + 1, gx);
    }
  }
}

// ---- fused fast path for "mse" and "cc": both depend on the shifts only through q = sum_f w |Sigma|^2
//      (Z_t = 2 b Sigma with b = -scale a^2 / T resp. -scale / (P (T-1))), so one kernel does it all. ----

// E[(g*T + t) * (KY + KX) + i]: i < KY -> exp(i cfy(i) s_y), else exp(i cfx(i - KY) s_x).
// exp(i theta) = exp(i cfy s_y) exp(i cfx s_x): 2 table reads + one complex multiply per bin and frame
// instead of a sincosf (differs from the reference's cos/sin of the summed angle by fp32 rounding only).
__global__ void phase_tables_kernel(const float* __restrict__ shifts, int T, BandGeom geom, float2* __restrict__ E) {
  const int gt = blockIdx.x;
  const float sy = shifts[2 * gt], sx = shifts[2 * gt + 1];
  const float c = -6.283185307179586f;
  for (int i = threadIdx.x; i < geom.KY + geom.KX; i += blockDim.x) {
    float ang;
    if (i < geom.KY) {
      int ky = geom.ky_start + i;
      ky = ((ky % geom.ny) + geom.ny) % geom.ny;
      if (ky >= (geom.ny + 1) / 2) ky -= geom.ny;
      ang = __fmul_rn(__fmul_rn(c, __fmul_rn((float)ky, (float)(1.0 / (double)geom.ny))), sy);
    } else {
      ang = __fmul_rn(__fmul_rn(c, __fmul_rn((float)(i - geom.KY), (float)(1.0 / (double)geom.nx))), sx);
    }
    float s, co;
    sincosf(ang, &s, &co);
    E[(long)gt * (geom.KY + geom.KX) + i] = make_float2(co, s);
  }
}

// q[g] += sum_f w |Sigma|^2 ; grad[g][t][:] += -2 b sum_f w (c f) Im(S_t conj Sigma)
// ("cc" on a self-paired column: Sigma = sum_t H_t, q[g] -= A_t(H) - A_t(S), Im(S_t conj (Sigma - H_t)); see the header)
// kFusedBins bins per thread amortise the per-frame warp reductions; UNROLL frames in flight hide load latency;
// MINB CTAs/SM caps the registers (the first version ran at 168 registers, 17 % occupancy: profiles/r01_final_*)
template <int kFusedBins, int UNROLL, int MINB>
__global__ void __launch_bounds__(kOptThreads, MINB)
loss_fused_kernel(const float2* __restrict__ spec, const float2* __restrict__ E, const float* __restrict__ patch_scale,
                  const int* __restrict__ iter_ptr, int G, int T, int Tp, BandGeom geom, int loss_type, int ph, int pw,
                  double* __restrict__ q, float* __restrict__ grad) {
  extern __shared__ float acc[];  // [T][2]
  const int g = blockIdx.y;
  const int bins = geom.KY * geom.KX;
  for (int i = threadIdx.x; i < 2 * T; i += kOptThreads) acc[i] = 0.f;
  const float sc = patch_scale[(long)(iter_ptr ? *iter_ptr : 0) * G + g];
  if (sc == 0.f || T < 2) return;
  float b;
  if (loss_type == 0) {
    const float a = (float)T / (float)(T - 1);
    b = -sc * a * a / (float)T;
  } else {
    b = -sc / ((float)ph * (float)pw * (float)(T - 1));
  }
  int bin[kFusedBins], kyb[kFusedBins], kx[kFusedBins], pyb[kFusedBins];
  float cfy[kFusedBins], cfx[kFusedBins], w[kFusedBins];
  float2 sum[kFusedBins];
#pragma unroll
  for (int i = 0; i < kFusedBins; ++i) {
    bin[i] = (blockIdx.x * kFusedBins + i) * kOptThreads + threadIdx.x;
    const bool live = bin[i] < bins;
    const int bb = live ? bin[i] : 0;
    float herm;
    bin_freqs(geom, bb, cfy[i], cfx[i], herm);
    w[i] = live ? (loss_type == 0 ? 1.0f : herm) : 0.0f;
    kyb[i] = bb / geom.KX;
    kx[i] = bb % geom.KX;
    pyb[i] = live && loss_type != 0 ? partner_row(geom, bb) : -1;
    bin[i] = bb;
    sum[i] = make_float2(0.f, 0.f);
  }
  double dq = 0.0;  // - sum_t (A_t(H) - A_t(S)) over this thread's self-paired bins
  const float2* sp = spec + (long)g * Tp * bins;
  const float2* Eg = E + (long)g * T * (geom.KY + geom.KX);
#pragma unroll UNROLL
  for (int t = 0; t < T; ++t) {
    const float2* Et = Eg + (long)t * (geom.KY + geom.KX);
#pragma unroll
    for (int i = 0; i < kFusedBins; ++i) {
      const float2 e = cmul(__ldg(Et + kyb[i]), __ldg(Et + geom.KY + kx[i]));
      float2 s = cmul(__ldg(sp + (long)t * bins + bin[i]), e);
      if (pyb[i] >= 0) {
        const float2 ep = cmul(__ldg(Et + pyb[i]), __ldg(Et + geom.KY + kx[i]));
        const float2 h = hermitian_part(s, cmul(__ldg(sp + (long)t * bins + pyb[i] * geom.KX + kx[i]), ep));
        dq -= (double)w[i] * (((double)h.x * h.x + (double)h.y * h.y) - ((double)s.x * s.x + (double)s.y * s.y));
        s = h;
      }
      sum[i] = cadd(sum[i], s);
    }
  }
  {
    double v = dq;
#pragma unroll
    for (int i = 0; i < kFusedBins; ++i) v += (double)w[i] * ((double)sum[i].x * sum[i].x + (double)sum[i].y * sum[i].y);
    v = warp_sum(v);
    if ((threadIdx.x & 31) == 0) atomicAdd(q + g, v);
  }
  __syncthreads();  // acc zeroed
#pragma unroll UNROLL
  for (int t = 0; t < T; ++t) {
    const float2* Et = Eg + (long)t * (geom.KY + geom.KX);
    float gy = 0.f, gx = 0.f;
#pragma unroll
    for (int i = 0; i < kFusedBins; ++i) {
      const float2 e = cmul(__ldg(Et + kyb[i]), __ldg(Et + geom.KY + kx[i]));
      const float2 s = cmul(__ldg(sp + (long)t * bins + bin[i]), e);
      float2 z = sum[i];
      if (pyb[i] >= 0) {
        const float2 ep = cmul(__ldg(Et + pyb[i]), __ldg(Et + geom.KY + kx[i]));
        const float2 h = hermitian_part(s, cmul(__ldg(sp + (long)t * bins + pyb[i] * geom.KX + kx[i]), ep));
        z = make_float2(z.x - h.x, z.y - h.y);
      }
      const float im = w[i] * (s.y * z.x - s.x * z.y);  // w Im(S conj Sigma)
      gy = fmaf(cfy[i], im, gy);
      gx = fmaf(cfx[i], im, gx);
    }
    gy = warp_sum(gy);
    gx = warp_sum(gx);
    if ((threadIdx.x & 31) == 0) {
      atomicAdd(acc + 2 * t, gy);
      atomicAdd(acc + 2 * t + 1, gx);
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 2 * T; i += kOptThreads) {
    const float v = -2.0f * b * acc[i];
    if (v != 0.f) atomicAdd(grad + (long)g * T * 2 + i, v);
  }
}

// loss = sum_g scale_g * l_g(q_g, sum_t A_t) ; grad_eval[t][g][c] = -(1/px) grad_shifts[g][t][c]
__global__ void loss_fused_finish_kernel(const double* __restrict__ norms, const double* __restrict__ q,
                                         const float* __restrict__ patch_scale, const int* __restrict__ iter_ptr, int G, int T,
                                         int ph, int pw, int loss_type, const float* __restrict__ grad_shifts,
                                         float pixel_spacing, double* __restrict__ loss, float* __restrict__ grad_eval) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < T * G * 2) {
    const int c = i & 1, r = i >> 1;
    const int t = r / G, g = r % G;
    grad_eval[i] = -grad_shifts[((long)g * T + t) * 2 + c] / pixel_spacing;
  }
  if (i < G && T >= 2) {
    const int g = i;
    const double sc = (double)patch_scale[(long)(iter_ptr ? *iter_ptr : 0) * G + g];
    if (sc != 0.0) {
      double sumA = 0.0;
      for (int t = 0; t < T; ++t) sumA += norms[((long)g * T + t) * 2 + (loss_type == 0 ? 0 : 1)];
      double l;
      if (loss_type == 0) {
        const double a = (double)T / (double)(T - 1);
        l = sc * a * a * (sumA - q[g] / T);
      } else {
        l = -sc * (q[g] - sumA) / ((double)ph * (double)pw * (double)(T - 1));
      }
      atomicAdd(loss, l);
    }
  }
}

__global__ void advance_counter_kernel(int* counter) { *counter += 1; }

// torch.optim.Adam (amsgrad=False, maximize=False), single-tensor formulas, step = *step_counter + 1:
//   g += wd p ; m = lerp(m, g, 1 - b1) ; v = b2 v + (1 - b2) g^2 ;
//   p -= (lr / (1 - b1^step)) * m / (sqrt(v) / sqrt(1 - b2^step) + eps)
__global__ void adam_step_kernel(float* __restrict__ param, const float* __restrict__ grad, float* __restrict__ exp_avg,
                                 float* __restrict__ exp_avg_sq, int n, double lr, double beta1, double beta2, double eps,
                                 double weight_decay, const int* __restrict__ step_counter) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  // scalars are formed in double on the "host side" of torch.optim and enter the tensor ops as fp32
  const double step = (double)(*step_counter + 1);
  const double bc1 = 1.0 - pow(beta1, step);
  const double bc2 = 1.0 - pow(beta2, step);
  const float step_size = (float)(lr / bc1);
  const float bc2_sqrt = (float)sqrt(bc2);
  const float w1 = (float)(1.0 - beta1), w2 = (float)(1.0 - beta2), b2 = (float)beta2, epsf = (float)eps;
  float g = grad[i];
  const float p = param[i];
  if (weight_decay != 0.0) g = __fadd_rn(g, __fmul_rn((float)weight_decay, p));
  const float m = __fadd_rn(exp_avg[i], __fmul_rn(w1, __fsub_rn(g, exp_avg[i])));   // lerp_(grad, 1 - beta1)
  const float v = __fadd_rn(__fmul_rn(exp_avg_sq[i], b2), __fmul_rn(w2, __fmul_rn(g, g)));  // mul_(b2).addcmul_(g, g, 1 - b2)
  exp_avg[i] = m;
  exp_avg_sq[i] = v;
  const float denom = __fadd_rn(__fdiv_rn(__fsqrt_rn(v), bc2_sqrt), epsf);
  param[i] = __fadd_rn(p, __fmul_rn(-step_size, __fdiv_rn(m, denom)));               // addcdiv_(m, denom, value=-step_size)
}

// shifts[g][t] = -(new[t][g] + base[t][g]) / pixel_spacing   (estimate_motion_optimizer.py:487-492)
__global__ void predicted_shifts_kernel(const float* __restrict__ eval_new, const float* __restrict__ eval_base, int T, int G,
                                        float pixel_spacing, float* __restrict__ shifts) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= T * G * 2) return;
  const int c = i & 1, r = i >> 1;
  const int t = r / G, g = r % G;
  const float v = __fmul_rn(-1.0f, __fadd_rn(eval_new[i], eval_base[i]));
  shifts[((long)g * T + t) * 2 + c] = __fdiv_rn(v, pixel_spacing);
}

// dL/d(eval_new[t][g][c]) = -(1/px) dL/ds[g][t][c]
__global__ void shifts_grad_to_eval_kernel(const float* __restrict__ grad_shifts, int T, int G, float pixel_spacing,
                                           float* __restrict__ grad_eval) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= T * G * 2) return;
  const int c = i & 1, r = i >> 1;
  const int t = r / G, g = r % G;
  grad_eval[i] = -grad_shifts[((long)g * T + t) * 2 + c] / pixel_spacing;
}

}  // namespace

// spec (G, Tp, KY, KX) complex64 -- or, frame_major != 0, (Tp / 2, G, 2, KY, KX): the plane order of frame-pair jobs
// listed frame pair by frame pair -- -> norms (G, T, 2) float64 (zeroed here)
TMC_API int tmc_local_spectra_norms(const void* spec, int g, int t, int tp, int ny, int nx, int ky_count, int kx_count,
                                    int ky_start, int frame_major, double* norms, cudaStream_t stream) {
  TMC_CHECK_ARG(spec && norms && g >= 1 && t >= 1 && tp >= t, "local_spectra_norms: bad arguments");
  TMC_CHECK_ARG(g <= kMaxGridYZ, "local_spectra_norms: at most %d patches, got %d", kMaxGridYZ, g);
  BandGeom geom{ny, nx, ky_count, kx_count, ky_start};
  TMC_CUDA(cudaMemsetAsync(norms, 0, sizeof(double) * (size_t)g * t * 2, stream));
  dim3 grid(tmc_div_up((long)ky_count * kx_count, kOptThreads), g);
  spectra_norms_kernel<<<grid, kOptThreads, 0, stream>>>((const float2*)spec, t, tp, geom, frame_major, norms); tmc_count_launch();
  TMC_CHECK_LAUNCH("tmc_local_spectra_norms");
  return TMC_OK;
}

// One loss + gradient evaluation.
//  eval_new / eval_base: (T, G, 2) spline values (Angstrom) at the patch centres; patch_scale (G) f32;
//  loss_type 0 mse / 1 cc / 2 ncc; outputs: loss (device double, zeroed here), grad_eval (T, G, 2) = dL/d eval_new.
//  patch_scale: (G) f32, or (n_iterations, G) when `iteration` (device int, nullable) selects the row -- this
//  lets a captured CUDA graph replay the step with a different mini-batch weighting every iteration;
//  workspace layout (floats): sigma 2*G*bins | phase tables 2*G*T*(KY+KX) | shifts 2*G*T | grad_shifts 2*G*T |
//                             alpha G*T | beta G | gamma G*T | then doubles q G | p G*T | dA G*T
static long local_loss_workspace_floats(int g, int t, int ky_count, int kx_count) {
  long bins = (long)ky_count * kx_count;
  long floats = 2 * g * bins + 2l * g * t * (ky_count + kx_count) + 2l * g * t + 2l * g * t + (long)g * t + g + (long)g * t;
  return (floats + 1) & ~1l;
}
TMC_API long tmc_local_loss_workspace_bytes(int g, int t, int ky_count, int kx_count) {
  return local_loss_workspace_floats(g, t, ky_count, kx_count) * 4 + 8l * (g + 2l * g * t);
}

TMC_API int tmc_local_loss_grad(const void* spec, const double* norms, const float* eval_new, const float* eval_base,
                                const float* patch_scale, const int* iteration, int g, int t, int tp, int ny, int nx,
                                int ky_count, int kx_count, int ky_start, float pixel_spacing, int loss_type, double* loss,
                                float* grad_eval, void* workspace, cudaStream_t stream) {
  TMC_CHECK_ARG(spec && norms && eval_new && eval_base && patch_scale && loss && grad_eval && workspace,
                "local_loss_grad: null pointer");
  TMC_CHECK_ARG(g >= 1 && t >= 1 && tp >= t && loss_type >= 0 && loss_type <= 2 && pixel_spacing > 0.f,
                "local_loss_grad: bad arguments");
  TMC_CHECK_ARG(g <= kMaxGridYZ, "local_loss_grad: at most %d patches, got %d", kMaxGridYZ, g);
  BandGeom geom{ny, nx, ky_count, kx_count, ky_start};
  const long bins = (long)ky_count * kx_count;
  float* wf = (float*)workspace;
  float2* sigma = (float2*)wf;
  float2* E = (float2*)(wf + 2 * g * bins);
  float* shifts = wf + 2 * g * bins + 2l * g * t * (ky_count + kx_count);
  float* grad_shifts = shifts + 2l * g * t;
  float* alpha = grad_shifts + 2l * g * t;
  float* beta = alpha + (long)g * t;
  float* gamma = beta + g;
  const long floats = local_loss_workspace_floats(g, t, ky_count, kx_count);
  double* q = (double*)(wf + floats);
  double* p = q + g;
  double* dA = p + (long)g * t;
  TMC_CUDA(cudaMemsetAsync(q, 0, sizeof(double) * ((size_t)g + 2 * (size_t)g * t), stream));
  TMC_CUDA(cudaMemsetAsync(grad_shifts, 0, sizeof(float) * 2 * (size_t)g * t, stream));
  TMC_CUDA(cudaMemsetAsync(loss, 0, sizeof(double), stream));
  const int n = t * g * 2;
  predicted_shifts_kernel<<<tmc_div_up(n, 128), 128, 0, stream>>>(eval_new, eval_base, t, g, pixel_spacing, shifts); tmc_count_launch();
  if (loss_type != 2) {
    phase_tables_kernel<<<g * t, 128, 0, stream>>>(shifts, t, geom, E); tmc_count_launch();
    // Measured alternatives that were SLOWER than this streaming kernel (C2, 100 iterations per movie: 16.3 ms):
    // all frames of a bin tile kept in shared memory (+20..75 %), all frames of one bin kept in registers with a
    // shared-memory transpose for the per-frame reductions (+45 %), 64-register / high-occupancy variants (+10..45 %).
    {
      // 4 bins per thread, 4 frames in flight: measured fastest (ILP beats occupancy here; the 64-register
      // variants with 2-8 CTAs/SM were 10-45 % slower)
      dim3 fgrid(tmc_div_up(bins, kOptThreads * 4), g);
      loss_fused_kernel<4, 4, 1><<<fgrid, kOptThreads, sizeof(float) * 2 * t, stream>>>(
          (const float2*)spec, E, patch_scale, iteration, g, t, tp, geom, loss_type, ny, nx, q, grad_shifts);
    }
    tmc_count_launch();
    loss_fused_finish_kernel<<<tmc_div_up(n > g ? n : g, 128), 128, 0, stream>>>(norms, q, patch_scale, iteration, g, t, ny, nx,
                                                                                 loss_type, grad_shifts, pixel_spacing, loss,
                                                                                 grad_eval); tmc_count_launch();
    TMC_CHECK_LAUNCH("tmc_local_loss_grad(fused)");
    return TMC_OK;
  }
  TMC_CHECK_ARG(iteration == nullptr, "local_loss_grad: the ncc path takes the per-iteration scale row directly");
  const int hermitian = loss_type != 0;
  dim3 grid(tmc_div_up(bins, kOptThreads), g);
  loss_forward_kernel<<<grid, kOptThreads, 0, stream>>>((const float2*)spec, shifts, t, tp, geom, hermitian, sigma, q, p, dA);
  tmc_count_launch();
  loss_scalars_kernel<<<tmc_div_up(g, 64), 64, 0, stream>>>(norms, q, p, dA, patch_scale, g, t, ny, nx, loss_type, alpha, beta, gamma,
                                                            loss); tmc_count_launch();
  loss_backward_kernel<<<grid, kOptThreads, 0, stream>>>((const float2*)spec, shifts, sigma, alpha, beta, gamma, t, tp, geom, hermitian,
                                                        loss_type != 0, grad_shifts); tmc_count_launch();
  shifts_grad_to_eval_kernel<<<tmc_div_up(n, 128), 128, 0, stream>>>(grad_shifts, t, g, pixel_spacing, grad_eval); tmc_count_launch();
  TMC_CHECK_LAUNCH("tmc_local_loss_grad");
  return TMC_OK;
}


// *counter += 1 on the stream (device-side iteration index of a captured optimiser step)
TMC_API int tmc_advance_counter(int* counter, cudaStream_t stream) {
  TMC_CHECK_ARG(counter, "advance_counter: null pointer");
  advance_counter_kernel<<<1, 1, 0, stream>>>(counter); tmc_count_launch();
  TMC_CHECK_LAUNCH("tmc_advance_counter");
  return TMC_OK;
}

// One torch.optim.Adam step (amsgrad off) on n parameters; step number = *step_counter + 1 (device int)
TMC_API int tmc_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int n, double lr, double beta1,
                          double beta2, double eps, double weight_decay, const int* step_counter, cudaStream_t stream) {
  TMC_CHECK_ARG(param && grad && exp_avg && exp_avg_sq && step_counter && n >= 1, "adam_step: bad arguments");
  adam_step_kernel<<<tmc_div_up(n, 128), 128, 0, stream>>>(param, grad, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps, weight_decay,
                                                          step_counter); tmc_count_launch();
  TMC_CHECK_LAUNCH("tmc_adam_step");
  return TMC_OK;
}

// Tail of estimate_motion_cross_correlation_patches on the (T, gh, gw) patch shifts, entirely on
// the device (the reference round-trips through the host per patch and per frame):
//   per-frame outlier rejection        estimate_motion_xc.py:538-627  (quirk Q8)
//   px -> Angstrom, add to base field  estimate_motion_xc.py:381-388
//   Savitzky-Golay (polyorder 1)       estimate_motion_xc.py:486-535  (quirk Q9, scipy mode="interp")
//   subtract ONE joint scalar mean     estimate_motion_xc.py:410      (quirk Q4)
// and of estimate_global_motion (px -> Angstrom into a (2, T, 1, 1) field, :131-133).
#include "common.cuh"

namespace {

// shifts (T, G, 2) px; field (2, T, G) Angstrom, updated in place; skip_frame: frame left untouched (-1: none)
__global__ void reject_and_accumulate_kernel(const float* __restrict__ shifts, int T, int G, int reject, float threshold,
                                             float pixel_spacing, int skip_frame, float* __restrict__ field) {
  const int k = blockIdx.x;
  if (k == skip_frame) return;
  extern __shared__ float sh[];  // [2][G] values, then flags
  float* vy = sh;
  float* vx = sh + G;
  int* bad = reinterpret_cast<int*>(sh + 2 * G);
  __shared__ float med[2], sd[2], mean_valid[2];
  __shared__ int n_valid;
  for (int g = threadIdx.x; g < G; g += blockDim.x) {
    vy[g] = shifts[((long)k * G + g) * 2 + 0];
    vx[g] = shifts[((long)k * G + g) * 2 + 1];
  }
  __syncthreads();
  if (reject) {
    // lower median by rank counting (torch.median), unbiased std (torch.std)
    for (int c = 0; c < 2; ++c) {
      const float* v = c == 0 ? vy : vx;
      for (int g = threadIdx.x; g < G; g += blockDim.x) {
        int rank = 0;
        for (int o = 0; o < G; ++o) rank += (v[o] < v[g]) || (v[o] == v[g] && o < g);
        if (rank == (G - 1) / 2) med[c] = v[g];
      }
      if (threadIdx.x == 0) {
        double s = 0.0;
        for (int g = 0; g < G; ++g) s += v[g];
        const double m = s / G;
        double ss = 0.0;
        for (int g = 0; g < G; ++g) ss += (v[g] - m) * (v[g] - m);
        sd[c] = G > 1 ? (float)sqrt(ss / (G - 1)) : NAN;
      }
    }
    __syncthreads();
    for (int g = threadIdx.x; g < G; g += blockDim.x) {
      // torch.max(std, 1e-6) propagates NaN (single patch): z is NaN, nothing is rejected
      const float sy = (sd[0] != sd[0]) ? sd[0] : fmaxf(sd[0], 1e-6f);
      const float sx = (sd[1] != sd[1]) ? sd[1] : fmaxf(sd[1], 1e-6f);
      const float zy = fabsf(vy[g] - med[0]) / sy, zx = fabsf(vx[g] - med[1]) / sx;
      bad[g] = (zy > threshold) || (zx > threshold);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      double sy = 0.0, sx = 0.0;
      int n = 0;
      for (int g = 0; g < G; ++g)
        if (!bad[g]) {
          sy += vy[g];
          sx += vx[g];
          ++n;
        }
      n_valid = n;
      mean_valid[0] = n > 0 ? (float)(sy / n) : med[0];
      mean_valid[1] = n > 0 ? (float)(sx / n) : med[1];
    }
    __syncthreads();
    for (int g = threadIdx.x; g < G; g += blockDim.x)
      if (bad[g]) {
        vy[g] = mean_valid[0];
        vx[g] = mean_valid[1];
      }
    __syncthreads();
  }
  for (int g = threadIdx.x; g < G; g += blockDim.x) {
    field[((long)0 * T + k) * G + g] += __fmul_rn(vy[g], pixel_spacing);
    field[((long)1 * T + k) * G + g] += __fmul_rn(vx[g], pixel_spacing);
  }
}

// Savitzky-Golay, polyorder 1, window w <= T, scipy mode="interp": moving average inside, least-squares line through
// the first / last w samples at the edges.  in/out (2, T, G).  An even window (the reference caps an odd window at an
// even frame count, quirk Q9; scipy >= 1.11 accepts it) averages x[i - w/2 + 1 .. i + w/2]: scipy evaluates the fit at
// pos = w/2 - 0.5 and ndimage's convolve1d places an even kernel one sample to the right.
__global__ void savgol_linear_kernel(const float* __restrict__ in, int T, int G, int window, float* __restrict__ out) {
  const int series = blockIdx.x * blockDim.x + threadIdx.x;  // (c, g)
  if (series >= 2 * G) return;
  const int c = series / G, g = series % G;
  const float* x = in + (long)c * T * G + g;
  float* y = out + (long)c * T * G + g;
  const int half = window / 2;
  const int left = (window & 1) ? half : half - 1;  // samples before i inside the window
  for (int i = half; i < T - half; ++i) {
    double s = 0.0;
    for (int j = -left; j <= half; ++j) s += (double)x[(long)(i + j) * G];
    y[(long)i * G] = (float)(s / window);
  }
  const double xm = 0.5 * (window - 1);
  double sxx = 0.0;
  for (int j = 0; j < window; ++j) sxx += (j - xm) * (j - xm);
  for (int side = 0; side < 2; ++side) {
    const int start = side == 0 ? 0 : T - window;
    double ym = 0.0;
    for (int j = 0; j < window; ++j) ym += (double)x[(long)(start + j) * G];
    ym /= window;
    double sxy = 0.0;
    for (int j = 0; j < window; ++j) sxy += (j - xm) * ((double)x[(long)(start + j) * G] - ym);
    const double slope = sxy / sxx;
    for (int j = 0; j < half; ++j) {
      const int pos = side == 0 ? j : window - half + j;  // position inside the fitted window
      y[(long)(start + pos) * G] = (float)(ym + slope * (pos - xm));
    }
  }
}

// field -= mean(field) (fp32 values, double accumulation); single CTA
__global__ void subtract_mean_kernel(float* __restrict__ field, long n) {
  __shared__ double sh[32];
  __shared__ float mean;
  double s = 0.0;
  for (long i = threadIdx.x; i < n; i += blockDim.x) s += (double)field[i];
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double tot = 0.0;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) tot += sh[i];
    mean = (float)(tot / (double)n);
  }
  __syncthreads();
  for (long i = threadIdx.x; i < n; i += blockDim.x) field[i] = __fsub_rn(field[i], mean);
}

// (T, 1, 2) px shifts -> (2, T, 1, 1) Angstrom field; frame `zero_frame` gets zero shift
__global__ void global_field_kernel(const float* __restrict__ shifts, int T, float pixel_spacing, int zero_frame,
                                    float* __restrict__ field) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= T) return;
  const float sy = k == zero_frame ? 0.f : shifts[2 * k], sx = k == zero_frame ? 0.f : shifts[2 * k + 1];
  field[k] = __fmul_rn(sy, pixel_spacing);
  field[T + k] = __fmul_rn(sx, pixel_spacing);
}

}  // namespace

// shifts (T, G, 2) px; field (2, T, G) Angstrom holds the base field on entry and the result on exit;
// scratch: 2*T*G floats (only used when smoothing is applied).
TMC_API int tmc_xc_postprocess(const float* shifts, int t, int g, float pixel_spacing, int skip_frame, int outlier_rejection,
                               float outlier_threshold, int temporal_smoothing, int smoothing_window, int subtract_mean,
                               float* field, float* scratch, cudaStream_t stream) {
  TMC_CHECK_ARG(shifts && field && scratch && t >= 1 && g >= 1, "xc_postprocess: bad arguments");
  const size_t smem = (size_t)g * (2 * sizeof(float) + sizeof(int));
  TMC_CHECK_ARG(smem <= 48 * 1024, "xc_postprocess: too many patches per frame (%d)", g);
  reject_and_accumulate_kernel<<<t, 128, smem, stream>>>(shifts, t, g, outlier_rejection, outlier_threshold, pixel_spacing,
                                                         skip_frame, field); tmc_count_launch();
  if (temporal_smoothing) {
    int window = smoothing_window;
    if (window % 2 == 0) window += 1;
    if (window > t) window = t;
    // an even t caps the window at an even value: savgol_filter accepts even windows since scipy 1.11
    if (window >= 3) {
      TMC_CUDA(cudaMemcpyAsync(scratch, field, sizeof(float) * 2 * (size_t)t * g, cudaMemcpyDeviceToDevice, stream));
      savgol_linear_kernel<<<tmc_div_up(2 * g, 64), 64, 0, stream>>>(scratch, t, g, window, field); tmc_count_launch();
    }
  }
  if (subtract_mean) {
    subtract_mean_kernel<<<1, 256, 0, stream>>>(field, 2l * t * g);
    tmc_count_launch();
  }
  TMC_CHECK_LAUNCH("tmc_xc_postprocess");
  return TMC_OK;
}

TMC_API int tmc_global_shifts_to_field(const float* shifts, int t, float pixel_spacing, int zero_frame, float* field,
                                       cudaStream_t stream) {
  TMC_CHECK_ARG(shifts && field && t >= 1, "global_shifts_to_field: bad arguments");
  global_field_kernel<<<tmc_div_up(t, 128), 128, 0, stream>>>(shifts, t, pixel_spacing, zero_frame, field); tmc_count_launch();
  TMC_CHECK_LAUNCH("tmc_global_shifts_to_field");
  return TMC_OK;
}

// data -= mean(data), one joint scalar (quirk Q4: estimate_motion_optimizer.py:148,432-434)
TMC_API int tmc_subtract_mean(float* data, long n, cudaStream_t stream) {
  TMC_CHECK_ARG(data && n >= 1, "subtract_mean: bad arguments");
  subtract_mean_kernel<<<1, 256, 0, stream>>>(data, n); tmc_count_launch();
  TMC_CHECK_LAUNCH("tmc_subtract_mean");
  return TMC_OK;
}

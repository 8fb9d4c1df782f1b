// One-off tables, built on the device so no estimator call ever touches the host:
//  * the soft-edged circular real-space mask  (torch_grid_utils.circle; SURVEY.md A.4)
//  * the band-limited Fourier weight  bandpass * b_envelope  (torch_fourier_filter; A.5),
//    evaluated only on the band-pass bounding box that the FFT kernels keep.
// Reference call sites: estimate_motion_xc.py:69-74,81-95,262-280; estimate_motion_optimizer.py:162-184;
// utils.py:87-114.
#include "common.cuh"

namespace {

// half-width of the disc on every row: largest dx with sqrt(dy^2 + dx^2) < radius (fp32, like
// coordinate_grid(norm=True) < radius), or -1 if the row misses the disc
__global__ void disc_rows_kernel(int h, int w, int cy, int cx, float radius, int* __restrict__ half_width) {
  const int y = blockIdx.x * blockDim.x + threadIdx.x;
  if (y >= h) return;
  const float dy = (float)(y - cy);
  const float dy2 = __fmul_rn(dy, dy);
  int r = -1;
  const int max_dx = max(cx, w - 1 - cx);
  for (int dx = 0; dx <= max_dx; ++dx) {
    const float fx = (float)dx;
    const float d = __fsqrt_rn(__fadd_rn(dy2, __fmul_rn(fx, fx)));
    if (d < radius)
      r = dx;
    else
      break;
  }
  half_width[y] = r;
}

// exact Euclidean distance transform of the complement of the disc, restricted to the soft edge
__global__ void soft_disc_kernel(int h, int w, int cy, int cx, float radius, float smoothing, const int* __restrict__ half_width,
                                 float* __restrict__ mask) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y;
  if (x >= w) return;
  const int adx = abs(x - cx);
  const int hw = half_width[y];
  float value = 0.f;
  if (hw >= 0 && adx <= hw) {
    value = 1.f;
  } else if (smoothing > 0.f &&
             sqrtf((float)(y - cy) * (float)(y - cy) + (float)(x - cx) * (float)(x - cx)) <= radius + smoothing + 2.f) {
    const int reach = (int)ceilf(smoothing) + 1;
    long best = -1;
    for (int yy = max(0, y - reach); yy <= min(h - 1, y + reach); ++yy) {
      const int r = half_width[yy];
      if (r < 0) continue;
      // nearest member of the run [cx - r, cx + r] clipped to the image
      const int lo = max(0, cx - r), hi = min(w - 1, cx + r);
      const long gx = x < lo ? lo - x : (x > hi ? x - hi : 0);
      const long gy = y - yy;
      const long d2 = gx * gx + gy * gy;
      if (best < 0 || d2 < best) best = d2;
    }
    if (best > 0) {
      const float edt = (float)sqrt((double)best);  // scipy EDT is float64, then .float()
      if (edt <= smoothing) value = cosf(__fmul_rn(1.5707963267948966f, __fdiv_rn(edt, smoothing)));
    }
  }
  mask[(long)y * w + x] = value;
}

// weight[kyb][kx] for ky = ky_start + kyb, kx in [0, KX): (low < f <= high) * exp(-B (f/px)^2 / 4)
__global__ void band_weight_kernel(int ny, int nx, int KY, int KX, int ky_start, float low, float high, int use_band,
                                   float b_factor, float pixel_size, int use_envelope, float* __restrict__ weight) {
  const int kx = blockIdx.x * blockDim.x + threadIdx.x;
  const int kyb = blockIdx.y;
  if (kx >= KX) return;
  int ky = ky_start + kyb;  // signed frequency index
  ky = ((ky % ny) + ny) % ny;
  if (ky >= (ny + 1) / 2) ky -= ny;
  // torch.fft.fftfreq / rfftfreq: integer index times fp32(1/n)
  const float fy = __fmul_rn((float)ky, (float)(1.0 / (double)ny));
  const float fx = __fmul_rn((float)kx, (float)(1.0 / (double)nx));
  const float f = __fsqrt_rn(__fadd_rn(__fmul_rn(fy, fy), __fmul_rn(fx, fx)));
  float v = 1.f;
  if (use_band && !(f > low && f <= high)) v = 0.f;
  if (use_envelope && v != 0.f) {
    const float fp = __fdiv_rn(f, pixel_size);
    v *= expf(-__fdiv_rn(__fmul_rn(b_factor, __fmul_rn(fp, fp)), 4.0f));
  }
  weight[(long)kyb * KX + kx] = v;
}

// Dose-weighted frame sum in Fourier space (examples/ttMotion.py:331-351 -> torch_fourier_filter.dose_weight_movie,
// SURVEY.md A.6): out[ky][kx] = sum_t spec[t][ky][kx] q_t(k) / sqrt(sum_t q_t(k)^2),
// q_t = exp(-N_t / (2 N_e(k))), N_t = pre_exposure + (t + 1) dose_per_frame, N_e(k) = scale (0.24499 k^-1.6649 + 2.8141),
// k = |f| / pixel_size in 1/Angstrom.  One thread per bin, frames streamed (coalesced over kx).
__global__ void dose_weighted_sum_kernel(const float2* __restrict__ spec, int T, int ny, int nx, float pixel_size,
                                         float pre_exposure, float dose_per_frame, float ne_scale, int frame_offset,
                                         float2* __restrict__ out_num, float* __restrict__ out_den2, int finalize) {
  const int kxn = nx / 2 + 1;
  const int kx = blockIdx.x * blockDim.x + threadIdx.x;
  const int kyi = blockIdx.y;
  if (kx >= kxn) return;
  const int ky = kyi < (ny + 1) / 2 ? kyi : kyi - ny;
  const float fy = __fmul_rn((float)ky, (float)(1.0 / (double)ny));
  const float fx = __fmul_rn((float)kx, (float)(1.0 / (double)nx));
  const float f = __fsqrt_rn(__fadd_rn(__fmul_rn(fy, fy), __fmul_rn(fx, fx)));
  const float k = fmaxf(__fdiv_rn(f, pixel_size), 1e-10f);
  const float ne = ne_scale * (0.24499f * powf(k, -1.6649f) + 2.8141f);
  const long bin = (long)kyi * kxn + kx;
  float2 num = make_float2(0.f, 0.f);
  float den2 = 0.f;
  for (int t = 0; t < T; ++t) {
    const float dose = pre_exposure + dose_per_frame * (float)(frame_offset + t + 1);
    const float q = expf(-0.5f * dose / ne);
    const float2 z = spec[(long)t * ny * kxn + bin];
    num.x = fmaf(q, z.x, num.x);
    num.y = fmaf(q, z.y, num.y);
    den2 = fmaf(q, q, den2);
  }
  if (out_den2) {  // frame blocks / frame-split ranks accumulate numerator and sum of squares, the last call finalises
    num.x += out_num[bin].x;
    num.y += out_num[bin].y;
    den2 += out_den2[bin];
    out_den2[bin] = den2;
  }
  if (finalize) {
    const float inv = rsqrtf(den2);
    num.x *= inv;
    num.y *= inv;
  }
  out_num[bin] = num;
}

// ---- exposure (dose) weights as a per-frame pre-filter of band-limited patch spectra ------------------------------------
// ne[kyb][kx] = N_e(k) and inv_norm[kyb][kx] = 1 / sqrt(sum_t q_t(k)^2) on the band box (ky = ky_start + kyb)
__global__ void dose_tables_kernel(int ny, int nx, int KY, int KX, int ky_start, int T, float pixel_size, float pre_exposure,
                                   float dose_per_frame, float ne_scale, float* __restrict__ ne_out, float* __restrict__ inv_norm) {
  const int kx = blockIdx.x * blockDim.x + threadIdx.x;
  const int kyb = blockIdx.y;
  if (kx >= KX) return;
  int ky = ky_start + kyb;
  ky = ((ky % ny) + ny) % ny;
  if (ky >= (ny + 1) / 2) ky -= ny;
  const float fy = __fmul_rn((float)ky, (float)(1.0 / (double)ny));
  const float fx = __fmul_rn((float)kx, (float)(1.0 / (double)nx));
  const float f = __fsqrt_rn(__fadd_rn(__fmul_rn(fy, fy), __fmul_rn(fx, fx)));
  const float k = fmaxf(__fdiv_rn(f, pixel_size), 1e-10f);
  const float ne = ne_scale * (0.24499f * powf(k, -1.6649f) + 2.8141f);
  float den2 = 0.f;
  for (int t = 0; t < T; ++t) {
    const float q = expf(-0.5f * (pre_exposure + dose_per_frame * (float)(t + 1)) / ne);
    den2 = fmaf(q, q, den2);
  }
  ne_out[(long)kyb * KX + kx] = ne;
  inv_norm[(long)kyb * KX + kx] = rsqrtf(den2);
}

// spec plane p (p = 2 job + {0: frame_a, 1: frame_b}) *= q_frame(k) / sqrt(sum_t q_t^2)
__global__ void dose_filter_spectra_kernel(float2* __restrict__ spec, const int* __restrict__ jobs, long bins,
                                           const float* __restrict__ ne, const float* __restrict__ inv_norm, float pre_exposure,
                                           float dose_per_frame) {
  const long bin = (long)blockIdx.x * blockDim.x + threadIdx.x;
  const int plane = blockIdx.y;
  if (bin >= bins) return;
  const int frame = jobs[(plane >> 1) * 6 + ((plane & 1) ? 2 : 0)];
  if (frame < 0) return;
  const float q = expf(-0.5f * (pre_exposure + dose_per_frame * (float)(frame + 1)) / __ldg(ne + bin)) * __ldg(inv_norm + bin);
  float2* z = spec + (long)plane * bins + bin;
  const float2 v = *z;
  *z = make_float2(v.x * q, v.y * q);
}

// ---- low-rank dose weighting (dose_weight.exposure_filter_lowrank) -------------------------------------------------------
// The normalised exposure weights w_t(k) = q_t(k) / sqrt(sum_t q_t(k)^2) depend on k only through x = 1 / N_e(k), and as a
// (frames x x) matrix they have very low rank: w_t(k) ~= sum_r U_r(t) v_r(x(k)) to 1e-6 (L2 over t) with R <= 8 for real
// exposures.  spec plane p holds the spectrum of the real-space sum sum_t U_r(t) c_t for one (group, r); table row p holds
// v_r on a uniform grid of x in [0, x_max].  out[o][bin] = sum over the planes p with bit o of plane_outputs[p] of
// lerp(table[p], x(k)) * spec[p][bin].  k as in dose_weighted_sum_kernel (same float operations, same N_e).
constexpr int kMaxLowRankOutputs = 3;
__global__ void dose_lowrank_combine_kernel(const float2* __restrict__ spec, int n_spec, int ny, int nx, float pixel_size,
                                            float ne_scale, const float* __restrict__ table, int n_table, float x_max,
                                            const int* __restrict__ plane_outputs, int n_out, float2* __restrict__ out) {
  const int kxn = nx / 2 + 1;
  const int kx = blockIdx.x * blockDim.x + threadIdx.x;
  const int kyi = blockIdx.y;
  if (kx >= kxn) return;
  const int ky = kyi < (ny + 1) / 2 ? kyi : kyi - ny;
  const float fy = __fmul_rn((float)ky, (float)(1.0 / (double)ny));
  const float fx = __fmul_rn((float)kx, (float)(1.0 / (double)nx));
  const float f = __fsqrt_rn(__fadd_rn(__fmul_rn(fy, fy), __fmul_rn(fx, fx)));
  const float k = fmaxf(__fdiv_rn(f, pixel_size), 1e-10f);
  const float ne = ne_scale * (0.24499f * powf(k, -1.6649f) + 2.8141f);
  const float pos = fminf(fmaxf(__fdiv_rn(1.0f, ne) / x_max * (float)(n_table - 1), 0.f), (float)(n_table - 1));
  const int i = min((int)pos, n_table - 2);
  const float frac = pos - (float)i;
  const long bins = (long)ny * kxn, bin = (long)kyi * kxn + kx;
  float2 acc[kMaxLowRankOutputs];
#pragma unroll
  for (int o = 0; o < kMaxLowRankOutputs; ++o) acc[o] = make_float2(0.f, 0.f);
  for (int p = 0; p < n_spec; ++p) {
    const float* row = table + (long)p * n_table + i;
    const float v = fmaf(frac, __ldg(row + 1) - __ldg(row), __ldg(row));
    const float2 z = spec[p * bins + bin];
    const int mask = __ldg(plane_outputs + p);
#pragma unroll
    for (int o = 0; o < kMaxLowRankOutputs; ++o)
      if (mask & (1 << o)) {
        acc[o].x = fmaf(v, z.x, acc[o].x);
        acc[o].y = fmaf(v, z.y, acc[o].y);
      }
  }
  for (int o = 0; o < n_out; ++o) out[o * bins + bin] = acc[o];
}

}  // namespace

// Exposure filter of torch_fourier_filter.dose_weight_movie (SURVEY.md A.6) applied per frame to the band-limited
// spectra of tmc_rfft2_band (planes 2 job + {0,1} <-> jobs[job].frame_a / frame_b): an additive pre-filter of the
// patch cross-correlation (the reference filters with band-pass and B-factor only, estimate_motion_xc.py:338-346).
// tables: 2 * ky_count * kx_count floats of scratch; total_frames = frames of the movie (normalisation).
TMC_API int tmc_dose_filter_spectra(void* spec, const int* jobs, int njobs, int ny, int nx, int ky_count, int kx_count,
                                    int ky_start, int total_frames, float pixel_size, float pre_exposure, float dose_per_frame,
                                    float voltage_kv, float* tables, cudaStream_t stream) {
  TMC_CHECK_ARG(spec && jobs && tables && njobs >= 1 && ky_count >= 1 && kx_count >= 1 && total_frames >= 1 && pixel_size > 0.f,
                "dose_filter_spectra: bad arguments");
  const long bins = (long)ky_count * kx_count;
  {
    dim3 grid(tmc_div_up(kx_count, 128), ky_count);
    dose_tables_kernel<<<grid, 128, 0, stream>>>(ny, nx, ky_count, kx_count, ky_start, total_frames, pixel_size, pre_exposure,
                                                dose_per_frame, voltage_kv >= 300.f ? 1.0f : 0.8f, tables, tables + bins);
    tmc_count_launch();
  }
  TMC_CHECK_ARG(2l * njobs <= kMaxGridYZ, "dose_filter_spectra: too many planes for one launch (chunk the jobs)");
  dim3 grid(tmc_div_up(bins, 256), 2 * njobs);
  dose_filter_spectra_kernel<<<grid, 256, 0, stream>>>((float2*)spec, jobs, bins, tables, tables + bins, pre_exposure,
                                                      dose_per_frame); tmc_count_launch();
  TMC_CHECK_LAUNCH("tmc_dose_filter_spectra");
  return TMC_OK;
}

// spec (t, ny, nx/2+1) complex64 spectra of t frames (frames frame_offset .. of the movie) -> out (ny, nx/2+1) complex64.
// den2 (ny, nx/2+1) f32 nullable: running sum of q^2 for accumulation over frame blocks (zero it before the first
// block; then out is accumulated too); finalize != 0 divides by sqrt(sum q^2).  voltage_kv < 300 uses the 0.8 scaling.
TMC_API int tmc_dose_weighted_sum(const void* spec, int t, int ny, int nx, float pixel_size, float pre_exposure,
                                  float dose_per_frame, float voltage_kv, int frame_offset, void* out, float* den2,
                                  int finalize, cudaStream_t stream) {
  TMC_CHECK_ARG(spec && out && t >= 1 && ny >= 1 && nx >= 2 && pixel_size > 0.f && frame_offset >= 0,
                "dose_weighted_sum: bad arguments");
  TMC_CHECK_ARG(ny <= kMaxGridYZ, "dose_weighted_sum: at most %d rows, got %d", kMaxGridYZ, ny);
  dim3 grid(tmc_div_up(nx / 2 + 1, 128), ny);
  dose_weighted_sum_kernel<<<grid, 128, 0, stream>>>((const float2*)spec, t, ny, nx, pixel_size, pre_exposure, dose_per_frame,
                                                    voltage_kv >= 300.f ? 1.0f : 0.8f, frame_offset, (float2*)out, den2,
                                                    finalize); tmc_count_launch();
  TMC_CHECK_LAUNCH("tmc_dose_weighted_sum");
  return TMC_OK;
}

// mask (h, w) f32; workspace: h ints.  Non-zero rows lie within |y - h/2| <= radius + smoothing_radius.
TMC_API int tmc_soft_disc_mask(int h, int w, float radius, float smoothing_radius, float* mask, int* workspace,
                               cudaStream_t stream) {
  TMC_CHECK_ARG(mask && workspace && h >= 1 && w >= 1 && radius >= 0.f && smoothing_radius >= 0.f,
                "soft_disc_mask: bad arguments");
  TMC_CHECK_ARG(h <= kMaxGridYZ, "soft_disc_mask: at most %d rows, got %d", kMaxGridYZ, h);
  const int cy = h / 2, cx = w / 2;  // torch_grid_utils: centre = shape // 2
  disc_rows_kernel<<<tmc_div_up(h, 128), 128, 0, stream>>>(h, w, cy, cx, radius, workspace); tmc_count_launch();
  dim3 grid(tmc_div_up(w, 128), h);
  soft_disc_kernel<<<grid, 128, 0, stream>>>(h, w, cy, cx, radius, smoothing_radius, workspace, mask); tmc_count_launch();
  TMC_CHECK_LAUNCH("tmc_soft_disc_mask");
  return TMC_OK;
}

TMC_API int tmc_band_weights(int ny, int nx, int ky_count, int kx_count, int ky_start, float low, float high, int use_band,
                             float b_factor, float pixel_size, int use_envelope, float* weight, cudaStream_t stream) {
  TMC_CHECK_ARG(weight && ny >= 1 && nx >= 1 && ky_count >= 1 && kx_count >= 1 && kx_count <= nx / 2 + 1 && pixel_size > 0.f,
                "band_weights: bad arguments");
  TMC_CHECK_ARG(ky_count <= kMaxGridYZ, "band_weights: at most %d rows, got %d", kMaxGridYZ, ky_count);
  dim3 grid(tmc_div_up(kx_count, 128), ky_count);
  band_weight_kernel<<<grid, 128, 0, stream>>>(ny, nx, ky_count, kx_count, ky_start, low, high, use_band, b_factor,
                                              pixel_size, use_envelope, weight); tmc_count_launch();
  TMC_CHECK_LAUNCH("tmc_band_weights");
  return TMC_OK;
}

// spec (n_spec, ny, nx/2+1) complex64 -> out (n_out, ny, nx/2+1) complex64, see dose_lowrank_combine_kernel.  table
// (n_spec, n_table) f32 and plane_outputs (n_spec) int32 (bit o: the plane adds to output o) are device arrays;
// n_out <= 3; voltage_kv < 300 uses the 0.8 scaling of N_e.
TMC_API int tmc_dose_lowrank_combine(const void* spec, int n_spec, int ny, int nx, float pixel_size, float voltage_kv,
                                     const float* table, int n_table, float x_max, const int* plane_outputs, int n_out,
                                     void* out, cudaStream_t stream) {
  TMC_CHECK_ARG(spec && table && plane_outputs && out, "dose_lowrank_combine: null pointer");
  TMC_CHECK_ARG(n_spec >= 1 && ny >= 1 && nx >= 2 && n_table >= 2, "dose_lowrank_combine: bad shape n_spec=%d ny=%d nx=%d "
                "n_table=%d", n_spec, ny, nx, n_table);
  TMC_CHECK_ARG(ny <= kMaxGridYZ, "dose_lowrank_combine: at most %d rows, got %d", kMaxGridYZ, ny);
  TMC_CHECK_ARG(n_out >= 1 && n_out <= kMaxLowRankOutputs, "dose_lowrank_combine: n_out=%d outside [1, %d]", n_out,
                kMaxLowRankOutputs);
  TMC_CHECK_ARG(pixel_size > 0.f && x_max > 0.f, "dose_lowrank_combine: pixel_size and x_max must be > 0");
  dim3 grid(tmc_div_up(nx / 2 + 1, 128), ny);
  TMC_TIMED("dose_lowrank_combine_kernel", stream,
            dose_lowrank_combine_kernel<<<grid, 128, 0, stream>>>((const float2*)spec, n_spec, ny, nx, pixel_size,
                                                                 voltage_kv >= 300.f ? 1.0f : 0.8f, table, n_table, x_max,
                                                                 plane_outputs, n_out, (float2*)out));
  TMC_CHECK_LAUNCH("tmc_dose_lowrank_combine");
  return TMC_OK;
}

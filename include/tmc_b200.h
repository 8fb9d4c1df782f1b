/* tmc_b200.h -- C ABI of libtmc_b200.so: B200 (sm_100a) kernels for the hot path of
 * teamtomo/torch-motion-correction (patch-based Fourier cross-correlation motion estimation and
 * cubic-spline deformation-field warping of cryo-EM movie stacks).
 *
 * The reference is a pure-Python/PyTorch package with no FFI of its own; its "operator interface" for
 * this path are the Python callables re-exported at src/torch_motion_correction/__init__.py:12-44.
 * Each entry point below replaces the arithmetic of one stage of those callables (cited as
 * reference `file:line`, relative to /root/reference/src/torch_motion_correction/); the Python shims in
 * torch_motion_correction_b200/ bind them with ctypes (see INTEGRATION.md for the binding a
 * maintainer of the reference would add).
 *
 * Conventions
 *   - plain pointers and sizes only; all pointers are DEVICE pointers unless stated otherwise;
 *   - no allocation inside: callers pass workspaces sized by the tmc_*_workspace_* queries;
 *   - every compute call is asynchronous on `stream` (a cudaStream_t) of the CURRENT device;
 *   - int-returning calls return 0 on success, 1 bad argument, 2 CUDA error, 3 unsupported;
 *     tmc_last_error() holds a thread-local message for the last non-zero status;
 *   - thread-safe for concurrent use from different host threads on different streams/devices;
 *   - images are float32, spectra complex64 (interleaved re,im), indices int32;
 *   - counts of any size: tmc_rfft2_band (njobs), tmc_xc_pair_products and tmc_xc_peaks (nitems) and
 *     tmc_irfft2_full (nitems) split longer calls into launches of at most 65535 planes / items themselves;
 *     counts limited to 65535 per call (status 1 beyond, split the call): frames t of tmc_convert_stack,
 *     tmc_remove_hot_pixels, tmc_subtract_frame_means, tmc_warp_dense_shifts, tmc_pixel_tyx, tmc_fourier_shift,
 *     tmc_fourier_shift_frames and tmc_fourier_crop; frame groups of tmc_group_frames; patches g of
 *     tmc_xc_leave_one_out_products, tmc_local_spectra_norms, tmc_local_loss_grad, tmc_local_steps and
 *     tmc_local_tile_spectra (which limits t too); 2 njobs of tmc_dose_filter_spectra; rows (h, ny, ky_count) of tmc_pixel_shifts,
 *     tmc_warp_dense_shifts, tmc_pixel_tyx, tmc_warp_lattice_backward, tmc_fourier_shift, tmc_dose_weighted_sum,
 *     tmc_dose_lowrank_combine, tmc_soft_disc_mask and tmc_band_weights;
 *   - deformation fields are (2 [y,x], nt, nh, nw) float32 in Angstrom, spline `kind` 0 = Catmull-Rom,
 *     1 = cubic B-spline on [0,1]^3 (t, y, x).
 */
#ifndef TMC_B200_H
#define TMC_B200_H

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CUstream_st* tmc_stream_t; /* == cudaStream_t */

/* ---- library ------------------------------------------------------------------------------- */
int tmc_version(void);            /* 100 = 0.1.0 */
const char* tmc_last_error(void); /* thread-local message of the last failing call (host pointer) */
int tmc_sm_count(void);           /* SM count of the current device, -1 on error */
long tmc_launch_count(void);      /* kernels launched by this library since load (bench bookkeeping) */
/* per-kernel device timing for the roofline report: while enabled, the hot kernels' launches are bracketed by CUDA events on
 * their stream (enable != 0 drops earlier records); the report is "kernel,launches,total_ms\n" lines (NUL-terminated,
 * truncated to size; waits for the recorded events) and returns the bytes the full report needs */
int tmc_kernel_timing(int enable);
long tmc_kernel_timing_report(char* buf, long size);
/* copy nbytes (multiple of 4) from PAGE-LOCKED host memory to device memory with a kernel reading the host mapping:
 * unlike cudaMemcpyAsync it does not queue behind a large host-to-device copy of a pipelined run */
int tmc_upload_pinned(const void* host_pinned, void* dst, long nbytes, tmc_stream_t stream);

/* ---- normalize_image statistics: utils.py:49-84 ------------------------------------------------ */
/* mean and unbiased std of image[:, y0:y1, x0:x1] over ALL frames -> mean_std[2] (device).
 * The affine (x - mean) / std itself is fused into the consumers (mean_std arguments below). */
int tmc_stack_stats_workspace_doubles(void);
int tmc_stack_stats(const float* image, int t, int h, int w, int y0, int y1, int x0, int x1, float* mean_std,
                    double* workspace, tmc_stream_t stream);

/* frame-split movies: raw moments {sum, sum of squares, count} (device double[3]) of the local frames;
 * ranks all-reduce (SUM) them and convert once. */
int tmc_stack_moments(const float* image, int t, int h, int w, int y0, int y1, int x0, int x1, double* moments,
                      double* workspace, tmc_stream_t stream);
int tmc_moments_to_mean_std(const double* moments, float* mean_std, tmc_stream_t stream);

/* ---- movie preparation: examples/ttMotion.py:90-202,357 (gain_correct, remove_hot_pixels, set_frames_mean_zero, the
 *      cast to float32) for movies that arrive in their detector-native type ------------------------------------------- */
/* src (t, n) of dtype 0 uint8 / 1 uint16 / 2 int16 / 3 float16 / 4 float32 / 5 int8 -> dst (t, n) fp32, times gain (n, nullable);
 * moments (t, 2) double (nullable) = per-frame {sum, sum of squares} of the result */
int tmc_convert_stack(const void* src, int dtype, int t, long n, const float* gain, float* dst, double* moments,
                      tmc_stream_t stream);
/* pixels further than `threshold` population standard deviations from their frame's mean are replaced by one of their (up to
 * 8) neighbours, picked by a hash of the position (the reference draws it with np.random.choice); moments are updated;
 * hot_count (device int, nullable) receives the number found, at most `capacity` are replaced.
 * workspace: tmc_hot_pixel_workspace_bytes(capacity) bytes */
long tmc_hot_pixel_workspace_bytes(int capacity);
int tmc_remove_hot_pixels(float* stack, int t, int h, int w, double* moments, float threshold, int capacity, void* workspace,
                          int* hot_count, tmc_stream_t stream);
/* every frame minus its own mean (moments[f][0] / n), in place */
int tmc_subtract_frame_means(float* stack, int t, long n, const double* moments, tmc_stream_t stream);
/* frame grouping (MotionCor2 -Group, RELION "group frames"): movie (t, h, w) -> groups (t / frame_group, h, w), the sums
 * of frame_group consecutive frames; the last group also takes the t % frame_group leftover frames.  At least 2 groups.
 * Each sum is movie[first] + movie[first + 1] + ... added left to right in fp32 (one rounding per add, no reordering). */
int tmc_group_frames(const float* movie, int t, int h, int w, int frame_group, float* groups, tmc_stream_t stream);
/* EER electron-event frames (Falcon 4 / 4i) -> counts (n_frames / frames_per_fraction, h, w) of uint8 (count_bytes 1,
 * frames_per_fraction <= 255) or uint16 (2, <= 65535): fraction k holds the electrons of frames [k F, (k + 1) F).
 * payload (device, 4-byte aligned, payload_bytes long): the frames' bit streams; frame f is bytes
 * [frame_offsets[f], frame_offsets[f + 1] - 8) followed by 8 zero bytes; frame_offsets (device int64, n_frames + 1).
 * Codes are rle_bits (1..16) run lengths, escape 2^rle_bits - 1, each electron followed by sub_bits sub-pixel bits that
 * are skipped (rle_bits + sub_bits <= 32).  counts (device, 4-byte aligned) must have room for the byte count rounded up
 * to a multiple of 4; every element is written.  status (device int32, n_frames): 0 decoded, 1 malformed stream (runs out
 * or moves past h * w before landing on it; contributes nothing), 2 offsets outside the payload.  No workspace. */
int tmc_eer_render(const void* payload, long payload_bytes, const long long* frame_offsets, int n_frames, int h, int w,
                   int rle_bits, int sub_bits, int frames_per_fraction, int count_bytes, void* counts, int* status,
                   tmc_stream_t stream);

/* ---- cubic spline grids: torch_cubic_spline_grids.Cubic{CatmullRom,BSpline}Grid3d as used at
 *      deformation_field_utils.py:9-93, estimate_motion_optimizer.py:487-490, correct_motion.py:288-305 */
long tmc_spline_workspace_floats(int c, int n0, int n1, int n2);
/* out (n, c) = grid(tyx (n, 3)) */
int tmc_spline_eval(const float* coeffs, int c, int n0, int n1, int n2, int kind, const float* tyx, long n, float* out,
                    float* workspace, tmc_stream_t stream);
/* grad_coeffs (c, n0, n1, n2) = scale * B^T grad_out (n, c): the autograd transpose of tmc_spline_eval */
int tmc_spline_eval_backward(int c, int n0, int n1, int n2, int kind, const float* tyx, long n, const float* grad_out,
                             float scale, float* grad_coeffs, float* workspace, tmc_stream_t stream);
/* evaluate_deformation_field_at_t for n_frames frames at once: lattice (n_frames, c, lh, lw) at
 * t = linspace(0,1,total_frames)[frame_offset + f], y = linspace(0,1,lh), x = linspace(0,1,lw);
 * coeffs2 (nullable, (c, m0, m1, m2), kind2) is added (correct_motion_two_grids).
 * workspace: tmc_spline_workspace_floats(coeffs) + tmc_spline_workspace_floats(coeffs2) floats. */
int tmc_spline_lattice(const float* coeffs, int c, int n0, int n1, int n2, int kind, const float* coeffs2, int m0, int m1,
                       int m2, int kind2, int n_frames, int frame_offset, int total_frames, int lh, int lw, float* lattice,
                       float* workspace, tmc_stream_t stream);
/* tmc_spline_lattice at t = times[f] (device, n_frames floats): a field estimated on frame-group sums evaluated at the
 * raw frames.  Times outside [0, 1] extend the end interval's cubic (the interval index is clamped, t is not). */
int tmc_spline_lattice_times(const float* coeffs, int c, int n0, int n1, int n2, int kind, const float* coeffs2, int m0,
                             int m1, int m2, int kind2, int n_frames, const float* times, int lh, int lw, float* lattice,
                             float* workspace, tmc_stream_t stream);

/* ---- warp: correct_motion.py:81-185 (_correct_frame, get_pixel_shifts) + sample_image_2d -------- */
long tmc_warp_workspace_floats(int t, int w, int lh); /* t * 2 * (lh + 3) * w: x-interpolated lattice, reflection-padded rows */
/* per pixel: bicubic(reflection) lookup of the frame's (2, lh, lw) Angstrom lattice -> / pixel_spacing ->
 * bicubic (border-clamped taps, zero outside) gather of the frame.  out_stack (t,h,w) and/or out_sum (h,w)
 * (fused sum over frames, never materialising the stack); accumulate_sum != 0 adds into out_sum (frame
 * blocks of one movie).  mean_std nullable: output is (v - mean) / std of the warped value. */
int tmc_warp_lattice(const float* image, int t, int h, int w, const float* lattice, int lh, int lw, float pixel_spacing,
                     const float* mean_std, float* out_stack, float* out_sum, int accumulate_sum, float* workspace,
                     tmc_stream_t stream);
/* frame-weighted sums in one pass over the movie: out_sums (n_sums, h, w) = sum_f frame_weights[s][f] * (frame f warped as
 * by tmc_warp_lattice), frame_weights (n_sums, t) f32.  At most 19 sums per call (3 plain sums + 2 x 8 low-rank dose
 * components; split larger requests into passes); an all-ones row gives the out_sum of tmc_warp_lattice bit for bit.
 * workspace: tmc_warp_workspace_floats(t, w, lh) floats. */
int tmc_warp_lattice_sums(const float* image, int t, int h, int w, const float* lattice, int lh, int lw, float pixel_spacing,
                          const float* frame_weights, int n_sums, float* out_sums, float* workspace, tmc_stream_t stream);
/* backward of tmc_warp_lattice w.r.t. the lattice (correct_motion_two_grids, grad=True; correct_motion.py:256-317):
 * grad_out (t,h,w) -> grad_lattice (t,2,lh,lw).  workspace: 2 * tmc_warp_workspace_floats(t, w, lh) floats. */
int tmc_warp_lattice_backward(const float* image, int t, int h, int w, const float* lattice, int lh, int lw,
                              float pixel_spacing, const float* grad_out, float* grad_lattice, float* workspace,
                              tmc_stream_t stream);
/* (t, y, x) in [0,1]^3 of every lattice node, (t, lh, lw, 3): the points tmc_spline_lattice evaluates */
int tmc_lattice_tyx(int t, int frame_offset, int total_frames, int lh, int lw, float* tyx, tmc_stream_t stream);
/* get_pixel_shifts: (2, lh, lw) lattice -> (h, w, 2) px shifts */
int tmc_pixel_shifts(const float* lattice, int lh, int lw, int h, int w, float pixel_spacing, float* out,
                     tmc_stream_t stream);
/* correct_motion_slow (correct_motion.py:371-427): out = bicubic(frame; pixel + shifts (t,h,w,2) px) */
int tmc_warp_dense_shifts(const float* image, int t, int h, int w, const float* shifts, float* out_stack,
                          tmc_stream_t stream);
/* normalised (t, y, x) of every pixel: tyx (t, h, w, 3)  (correct_motion.py:401-409) */
int tmc_pixel_tyx(int h, int w, int t, int frame_offset, int total_frames, float* tyx, tmc_stream_t stream);

/* ---- tables: torch_grid_utils.circle, torch_fourier_filter.{bandpass_filter,b_envelope} as used at
 *      estimate_motion_xc.py:69-95,262-280, estimate_motion_optimizer.py:162-184, utils.py:87-114 ---- */
/* soft-edged disc centred at (h/2, w/2): 1 inside radius, cos roll-off over the exact Euclidean distance
 * transform up to smoothing_radius.  workspace: h ints. */
int tmc_soft_disc_mask(int h, int w, float radius, float smoothing_radius, float* mask, int* workspace,
                       tmc_stream_t stream);
/* weight[kyb][kx] = (low < f <= high) * exp(-b_factor (f / pixel_size)^2 / 4) on the band box
 * ky = ky_start + kyb (kyb < ky_count), kx < kx_count; f in cycles/px on the (ny, nx) rfft grid */
int tmc_band_weights(int ny, int nx, int ky_count, int kx_count, int ky_start, float low, float high, int use_band,
                     float b_factor, float pixel_size, int use_envelope, float* weight, tmc_stream_t stream);

/* dose-weighted frame sum in Fourier space: examples/ttMotion.py:331-351 + torch_fourier_filter.dose_weight_movie
 * (Grant & Grigorieff critical exposure).  spec (t, ny, nx/2+1) complex64 -> out (ny, nx/2+1) complex64 =
 * sum_t spec_t q_t / sqrt(sum_t q_t^2); den2 (ny, nx/2+1) f32 nullable accumulates sum q^2 over frame blocks (then out
 * accumulates too and only the call with finalize != 0 normalises); frames are frame_offset .. frame_offset + t - 1 */
int tmc_dose_weighted_sum(const void* spec, int t, int ny, int nx, float pixel_size, float pre_exposure,
                          float dose_per_frame, float voltage_kv, int frame_offset, void* out, float* den2, int finalize,
                          tmc_stream_t stream);

/* low-rank dose weighting (correct_motion_sums): the normalised weights w_t(k) = q_t(k) / sqrt(sum_t q_t(k)^2) depend on k
 * only through x = 1 / N_e(k) and are approximated as sum_r U_r(t) v_r(x) with a worst L2 residual over t of 1e-6 (R <= 8
 * for real exposures).  spec (n_spec, ny, nx/2+1) complex64: spectra of the weighted sums sum_t U_r(t) c_t; table
 * (n_spec, n_table) f32: v_r of each plane on n_table uniform nodes of x in [0, x_max], linearly interpolated;
 * plane_outputs (n_spec) int32: bit o set = the plane adds to output o.  out (n_out <= 3, ny, nx/2+1) complex64. */
int tmc_dose_lowrank_combine(const void* spec, int n_spec, int ny, int nx, float pixel_size, float voltage_kv,
                             const float* table, int n_table, float x_max, const int* plane_outputs, int n_out, void* out,
                             tmc_stream_t stream);

/* the same exposure filter q_frame / sqrt(sum_t q_t^2) applied per frame to the band-limited spectra of tmc_rfft2_band
 * (planes 2 job + {0, 1} belong to jobs[job].frame_a / frame_b): additive pre-filter of the patch cross-correlation
 * (the reference filters with band-pass and B-factor only, estimate_motion_xc.py:338-346).
 * tables: 2 * ky_count * kx_count floats of scratch; 2 * njobs <= 65535 per call */
int tmc_dose_filter_spectra(void* spec, const int* jobs, int njobs, int ny, int nx, int ky_count, int kx_count, int ky_start,
                            int total_frames, float pixel_size, float pre_exposure, float dose_per_frame, float voltage_kv,
                            float* tables, tmc_stream_t stream);

/* ---- FFT plans ------------------------------------------------------------------------------------ */
/* 1: full and band-limited transforms: powers of two in [16, 8192], any other n in [2, 4096] (Bluestein), and 2..8
 *    times such a length (the axis is decimated, n = R n', and the R sub-transforms are combined) while the accumulators
 *    of a full spectrum fit in shared memory (n <= 12158, 12288, 16384: K3 5760 x 4092, super-resolution 11520 x 8184);
 * 2: longer decimated axes (<= 32768): band-limited transforms only (tmc_rfft2_band with a narrow band, tmc_xc_peaks);
 * 0: unsupported */
int tmc_fft_supported_length(int n);
long tmc_fft_plan_elems(int n);      /* complex64 elements of a plan buffer, 0 if unsupported */
int tmc_fft_plan_init(int n, void* plan, tmc_stream_t stream);
/* out[r] = DFT_n(in[r]) for `rows` complex64 rows (utility / tests) */
int tmc_fft_c2c_rows(const void* in, int rows, int n, const void* plan, void* out, tmc_stream_t stream);

/* ---- band-limited forward transform: torch.fft.rfftn(patch * mask) * bandpass * b_envelope at
 *      estimate_motion_xc.py:77-98,338-346, estimate_motion_optimizer.py:371-372, correct_motion.py:484 */
/* jobs (njobs, 6) int32 = {frame_a, mask_power_a, frame_b (-1: none), mask_power_b, y0, x0}: the (ny, nx)
 * window at (y0, x0) of frame_a / frame_b, normalised with mean_std (nullable), times mask^power, packed as
 * real / imaginary part of ONE complex transform.  Only rows [ylo, yhi) of the mask are non-zero.
 * out (2 * njobs, ky_count, kx_count) complex64: plane 2*job = a, 2*job + 1 = b; ky = ky_start + kyb.
 * job_mode: 0 generic; 1 all jobs are {f, 1, f, 2, ..} (one frame, mask powers 1 and 2); 2 all jobs use power 1.
 * tmp: 2 * njobs * ny * kx_count complex64. */
int tmc_rfft2_band(const float* image, int t, int h, int w, const float* mean_std, const float* mask, int ny, int nx,
                   const int* jobs, int njobs, int job_mode, const int* frame_shifts, int x_margin, int ylo, int yhi,
                   int kx_count, int ky_count, int ky_start, const float* weight, const void* plan_x, const void* plan_y,
                   void* tmp, void* out, tmc_stream_t stream);
/* frame_shifts (nullable, (t, 2) int32 device): whole-pixel (dy, dx) added to the window origin of every frame, the
 * window wrapping around the frame edges -- the patches of the frames rolled by an integer Fourier shift, which is what
 * the rigid pre-correction of estimate_motion_xc.py:232-241 (correct_motion_fast, correct_motion.py:430-498) produces for
 * whole-pixel fields such as estimate_global_motion's (quirk Q5), without a pass over the stack.  x_margin: the first
 * and last x_margin columns of `mask` are all zero (0 if unknown).
 * tmc_integer_shifts: shifts[f] = rint(scale * field[c][f]) for a (2, t) field; *not_integer (device int) = 1 when a
 * scaled value is further than 1e-4 from a whole number. */
int tmc_integer_shifts(const float* field, int t, float scale, int* shifts, int* not_integer, tmc_stream_t stream);

/* ---- cross-correlation products: estimate_motion_xc.py:112,310-349 ---------------------------------- */
/* out[i] = conj(spec[ref_plane[i]]) * spec[cur_plane[i]] */
int tmc_xc_pair_products(const void* spec, const int* ref_plane, const int* cur_plane, int nitems, long plane_elems,
                         void* out, tmc_stream_t stream);
/* leave-one-out mean reference incl. the reference's cache aliasing (SURVEY.md quirk Q1).  spec planes
 * [t][g][2] (mask^1, mask^2) for ALL t frames; out items [k_count][g] for frames k_begin.. (a rank of a
 * frame-split movie computes only its own frames); delta_offsets (t+1) / deltas: for frame k the signed
 * (j+1) entries that toggle "frame j is double-masked" relative to frame k-1. */
int tmc_xc_leave_one_out_products(const void* spec, int t, int g, long plane_elems, const int* delta_offsets,
                                  const int* deltas, int k_begin, int k_count, void* out, tmc_stream_t stream);

/* ---- inverse transform + peak: irfftn, argmax, parabola, wrap at estimate_motion_xc.py:113-121,350-369,414-483 */
int tmc_xc_peak_partials(int ny, int nx);
/* prod (nitems, ky_count, kx_count) -> shifts (nitems, 2) = (dy, dx) px.  tmp: nitems*ny*kx_count complex64;
 * partial: nitems * tmc_xc_peak_partials(ny, nx) * 8 bytes. */
int tmc_xc_peaks(const void* prod, int nitems, int ny, int nx, int kx_count, int ky_count, int ky_start, int sub_pixel,
                 const void* plan_x, const void* plan_y, void* tmp, void* partial, float* shifts, tmc_stream_t stream);

/* ---- whole-frame Fourier shift: correct_motion.py:484-496 + torch_fourier_shift.fourier_shift_dft_2d */
/* spec (t, ny, nx/2+1) *= exp(-2 pi i (f_y s_y + f_x s_x)), (s_y, s_x)[f] = sign * field[(0|1) * t + f] */
int tmc_fourier_shift(void* spec, int t, int ny, int nx, const float* field, float sign, tmc_stream_t stream);
/* torch.fft.irfftn(spec, s=(ny, nx)): spec (nitems, ny, nx/2+1) -> out (nitems, ny, nx); tmp like spec */
int tmc_irfft2_full(const void* spec, int nitems, int ny, int nx, const void* plan_x, const void* plan_y, void* tmp,
                    float* out, tmc_stream_t stream);

/* ---- Fourier crop ("binning", MotionCor2 -FtBin) of whole frames ---------------------------------------------------- */
/* image (t, h, w) -> out (t, out_h, out_w): rfft2, keep ky in [-out_h/2, out_h/2) and kx in [0, out_w/2], irfft2 at
 * (out_h, out_w), times out_h out_w / (h w) so the mean pixel value is kept (the self-paired columns kx = 0 and
 * kx = out_w/2 enter through their Hermitian part, as in numpy's irfft2).  All four sides even, out sides <= in sides,
 * all four full-spectrum lengths (tmc_fft_supported_length == 1).  jobs: frame-pair jobs as for tmc_rfft2_band
 * (job_mode 2) covering the t frames in order; plan_x / plan_y / plan_x_out / plan_y_out: plans of w, h, out_w, out_h;
 * workspace: tmc_fourier_crop_workspace_bytes(t, h, w, out_h, out_w) bytes (-1: bad arguments).  Power-of-two heights
 * cropped by 2 or 4 to >= 256 rows run the column passes as one kernel that keeps the cropped spectrum on chip
 * (environment TMC_FFT_CROP_FUSED=0, read per call: two passes through HBM instead; the result is the same). */
long tmc_fourier_crop_workspace_bytes(int t, int h, int w, int out_h, int out_w);
int tmc_fourier_crop(const float* image, int t, int h, int w, int out_h, int out_w, const int* jobs, int njobs,
                     const void* plan_x, const void* plan_y, const void* plan_x_out, const void* plan_y_out, void* workspace,
                     float* out, tmc_stream_t stream);

/* fused correct_motion_fast (power-of-two frame sides >= 256): rows r2c -> columns (FFT, phase, inverse FFT in one
 * kernel) -> rows c2r.  jobs: frame-pair jobs as for tmc_rfft2_band (job_mode 2) covering the t frames in order;
 * tmp: 2*njobs*ny*(nx/2+1) complex64; phase: t*ny complex64; out (t, ny, nx). */
int tmc_fourier_shift_frames_supported(int ny, int nx);
int tmc_fourier_shift_frames(const float* image, int t, int ny, int nx, const float* mean_std, const int* jobs, int njobs,
                             const float* field, float sign, const void* plan_x, const void* plan_y, void* tmp, void* phase,
                             float* out, tmc_stream_t stream);

/* ---- tail of the estimators: estimate_motion_xc.py:131-133,376-410,486-627 -------------------------- */
/* shifts (t, g, 2) px; field (2, t, g) Angstrom = base field in, result out: per-frame outlier rejection,
 * px -> Angstrom accumulate, Savitzky-Golay (polyorder 1, scipy mode="interp"), one joint mean removed.
 * skip_frame: frame left untouched (middle_frame reference), -1 none.  scratch: 2*t*g floats. */
int tmc_xc_postprocess(const float* shifts, int t, int g, float pixel_spacing, int skip_frame, int outlier_rejection,
                       float outlier_threshold, int temporal_smoothing, int smoothing_window, int subtract_mean,
                       float* field, float* scratch, tmc_stream_t stream);
/* (t, 2) px -> (2, t, 1, 1) Angstrom, zero_frame forced to 0 (deformation_field_utils.py:129-162) */
int tmc_global_shifts_to_field(const float* shifts, int t, float pixel_spacing, int zero_frame, float* field,
                               tmc_stream_t stream);
/* data -= mean(data): one joint scalar (estimate_motion_optimizer.py:148,432-434) */
int tmc_subtract_mean(float* data, long n, tmc_stream_t stream);

/* ---- spline-coefficient optimiser: estimate_motion_optimizer.py:371-407,442-510,611-671 -------------- */
/* spec (g, tp, ky_count, kx_count): band-limited filtered spectra of every patch and frame (tp >= t planes
 * per patch); with frame_major != 0 the planes are ordered (tp / 2, g, 2, ...) instead, i.e. as tmc_rfft2_band writes
 * them for frame-pair jobs listed frame pair by frame pair (every frame is then read from HBM once: the overlapping
 * patches of a frame pair run back to back and hit L2).  norms (g, t, 2) float64 = sum_f w |spec|^2 for w = 1 and
 * Hermitian weights. */
int tmc_local_spectra_norms(const void* spec, int g, int t, int tp, int ny, int nx, int ky_count, int kx_count,
                            int ky_start, int frame_major, double* norms, tmc_stream_t stream);
long tmc_local_loss_workspace_bytes(int g, int t, int ky_count, int kx_count);
/* one loss + gradient evaluation: eval_new / eval_base (t, g, 2) spline values (Angstrom) at the patch
 * centres; patch_scale (g): weight of each patch's mean-reduced mini-batch loss; loss_type 0 mse, 1 cc,
 * 2 ncc.  Outputs: loss (device double, sum over mini-batches) and grad_eval (t, g, 2) = dloss/d eval_new. */
int tmc_local_loss_grad(const void* spec, const double* norms, const float* eval_new, const float* eval_base,
                        const float* patch_scale, const int* iteration, int g, int t, int tp, int ny, int nx, int ky_count,
                        int kx_count, int ky_start, float pixel_spacing, int loss_type, double* loss, float* grad_eval,
                        void* workspace, tmc_stream_t stream);
/* *counter += 1 on the stream: device-side iteration index so a captured optimiser step can be replayed
 * (patch_scale may then be (n_iterations, g) with `iteration` = counter; mse / cc only) */
int tmc_advance_counter(int* counter, tmc_stream_t stream);
/* one torch.optim.Adam step (amsgrad off; estimate_motion_optimizer.py:535-548 defaults) on n parameters, fused in
 * one kernel; the step number is *step_counter + 1 (device int, so the call can live in a CUDA graph) */
int tmc_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int n, double lr, double beta1,
                  double beta2, double eps, double weight_decay, const int* step_counter, tmc_stream_t stream);

/* ---- one optimiser iteration as two launches ("mse" / "cc"): estimate_motion_optimizer.py:361-416 (loop over the
 *      shuffled mini-batches, loss.backward(), optimizer.step()) with the spline evaluation of :487-490, the Fourier
 *      shift + filters of :495-508, the leave-one-out reference of :391-399 and _compute_loss :611-671 inside ---- */
/* 1 if tmc_local_steps supports the problem (t frames fit the shared-memory tile of t KB, ...), else 0 (use
 * tmc_local_loss_grad) */
int tmc_local_steps_supported(int g, int t, int nt, int nhw);
/* re-lay spec (g, tp, ky_count, kx_count) complex64 into tiles of 8 (ky) x 16 (kx) bins with the t frames of a tile
 * contiguous, real and imaginary parts in separate planes: out (g, n_tiles, t, 2, 128) float32, zero padded
 * (frame_major: plane order of spec as for tmc_local_spectra_norms);
 * tiles (n_tiles, 2) int32 = (ty, tx) lists the tiles that hold at least one pass-band bin */
int tmc_local_tile_spectra(const void* spec, int g, int t, int tp, int ky_count, int kx_count, const int* tiles,
                           int n_tiles, int frame_major, void* out, tmc_stream_t stream);
long tmc_local_steps_workspace_bytes(int g, int t, int nt);
/* n_steps iterations (1 + 2 n_steps launches).  sum_norms (g) double = sum_t A_t; eval_base (t, g, 2) Angstrom; w_t (t, nt)
 * and w_sp (g, nhw): dense separable spline weights of the patch centres (time / space); patch_scale (rows, g), step i
 * uses row first_row + i; coef (2, nt, nhw).  mode 0: Adam update in place (step number first_row + i + 1),
 * loss_out[first_row + i]; mode 1 (n_steps == 1): gradient only -> grad_out (2, nt, nhw), loss_out[0];
 * modes 2 / 3 (n_steps == 1; one movie split over several GPUs, the caller all-reduces grad_out between calls and keeps the
 * workspace of the preceding mode 1 / 2 call untouched): mode 2 = Adam step number first_row on the gradient found in
 * grad_out, then gradient and loss_out[0] of the updated coefficients under patch_scale row first_row; mode 3 = that Adam
 * step only. */
int tmc_local_steps(const void* tiled, const int* tiles, int n_tiles, int g, int t, int ny, int nx, int ky_count,
                    int kx_count, int ky_start, const double* sum_norms, const float* eval_base, const float* w_t,
                    const float* w_sp, int nt, int nhw, const float* patch_scale, float pixel_spacing, int loss_type,
                    float* coef, float* exp_avg, float* exp_avg_sq, double lr, double beta1, double beta2, double eps,
                    double weight_decay, int first_row, int mode, int n_steps, double* loss_out, float* grad_out,
                    void* workspace, tmc_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* TMC_B200_H */

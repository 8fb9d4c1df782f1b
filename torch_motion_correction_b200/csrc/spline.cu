// Uniform cubic spline grids (B-spline / Catmull-Rom) on [0,1]^3: evaluation, its transpose
// (gradient w.r.t. the coefficients) and the per-frame 10x lattice used by the warp.
//
// Replaces torch_cubic_spline_grids.Cubic{BSpline,CatmullRom}Grid3d as called from the
// reference at deformation_field_utils.py:30-38,84-92, estimate_motion_optimizer.py:487-490
// and correct_motion.py:299-302 (semantics: SURVEY.md Appendix A.1).
#include "common.cuh"

namespace {

// weights = [1, u, u^2, u^3] @ M ; M row-major [power][tap]
struct SplineMatrix {
  float m[4][4];
};

__device__ __forceinline__ SplineMatrix spline_matrix(int kind) {
  SplineMatrix s;
  if (kind == 0) {  // Catmull-Rom: 0.5 * [[0,2,0,0],[-1,0,1,0],[2,-5,4,-1],[-1,3,-3,1]]
    const float h = 0.5f;
    const float r[4][4] = {{0.f, 2.f, 0.f, 0.f}, {-1.f, 0.f, 1.f, 0.f}, {2.f, -5.f, 4.f, -1.f}, {-1.f, 3.f, -3.f, 1.f}};
#pragma unroll
    for (int p = 0; p < 4; ++p)
#pragma unroll
      for (int j = 0; j < 4; ++j) s.m[p][j] = h * r[p][j];
  } else {  // B-spline: (1/6) * [[1,4,1,0],[-3,0,3,0],[3,-6,3,0],[-1,3,-3,1]]
    const float h = (float)(1.0 / 6.0);
    const float r[4][4] = {{1.f, 4.f, 1.f, 0.f}, {-3.f, 0.f, 3.f, 0.f}, {3.f, -6.f, 3.f, 0.f}, {-1.f, 3.f, -3.f, 1.f}};
#pragma unroll
    for (int p = 0; p < 4; ++p)
#pragma unroll
      for (int j = 0; j < 4; ++j) s.m[p][j] = __fmul_rn(h, r[p][j]);
  }
  return s;
}

// e = expanded node count (>= 2); returns first padded tap index and the 4 weights
__device__ __forceinline__ int axis_taps(float u, int e, const SplineMatrix& M, float (&w)[4]) {
  float x = __fmul_rn(u, (float)(e - 1));
  float fi = fminf(fmaxf(floorf(x), 0.0f), (float)(e - 2));
  float tau = __fsub_rn(x, fi);
  float t2 = __fmul_rn(tau, tau);
  float t3 = __fmul_rn(t2, tau);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    float acc = M.m[0][j];
    acc = __fadd_rn(acc, __fmul_rn(tau, M.m[1][j]));
    acc = __fadd_rn(acc, __fmul_rn(t2, M.m[2][j]));
    acc = __fadd_rn(acc, __fmul_rn(t3, M.m[3][j]));
    w[j] = acc;
  }
  return (int)fi;  // padded index of tap 0 (original node fi-1)
}

struct PaddedGrid {
  const float* data;  // (c, p0, p1, p2)
  int c, p0, p1, p2;  // padded dims = expanded + 2
};

__device__ __forceinline__ void spline_eval_point(const PaddedGrid& g, const SplineMatrix& M, float u0, float u1, float u2,
                                                  float* out, int out_stride, bool accumulate) {
  float w0[4], w1[4], w2[4];
  int i0 = axis_taps(u0, g.p0 - 2, M, w0);
  int i1 = axis_taps(u1, g.p1 - 2, M, w1);
  int i2 = axis_taps(u2, g.p2 - 2, M, w2);
  const long s0 = (long)g.p1 * g.p2, s1 = g.p2;
  for (int ch = 0; ch < g.c; ++ch) {
    const float* base = g.data + (long)ch * g.p0 * s0 + (long)i0 * s0 + (long)i1 * s1 + i2;
    float acc = 0.f;
#pragma unroll
    for (int a = 0; a < 4; ++a) {
      float acc1 = 0.f;
#pragma unroll
      for (int b = 0; b < 4; ++b) {
        const float* p = base + a * s0 + b * s1;
        float acc2 = w2[0] * __ldg(p) + w2[1] * __ldg(p + 1) + w2[2] * __ldg(p + 2) + w2[3] * __ldg(p + 3);
        acc1 += w1[b] * acc2;
      }
      acc += w0[a] * acc1;
    }
    if (accumulate)
      out[ch * out_stride] += acc;
    else
      out[ch * out_stride] = acc;
  }
}

// ---- padding (linear-extrapolated phantom nodes; singleton axes repeated) ---------------

__global__ void spline_pad_kernel(const float* __restrict__ coeffs, int c, int n0, int n1, int n2, float* __restrict__ P) {
  const int e0 = max(n0, 2), e1 = max(n1, 2), e2 = max(n2, 2);
  const int p0 = e0 + 2, p1 = e1 + 2, p2 = e2 + 2;
  const long s0 = (long)p1 * p2, s1 = p2, sc = (long)p0 * s0;
  const int tid = threadIdx.x, nth = blockDim.x;
  // interior
  for (long i = tid; i < (long)c * e0 * e1 * e2; i += nth) {
    int d = i % e2;
    long r = i / e2;
    int b = r % e1;
    r /= e1;
    int a = r % e0;
    int ch = r / e0;
    int sa = (n0 == 1) ? 0 : a, sb = (n1 == 1) ? 0 : b, sd = (n2 == 1) ? 0 : d;
    P[ch * sc + (a + 1) * s0 + (b + 1) * s1 + (d + 1)] = coeffs[((long)(ch * n0 + sa) * n1 + sb) * n2 + sd];
  }
  __syncthreads();
  // axis 0 (only interior of axes 1,2 is defined yet)
  for (long i = tid; i < (long)c * e1 * e2; i += nth) {
    int d = i % e2;
    long r = i / e2;
    int b = r % e1;
    int ch = r / e1;
    float* q = P + ch * sc + (b + 1) * s1 + (d + 1);
    q[0] = 2.f * q[s0] - q[2 * s0];
    q[(p0 - 1) * s0] = 2.f * q[(p0 - 2) * s0] - q[(p0 - 3) * s0];
  }
  __syncthreads();
  // axis 1 over the full padded axis 0
  for (long i = tid; i < (long)c * p0 * e2; i += nth) {
    int d = i % e2;
    long r = i / e2;
    int a = r % p0;
    int ch = r / p0;
    float* q = P + ch * sc + a * s0 + (d + 1);
    q[0] = 2.f * q[s1] - q[2 * s1];
    q[(p1 - 1) * s1] = 2.f * q[(p1 - 2) * s1] - q[(p1 - 3) * s1];
  }
  __syncthreads();
  // axis 2 over full padded axes 0,1
  for (long i = tid; i < (long)c * p0 * p1; i += nth) {
    int b = i % p1;
    long r = i / p1;
    int a = r % p0;
    int ch = r / p0;
    float* q = P + ch * sc + a * s0 + b * s1;
    q[0] = 2.f * q[1] - q[2];
    q[p2 - 1] = 2.f * q[p2 - 2] - q[p2 - 3];
  }
}

// adjoint of spline_pad_kernel: gP (c,p0,p1,p2) -> gcoeffs (c,n0,n1,n2). gP is destroyed.
__global__ void spline_unpad_kernel(float* __restrict__ gP, int c, int n0, int n1, int n2, float* __restrict__ gcoeffs,
                                    float scale) {
  const int e0 = max(n0, 2), e1 = max(n1, 2), e2 = max(n2, 2);
  const int p0 = e0 + 2, p1 = e1 + 2, p2 = e2 + 2;
  const long s0 = (long)p1 * p2, s1 = p2, sc = (long)p0 * s0;
  const int tid = threadIdx.x, nth = blockDim.x;
  for (long i = tid; i < (long)c * p0 * p1; i += nth) {
    int b = i % p1;
    long r = i / p1;
    int a = r % p0;
    int ch = r / p0;
    float* q = gP + ch * sc + a * s0 + b * s1;
    float lo = q[0], hi = q[p2 - 1];
    // NB: with e2 == 2 the two ends touch the same interior nodes: apply sequentially
    q[1] += 2.f * lo;
    q[2] -= lo;
    q[p2 - 2] += 2.f * hi;
    q[p2 - 3] -= hi;
  }
  __syncthreads();
  for (long i = tid; i < (long)c * p0 * e2; i += nth) {
    int d = i % e2;
    long r = i / e2;
    int a = r % p0;
    int ch = r / p0;
    float* q = gP + ch * sc + a * s0 + (d + 1);
    float lo = q[0], hi = q[(p1 - 1) * s1];
    q[s1] += 2.f * lo;
    q[2 * s1] -= lo;
    q[(p1 - 2) * s1] += 2.f * hi;
    q[(p1 - 3) * s1] -= hi;
  }
  __syncthreads();
  for (long i = tid; i < (long)c * e1 * e2; i += nth) {
    int d = i % e2;
    long r = i / e2;
    int b = r % e1;
    int ch = r / e1;
    float* q = gP + ch * sc + (b + 1) * s1 + (d + 1);
    float lo = q[0], hi = q[(p0 - 1) * s0];
    q[s0] += 2.f * lo;
    q[2 * s0] -= lo;
    q[(p0 - 2) * s0] += 2.f * hi;
    q[(p0 - 3) * s0] -= hi;
  }
  __syncthreads();
  for (long i = tid; i < (long)c * n0 * n1 * n2; i += nth) {
    int d = i % n2;
    long r = i / n2;
    int b = r % n1;
    r /= n1;
    int a = r % n0;
    int ch = r / n0;
    float acc = 0.f;
    for (int da = 0; da < (n0 == 1 ? 2 : 1); ++da)
      for (int db = 0; db < (n1 == 1 ? 2 : 1); ++db)
        for (int dd = 0; dd < (n2 == 1 ? 2 : 1); ++dd)
          acc += gP[ch * sc + (a + da + 1) * s0 + (b + db + 1) * s1 + (d + dd + 1)];
    gcoeffs[i] = acc * scale;
  }
}

__global__ void spline_eval_kernel(PaddedGrid g, int kind, const float* __restrict__ tyx, long n, float* __restrict__ out) {
  long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  SplineMatrix M = spline_matrix(kind);
  spline_eval_point(g, M, tyx[3 * i], tyx[3 * i + 1], tyx[3 * i + 2], out + i * g.c, 1, false);
}

__global__ void spline_eval_backward_kernel(int c, int p0, int p1, int p2, int kind, const float* __restrict__ tyx, long n,
                                            const float* __restrict__ gout, float* __restrict__ gP) {
  long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  SplineMatrix M = spline_matrix(kind);
  float w0[4], w1[4], w2[4];
  int i0 = axis_taps(tyx[3 * i], p0 - 2, M, w0);
  int i1 = axis_taps(tyx[3 * i + 1], p1 - 2, M, w1);
  int i2 = axis_taps(tyx[3 * i + 2], p2 - 2, M, w2);
  const long s0 = (long)p1 * p2, s1 = p2;
  for (int ch = 0; ch < c; ++ch) {
    float go = gout[i * c + ch];
    float* base = gP + (long)ch * p0 * s0 + (long)i0 * s0 + (long)i1 * s1 + i2;
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int b = 0; b < 4; ++b)
#pragma unroll
        for (int d = 0; d < 4; ++d) atomicAdd(base + a * s0 + b * s1 + d, go * w0[a] * w1[b] * w2[d]);
  }
}

// where the lattice's normalised frame times come from: t_f = linspace(0,1,total_frames)[frame_offset + f] ...
struct LinspaceTimes {
  int frame_offset, total_frames;
  __device__ __forceinline__ float operator()(int f) const { return linspace01(f + frame_offset, total_frames); }
};
// ... or a per-frame table (frame grouping: times of the raw frames on the group time axis, may leave [0, 1])
struct TableTimes {
  const float* times;
  __device__ __forceinline__ float operator()(int f) const { return __ldg(times + f); }
};

// lattice[f][ch][iy][ix] = G1(t_f, y_iy, x_ix) (+ G2(...))
template <class Times>
__global__ void spline_lattice_kernel(PaddedGrid g1, int kind1, PaddedGrid g2, int kind2, int has2, int T, Times times, int lh,
                                      int lw, float* __restrict__ lattice) {
  long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  long total = (long)T * lh * lw;
  if (i >= total) return;
  int ix = i % lw;
  long r = i / lw;
  int iy = r % lh;
  int f = r / lh;
  float ut = times(f), uy = linspace01(iy, lh), ux = linspace01(ix, lw);
  float* out = lattice + ((long)f * g1.c * lh + iy) * lw + ix;
  SplineMatrix M = spline_matrix(kind1);
  spline_eval_point(g1, M, ut, uy, ux, out, lh * lw, false);
  if (has2) {
    SplineMatrix M2 = spline_matrix(kind2);
    spline_eval_point(g2, M2, ut, uy, ux, out, lh * lw, true);
  }
}

inline void padded_dims(int n0, int n1, int n2, int& p0, int& p1, int& p2) {
  p0 = (n0 > 2 ? n0 : 2) + 2;
  p1 = (n1 > 2 ? n1 : 2) + 2;
  p2 = (n2 > 2 ? n2 : 2) + 2;
}

}  // namespace

TMC_API long tmc_spline_workspace_floats(int c, int n0, int n1, int n2) {
  int p0, p1, p2;
  padded_dims(n0, n1, n2, p0, p1, p2);
  return (long)c * p0 * p1 * p2;
}

static int check_grid(const void* coeffs, int c, int n0, int n1, int n2, int kind) {
  TMC_CHECK_ARG(coeffs != nullptr, "spline: null coefficient pointer");
  TMC_CHECK_ARG(c >= 1 && n0 >= 1 && n1 >= 1 && n2 >= 1, "spline: bad grid shape (%d,%d,%d,%d)", c, n0, n1, n2);
  TMC_CHECK_ARG(kind == 0 || kind == 1, "spline: kind must be 0 (catmull_rom) or 1 (bspline), got %d", kind);
  return TMC_OK;
}

TMC_API int tmc_spline_eval(const float* coeffs, int c, int n0, int n1, int n2, int kind, const float* tyx, long n,
                            float* out, float* workspace, cudaStream_t stream) {
  if (int e = check_grid(coeffs, c, n0, n1, n2, kind)) return e;
  TMC_CHECK_ARG(workspace != nullptr && (n == 0 || (tyx && out)), "spline_eval: null pointer");
  PaddedGrid g;
  g.data = workspace;
  g.c = c;
  padded_dims(n0, n1, n2, g.p0, g.p1, g.p2);
  spline_pad_kernel<<<1, 256, 0, stream>>>(coeffs, c, n0, n1, n2, workspace); tmc_count_launch();
  if (n > 0) spline_eval_kernel<<<tmc_div_up(n, 128), 128, 0, stream>>>(g, kind, tyx, n, out); tmc_count_launch();
  TMC_CHECK_LAUNCH("tmc_spline_eval");
  return TMC_OK;
}

// grad_coeffs = scale * B^T grad_out ; workspace as for tmc_spline_eval
TMC_API int tmc_spline_eval_backward(int c, int n0, int n1, int n2, int kind, const float* tyx, long n,
                                     const float* grad_out, float scale, float* grad_coeffs, float* workspace,
                                     cudaStream_t stream) {
  TMC_CHECK_ARG(c >= 1 && n0 >= 1 && n1 >= 1 && n2 >= 1, "spline_eval_backward: bad grid shape");
  TMC_CHECK_ARG(kind == 0 || kind == 1, "spline_eval_backward: bad kind %d", kind);
  TMC_CHECK_ARG(grad_coeffs && workspace && (n == 0 || (tyx && grad_out)), "spline_eval_backward: null pointer");
  int p0, p1, p2;
  padded_dims(n0, n1, n2, p0, p1, p2);
  TMC_CUDA(cudaMemsetAsync(workspace, 0, sizeof(float) * (size_t)c * p0 * p1 * p2, stream));
  if (n > 0)
    spline_eval_backward_kernel<<<tmc_div_up(n, 128), 128, 0, stream>>>(c, p0, p1, p2, kind, tyx, n, grad_out, workspace); tmc_count_launch();
  spline_unpad_kernel<<<1, 256, 0, stream>>>(workspace, c, n0, n1, n2, grad_coeffs, scale); tmc_count_launch();
  TMC_CHECK_LAUNCH("tmc_spline_eval_backward");
  return TMC_OK;
}

// padding of the grid(s) + spline_lattice_kernel: the common body of tmc_spline_lattice and tmc_spline_lattice_times
template <class Times>
static int spline_lattice_launch(const char* name, const float* coeffs, int c, int n0, int n1, int n2, int kind,
                                 const float* coeffs2, int m0, int m1, int m2, int kind2, int n_frames, Times times, int lh,
                                 int lw, float* lattice, float* workspace, cudaStream_t stream) {
  if (coeffs2)
    if (int e = check_grid(coeffs2, c, m0, m1, m2, kind2)) return e;
  PaddedGrid g1, g2;
  g1.data = workspace;
  g1.c = c;
  padded_dims(n0, n1, n2, g1.p0, g1.p1, g1.p2);
  spline_pad_kernel<<<1, 256, 0, stream>>>(coeffs, c, n0, n1, n2, workspace); tmc_count_launch();
  g2 = g1;
  if (coeffs2) {
    float* ws2 = workspace + tmc_spline_workspace_floats(c, n0, n1, n2);
    g2.data = ws2;
    padded_dims(m0, m1, m2, g2.p0, g2.p1, g2.p2);
    spline_pad_kernel<<<1, 256, 0, stream>>>(coeffs2, c, m0, m1, m2, ws2); tmc_count_launch();
  }
  long total = (long)n_frames * lh * lw;
  spline_lattice_kernel<Times><<<tmc_div_up(total, 128), 128, 0, stream>>>(g1, kind, g2, kind2, coeffs2 != nullptr, n_frames,
                                                                          times, lh, lw, lattice); tmc_count_launch();
  TMC_CHECK_LAUNCH(name);
  return TMC_OK;
}

// deformation_field_utils.py:42-93 for all frames at once: lattice (T, c, lh, lw).
// coeffs2 (optional, may be null) is added (correct_motion.py:297-305).
TMC_API int tmc_spline_lattice(const float* coeffs, int c, int n0, int n1, int n2, int kind, const float* coeffs2, int m0,
                               int m1, int m2, int kind2, int n_frames, int frame_offset, int total_frames, int lh,
                               int lw, float* lattice, float* workspace, cudaStream_t stream) {
  if (int e = check_grid(coeffs, c, n0, n1, n2, kind)) return e;
  TMC_CHECK_ARG(lattice && workspace && n_frames >= 1 && lh >= 1 && lw >= 1, "spline_lattice: bad arguments");
  TMC_CHECK_ARG(frame_offset >= 0 && frame_offset + n_frames <= total_frames, "spline_lattice: frame range outside the movie");
  return spline_lattice_launch("tmc_spline_lattice", coeffs, c, n0, n1, n2, kind, coeffs2, m0, m1, m2, kind2, n_frames,
                               LinspaceTimes{frame_offset, total_frames}, lh, lw, lattice, workspace, stream);
}

// tmc_spline_lattice at the normalised times times[f] (device, n_frames floats) instead of linspace(0,1,total)[offset + f]
TMC_API int tmc_spline_lattice_times(const float* coeffs, int c, int n0, int n1, int n2, int kind, const float* coeffs2,
                                     int m0, int m1, int m2, int kind2, int n_frames, const float* times, int lh, int lw,
                                     float* lattice, float* workspace, cudaStream_t stream) {
  if (int e = check_grid(coeffs, c, n0, n1, n2, kind)) return e;
  TMC_CHECK_ARG(times && lattice && workspace, "spline_lattice_times: null pointer");
  TMC_CHECK_ARG(n_frames >= 1 && lh >= 1 && lw >= 1, "spline_lattice_times: bad sizes (%d frames, %d x %d lattice)",
                n_frames, lh, lw);
  return spline_lattice_launch("tmc_spline_lattice_times", coeffs, c, n0, n1, n2, kind, coeffs2, m0, m1, m2, kind2,
                               n_frames, TableTimes{times}, lh, lw, lattice, workspace, stream);
}

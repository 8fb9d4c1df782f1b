// One iteration of the spline-coefficient optimisation ("mse" / "cc" losses) as two kernels: a streaming
// loss/gradient kernel over tiled spectra and a single-CTA coefficient kernel.
//
// Replaces, per optimiser iteration, the reference's loop over shuffled mini-batches with autograd through
// the spline evaluation, fourier_shift_dft_2d, the Fourier filters, the leave-one-out reference and
// _compute_loss, followed by optimizer.step() (estimate_motion_optimizer.py:361-416,442-510,611-671;
// closed form of loss and gradient: SURVEY.md Appendix E, optimizer.cu header).
//
// Data layout: the band-limited, filtered patch spectra FW[g][t] are re-laid once per call into tiles of
// 8 (ky) x 16 (kx) bins with all T frames of a tile contiguous and real / imaginary parts in separate
// planes: (G, n_tiles, T, 2 [re, im], 128) float32.  Tiles that hold no pass-band bin are dropped.
//
// local_loss_tile_kernel, one CTA = one (patch, tile):
//   1. one elected thread issues 1-D bulk (TMA) copies of the tile's T KB into shared memory, 8 frames per
//      mbarrier; meanwhile the CTA turns the patch's per-frame shifts into the 8 + 16 phase factors per frame;
//   2. pass 1 (thread = 2 adjacent bins, packed fp32x2 arithmetic): S_t = FW_t exp(i theta_t) written back in
//      place, Sigma = sum_t S_t;
//   3. pass 2 (half-warp = frame): dL/ds_t = -2 b sum_f w (c f) Im(S_t conj Sigma) from shared memory.
//   The spectra are read from HBM exactly once per iteration.
// local_coefficient_kernel (one CTA): dL/ds -> dL/dcoefficients through the transposed separable dense spline
//   weights W_t (T, nt), W_sp (G, nh nw); loss; Adam update; the next iteration's shifts; re-arms the accumulators.
#include "common.cuh"
#include <math.h>

namespace {

constexpr int kTileKy = 8, kTileKx = 16, kTileBins = kTileKy * kTileKx;
constexpr int kChunkFrames = 8;  // frames per bulk copy
constexpr int kMaxChunks = 256 / kChunkFrames;  // T <= 256
constexpr int kTileThreads = 256;
constexpr int kCoefThreads = 1024;

struct StepParams {
  const float* spec;  // (G, n_tiles, T, 2 [re, im], 128)
  const int* tiles;   // (n_tiles, 2) = (ty, tx)
  int n_tiles, G, T;
  int ny, nx, KY, KX, ky_start;
  float inv_ny, inv_nx;     // fp32(1/ny), fp32(1/nx)
  const double* sum_norms;  // (G): sum_t A_t under the loss's weighting
  const float* eval_base;   // (T, G, 2) Angstrom
  const float* w_t;         // (T, nt)
  const float* w_sp;        // (G, nhw)
  int nt, nhw;
  const float* patch_scale;  // (G): the row of this iteration
  float pixel_spacing;
  int loss_type;  // 0 mse, 1 cc
  float* coef;    // (2, nt, nhw) learnable grid
  float* exp_avg;
  float* exp_avg_sq;
  // torch.optim.Adam scalars, formed in double on the host like torch does: step_size = lr / (1 - beta1^step),
  // bc2_sqrt = sqrt(1 - beta2^step)
  float step_size, bc2_sqrt, w1, w2, b2, epsf, weight_decay;
  double* loss_out;  // where this iteration's loss goes
  float* grad_out;   // (2, nt, nhw)
  float* shifts;       // (G, T, 2) px, written by the coefficient kernel
  float* grad_shifts;  // (G, T, 2) accumulator, zero on entry, zero on exit
  double* q;           // (G) accumulator, zero on entry, zero on exit
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_load(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void mbar_wait_addr(uint32_t bar_addr, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "LAB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
      "@P1 bra DONE;\n"
      "bra LAB_WAIT;\n"
      "DONE:\n"
      "}" ::"r"(bar_addr),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "LAB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
      "@P1 bra DONE;\n"
      "bra LAB_WAIT;\n"
      "DONE:\n"
      "}" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}

// exp(i x): two-term Cody-Waite reduction to [-pi, pi], then the SFU sine / cosine (absolute error <= 2^-21.2 there,
// the size of the fp32 rounding of the angle itself); ~5x fewer instructions than sincosf
__device__ __forceinline__ float2 fast_cis(float x) {
  const float k = rintf(x * 0.15915494309189535f);
  float r = fmaf(k, -6.2831854820251465f, x);
  r = fmaf(k, 1.7484555e-7f, r);  // fp32(2 pi) - 2 pi
  return make_float2(__cosf(r), __sinf(r));
}

// ---- the coefficient kernel -------------------------------------------------------------------------------------------
// flags: 1 = backward (gradient, loss, re-arm), 2 = Adam update with that gradient, 4 = shifts of the (updated)
// coefficients, 8 = Adam update with the gradient found in grad_out (complete: all-reduced over the ranks of a
// frame-split movie by the caller), before the shifts
// dynamic shared memory (floats): grad_shifts 2GT | eval_base 2GT | W_t T nt | W_sp G nhw | coef 2 nt nhw | u G 2 nt |
// exp_avg, exp_avg_sq 2 nt nhw each
// Everything the kernel reads is staged with one batch of independent loads (one memory latency), the rest is
// shared-memory arithmetic: the kernel sits on the critical path of every iteration.
__global__ void __launch_bounds__(kCoefThreads) local_coefficient_kernel(const StepParams p, int flags) {
  extern __shared__ float csm[];
  __shared__ double red[kCoefThreads / 32];
  const int tid = threadIdx.x;
  const int G = p.G, T = p.T, nt = p.nt, nhw = p.nhw;
  const int ncoef = 2 * nt * nhw, ngt = 2 * G * T;
  float* gs_s = csm;
  float* eb_s = gs_s + ngt;
  float* wt_s = eb_s + ngt;
  float* wsp_s = wt_s + T * nt;
  float* coef_s = wsp_s + G * nhw;
  float* u_s = coef_s + ncoef;
  float* ea_s = u_s + G * 2 * nt;  // Adam state, staged with everything else
  float* eas_s = ea_s + ncoef;
  // the next loss kernel may start its prologue (bulk copies of the spectra) now; it waits for this grid to
  // complete before it reads the shifts (programmatic dependent launch)
  asm volatile("griddepcontrol.launch_dependents;");
  const float neg_inv_px = -1.0f / p.pixel_spacing;
  // constants first: they do not depend on the loss kernel this launch is a programmatic dependent of
  if (flags & 4)
    for (int i = tid; i < ngt; i += kCoefThreads) eb_s[i] = __ldg(p.eval_base + i);
  for (int i = tid; i < T * nt; i += kCoefThreads) wt_s[i] = __ldg(p.w_t + i);
  for (int i = tid; i < G * nhw; i += kCoefThreads) wsp_s[i] = __ldg(p.w_sp + i);
  asm volatile("griddepcontrol.wait;" ::: "memory");  // the preceding loss kernel (and everything before it) is complete
  if (flags & 1)
    for (int i = tid; i < ngt; i += kCoefThreads) gs_s[i] = p.grad_shifts[i] * neg_inv_px;  // dL/d eval_new = -(1/px) dL/ds
  for (int i = tid; i < ncoef; i += kCoefThreads) coef_s[i] = p.coef[i];
  if (flags & (2 | 8))
    for (int i = tid; i < ncoef; i += kCoefThreads) {
      ea_s[i] = p.exp_avg[i];
      eas_s[i] = p.exp_avg_sq[i];
    }
  double l = 0.0;
  if (flags & 1) {
    // loss = sum_g scale_g l_g(q_g, sum_t A_t)
    for (int g = tid; g < G; g += kCoefThreads) {
      const double sc = (double)p.patch_scale[g];
      if (sc != 0.0) {
        const double sumA = p.sum_norms[g], qg = p.q[g];
        if (p.loss_type == 0) {
          const double a = (double)T / (double)(T - 1);
          l += sc * a * a * (sumA - qg / T);
        } else {
          l += -sc * (qg - sumA) / ((double)p.ny * (double)p.nx * (double)(T - 1));
        }
      }
    }
    l = warp_sum(l);
    if ((tid & 31) == 0) red[tid >> 5] = l;
  }
  __syncthreads();
  if (flags & 1) {
    if (tid == 0) {
      double s = 0.0;
      for (int i = 0; i < kCoefThreads / 32; ++i) s += red[i];
      *p.loss_out = s;
    }
    // re-arm the accumulators for the next iteration
    for (int i = tid; i < ngt; i += kCoefThreads) p.grad_shifts[i] = 0.f;
    for (int i = tid; i < G; i += kCoefThreads) p.q[i] = 0.0;
    // (a) gu[g][c][k] = sum_t W_t[t][k] * dL/d eval_new[t][g][c],  dL/d eval_new = -(1/px) dL/ds
    for (int o = tid; o < G * 2 * nt; o += kCoefThreads) {
      const int k = o % nt, c = (o / nt) & 1, g = o / (2 * nt);
      float acc = 0.f;
      for (int t = 0; t < T; ++t) acc = fmaf(wt_s[t * nt + k], gs_s[(g * T + t) * 2 + c], acc);
      u_s[o] = acc;
    }
    __syncthreads();
    // (b) dL/dcoef[c][k][j] = sum_g W_sp[g][j] gu[g][c][k]; then the Adam update (torch.optim.Adam, amsgrad off)
    const float step_size = p.step_size, bc2_sqrt = p.bc2_sqrt, w1 = p.w1, w2 = p.w2, b2 = p.b2, epsf = p.epsf;
    for (int o = tid; o < ncoef; o += kCoefThreads) {
      const int j = o % nhw, ck = o / nhw;  // ck = c * nt + k
      float acc = 0.f;
      for (int g = 0; g < G; ++g) acc = fmaf(wsp_s[g * nhw + j], u_s[g * 2 * nt + ck], acc);
      p.grad_out[o] = acc;
      if (flags & 2) {
        float gr = acc;
        float par = coef_s[o];
        if (p.weight_decay != 0.f) gr = __fadd_rn(gr, __fmul_rn(p.weight_decay, par));
        const float m = __fadd_rn(ea_s[o], __fmul_rn(w1, __fsub_rn(gr, ea_s[o])));
        const float v = __fadd_rn(__fmul_rn(eas_s[o], b2), __fmul_rn(w2, __fmul_rn(gr, gr)));
        p.exp_avg[o] = m;
        p.exp_avg_sq[o] = v;
        const float denom = __fadd_rn(__fdiv_rn(__fsqrt_rn(v), bc2_sqrt), epsf);
        par = __fadd_rn(par, __fmul_rn(-step_size, __fdiv_rn(m, denom)));
        p.coef[o] = par;
        coef_s[o] = par;
      }
    }
    __syncthreads();  // coef_s updated, u_s (as gu) consumed
  }
  if (flags & 8) {
    // torch.optim.Adam on the gradient the caller completed (same formulas as above)
    const float step_size = p.step_size, bc2_sqrt = p.bc2_sqrt, w1 = p.w1, w2 = p.w2, b2 = p.b2, epsf = p.epsf;
    for (int o = tid; o < ncoef; o += kCoefThreads) {
      float gr = p.grad_out[o];
      float par = coef_s[o];
      if (p.weight_decay != 0.f) gr = __fadd_rn(gr, __fmul_rn(p.weight_decay, par));
      const float m = __fadd_rn(ea_s[o], __fmul_rn(w1, __fsub_rn(gr, ea_s[o])));
      const float v = __fadd_rn(__fmul_rn(eas_s[o], b2), __fmul_rn(w2, __fmul_rn(gr, gr)));
      p.exp_avg[o] = m;
      p.exp_avg_sq[o] = v;
      const float denom = __fadd_rn(__fdiv_rn(__fsqrt_rn(v), bc2_sqrt), epsf);
      par = __fadd_rn(par, __fmul_rn(-step_size, __fdiv_rn(m, denom)));
      p.coef[o] = par;
      coef_s[o] = par;
    }
    __syncthreads();
  }
  if (!(flags & 4)) return;
  // u[g][c][k] = sum_j W_sp[g][j] coef[c][k][j]
  for (int o = tid; o < G * 2 * nt; o += kCoefThreads) {
    const int ck = o % (2 * nt), g = o / (2 * nt);
    float acc = 0.f;
    for (int j = 0; j < nhw; ++j) acc = fmaf(wsp_s[g * nhw + j], coef_s[ck * nhw + j], acc);
    u_s[o] = acc;
  }
  __syncthreads();
  // shifts[g][t][c] = -(eval_new + eval_base) / px   (estimate_motion_optimizer.py:487-492)
  for (int i = tid; i < ngt; i += kCoefThreads) {
    const int c = i & 1, t = (i >> 1) % T, g = (i >> 1) / T;
    float ev = 0.f;
    for (int k = 0; k < nt; ++k) ev = fmaf(wt_s[t * nt + k], u_s[(g * 2 + c) * nt + k], ev);
    const float v = __fmul_rn(-1.0f, __fadd_rn(ev, eb_s[(t * G + g) * 2 + c]));
    p.shifts[i] = __fdiv_rn(v, p.pixel_spacing);
  }
}

// ---- the loss / gradient kernel ---------------------------------------------------------------------------------------
// dynamic shared memory (floats): tile T*256 (re[128] | im[128] per frame) | Ey T*8 float4 (c,c,s,s) |
// Ex T*8 float4 (c0,c1,s0,s1) per column pair | Cy, Cx 64 float4 each | sigma 256 | cf 24 | red | bars
__global__ void __launch_bounds__(kTileThreads) local_loss_tile_kernel(const StepParams p) {
  constexpr int THREADS = kTileThreads;
  constexpr int NW = THREADS / 64;  // frame interleave of pass 1 (thread = 2 adjacent kx bins)
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int T = p.T;
  float* tile = reinterpret_cast<float*>(smem_raw);               // [T][2][128]
  float4* Ey = reinterpret_cast<float4*>(tile + (long)T * 256);   // [T][8]
  float4* Ex = Ey + T * 8;                                        // [T][8]
  float4* Cy = Ex + T * 8;                                        // [64] (cfy w Sig_re x2, -cfy w Sig_im x2)
  float4* Cx = Cy + 64;                                           // [64] the same with cfx
  float* sigma = reinterpret_cast<float*>(Cx + 64);               // [4][64]: re even / re odd / im even / im odd columns
  float* cf = sigma + 256;                                        // [24]
  double* red = reinterpret_cast<double*>(cf + 24);               // [2]
  uint64_t* bars = reinterpret_cast<uint64_t*>(red + 2);          // [nchunks]

  const int tid = threadIdx.x;
  const int g = blockIdx.y, tile_id = blockIdx.x;
  const int nchunks = (T + kChunkFrames - 1) / kChunkFrames;
  // the coefficient kernel that follows may be scheduled as soon as every CTA of this grid has started; it waits
  // for this grid to complete before it reads the accumulators
  asm volatile("griddepcontrol.launch_dependents;");

  if (tid == 0) {
    for (int c = 0; c < nchunks; ++c) mbar_init(bars + c, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    const float* src = p.spec + ((long)g * p.n_tiles + tile_id) * T * 256;
    for (int c = 0; c < nchunks; ++c) {
      const int frames = min(kChunkFrames, T - c * kChunkFrames);
      const uint32_t bytes = (uint32_t)frames * 256 * sizeof(float);
      mbar_expect_tx(bars + c, bytes);
      bulk_load(tile + (long)c * kChunkFrames * 256, src + (long)c * kChunkFrames * 256, bytes, bars + c);
    }
  }
  const float sc = __ldg(p.patch_scale + g);
  const int ty = __ldg(p.tiles + 2 * tile_id), tx = __ldg(p.tiles + 2 * tile_id + 1);
  // frequency factors fp32(-2 pi) * fp32(k * fp32(1/n)) (torch_fourier_shift on torch.fft.fftfreq grids) of the tile's
  // 8 rows and 16 columns (clamped inside the band box: the padding holds zeros); every thread forms the one it needs
  // for the phase table below; one thread per slot also publishes it (cf[24]) for the gradient factors
  // phase-table slot of this thread (see the loops below): 96 threads share the 8 rows, 160 threads the 16 columns, so that
  // both halves of the table take the same number of sweeps over the frames (T = 40: 4 and 4 instead of 3 and 5)
  constexpr int kRowThreads = 96;
  const int my_r = tid < kRowThreads ? (tid & 7) : kTileKy + ((tid - kRowThreads) & 15);
  float my_cf;
  {
    if (my_r < kTileKy) {
      int ky = p.ky_start + min(ty * kTileKy + my_r, p.KY - 1);
      if (ky >= (p.ny + 1) / 2) ky -= p.ny;
      if (ky < -(p.ny / 2)) ky += p.ny;
      my_cf = __fmul_rn(-6.283185307179586f, __fmul_rn((float)ky, p.inv_ny));
    } else {
      my_cf = __fmul_rn(-6.283185307179586f, __fmul_rn((float)min(tx * kTileKx + my_r - kTileKy, p.KX - 1), p.inv_nx));
    }
    if (tid < kTileKy) cf[tid] = my_cf;
    if (tid >= kRowThreads && tid < kRowThreads + kTileKx) cf[kTileKy + tid - kRowThreads] = my_cf;
  }
  sigma[tid] = 0.f;
  // everything above is independent of the coefficient kernel that precedes this launch (programmatic dependent
  // launch): wait for it to complete before touching the shifts and the accumulators
  asm volatile("griddepcontrol.wait;" ::: "memory");
  if (sc == 0.f || T < 2) {
    // nothing to add for this patch, but the bulk copies must land before the CTA may retire
    __syncthreads();  // barriers initialised
    for (int c = 0; c < nchunks; ++c) mbar_wait(bars + c, 0);
    return;
  }
  // phase factors exp(i c f_y s_y) of the 8 rows (duplicated for the packed arithmetic: threads 0..95, 12 frames per
  // sweep) and exp(i c f_x s_x) of the 8 column pairs (threads 96..255, 10 frames per sweep), every frame; the shifts
  // come straight from the coefficient kernel's (G, T, 2) table
  const float* shg = p.shifts + (long)g * T * 2;
  if (tid < kRowThreads) {
    for (int t = tid >> 3; t < T; t += kRowThreads / 8) {
      const float2 e = fast_cis(__fmul_rn(my_cf, shg[2 * t]));
      Ey[t * 8 + my_r] = make_float4(e.x, e.x, e.y, e.y);
    }
  } else {
    const int j = (tid - kRowThreads) & 15;
    for (int t = (tid - kRowThreads) >> 4; t < T; t += (kTileThreads - kRowThreads) / 16) {
      const float2 e = fast_cis(__fmul_rn(my_cf, shg[2 * t + 1]));
      float* o = reinterpret_cast<float*>(Ex + t * 8 + (j >> 1)) + (j & 1);
      o[0] = e.x;
      o[2] = e.y;
    }
  }
  __syncthreads();  // barriers initialised; cf, sigma, Ey, Ex complete

  // pass 1 (thread = 2 adjacent columns of one row, every NW-th frame): S_t = FW_t e_t in place, Sigma
  {
    const int pb = tid & 63, th = tid >> 6;
    // running pointers: frame t0 = th of the current chunk
    const float4* ey = Ey + (pb >> 3) + th * 8;
    const float4* ex = Ex + (pb & 7) + th * 8;
    float2* col = reinterpret_cast<float2*>(tile) + pb + th * 128;  // re pair; im pair at +64
    float2 sre = make_float2(0.f, 0.f), sim = make_float2(0.f, 0.f);
    auto body = [&](const float4* eyp, const float4* exp_, float2* cp) {
      const float4 y = *eyp, x = *exp_;
      const float2 cy = make_float2(y.x, y.y), sy = make_float2(y.z, y.w);
      const float2 cx = make_float2(x.x, x.y), sx = make_float2(x.z, x.w);
      // e = ey * ex
      const float2 ere = __ffma2_rn(make_float2(-sy.x, -sy.y), sx, __fmul2_rn(cy, cx));
      const float2 eim = __ffma2_rn(sy, cx, __fmul2_rn(cy, sx));
      const float2 a = cp[0], b = cp[64];
      const float2 re = __ffma2_rn(make_float2(-b.x, -b.y), eim, __fmul2_rn(a, ere));
      const float2 im = __ffma2_rn(b, ere, __fmul2_rn(a, eim));
      cp[0] = re;
      cp[64] = im;
      sre = __fadd2_rn(sre, re);
      sim = __fadd2_rn(sim, im);
    };
    const uint32_t bar0 = smem_u32(bars);
    for (int c = 0; c < nchunks; ++c) {
      mbar_wait_addr(bar0 + 8u * c, 0);
      if ((c + 1) * kChunkFrames <= T) {
#pragma unroll
        for (int i = 0; i < kChunkFrames / NW; ++i) body(ey + i * NW * 8, ex + i * NW * 8, col + i * NW * 128);
      } else {
        for (int t = c * kChunkFrames + th, i = 0; t < T; t += NW, ++i) body(ey + i * NW * 8, ex + i * NW * 8, col + i * NW * 128);
      }
      ey += kChunkFrames * 8;
      ex += kChunkFrames * 8;
      col += kChunkFrames * 128;
    }
    atomicAdd(sigma + pb, sre.x);
    atomicAdd(sigma + 64 + pb, sre.y);
    atomicAdd(sigma + 128 + pb, sim.x);
    atomicAdd(sigma + 192 + pb, sim.y);
  }
  __syncthreads();  // S and Sigma complete
  if (tid < 64) {
    const int pb = tid;
    const float2 re = make_float2(sigma[pb], sigma[64 + pb]), im = make_float2(sigma[128 + pb], sigma[192 + pb]);
    const int kx0 = tx * kTileKx + 2 * (pb & 7);
    const float w0 = (p.loss_type == 0 || kx0 == 0 || 2 * kx0 == p.nx) ? 1.0f : 2.0f;
    const float w1 = (p.loss_type == 0 || 2 * (kx0 + 1) == p.nx) ? 1.0f : 2.0f;
    const float cfy = cf[pb >> 3], cfx0 = cf[8 + 2 * (pb & 7)], cfx1 = cf[9 + 2 * (pb & 7)];
    const float wr0 = w0 * re.x, wr1 = w1 * re.y, wi0 = w0 * im.x, wi1 = w1 * im.y;
    // gy += S_im (cfy w Sig_re) - S_re (cfy w Sig_im); the same with cfx
    Cy[pb] = make_float4(cfy * wr0, cfy * wr1, -cfy * wi0, -cfy * wi1);
    Cx[pb] = make_float4(cfx0 * wr0, cfx1 * wr1, -cfx0 * wi0, -cfx1 * wi1);
  }
  __syncthreads();  // Ctab complete

  // pass 2: half-warp per frame, lane = 2 adjacent bins, 4 steps over the 128 bins
  float bscale;
  if (p.loss_type == 0) {
    const float a = (float)T / (float)(T - 1);
    bscale = -sc * a * a / (float)T;
  } else {
    bscale = -sc / ((float)p.ny * (float)p.nx * (float)(T - 1));
  }
  const int lane = tid & 31, warp = tid >> 5;
  const int half = lane >> 4, l16 = lane & 15;
  for (int pi = warp; 2 * pi < T; pi += THREADS / 32) {
    const int t = 2 * pi + half;
    const bool ok = t < T;
    const float2* row = reinterpret_cast<const float2*>(tile + (long)(ok ? t : 0) * 256) + l16;
    float2 ay = make_float2(0.f, 0.f), ax = make_float2(0.f, 0.f);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float2 re = row[16 * k], im = row[64 + 16 * k];
      const float4 cy = Cy[l16 + 16 * k], cx = Cx[l16 + 16 * k];
      ay = __ffma2_rn(im, make_float2(cy.x, cy.y), ay);
      ay = __ffma2_rn(re, make_float2(cy.z, cy.w), ay);
      ax = __ffma2_rn(im, make_float2(cx.x, cx.y), ax);
      ax = __ffma2_rn(re, make_float2(cx.z, cx.w), ax);
    }
    const float gy = ay.x + ay.y, gx = ax.x + ax.y;
    // lanes with bit 3 clear keep the y sum, the others the x sum: one exchange, then 3 single-value stages
    const bool keep_x = (l16 & 8) != 0;
    float v = (keep_x ? gx : gy) + __shfl_xor_sync(0xffffffffu, keep_x ? gy : gx, 8);
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (ok && (l16 & 7) == 0) {
      v *= -2.0f * bscale;
      if (v != 0.f) atomicAdd(p.grad_shifts + ((long)g * T + t) * 2 + (keep_x ? 1 : 0), v);
    }
  }
  // q_g += sum_bins w |Sigma|^2 (the loss value; double): after the gradient pass, off the critical path of the CTA
  if (tid < 64) {
    const int pb = tid;
    const float2 re = make_float2(sigma[pb], sigma[64 + pb]), im = make_float2(sigma[128 + pb], sigma[192 + pb]);
    const int kx0 = tx * kTileKx + 2 * (pb & 7);
    const float w0 = (p.loss_type == 0 || kx0 == 0 || 2 * kx0 == p.nx) ? 1.0f : 2.0f;
    const float w1 = (p.loss_type == 0 || 2 * (kx0 + 1) == p.nx) ? 1.0f : 2.0f;
    double v = (double)w0 * ((double)re.x * re.x + (double)im.x * im.x) + (double)w1 * ((double)re.y * re.y + (double)im.y * im.y);
    v = warp_sum(v);
    if ((tid & 31) == 0 && v != 0.0) atomicAdd(p.q + g, v);
  }
}

// spec (G, Tp, KY, KX) -> tiled (G, n_tiles, T, 2 [re, im], 128), zero padded
__global__ void tile_spectra_kernel(const float2* __restrict__ spec, int T, int Tp, int KY, int KX, const int* __restrict__ tiles,
                                    int n_tiles, int frame_major, float* __restrict__ out) {
  const int tile_id = blockIdx.x, t = blockIdx.y, g = blockIdx.z, G = gridDim.z;
  const int b = threadIdx.x;
  const int kyb = tiles[2 * tile_id] * kTileKy + b / kTileKx, kx = tiles[2 * tile_id + 1] * kTileKx + b % kTileKx;
  float2 v = make_float2(0.f, 0.f);
  const long plane = frame_major ? ((long)(t >> 1) * G + g) * 2 + (t & 1) : (long)g * Tp + t;
  if (kyb < KY && kx < KX) v = spec[(plane * KY + kyb) * KX + kx];
  float* o = out + (((long)g * n_tiles + tile_id) * T + t) * 2 * kTileBins;
  o[b] = v.x;
  o[kTileBins + b] = v.y;
}

size_t tile_smem_bytes(int t) {
  return (size_t)t * kTileBins * 8 + (size_t)t * 16 * 16 + 128 * 16 + 256 * 4 + 24 * 4 + 2 * 8 +
         (size_t)((t + kChunkFrames - 1) / kChunkFrames) * 8;
}
size_t coef_smem_bytes(int g, int t, int nt, int nhw) {
  return ((size_t)4 * g * t + (size_t)t * nt + (size_t)g * nhw + (size_t)6 * nt * nhw + (size_t)g * 2 * nt) * 4;
}

}  // namespace

// 1 if the two-kernel iteration supports this problem (shared-memory tile of t KB, coefficient scratch), else 0
TMC_API int tmc_local_steps_supported(int g, int t, int nt, int nhw) {
  if (t < 2 || t > kChunkFrames * kMaxChunks || g < 1 || g > 65535 || nt < 1 || nhw < 1) return 0;
  if (tile_smem_bytes(t) > 200 * 1024) return 0;
  return coef_smem_bytes(g, t, nt, nhw) <= 160 * 1024 ? 1 : 0;
}

// spec (g, tp, ky_count, kx_count) complex64 (frame_major != 0: (tp / 2, g, 2, ky_count, kx_count), see
// tmc_local_spectra_norms) -> out (g, n_tiles, t, 2, 128) float32; tiles (n_tiles, 2) int32 (ty, tx)
TMC_API int tmc_local_tile_spectra(const void* spec, int g, int t, int tp, int ky_count, int kx_count, const int* tiles,
                                   int n_tiles, int frame_major, void* out, cudaStream_t stream) {
  TMC_CHECK_ARG(spec && tiles && out && g >= 1 && t >= 1 && tp >= t && n_tiles >= 1 && t <= 65535 && g <= 65535,
                "local_tile_spectra: bad arguments");
  dim3 grid(n_tiles, t, g);
  tile_spectra_kernel<<<grid, kTileBins, 0, stream>>>((const float2*)spec, t, tp, ky_count, kx_count, tiles, n_tiles, frame_major, (float*)out);
  tmc_count_launch();
  TMC_CHECK_LAUNCH("tmc_local_tile_spectra");
  return TMC_OK;
}

// workspace of tmc_local_steps: shifts 2*g*t | grad_shifts 2*g*t floats | q g doubles
TMC_API long tmc_local_steps_workspace_bytes(int g, int t, int nt) {
  (void)nt;
  long floats = 4l * g * t;
  floats = (floats + 1) & ~1l;
  return floats * 4 + 8l * g;
}

// n_steps iterations of the optimisation: a coefficient launch, then per step a loss/gradient launch and a coefficient launch.
//  tiled (g, n_tiles, t, 2, 128) from tmc_local_tile_spectra; sum_norms (g) double; eval_base (t, g, 2);
//  w_t (t, nt), w_sp (g, nhw): dense separable spline weights of the patch centres (time axis / spatial axes);
//  patch_scale (rows, g): step i uses row first_row + i; coef (2, nt, nhw);
//  mode 0: Adam (exp_avg, exp_avg_sq, lr, betas, eps, weight_decay; step number first_row + i + 1) updates coef in
//          place, loss_out[first_row + i];
//  mode 1: n_steps must be 1; only grad_out (2, nt, nhw) and loss_out[0] are produced.
TMC_API int tmc_local_steps(const void* tiled, const int* tiles, int n_tiles, int g, int t, int ny, int nx, int ky_count,
                            int kx_count, int ky_start, const double* sum_norms, const float* eval_base, const float* w_t,
                            const float* w_sp, int nt, int nhw, const float* patch_scale, float pixel_spacing, int loss_type,
                            float* coef, float* exp_avg, float* exp_avg_sq, double lr, double beta1, double beta2, double eps,
                            double weight_decay, int first_row, int mode, int n_steps, double* loss_out, float* grad_out,
                            void* workspace, cudaStream_t stream) {
  TMC_CHECK_ARG(tiled && tiles && sum_norms && eval_base && w_t && w_sp && patch_scale && coef && loss_out && grad_out && workspace,
                "local_steps: null pointer");
  TMC_CHECK_ARG(g >= 1 && g <= kMaxGridYZ, "local_steps: at most %d patches, got %d", kMaxGridYZ, g);
  TMC_CHECK_ARG(mode >= 0 && mode <= 3, "local_steps: mode must be 0 .. 3");
  TMC_CHECK_ARG(mode == 1 || (exp_avg && exp_avg_sq), "local_steps: Adam state missing");
  TMC_CHECK_ARG(mode == 0 || n_steps == 1, "local_steps: modes 1 .. 3 take one step");
  TMC_CHECK_ARG(n_tiles >= 1 && n_steps >= 1 && first_row >= 0 && pixel_spacing > 0.f && (loss_type == 0 || loss_type == 1),
                "local_steps: bad arguments");
  if (!tmc_local_steps_supported(g, t, nt, nhw)) {
    tmc_set_error("local_steps: unsupported problem size (g=%d t=%d nt=%d nhw=%d)", g, t, nt, nhw);
    return TMC_ERR_UNSUPPORTED;
  }
  StepParams p;
  p.spec = (const float*)tiled;
  p.tiles = tiles;
  p.n_tiles = n_tiles;
  p.G = g;
  p.T = t;
  p.ny = ny;
  p.nx = nx;
  p.KY = ky_count;
  p.KX = kx_count;
  p.ky_start = ky_start;
  p.inv_ny = (float)(1.0 / (double)ny);
  p.inv_nx = (float)(1.0 / (double)nx);
  p.sum_norms = sum_norms;
  p.eval_base = eval_base;
  p.w_t = w_t;
  p.w_sp = w_sp;
  p.nt = nt;
  p.nhw = nhw;
  p.pixel_spacing = pixel_spacing;
  p.loss_type = loss_type;
  p.coef = coef;
  p.exp_avg = exp_avg;
  p.exp_avg_sq = exp_avg_sq;
  p.w1 = (float)(1.0 - beta1);
  p.w2 = (float)(1.0 - beta2);
  p.b2 = (float)beta2;
  p.epsf = (float)eps;
  p.weight_decay = (float)weight_decay;
  p.step_size = 0.f;
  p.bc2_sqrt = 1.f;
  p.grad_out = grad_out;
  float* wf = (float*)workspace;
  p.shifts = wf;
  p.grad_shifts = wf + 2l * g * t;
  const long floats = (4l * g * t + 1) & ~1l;
  p.q = (double*)(wf + floats);
  if (mode < 2) TMC_CUDA(cudaMemsetAsync(workspace, 0, (size_t)tmc_local_steps_workspace_bytes(g, t, nt), stream));
  const size_t smem = tile_smem_bytes(t), csmem = coef_smem_bytes(g, t, nt, nhw);
  // per-device attributes: set on every call (cheap) so whichever device is current is configured
  TMC_CUDA(cudaFuncSetAttribute(local_loss_tile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(200 * 1024)));
  TMC_CUDA(cudaFuncSetAttribute(local_coefficient_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(160 * 1024)));
  dim3 grid(n_tiles, g);
  p.patch_scale = patch_scale + (long)first_row * g;
  p.loss_out = loss_out;
  if (mode >= 2) {
    // Adam step number first_row on the caller's (all-reduced) gradient [+ the shifts of the updated coefficients]
    const double step = (double)first_row;
    p.step_size = (float)(lr / (1.0 - pow(beta1, step)));
    p.bc2_sqrt = (float)sqrt(1.0 - pow(beta2, step));
  }
  local_coefficient_kernel<<<1, kCoefThreads, csmem, stream>>>(p, mode == 2 ? (8 | 4) : (mode == 3 ? 8 : 4));
  tmc_count_launch();
  if (mode == 3) {
    TMC_CHECK_LAUNCH("tmc_local_steps");
    return TMC_OK;
  }
  // the loss kernel is a programmatic dependent of the coefficient kernel before it: its CTAs become resident and
  // start their bulk copies while the (single-CTA) coefficient kernel still runs
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = dim3(kTileThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaLaunchConfig_t ccfg = {};  // the coefficient kernel as a programmatic dependent of the loss kernel before it
  ccfg.gridDim = dim3(1);
  ccfg.blockDim = dim3(kCoefThreads);
  ccfg.dynamicSmemBytes = csmem;
  ccfg.stream = stream;
  ccfg.attrs = attr;
  ccfg.numAttrs = 1;
  for (int i = 0; i < n_steps; ++i) {
    const int row = first_row + i;
    p.patch_scale = patch_scale + (long)row * g;
    const double step = (double)(row + 1);
    p.step_size = (float)(lr / (1.0 - pow(beta1, step)));
    p.bc2_sqrt = (float)sqrt(1.0 - pow(beta2, step));
    p.loss_out = loss_out + (mode == 0 ? row : 0);
    TMC_CUDA(cudaLaunchKernelEx(&cfg, local_loss_tile_kernel, p));
    tmc_count_launch();
    const int last = i == n_steps - 1;
    TMC_CUDA(cudaLaunchKernelEx(&ccfg, local_coefficient_kernel, p, mode == 0 ? (last ? 3 : 7) : 1));  // modes 1, 2: backward only
    tmc_count_launch();
  }
  TMC_CHECK_LAUNCH("tmc_local_steps");
  return TMC_OK;
}

// Fused resample-and-sum with frame tiles staged by TMA (included by warp.cu inside its anonymous namespace).
//
// Replaces the per-pixel global-memory gathers of warp_lattice_kernel for images whose rows are 16-byte aligned
// (W % 4 == 0); same arithmetic, same results (correct_motion.py:81-185, SURVEY.md Appendix A.2).
//
// One persistent CTA per SM walks over 32 x 60 output tiles; for every tile it visits the T frames in order:
//   * a producer warp computes, per frame, where the tile lands in the frame (tile origin + the field's shift at the tile
//     centre) and issues two tensor-map TMA loads (cp.async.bulk.tensor) into one slot of a ring of shared-memory stages:
//     the 48 x 71 pixel box of the frame around that landing point (hardware zero-fill outside the frame) and the
//     64 x 16 x 2 block of the x-interpolated shift lattice the tile's pixels need;
//   * 15 consumer warps (thread = one column x 4 rows of the tile) wait on the stage's "full" mbarrier, evaluate the
//     shift of their pixels from the staged lattice rows, run the reference's fp32 coordinate chain (packed fp32x2,
//     both axes at once), read their 4 x 4 taps from the staged box at immediate offsets of one address (7 x 4 loads
//     shared by the 4 vertically stacked pixels whenever their sampling points are stacked too) and release the stage
//     through its "empty" mbarrier.  No block-wide barrier in the frame loop; frame sums live in registers.
//   Pixels whose taps leave the box (shift varying by more than the 4-px margin inside one tile) or touch the image
//   border (border-clamped taps / zero outside) take the generic global-memory path.
// The WEIGHTED instantiation forms n_sums frame-weighted sums at once (tmc_warp_lattice_sums): the accumulators of a
// thread's 4 pixels are one float4 per sum in thread-private shared memory, in front of the (then shallower) ring.
#pragma once
#include <cuda.h>
#include <type_traits>

namespace tma {

// output tile: one consumer warp per 4 image rows.  32 x 60 = 15 consumer warps + the producer warp = 16 warps of 128
// registers, 4 per scheduler (with 14 warps two schedulers would idle a quarter of the time)
constexpr int kTX = 32, kTY = 60;
constexpr int kMargin = 4;              // how far a pixel's shift may differ from the tile-centre shift
constexpr int kBoxW = kTX + 2 * kMargin + 8;   // 48: + 3 tap columns + up to 3 columns of alignment slack (see below), 16-byte rows
constexpr int kBoxH = kTY + 2 * kMargin + 3;   // 71
constexpr int kRxRows = 16;             // lattice rows staged per tile and channel
constexpr int kImgBytes = kBoxW * kBoxH * 4;                      // 13632
constexpr int kImgBytesPadded = (kImgBytes + 127) / 128 * 128;    // 13696
// The ring is as deep as shared memory allows (a stage holds only the lattice rows actually staged, rx_rows = 5..16, so
// 13-15 stages fit).  Measured on C2: 4 stages 2.37 ms, 8 stages 2.34 ms, 15 stages 2.33 ms -- one frame of a tile takes
// a CTA ~1 us, several DRAM round trips, so the ring never runs dry; the kernel is bound by instruction issue (about
// 300 warp instructions per warp and frame at 0.65 per cycle and scheduler: the packed fp32 instructions hold the fp32
// pipe for two cycles each and collide between the 4 warps of a scheduler), not by memory (0.64 ms with the
// arithmetic switched off).
constexpr int kMaxStages = 16;
constexpr int kMaxSmemBytes = 227 * 1024 - 2048;  // dynamic part: the static barriers / headers and alignment slack stay below 2 KB
constexpr int kConsumers = kTX * (kTY / kRows);  // 480 threads, 15 warps
static_assert(kTX % 32 == 0 && kTY % kRows == 0 && (kTX & (kTX - 1)) == 0, "tile shape");
constexpr int kThreads = kConsumers + 32;        // + the producer warp
constexpr int kConsumerWarps = kConsumers / 32;
__host__ __device__ constexpr int stage_bytes_for(int rx_rows) { return kImgBytesPadded + (rx_rows * kTX * 2 * 4 + 127) / 128 * 128; }
inline int stages_for(int rx_rows) {
  const int n = (kMaxSmemBytes - 128) / stage_bytes_for(rx_rows);
  return n < kMaxStages ? n : kMaxStages;
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
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
// the same on 32-bit shared-window addresses formed once outside the loops (the generic -> shared conversion of a
// __shared__ array element costs an S2R and two LEAs every time it is written inside a loop)
__device__ __forceinline__ void mbar_wait_addr(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "LAB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
      "@P1 bra DONE;\n"
      "bra LAB_WAIT;\n"
      "DONE:\n"
      "}" ::"r"(bar),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void mbar_arrive_addr(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ int4 lds_int4(uint32_t addr) {
  int4 v;
  asm volatile("ld.shared.v4.s32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ int2 lds_int2(uint32_t addr) {
  int2 v;
  asm volatile("ld.shared.v2.s32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(addr));
  return v;
}
// 3-D tiled tensor-map load: box at (c0, c1, c2) (innermost first) -> shared memory, completion on an mbarrier
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* map, int c0, int c1, int c2, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(
          smem_u32(dst)),
      "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(smem_u32(bar))
      : "memory");
}

// packed fp32x2 arithmetic (FFMA2 / FMUL2 / FADD2)
__device__ __forceinline__ float2 pk_fma(float2 a, float2 b, float2 c) { return __ffma2_rn(a, b, c); }
__device__ __forceinline__ float2 pk_mul(float2 a, float2 b) { return __fmul2_rn(a, b); }
__device__ __forceinline__ float2 pk_add(float2 a, float2 b) { return __fadd2_rn(a, b); }

// Keys cubic-convolution weights (A = -0.75, ATen's bicubic) of two fractions at once (.x = y axis, .y = x axis) in
// factored form: w0 = A t (1 - t)^2, w3 = A t^2 (1 - t), w1 = ((A + 2) t - (A + 3)) t^2 + 1, w2 = w1(1 - t).  Same
// polynomials as get_cubic_upsample_coefficients (cubic_weights2), 10 instead of 15 packed instructions; the results
// differ from ATen's evaluation order by rounding only (<= 2e-7 absolute, against a 1e-4 tolerance on the frame sum).
__device__ __forceinline__ void keys_weights2(float2 t, float2 (&w)[4]) {
  const float2 A = dup(kA), A2 = dup(kA + 2.0f), mA3 = dup(-(kA + 3.0f)), one = dup(1.0f);
  const float2 u = pk_fma(t, dup(-1.0f), one);
  const float2 a = pk_mul(A, pk_mul(t, u));
  w[0] = pk_mul(a, u);
  w[3] = pk_mul(a, t);
  w[1] = pk_fma(pk_fma(A2, t, mA3), pk_mul(t, t), one);
  w[2] = pk_add(pk_fma(a, dup(-1.0f), one), pk_mul(w[1], dup(-1.0f)));  // w0 + w1 + w2 + w3 = 1 and w0 + w3 = A t (1 - t)
}

// the same with an L2 eviction-priority hint (createpolicy)
__device__ __forceinline__ void tma_load_3d_hint(void* dst, const CUtensorMap* map, int c0, int c1, int c2, uint64_t* bar,
                                                 uint64_t policy) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%2, %3, "
      "%4}], [%5], %6;" ::"r"(smem_u32(dst)),
      "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(smem_u32(bar)), "l"(policy)
      : "memory");
}

template <bool V>
struct BoolTag {
  static constexpr bool value = V;
};

struct Params {
  const float* image;
  int T, H, W;
  const float* rx;  // (T, lh + 3, 2, W): x-interpolated lattice, rows padded by reflection (row p <-> lattice row p - 1)
  int rx_rows;      // lattice rows staged per tile (5 .. kRxRows)
  int n_stages, stage_bytes;  // depth of the ring and bytes per stage (stages_for / stage_bytes_for)
  int lh;
  float pixel_spacing;
  const float* mean_std;
  float* out_stack;
  float* out_sum;
  int accumulate_sum;
  int tiles_x, n_tiles;
  // constants of the coordinate chain, formed on the host so that they reach the arithmetic as constant-bank operands
  // (the kernel is bound by register-file reads: a register operand less per instruction is what counts)
  float2 nden, rcp, half_scale;  // .x = y axis, .y = x axis
  float inv_px;
};
// the weighted instantiation's parameters (a separate type: growing Params changes the register allocation of the others)
struct SumsParams : Params {
  const float* weights;  // (n_sums, T) frame weights
  int n_sums;
  float* out_sums;  // (n_sums, H, W)
  int acc_bytes;    // shared-memory accumulators in front of the ring: n_sums * kConsumers float4s
};
template <bool WEIGHTED>
using KernelParams = typename std::conditional<WEIGHTED, SumsParams, Params>::type;

template <bool WRITE_STACK, bool WRITE_SUM, bool NORMALISE, bool WEIGHTED = false>
__global__ void __launch_bounds__(kThreads, 1)
warp_tma_kernel(const __grid_constant__ CUtensorMap img_map, const __grid_constant__ CUtensorMap rx_map,
                const KernelParams<WEIGHTED> p) {
  extern __shared__ unsigned char smem_raw[];
  __shared__ __align__(8) uint64_t full_bar[kMaxStages];
  __shared__ __align__(8) uint64_t empty_bar[kMaxStages];
  // per stage: {oy + 1, ox + 1, by_lo, by_n, bx_lo, bx_n, -, -}: box origin (+1: the first tap is one before the floor) and
  // the first-tap positions (by - by_lo <= by_n, unsigned) that keep 4 + 3 stacked tap rows / 4 tap columns inside the
  // box AND inside the image (the zero-filled part of a box that hangs over the frame edge is never used)
  __shared__ __align__(16) int stage_hdr[kMaxStages][8];
  unsigned char* stages = smem_raw + ((128u - (smem_u32(smem_raw) & 127u)) & 127u);
  static_assert(!WEIGHTED || (kRows == 4 && !WRITE_STACK && !WRITE_SUM && !NORMALISE), "weighted sums: 4 rows, no other output");
  float4* sums_acc = nullptr;
  if constexpr (WEIGHTED) {
    sums_acc = reinterpret_cast<float4*>(stages);
    stages += p.acc_bytes;
  }
  const int tid = threadIdx.x;
  const int T = p.T, H = p.H, W = p.W, lh = p.lh;
  const int lhp = lh + 3;
  if (tid == 0) {
    for (int s = 0; s < kMaxStages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], kConsumerWarps);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  __syncthreads();
  const float inv_px_s = 1.0f / p.pixel_spacing;

  if (tid >= kConsumers) {
    // ---------------- producer warp ----------------
    const int lane = tid - kConsumers;
    uint32_t stage = 0, phase = 0;
    uint64_t keep_policy;  // the lattice rows are re-read by every tile of the same lattice cells: keep them in L2
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(keep_policy));
    const uint32_t stage_tx = kImgBytes + (uint32_t)p.rx_rows * kTX * 2 * 4;
    // work = chunks of up to 32 frames of one tile; lane l owns frame f0 + l of the chunk: where the tile lands in that
    // frame (tile origin + the shift of the tile centre, rounded down).  The next chunk's landing points are computed
    // (global loads in flight) while the current chunk's loads are being issued.
    auto landing = [&](int tile, int f0, int& oy, int& ox, int& x0, int& i0_tile) {
      x0 = (tile % p.tiles_x) * kTX;
      const int y0 = (tile / p.tiles_x) * kTY;
      const int yc = min(y0 + kTY / 2, H - 1), xc = min(x0 + kTX / 2, W - 1);
      const LatticeAxis ac = lattice_axis(yc, H, lh);
      i0_tile = lattice_axis(y0, H, lh).i0;
      oy = ox = 0;
      if (f0 + lane < T) {
        const float* Ry = p.rx + ((size_t)(f0 + lane) * lhp + ac.i0) * 2 * W + xc;
        float sy = 0.f, sx = 0.f;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          sy = fmaf(ac.w[k], __ldg(Ry + (size_t)k * 2 * W), sy);
          sx = fmaf(ac.w[k], __ldg(Ry + (size_t)(k * 2 + 1) * W), sx);
        }
        // clamped: a wild (or NaN) shift must not overflow the int conversion; such tiles take the generic path
        oy = y0 + (int)fminf(fmaxf(floorf(sy * inv_px_s), -1e6f), 1e6f) - kMargin - 1;
        // TMA wants the innermost box coordinate on a 16-byte boundary (measured: any other x raises "illegal
        // instruction"; tools/tma_probe.cu): rounded down to 4 pixels, the box is 3 columns wider for it
        ox = (x0 + (int)fminf(fmaxf(floorf(sx * inv_px_s), -1e6f), 1e6f) - kMargin - 1) & ~3;
      }
    };
    int tile = blockIdx.x, f0 = 0;
    int oy, ox, x0, i0_tile;
    if (tile < p.n_tiles) landing(tile, f0, oy, ox, x0, i0_tile);
    while (tile < p.n_tiles) {
      int ntile = tile, nf0 = f0 + 32;
      if (nf0 >= T) {
        nf0 = 0;
        ntile += gridDim.x;
      }
      int noy = 0, nox = 0, nx0 = 0, ni0 = 0;
      if (ntile < p.n_tiles) landing(ntile, nf0, noy, nox, nx0, ni0);
      const int nf = min(32, T - f0);
      for (int i = 0; i < nf; ++i) {
        const int foy = __shfl_sync(0xffffffffu, oy, i), fox = __shfl_sync(0xffffffffu, ox, i);
        if (lane == 0) {
          mbar_wait(&empty_bar[stage], phase ^ 1u);  // the consumers have released this slot
          {
            const int by_lo = max(0, -foy), by_n = min(kBoxH - 4, H - 4 - foy) - by_lo - (kRows - 1);
            const int bx_lo = max(0, -fox), bx_n = min(kBoxW - 4, W - 4 - fox) - bx_lo;
            int* hdr = stage_hdr[stage];
            hdr[0] = foy + 1;
            hdr[1] = fox + 1;
            hdr[2] = by_n >= 0 ? by_lo : 0x40000000;  // empty range: nothing passes
            hdr[3] = by_n >= 0 ? by_n : 0;
            hdr[4] = bx_n >= 0 ? bx_lo : 0x40000000;
            hdr[5] = bx_n >= 0 ? bx_n : 0;
          }
          unsigned char* dst = stages + (size_t)stage * p.stage_bytes;
          mbar_expect_tx(&full_bar[stage], stage_tx);
          tma_load_3d(dst, &img_map, fox, foy, f0 + i, &full_bar[stage]);
          tma_load_3d_hint(dst + kImgBytesPadded, &rx_map, x0, 0, (f0 + i) * lhp + i0_tile, &full_bar[stage], keep_policy);
        }
        if (++stage == (uint32_t)p.n_stages) {
          stage = 0;
          phase ^= 1u;
        }
      }
      __syncwarp();
      tile = ntile;
      f0 = nf0;
      oy = noy;
      ox = nox;
      x0 = nx0;
      i0_tile = ni0;
    }
    return;
  }

  // ---------------- consumer warps ----------------
  const int tx = tid & (kTX - 1), tyg = tid / kTX;
  const int lane = tid & 31;
  float mean = 0.f, inv_std = 1.f;
  if (NORMALISE) {
    mean = __ldg(p.mean_std);
    inv_std = 1.0f / __ldg(p.mean_std + 1);
  }
  // grid_sample round trip constants, .x = y axis (H), .y = x axis (W); see warp_lattice_kernel
  // nden = -(0.5 n - 0.5), rcp = fl(1 / (0.5 n - 0.5)), half_scale = 0.5 (n - 1): ((g + 1) * 0.5) * (n - 1) ==
  // (g + 1) * (0.5 * (n - 1)) bit for bit (the halving is exact, so is 0.5 * (n - 1)); see fill_constants
  const float2 nden = p.nden, rcp = p.rcp, half_scale = p.half_scale;
  const float2 inv_px = dup(p.inv_px);
  uint32_t stage = 0, phase = 0;
  const uint32_t full0 = smem_u32(full_bar), empty0 = smem_u32(empty_bar), hdr0 = smem_u32(stage_hdr);
  for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {
    const int x0 = (tile % p.tiles_x) * kTX, y0 = (tile / p.tiles_x) * kTY;
    const int x = x0 + tx, y_base = y0 + tyg * kRows;
    const bool active = x < W && y_base < H;
    const int y_last = H - 1;
    // lattice taps along y of the thread's rows: staged row (i0 - i0_tile + k) of the block.  One lattice_axis per lane
    // (lanes 0..3: the thread's rows -- every lane of a warp has the same rows; lane 4: the tile's first row), shuffled
    float wy[kRows][4];
    int lat[kRows];
    float yf[kRows];
    bool same_cell = true;
    {
      const LatticeAxis mine = lattice_axis(lane < kRows ? min(y_base + lane, y_last) : y0, H, lh);
      const int i0_tile = __shfl_sync(0xffffffffu, mine.i0, kRows);
#pragma unroll
      for (int r = 0; r < kRows; ++r) {
        yf[r] = (float)min(y_base + r, y_last);
        const int i0 = __shfl_sync(0xffffffffu, mine.i0, r);
        lat[r] = min(max(i0 - i0_tile, 0), p.rx_rows - 4) * (2 * kTX) + tx;
#pragma unroll
        for (int k = 0; k < 4; ++k) wy[r][k] = __shfl_sync(0xffffffffu, mine.w[k], r);
        same_cell = same_cell && (lat[r] == lat[0]);
      }
    }
    const float xf = (float)min(x, W - 1);
    float acc[kRows];
#pragma unroll
    for (int r = 0; r < kRows; ++r) acc[r] = 0.f;
    if constexpr (WEIGHTED) zero_sums(sums_acc + tid, kConsumers, p.n_sums);

    // the frame loop, specialised on whether the thread's 4 rows read the same lattice rows (warp-uniform, true for all
    // but the few row groups that straddle a lattice cell boundary): no branch inside the coordinate arithmetic, so
    // the 4 pixels' dependent chains interleave
    auto frames = [&](auto same_tag) {
    constexpr bool SAME = decltype(same_tag)::value;
    for (int f = 0; f < T; ++f) {
      mbar_wait_addr(full0 + 8u * stage, phase);
      if (active) {
        const float* simg = reinterpret_cast<const float*>(stages + (size_t)stage * p.stage_bytes);
        const float* srx = simg + kImgBytesPadded / 4;
        const int4 org = lds_int4(hdr0 + 32u * stage);       // oy + 1, ox + 1, by_lo, by_n
        const int2 xr = lds_int2(hdr0 + 32u * stage + 16u);  // bx_lo, bx_n
        float2 R[SAME ? 1 : kRows][4];
#pragma unroll
        for (int r = 0; r < (SAME ? 1 : kRows); ++r)
#pragma unroll
          for (int k = 0; k < 4; ++k) R[r][k] = f2(srx[lat[r] + k * 2 * kTX], srx[lat[r] + (k * 2 + 1) * kTX]);
        float2 c[kRows], fl[kRows], frac[kRows];
#pragma unroll
        for (int r = 0; r < kRows; ++r) {
          const float2* Rr = R[SAME ? 0 : r];
          float2 s = pk_mul(dup(wy[r][0]), Rr[0]);
          s = pk_fma(dup(wy[r][1]), Rr[1], s);
          s = pk_fma(dup(wy[r][2]), Rr[2], s);
          s = pk_fma(dup(wy[r][3]), Rr[3], s);
          // Angstrom -> px, then pixel_grid + pixel_shifts (two roundings, like the reference)
          c[r] = pk_add(f2(yf[r], xf), pk_mul(s, inv_px));
          // grid_sample round trip: g = c / (0.5 n - 0.5) - 1 ; u = ((g + 1) / 2) (n - 1); the division as
          // q0 = c * rcp and one Newton step on the residual (correctly rounded, see Divisor)
          const float2 q0 = pk_mul(c[r], rcp);
          const float2 q = pk_fma(pk_fma(q0, nden, c[r]), rcp, q0);
          const float2 g = pk_add(q, dup(-1.0f));
          const float2 u = pk_mul(pk_add(g, dup(1.0f)), half_scale);
          fl[r] = f2(floorf(u.x), floorf(u.y));
          frac[r] = pk_fma(fl[r], dup(-1.0f), u);
        }
        // the 4 sampling points are vertically adjacent (same tap columns, consecutive tap rows: the shifts differ by
        // ~1e-3 px per row, so almost always) and their 7 x 4 taps lie inside the box and inside the image
        const int by0 = (int)fl[0].x - org.x, bx0 = (int)fl[0].y - org.y;
        bool stacked = (unsigned)(by0 - org.z) <= (unsigned)org.w && (unsigned)(bx0 - xr.x) <= (unsigned)xr.y;
#pragma unroll
        for (int r = 1; r < kRows; ++r) stacked = stacked && fl[r].x == fl[0].x + (float)r && fl[r].y == fl[0].y;
        float v[kRows];
        if (stacked) {
          // 7 rows of 4 taps serve all 4 pixels; rows (0,1), (2,3), (4,5) are kept as register pairs so that the x pass of
          // two tap rows is one packed instruction (the x weight enters as a scalar operand)
          const float* q = simg + by0 * kBoxW + bx0;
          float2 p01[4], p23[4], p45[4];
          float r6[4];
#pragma unroll
          for (int b = 0; b < 4; ++b) {
            p01[b] = f2(q[b], q[kBoxW + b]);
            p23[b] = f2(q[2 * kBoxW + b], q[3 * kBoxW + b]);
            p45[b] = f2(q[4 * kBoxW + b], q[5 * kBoxW + b]);
            r6[b] = q[6 * kBoxW + b];
          }
          float2 w[4];  // .x = weight along y, .y = weight along x
          // pixel 0: tap rows 0..3
          keys_weights2(frac[0], w);
          {
            float2 h01 = pk_mul(dup(w[0].y), p01[0]), h23 = pk_mul(dup(w[0].y), p23[0]);
#pragma unroll
            for (int b = 1; b < 4; ++b) {
              h01 = pk_fma(dup(w[b].y), p01[b], h01);
              h23 = pk_fma(dup(w[b].y), p23[b], h23);
            }
            v[0] = fmaf(w[3].x, h23.y, fmaf(w[2].x, h23.x, fmaf(w[1].x, h01.y, w[0].x * h01.x)));
          }
          // pixel 1: tap rows 1..4
          keys_weights2(frac[1], w);
          {
            float h1 = w[0].y * p01[0].y, h4 = w[0].y * p45[0].x;
            float2 h23 = pk_mul(dup(w[0].y), p23[0]);
#pragma unroll
            for (int b = 1; b < 4; ++b) {
              h1 = fmaf(w[b].y, p01[b].y, h1);
              h4 = fmaf(w[b].y, p45[b].x, h4);
              h23 = pk_fma(dup(w[b].y), p23[b], h23);
            }
            v[1] = fmaf(w[3].x, h4, fmaf(w[2].x, h23.y, fmaf(w[1].x, h23.x, w[0].x * h1)));
          }
          // pixel 2: tap rows 2..5
          keys_weights2(frac[2], w);
          {
            float2 h23 = pk_mul(dup(w[0].y), p23[0]), h45 = pk_mul(dup(w[0].y), p45[0]);
#pragma unroll
            for (int b = 1; b < 4; ++b) {
              h23 = pk_fma(dup(w[b].y), p23[b], h23);
              h45 = pk_fma(dup(w[b].y), p45[b], h45);
            }
            v[2] = fmaf(w[3].x, h45.y, fmaf(w[2].x, h45.x, fmaf(w[1].x, h23.y, w[0].x * h23.x)));
          }
          // pixel 3: tap rows 3..6
          keys_weights2(frac[3], w);
          {
            float h3 = w[0].y * p23[0].y, h6 = w[0].y * r6[0];
            float2 h45 = pk_mul(dup(w[0].y), p45[0]);
#pragma unroll
            for (int b = 1; b < 4; ++b) {
              h3 = fmaf(w[b].y, p23[b].y, h3);
              h6 = fmaf(w[b].y, r6[b], h6);
              h45 = pk_fma(dup(w[b].y), p45[b], h45);
            }
            v[3] = fmaf(w[3].x, h6, fmaf(w[2].x, h45.y, fmaf(w[1].x, h45.x, w[0].x * h3)));
          }
        } else {
          // rare: sampling points not stacked, taps outside the box (shift varying by more than the margin inside the
          // tile) or at the image border (border-clamped taps / zero outside): per pixel, from the box or from global memory
#pragma unroll
          for (int r = 0; r < kRows; ++r) {
            const int by = (int)fl[r].x - org.x, bx = (int)fl[r].y - org.y;
            if ((unsigned)(by - org.z) <= (unsigned)(org.w + kRows - 1) && (unsigned)(bx - xr.x) <= (unsigned)xr.y) {
              const float* q = simg + by * kBoxW + bx;
              float2 w[4];
              keys_weights2(frac[r], w);
              float h[4];
#pragma unroll
              for (int a = 0; a < 4; ++a)
                h[a] = fmaf(w[3].y, q[a * kBoxW + 3], fmaf(w[2].y, q[a * kBoxW + 2], fmaf(w[1].y, q[a * kBoxW + 1], w[0].y * q[a * kBoxW])));
              v[r] = fmaf(w[3].x, h[3], fmaf(w[2].x, h[2], fmaf(w[1].x, h[1], w[0].x * h[0])));
            } else {
              v[r] = gather_border(p.image + (size_t)f * H * W, H, W, c[r].x, c[r].y);
            }
          }
        }
#pragma unroll
        for (int r = 0; r < kRows; ++r) {
          float o = v[r];
          if (NORMALISE) o = (o - mean) * inv_std;
          if (WRITE_STACK && y_base + r < H) p.out_stack[((size_t)f * H + y_base + r) * W + x] = o;
          if (WRITE_SUM) acc[r] += o;
        }
        if constexpr (WEIGHTED) accumulate_sums(sums_acc + tid, kConsumers, p.weights, T, f, p.n_sums, v);
      }
      __syncwarp();
      if (lane == 0) mbar_arrive_addr(empty0 + 8u * stage);
      if (++stage == (uint32_t)p.n_stages) {
        stage = 0;
        phase ^= 1u;
      }
    }
    };
    if (same_cell) frames(BoolTag<true>{}); else frames(BoolTag<false>{});
    if (WRITE_SUM && active) {
#pragma unroll
      for (int r = 0; r < kRows; ++r) {
        if (y_base + r < H) {
          float* o = p.out_sum + (size_t)(y_base + r) * W + x;
          *o = p.accumulate_sum ? (*o + acc[r]) : acc[r];
        }
      }
    }
    if constexpr (WEIGHTED) if (active) store_sums(sums_acc + tid, kConsumers, p.n_sums, p.out_sums, H, W, x, y_base, H);
  }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// the driver's tensor-map encoder, looked up through the runtime (no link-time dependency on libcuda)
inline EncodeTiledFn encode_tiled() {
  static EncodeTiledFn fn = [] {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult status;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &status) != cudaSuccess ||
        status != cudaDriverEntryPointSuccess)
      ptr = nullptr;
    return (EncodeTiledFn)ptr;
  }();
  return fn;
}

// fp32 tensor (d2, d1, d0) contiguous, innermost d0; box (b2, b1, b0); out-of-bounds elements read as zero
inline bool make_map_3d(CUtensorMap* map, const float* base, uint64_t d0, uint64_t d1, uint64_t d2, uint32_t b0, uint32_t b1,
                        uint32_t b2) {
  EncodeTiledFn enc = encode_tiled();
  if (!enc) return false;
  const cuuint64_t dims[3] = {d0, d1, d2};
  const cuuint64_t strides[2] = {d0 * sizeof(float), d0 * d1 * sizeof(float)};
  const cuuint32_t box[3] = {b0, b1, b2};
  const cuuint32_t elem[3] = {1, 1, 1};
  // 64-byte L2 promotion: measured DRAM reads of the C2 warp 4.64 GB against 6.13 GB with none / 128 B and 6.62 GB with
  // 256 B (box rows are 192 bytes at arbitrary 16-byte offsets; same kernel time)
  return enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(base), dims, strides, box, elem,
             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_64B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// the coordinate-chain constants of Params, rounded exactly as the device code of warp_lattice_kernel rounds them
inline void fill_constants(Params& p) {
  const float dy = 0.5f * (float)p.H - 0.5f, dx = 0.5f * (float)p.W - 0.5f;  // both exact in fp32
  p.nden = make_float2(-dy, -dx);
  p.rcp = make_float2(1.0f / dy, 1.0f / dx);  // IEEE division == __frcp_rn
  p.half_scale = make_float2(0.5f * (float)(p.H - 1), 0.5f * (float)(p.W - 1));
  p.inv_px = 1.0f / p.pixel_spacing;
}

// lattice rows a tile needs: its kTY image rows span at most floor((kTY - 1) / cell) + 2 lattice cells (+ 3 taps)
inline int staged_lattice_rows(int h, int lh) {
  if (lh < 2) return 5;
  const double cell = (double)(h - 1) / (double)(lh - 1);  // image rows per lattice row
  return (int)((kTY - 1) / cell) + 6;  // one spare row against the fp32 rounding of the lattice coordinate
}

// the kernel serves this problem: 16-byte aligned rows and lattice cells tall enough for the staged lattice block
inline bool supported(const float* image, const float* rx, int t, int h, int w, int lh) {
  if (w % 4 != 0 || (reinterpret_cast<uintptr_t>(image) & 15) != 0 || (reinterpret_cast<uintptr_t>(rx) & 15) != 0) return false;
  if (h < kTY || w < kTX) return false;
  if (staged_lattice_rows(h, lh) > kRxRows) return false;
  if ((long)t * 2 > 0x7fffffffl) return false;
  return encode_tiled() != nullptr;
}

}  // namespace tma

// Second-generation shared-memory FFT core for power-of-two lengths (fast path).
//
// Differences to fft_core.cuh (which remains the generic / Bluestein engine):
//  * every thread owns exactly 16 complex values per pass (G butterflies of radix R, G*R = 16), so
//    the FIRST pass takes its inputs from registers (loaded straight from global memory by the
//    calling kernel) and the LAST pass leaves its outputs in registers (consumed by the caller:
//    argmax, coalesced global stores) -- no shared-memory staging at either end;
//  * passes run in place in ONE buffer (read all -> barrier -> write all), halving shared memory
//    and doubling the resident CTAs per SM;
//  * twiddles come from a factorised shared-memory table (W^m = hi[m >> 6] * lo[m & 63]); per
//    radix-16 butterfly only w^1, w^2, w^4, w^8 are looked up, the rest are products (<= 3 deep);
//  * all index arithmetic is compile-time strength-reduced.
#pragma once
#include "common.cuh"
#include "fft_core.cuh"

namespace fft2 {

using tmcfft::bitrev;
using tmcfft::pad_idx;
using tmcfft::padded_len;

constexpr int kThreads = 256;

template <int N>
struct Cfg {
  static_assert(N >= 256 && N <= 8192 && (N & (N - 1)) == 0, "fast path covers 256..8192");
  static constexpr int NB16 = N / 16;                                    // threads per sequence
  static constexpr int B = (kThreads / NB16) > 0 ? (kThreads / NB16) : 1;  // sequences per CTA pass
  static constexpr int TPS = NB16 < kThreads ? NB16 : kThreads;          // threads per sequence (<= 256)
  static constexpr int VPT = N / TPS;                                    // values per thread: 16 (32 for N = 8192)
  // sequence stride: padded length, nudged so that neighbouring sequences start 8 banks apart
  static constexpr int STRIDE = padded_len(N) + ((4 - (padded_len(N) & 15)) & 15);
  static constexpr int TW_HI = N / 64;
  static constexpr size_t smem_bytes = (size_t)(B * STRIDE + 64 + TW_HI) * sizeof(float2);
};

template <int N>
struct Smem {
  float2* data;   // B sequences, stride Cfg<N>::STRIDE
  float2* tw_lo;  // W_N^i, i < 64
  float2* tw_hi;  // W_N^(64 i), i < N/64
  __device__ explicit Smem(float2* base) : data(base), tw_lo(base + Cfg<N>::B * Cfg<N>::STRIDE), tw_hi(tw_lo + 64) {}
};

// fill the factorised twiddle tables from the global W_N^m table (or, stride s, from the W_{sN}^m table of a transform
// s times longer: W_N^m = W_{sN}^{s m}); caller syncs afterwards
template <int N>
__device__ __forceinline__ void load_twiddles(const Smem<N>& sm, const float2* __restrict__ tw, int stride = 1) {
  for (int i = threadIdx.x; i < 64 + Cfg<N>::TW_HI; i += kThreads)
    sm.tw_lo[i] = i < 64 ? __ldg(tw + stride * i) : __ldg(tw + stride * (i - 64) * 64);
}

template <int N>
__device__ __forceinline__ float2 twiddle(const Smem<N>& sm, int m) {  // m < N
  return cmul(sm.tw_hi[m >> 6], sm.tw_lo[m & 63]);
}

// v[r] *= w^r for r = 1..R-1 given the table index m of w (w = W_N^m, r*m < N guaranteed by the caller)
template <int N, int R>
__device__ __forceinline__ void apply_twiddles(const Smem<N>& sm, int m, float2* v) {
  if constexpr (R == 2) {
    v[1] = cmul(v[1], twiddle<N>(sm, m));
  } else if constexpr (R == 4) {
    const float2 w1 = twiddle<N>(sm, m), w2 = twiddle<N>(sm, 2 * m);
    v[1] = cmul(v[1], w1);
    v[2] = cmul(v[2], w2);
    v[3] = cmul(v[3], cmul(w1, w2));
  } else if constexpr (R == 8) {
    const float2 w1 = twiddle<N>(sm, m), w2 = twiddle<N>(sm, 2 * m), w4 = twiddle<N>(sm, 4 * m);
    const float2 w3 = cmul(w1, w2);
    v[1] = cmul(v[1], w1);
    v[2] = cmul(v[2], w2);
    v[3] = cmul(v[3], w3);
    v[4] = cmul(v[4], w4);
    v[5] = cmul(v[5], cmul(w4, w1));
    v[6] = cmul(v[6], cmul(w4, w2));
    v[7] = cmul(v[7], cmul(w4, w3));
  } else {
    static_assert(R == 16, "radix");
    const float2 w1 = twiddle<N>(sm, m), w2 = twiddle<N>(sm, 2 * m), w4 = twiddle<N>(sm, 4 * m), w8 = twiddle<N>(sm, 8 * m);
    const float2 w3 = cmul(w1, w2), w5 = cmul(w4, w1), w6 = cmul(w4, w2);
    const float2 w7 = cmul(w4, w3);
    v[1] = cmul(v[1], w1);
    v[2] = cmul(v[2], w2);
    v[3] = cmul(v[3], w3);
    v[4] = cmul(v[4], w4);
    v[5] = cmul(v[5], w5);
    v[6] = cmul(v[6], w6);
    v[7] = cmul(v[7], w7);
    v[8] = cmul(v[8], w8);
    v[9] = cmul(v[9], cmul(w8, w1));
    v[10] = cmul(v[10], cmul(w8, w2));
    v[11] = cmul(v[11], cmul(w8, w3));
    v[12] = cmul(v[12], cmul(w8, w4));
    v[13] = cmul(v[13], cmul(w8, w5));
    v[14] = cmul(v[14], cmul(w8, w6));
    v[15] = cmul(v[15], cmul(w8, w7));
  }
}

// radix of the pass that starts at sub-transform length NS
template <int N, int NS>
struct Radix {
  static constexpr int rem = N / NS;
  static constexpr int value = rem >= 16 ? 16 : rem;
};

// Geometry of one pass for thread (sequence-local index j in [0, TPS)):
// the thread owns G butterflies jb = j + g * TPS (g < G), each over inputs x[jb + r * NBR] (r < R),
// producing X[j0 + r * NS] with j0 = (jb / NS) * NS * R + jb % NS.
template <int N, int NS>
struct Pass {
  static constexpr int R = Radix<N, NS>::value;
  static constexpr int NBR = N / R;
  static constexpr int G = Cfg<N>::VPT / R;
  static constexpr int STEP = N / (NS * R);
  __device__ static __forceinline__ int in_index(int j, int g, int r) { return j + g * Cfg<N>::TPS + r * NBR; }
  __device__ static __forceinline__ int out_index(int j, int g, int r) {
    const int jb = j + g * Cfg<N>::TPS;
    return (jb / NS) * NS * R + (jb % NS) + r * NS;
  }
  // twiddle + butterflies on the VPT register values laid out v[g * R + r]
  __device__ static __forceinline__ void compute(const Smem<N>& sm, int j, float2* v) {
#pragma unroll
    for (int g = 0; g < G; ++g) {
      if constexpr (NS > 1) {
        const int k = (j + g * Cfg<N>::TPS) % NS;
        apply_twiddles<N, R>(sm, k * STEP, v + g * R);
      }
      tmcfft::fft_reg_ptr<R>(v + g * R);
    }
  }
  __device__ static __forceinline__ void load(const float2* __restrict__ seq, int j, float2* v) {
#pragma unroll
    for (int g = 0; g < G; ++g)
#pragma unroll
      for (int r = 0; r < R; ++r) v[g * R + r] = seq[pad_idx(in_index(j, g, r))];
  }
  __device__ static __forceinline__ void store(float2* __restrict__ seq, int j, const float2* v) {
#pragma unroll
    for (int g = 0; g < G; ++g)
#pragma unroll
      for (int r = 0; r < R; ++r) seq[pad_idx(out_index(j, g, r))] = v[g * R + bitrev<R>(r)];
  }
  // value of output slot (g, r) after compute()
  __device__ static __forceinline__ float2 result(const float2* v, int g, int r) { return v[g * R + bitrev<R>(r)]; }
};

template <int N>
struct Plan {
  static constexpr int R0 = Radix<N, 1>::value;
  static constexpr int NS1 = R0;
  static constexpr int R1 = Radix<N, NS1>::value;
  static constexpr int NS2 = NS1 * R1;
  static constexpr bool two_pass = NS2 >= N;
  static constexpr int R2 = two_pass ? 1 : Radix<N, NS2 < N ? NS2 : 1>::value;
  static constexpr int NS3 = two_pass ? N : NS2 * R2;
  static constexpr bool three_pass = !two_pass && NS3 >= N;
  static_assert(two_pass || three_pass || NS3 * Radix<N, NS3 < N ? NS3 : 1>::value >= N, "at most four passes");
  static constexpr int LAST_NS = two_pass ? NS1 : (three_pass ? NS2 : NS3);
  using First = Pass<N, 1>;
  using Last = Pass<N, LAST_NS>;
};

// Middle passes (everything between the first and the last), in place, for the calling thread's
// sequence `seq` and index j.  All threads of the CTA must call it (barriers inside).
template <int N>
__device__ __forceinline__ void middle_passes(const Smem<N>& sm, float2* seq, int j) {
  using P = Plan<N>;
  if constexpr (!P::two_pass) {
    float2 v[Cfg<N>::VPT];
    {
      using M1 = Pass<N, P::NS1>;
      M1::load(seq, j, v);
      M1::compute(sm, j, v);
      __syncthreads();
      M1::store(seq, j, v);
      __syncthreads();
    }
    if constexpr (!P::three_pass) {
      using M2 = Pass<N, P::NS2>;
      M2::load(seq, j, v);
      M2::compute(sm, j, v);
      __syncthreads();
      M2::store(seq, j, v);
      __syncthreads();
    }
  }
}

// Full transform with the first-pass inputs in registers (v[g*R0 + r] = x[First::in_index(j, g, r)])
// and the last-pass outputs left in registers (v[...] via Last::result / Last::out_index).
// `seq` = this thread's sequence buffer.  All threads of the CTA call it.
template <int N>
__device__ __forceinline__ void fft_regs_to_regs(const Smem<N>& sm, float2* seq, int j, float2* v) {
  using P = Plan<N>;
  P::First::compute(sm, j, v);
  P::First::store(seq, j, v);
  __syncthreads();
  middle_passes<N>(sm, seq, j);
  P::Last::load(seq, j, v);
  P::Last::compute(sm, j, v);
}

}  // namespace fft2

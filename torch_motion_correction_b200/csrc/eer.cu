// EER (Falcon electron-event list) frames -> electron counts per pixel, summed over frame fractions.
//
// A frame's stream is a sequence of codes read LSB-first: rle_bits bits `s` move the pixel cursor p by s; s == 2^rle_bits
// - 1 is an escape (no electron), any other s puts an electron at p and is followed by sub_bits sub-pixel bits (skipped:
// 4K rendering) and p += 1.  The frame ends at the first code after which p == h * w.
//
// One CTA per frame, one chunk of the bit stream per thread.  A code begins within L = rle_bits + sub_bits bits of any
// chunk's start, and every code length is a multiple of g = gcd(rle_bits, L), so with chunk lengths that are multiples of
// g a chunk can be entered at one of L / g offsets ("tracks").
//   pass 1  every thread decodes its chunk from each track and records where it leaves (the next chunk's track), how far
//           it moves p, and whether its last code was an escape; tracks are run against track 0 and stop when they reach
//           one of its code boundaries (the codes resynchronise within a few codes);
//   chain   thread 0 walks the chunk tables from chunk 0 / track 0: every chunk's true entry and starting pixel;
//   check   thread 0 decodes the chunk holding the end of the frame: a frame is well formed iff a code there lands on
//           p == h * w exactly and lies inside the stream;
//   pass 2  well-formed frames only: every thread decodes its chunk once more from its true entry and adds its electrons.
// The decoder never depends on the data for where it reads: every word load lies between the frame's start (rounded down
// to 4 bytes) and its end including the 8 zero bytes of padding, and a count is written only for p < h * w.
#include "common.cuh"

namespace {

// 256 threads, five CTAs per SM; 1024-thread CTAs (one per SM, fewer counts planes in flight) measured 1.9x slower: the
// serial chain and check of thread 0 grow with the chunk count while the SM has no other CTA to run (DESIGN §3)
constexpr int kEerThreads = 256;
constexpr int kEerMaxBits = 32;                // rle_bits + sub_bits: a code and its refill fit one 64-bit buffer
constexpr long long kEerMaxFrameBytes = 1LL << 27;  // bit positions (plus L) stay in int32

// LSB-first reader of one frame's bit stream: `buf` holds the `nb` bits from bit `pos` on
struct BitReader {
  const unsigned* words;  // payload as 32-bit words (the payload buffer is 4-byte aligned)
  long long base;         // bit index of the frame's first bit inside the payload
  unsigned long long buf;
  long long wi;
  int nb, pos;

  __device__ __forceinline__ void seek(int p, int max_pos) {
    pos = p;
    const long long abs = base + min(p, max_pos);  // clamped: a seek past the stream still loads inside the padding
    wi = abs >> 5;
    buf = (unsigned long long)(__ldg(words + wi) >> (abs & 31));
    nb = 32 - (int)(abs & 31);
    ++wi;
  }
  // one code at pos (< stream length): its rle field s; the reader moves past the code
  __device__ __forceinline__ unsigned next(int rle_bits, int code_bits, unsigned escape) {
    if (nb < code_bits) {
      buf |= (unsigned long long)__ldg(words + wi) << nb;
      ++wi;
      nb += 32;
    }
    const unsigned s = (unsigned)buf & escape;
    const int len = s == escape ? rle_bits : code_bits;
    buf >>= len;
    nb -= len;
    pos += len;
    return s;
  }
};

__device__ __forceinline__ int gcd_int(int a, int b) {
  while (b) {
    const int t = a % b;
    a = b;
    b = t;
  }
  return a;
}

__global__ void __launch_bounds__(kEerThreads)
eer_render_kernel(const unsigned char* __restrict__ payload, long long payload_bytes,
                  const long long* __restrict__ frame_offsets, int h, int w, int rle_bits, int sub_bits,
                  int frames_per_fraction, int count_bytes, unsigned* __restrict__ counts, int* __restrict__ status) {
  extern __shared__ unsigned char smem[];
  const int f = blockIdx.x;
  const int tid = threadIdx.x;
  const int L = rle_bits + sub_bits;
  const int g = gcd_int(rle_bits, L);
  const int ntracks = L / g;
  const unsigned escape = (1u << rle_bits) - 1u;
  const long long npix = (long long)h * w;

  unsigned* adv_tab = reinterpret_cast<unsigned*>(smem);                       // [ntracks][T] pixel advance (saturated)
  unsigned char* meta_tab = smem + sizeof(unsigned) * ntracks * kEerThreads;  // [ntracks][T] exit track | escape << 7
  int* p_start = reinterpret_cast<int*>(smem + ((5 * ntracks * kEerThreads + 3) & ~3));  // [T] starting pixel
  unsigned char* entry = reinterpret_cast<unsigned char*>(p_start + kEerThreads);     // [T] entry track
  __shared__ int s_nactive, s_ok;

  const long long lo = frame_offsets[f], hi = frame_offsets[f + 1];
  if (lo < 0 || hi > payload_bytes || hi - lo < 8 || hi - lo - 8 > kEerMaxFrameBytes) {
    if (tid == 0) status[f] = 2;  // the offset table does not describe a frame inside the payload
    return;
  }
  const int nbits = (int)(8 * (hi - lo - 8));
  // chunk length: a multiple of g and >= L, so that every chunk but the last holds the start of a code
  int C = max((nbits + kEerThreads - 1) / kEerThreads, L);
  C = (C + g - 1) / g * g;
  const int nchunks = (nbits + C - 1) / C;

  BitReader a, b;
  a.words = b.words = reinterpret_cast<const unsigned*>(payload);
  a.base = b.base = 8 * lo;
  const int cs = tid * C, ce = min(cs + C, nbits);

  // ---- pass 1: the chunk's map track -> (exit track, pixel advance, last code escape) ----
  if (tid < nchunks) {
    a.seek(cs, nbits);
    unsigned long long adv0 = 0;
    bool esc0 = false;
    while (a.pos < ce) {
      const unsigned s = a.next(rle_bits, L, escape);
      esc0 = s == escape;
      adv0 += s + (esc0 ? 0u : 1u);
    }
    const int exit0 = (a.pos - ce) / g;  // < ntracks for every chunk but the last, whose exit nobody reads
    adv_tab[tid] = (unsigned)min(adv0, 0xffffffffull);
    meta_tab[tid] = (unsigned char)(min(exit0, ntracks - 1) | (esc0 ? 0x80 : 0));
    for (int j = 1; j < ntracks; ++j) {
      unsigned long long aa = 0, ab = 0;
      bool escb = false, merged = false;
      const int start = cs + j * g;
      if (start < ce) {
        a.seek(cs, nbits);
        b.seek(start, nbits);
        while (b.pos < ce) {
          if (a.pos == b.pos) {  // same code boundary: the rest of the chunk decodes as track 0 does
            merged = true;
            break;
          }
          if (a.pos < b.pos) {
            const unsigned s = a.next(rle_bits, L, escape);
            aa += s + (s == escape ? 0u : 1u);
          } else {
            const unsigned s = b.next(rle_bits, L, escape);
            escb = s == escape;
            ab += s + (escb ? 0u : 1u);
          }
        }
      } else {
        b.pos = start;
      }
      unsigned long long adv;
      int ex;
      bool esc;
      if (merged) {
        adv = adv0 - aa + ab;
        ex = exit0;
        esc = esc0;
      } else {
        adv = ab;
        ex = (b.pos - ce) / g;
        esc = escb;
      }
      adv_tab[j * kEerThreads + tid] = (unsigned)min(adv, 0xffffffffull);
      meta_tab[j * kEerThreads + tid] = (unsigned char)(min(max(ex, 0), ntracks - 1) | (esc ? 0x80 : 0));
    }
  }
  __syncthreads();

  // ---- chain: true entry and starting pixel of every chunk up to the one holding the end of the frame ----
  if (tid == 0) {
    long long p = 0;
    int e = 0, k = 0;
    bool prev_esc = false;
    for (; k < nchunks; ++k) {
      // p only grows and every chunk moves it by >= 1: once a chunk starts past the end (or at it right after an
      // escape that landed there) so do all later ones
      if (!(p < npix || (p == npix && !prev_esc))) break;
      p_start[k] = (int)p;
      entry[k] = (unsigned char)e;
      const int idx = e * kEerThreads + k;
      p = min(p + (long long)adv_tab[idx], npix + 1);
      e = meta_tab[idx] & 0x7f;
      prev_esc = (meta_tab[idx] & 0x80) != 0;
    }
    s_nactive = k;
    // ---- check: the last active chunk must end the frame exactly, with its code inside the stream ----
    int ok = 0;
    if (k > 0) {
      const int kl = k - 1;
      const int lim = min(kl * C + C, nbits);
      long long q = p_start[kl];
      a.seek(kl * C + entry[kl] * g, nbits);
      while (a.pos < lim) {
        if (a.pos + rle_bits > nbits) break;  // ran out of bytes
        const unsigned s = a.next(rle_bits, L, escape);
        q += s;
        if (q >= npix) {
          ok = q == npix;
          break;
        }
        if (s != escape) ++q;
      }
    }
    s_ok = ok;
    status[f] = ok ? 0 : 1;
  }
  __syncthreads();
  if (!s_ok || tid >= s_nactive) return;

  // ---- pass 2: the electrons of the chunk ----
  const long long frac_base = (long long)(f / frames_per_fraction) * npix * count_bytes;
  long long q = p_start[tid];
  a.seek(cs + entry[tid] * g, nbits);
  while (a.pos < ce) {
    const unsigned s = a.next(rle_bits, L, escape);
    q += s;
    if (q >= npix) break;  // == npix: the end of the frame (checked above)
    if (s != escape) {
      const long long byte = frac_base + q * count_bytes;
      atomicAdd(counts + (byte >> 2), 1u << (8 * (int)(byte & 3)));  // a fraction's count <= F: no carry out of the pixel
      ++q;
    }
  }
}

size_t eer_smem_bytes(int rle_bits, int sub_bits) {
  const int L = rle_bits + sub_bits;
  int a = rle_bits, b = L;
  while (b) {
    const int t = a % b;
    a = b;
    b = t;
  }
  const int ntracks = L / a;
  return (((size_t)5 * ntracks * kEerThreads + 3) & ~(size_t)3) + (size_t)5 * kEerThreads;  // <= 42 KB
}

}  // namespace

// EER frames -> counts (n_frames / F, h, w) of uint8 (count_bytes 1) or uint16 (2); see include/tmc_b200.h
TMC_API int tmc_eer_render(const void* payload, long payload_bytes, const long long* frame_offsets, int n_frames, int h,
                           int w, int rle_bits, int sub_bits, int frames_per_fraction, int count_bytes, void* counts,
                           int* status, cudaStream_t stream) {
  TMC_CHECK_ARG(payload && frame_offsets && counts && status, "eer_render: null pointer");
  TMC_CHECK_ARG((reinterpret_cast<uintptr_t>(payload) & 3) == 0 && (reinterpret_cast<uintptr_t>(counts) & 3) == 0,
                "eer_render: payload and counts must be 4-byte aligned");
  TMC_CHECK_ARG(payload_bytes >= 8, "eer_render: payload of %ld bytes", payload_bytes);
  TMC_CHECK_ARG(h >= 1 && w >= 1 && (long long)h * w < (1LL << 31) - 1, "eer_render: bad frame size (%d, %d)", h, w);
  TMC_CHECK_ARG(rle_bits >= 1 && rle_bits <= 16 && sub_bits >= 0 && rle_bits + sub_bits <= kEerMaxBits,
                "eer_render: rle_bits %d / sub_bits %d: need 1 <= rle_bits <= 16 and rle_bits + sub_bits <= %d", rle_bits,
                sub_bits, kEerMaxBits);
  TMC_CHECK_ARG(count_bytes == 1 || count_bytes == 2, "eer_render: count_bytes must be 1 or 2, got %d", count_bytes);
  TMC_CHECK_ARG(frames_per_fraction >= 1 && frames_per_fraction <= (count_bytes == 1 ? 255 : 65535),
                "eer_render: %d frames per fraction overflow %d-byte counts", frames_per_fraction, count_bytes);
  TMC_CHECK_ARG(n_frames >= frames_per_fraction && n_frames % frames_per_fraction == 0,
                "eer_render: %d frames are not a whole number of fractions of %d", n_frames, frames_per_fraction);
  const long long n_fractions = n_frames / frames_per_fraction;
  const long long bytes = n_fractions * h * w * count_bytes;
  TMC_CUDA(cudaMemsetAsync(counts, 0, (size_t)((bytes + 3) & ~3LL), stream));
  const size_t smem = eer_smem_bytes(rle_bits, sub_bits);
  TMC_TIMED("eer_render_kernel", stream, eer_render_kernel<<<n_frames, kEerThreads, smem, stream>>>(
      static_cast<const unsigned char*>(payload), payload_bytes, frame_offsets, h, w, rle_bits, sub_bits,
      frames_per_fraction, count_bytes, static_cast<unsigned*>(counts), status));
  TMC_CHECK_LAUNCH("tmc_eer_render");
  return TMC_OK;
}

// TIFF LZW strips (compression 5, TIFF 6.0 §13) -> rows of a uint8 / uint16 stack, with Predictor 2 undone.
//
// A strip's stream is a sequence of codes packed MSB-first.  A Clear code (256) starts a segment, EOI (257) ends the
// stream; inside a segment code k (0-based, the Clear that opened it not counted) is 9 bits for k < 254, 10 for k < 766,
// 11 for k < 1790 and 12 after that ("early change"), so a code's position follows from its index alone.  Code k >= 1
// defines entry 257 + k; the entry created by code j + 1 (entry 258 + j) is the output of code j plus the first byte of
// code j + 1, i.e. the output bytes [off(j), off(j) + len(j) + 1).  A code c >= 258 therefore copies earlier output of
// its own segment, as in an LZ77 decoder, and no string storage is needed: only the output offset of every code.
//
//   scan     one CTA per strip walks its segments: all threads test the codes of a segment at once for the first
//            Clear / EOI / invalid code, thread 0 chains the segments.  The strip is cut into units at Clear codes, each
//            unit but the last holding >= kUnitCodes codes; the walk stops early once the strip's rows are certainly full
//            (every data code yields >= 1 byte), so codes after the rows are never read;
//   lengths  one warp per unit that is not its strip's last: the number of bytes it decodes to;
//   decode   one warp per unit: its output offset is the sum of its strip's earlier unit lengths; 32 codes at a time it
//            resolves their lengths (pointer jumping over in-batch references), their offsets (warp scan) and then the
//            batch's output bytes, one byte per lane, chasing in-batch references down to a literal or to output written
//            by an earlier batch.  The strip's last unit sets the status and zero-fills rows a short stream leaves empty;
//   predict  Predictor 2 only: a prefix sum along every row, modulo 2^8 or 2^16.
//
// Malformed (status 1): a code names an entry that is not yet defined (the first code of a segment must be a literal),
// a segment defines entry 4096 without a Clear, or the stream ends (EOI, or a code running past the strip's bytes)
// before the strip's rows are filled.  Like libtiff, a strip without a leading Clear or a trailing EOI decodes normally
// and codes after the rows are full are ignored.  Status 2: the offset tables do not describe a strip inside the payload
// and the stack.
//
// Memory safety whatever the data: a code is loaded only when it lies inside its strip's bytes, so every payload load
// is inside [strip_offsets[s], strip_offsets[s + 1]) (the last code's 3-byte window reaches at most 2 bytes into the 8
// bytes of padding); a unit record is written only inside the strip's own slot range; every output store is inside
// [out_offsets[s], out_offsets[s + 1]), and every output load is at an earlier position of the same strip that the same
// warp has already written.
#include "common.cuh"

namespace {

constexpr int kScanThreads = 256;
constexpr int kScanPerThread = 4;               // codes each scan thread tests per round
constexpr int kSegCodes = 3840;                 // indices 0..3838 may be data codes (entries up to 4095); 3839 must end
constexpr int kUnitCodes = 512;                 // a unit closes at the first Clear after this many codes ...
constexpr long long kUnitBits = 9LL * kUnitCodes;  // ... so it spans at least this many bits
constexpr int kWarpsPerCta = 2;                 // decode / lengths: each warp keeps a kSegCodes + 1 offset table
constexpr int kPadBytes = 8;

// bit offset of code k inside its segment, and its width
__device__ __forceinline__ long long code_bits_before(int k) {
  return 9LL * min(k, 254) + 10LL * min(max(k - 254, 0), 512) + 11LL * min(max(k - 766, 0), 1024) +
         12LL * max(k - 1790, 0);
}
__device__ __forceinline__ int code_width(int k) { return k < 254 ? 9 : k < 766 ? 10 : k < 1790 ? 11 : 12; }

// the code of `width` bits at bit `pos` (MSB-first); the caller checks pos + width <= the strip's bits
__device__ __forceinline__ int read_code(const unsigned char* __restrict__ strip, long long pos, int width) {
  const long long b = pos >> 3;
  const unsigned v = ((unsigned)__ldg(strip + b) << 16) | ((unsigned)__ldg(strip + b + 1) << 8) | __ldg(strip + b + 2);
  return (int)((v >> (24 - (int)(pos & 7) - width)) & ((1u << width) - 1u));
}

// first unit slot of strip s: slots [slot_base(s), slot_base(s + 1)) hold at least floor(bits / kUnitBits) + 1 units
__device__ __forceinline__ long long slot_base(long long payload_offset, int s) {
  return (8 * payload_offset) / kUnitBits + s;
}

__device__ __forceinline__ long long strip_bits(const long long* strip_offsets, int s) {
  return 8 * (strip_offsets[s + 1] - strip_offsets[s] - kPadBytes);
}

struct Strip {
  long long lo, bits, out_lo, out_bytes;
  bool ok;
};

__device__ __forceinline__ Strip strip_of(const long long* strip_offsets, const long long* out_offsets, int s,
                                          long long payload_bytes, long long out_bytes) {
  Strip st;
  st.lo = strip_offsets[s];
  const long long hi = strip_offsets[s + 1];
  st.out_lo = out_offsets[s];
  const long long out_hi = out_offsets[s + 1];
  st.ok = st.lo >= 0 && hi <= payload_bytes && hi - st.lo >= kPadBytes && st.out_lo >= 0 && out_hi <= out_bytes &&
          out_hi >= st.out_lo && out_hi - st.out_lo < (1LL << 31);
  st.bits = st.ok ? 8 * (hi - st.lo - kPadBytes) : 0;
  st.out_bytes = st.ok ? out_hi - st.out_lo : 0;
  return st;
}

// kinds of the code at segment index k
enum { kData = 0, kClear = 1, kStop = 2 };

__device__ __forceinline__ int classify(int c, int k) {
  if (c == 256) return kClear;
  if (c == 257 || k >= kSegCodes - 1) return kStop;  // EOI, or a data code that would define entry 4096
  if (c < 256) return kData;
  return c - 258 <= k - 1 ? kData : kStop;         // entry 258 + j is defined once code j + 1 has been read
}

__global__ void __launch_bounds__(kScanThreads)
lzw_scan_kernel(const unsigned char* __restrict__ payload, long long payload_bytes,
                const long long* __restrict__ strip_offsets, const long long* __restrict__ out_offsets,
                long long out_bytes, int n_strips, long long* __restrict__ unit_bits, int* __restrict__ unit_strip,
                int* __restrict__ status, unsigned char* __restrict__ out) {
  const int s = blockIdx.x;
  const int tid = threadIdx.x;
  __shared__ int s_first;      // 4 k + kind of the first Clear / stop code of the segment, 4 kSegCodes if none
  __shared__ int s_kmax;       // codes of the segment worth testing
  __shared__ long long s_seg;  // bit where the current segment starts; -1: the walk is over
  const Strip st = strip_of(strip_offsets, out_offsets, s, payload_bytes, out_bytes);
  const long long base = slot_base(strip_offsets[s], s);
  const long long slots = st.ok ? slot_base(strip_offsets[s + 1], s + 1) - base : 0;
  if (!st.ok) {
    if (tid == 0) status[s] = 2;
    return;
  }
  const unsigned char* strip = payload + st.lo;
  // thread 0's chain state
  long long unit_start = 0, data = 0;
  int unit_codes = 0, nunits = 0;
  bool full = false;
  if (tid == 0) s_seg = 0;
  __syncthreads();
  while (true) {
    const long long seg = s_seg;
    if (seg < 0) break;
    if (tid == 0) {
      s_first = kSegCodes * 4;
      // codes beyond this many data codes are not needed: the rows are full before them
      s_kmax = (int)min((long long)kSegCodes, st.out_bytes - data);
    }
    __syncthreads();
    const int kmax = s_kmax;
    for (int r = 0; r < kmax; r += kScanThreads * kScanPerThread) {
      int best = kSegCodes, kind = kData;
#pragma unroll
      for (int i = 0; i < kScanPerThread; ++i) {
        const int k = r + i * kScanThreads + tid;
        if (k >= kmax) break;
        const long long pos = seg + code_bits_before(k);
        const int width = code_width(k);
        const int kd = pos + width > st.bits ? kStop : classify(read_code(strip, pos, width), k);
        if (kd != kData && k < best) {
          best = k;
          kind = kd;
        }
      }
      if (best < kSegCodes) atomicMin(&s_first, best * 4 + kind);
      __syncthreads();
      const int found = s_first;
      __syncthreads();
      if (found < kSegCodes * 4) break;
    }
    if (tid == 0) {
      const int f = s_first;
      long long next = -1, end = -1;
      if (f < kSegCodes * 4) {
        const int k = f >> 2, kind = f & 3;
        data += k;
        unit_codes += k + 1;
        if (kind == kClear) {
          next = seg + code_bits_before(k) + code_width(k);
          if (unit_codes >= kUnitCodes) {  // close the unit after this Clear
            unit_bits[2 * (base + nunits)] = unit_start;
            unit_bits[2 * (base + nunits) + 1] = next;
            unit_strip[base + nunits] = s;
            ++nunits;
            unit_start = next;
            unit_codes = 0;
          }
        } else {
          end = seg + code_bits_before(k);  // EOI, an invalid code, or the end of the bytes
        }
      } else {  // no stop before kmax: the rows are full after code kmax - 1
        data += kmax;
        unit_codes += kmax;
        end = seg + code_bits_before(kmax);
        full = true;
      }
      if (next < 0) {
        if (end > unit_start || nunits == 0) {
          unit_bits[2 * (base + nunits)] = unit_start;
          unit_bits[2 * (base + nunits) + 1] = end;
          unit_strip[base + nunits] = s;
          ++nunits;
        }
        // a strip that decodes to nothing has no unit that could report it short
        status[s] = (full || data >= st.out_bytes) ? 0 : (data == 0 ? 1 : 0);
        s_first = nunits;  // hand the unit count to every thread
      }
      s_seg = next;
    }
    __syncthreads();
  }
  // the walk is over: s_first holds the unit count
  const int nu = s_first;
  for (long long u = nu + tid; u < slots; u += kScanThreads) unit_strip[base + u] = -1;
  if (status[s] == 1) {  // no data code at all: the rows are zeros
    for (long long i = tid; i < st.out_bytes; i += kScanThreads) out[st.out_lo + i] = 0;
  }
}

// Walk one unit 32 codes at a time.  DECODE: also write its bytes at out + dst (dst: the strip-relative offset of the
// unit's first byte) up to the strip's end.  Returns the number of bytes the unit decodes to (DECODE: it stops counting
// once the strip is full).
template <bool DECODE>
__device__ long long walk_unit(const unsigned char* __restrict__ strip, long long bits, long long start, long long end,
                               unsigned char* __restrict__ out_strip, long long dst, long long strip_bytes, int* off,
                               int* codes) {
  const int lane = threadIdx.x & 31;
  long long seg = start;  // bit of the current segment's first code
  long long seg_out = 0;  // unit-relative output offset of the current segment
  int kb = 0;             // segment index of the batch's first code
  if (lane == 0) off[0] = 0;
  __syncwarp();
  while (true) {
    const int k = kb + lane;
    const long long pos = seg + code_bits_before(k);
    const int width = code_width(k);
    const bool active = k < kSegCodes && pos >= 0 && pos < end && pos + width <= bits;
    const int c = active ? read_code(strip, pos, width) : -1;
    const unsigned active_mask = __ballot_sync(0xffffffffu, active);
    const unsigned stop_mask = __ballot_sync(0xffffffffu, !active || c == 256);
    const int n = stop_mask ? __ffs(stop_mask) - 1 : 32;  // data codes of this batch
    const bool is_data = lane < n;
    // lengths: literal 1, else len(j) + 1 with j = c - 258 (the scan checked 0 <= j < k; clamped all the same)
    const bool literal = c < 256 || k == 0;
    const int j = is_data && !literal ? min(max(c - 258, 0), k - 1) : -1;
    int ptr = j >= kb ? j - kb : -1;
    int len = !is_data ? 0 : literal ? 1 : ptr >= 0 ? 1 : off[j + 1] - off[j] + 1;
#pragma unroll
    for (int d = 0; d < 5; ++d) {
      const int src = ptr >= 0 ? ptr : lane;
      const int pl = __shfl_sync(0xffffffffu, len, src);
      const int pp = __shfl_sync(0xffffffffu, ptr, src);
      if (ptr >= 0) {
        len += pl;
        ptr = pp;
      }
    }
    int incl = len;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int v = __shfl_up_sync(0xffffffffu, incl, d);
      if (lane >= d) incl += v;
    }
    const int base_off = off[kb];
    if (is_data) {
      off[k + 1] = base_off + incl;
      if (DECODE) codes[lane] = c;
    }
    __syncwarp();
    const int batch_end = off[kb + n];
    if (DECODE && n > 0) {
      // one output byte per lane; q is segment-relative
      const long long seg_dst = dst + seg_out;
      const long long limit = min((long long)batch_end, strip_bytes - seg_dst);
      for (long long q = base_off + lane; q < limit; q += 32) {
        const int qi = (int)q;
        // the batch code holding byte q: the last i with off[kb + i] <= q
        int lo = 0, hi = n - 1;
        while (lo < hi) {
          const int mid = (lo + hi + 1) >> 1;
          if (off[kb + mid] <= qi) lo = mid; else hi = mid - 1;
        }
        int kk = kb + lo, p = qi - off[kk];
        unsigned char byte;
        while (true) {
          const int cc = codes[kk - kb];
          if (cc < 256 || kk == 0) {
            byte = (unsigned char)cc;
            break;
          }
          const int jj = min(max(cc - 258, 0), kk - 1);
          if (p < off[jj + 1] - off[jj]) {      // inside the output of code jj
            if (jj < kb) {
              byte = out_strip[seg_dst + off[jj] + p];
              break;
            }
            kk = jj;
          } else {                              // the first byte of code jj + 1
            if (jj + 1 < kb) {
              byte = out_strip[seg_dst + off[jj + 1]];
              break;
            }
            kk = jj + 1;
            p = 0;
          }
        }
        out_strip[seg_dst + q] = byte;
      }
      __syncwarp();
      if (seg_dst + batch_end >= strip_bytes) return seg_out + batch_end;  // the strip is full
    }
    if (n < 32 && ((active_mask >> n) & 1u)) {  // a Clear: the next segment starts after it
      const long long cpos = __shfl_sync(0xffffffffu, pos, n);
      const int cw = __shfl_sync(0xffffffffu, width, n);
      seg = cpos + cw;
      seg_out += batch_end;
      kb = 0;
      __syncwarp();
      if (lane == 0) off[0] = 0;
      __syncwarp();
    } else if (n < 32) {
      return seg_out + batch_end;  // the unit ends inside this batch
    } else {
      kb += 32;
    }
  }
}

__global__ void __launch_bounds__(32 * kWarpsPerCta)
lzw_lengths_kernel(const unsigned char* __restrict__ payload, const long long* __restrict__ strip_offsets,
                   long long n_slots, const long long* __restrict__ unit_bits, const int* __restrict__ unit_strip,
                   long long* __restrict__ unit_len) {
  extern __shared__ int lzw_smem[];
  const int warp = threadIdx.x >> 5;
  const long long u = (long long)blockIdx.x * kWarpsPerCta + warp;
  if (u >= n_slots) return;
  const int s = unit_strip[u];
  if (s < 0) return;
  // a strip's last unit needs no length (nothing follows it): it is computed by the decode
  if (u + 1 < n_slots && unit_strip[u + 1] != s) return;
  if (u + 1 == n_slots) return;
  int* off = lzw_smem + warp * (kSegCodes + 1 + 32);
  const long long len = walk_unit<false>(payload + strip_offsets[s], strip_bits(strip_offsets, s), unit_bits[2 * u],
                                         unit_bits[2 * u + 1], nullptr, 0, 0, off, off + kSegCodes + 1);
  if ((threadIdx.x & 31) == 0) unit_len[u] = len;
}

__global__ void __launch_bounds__(32 * kWarpsPerCta)
lzw_decode_kernel(const unsigned char* __restrict__ payload, const long long* __restrict__ strip_offsets,
                  const long long* __restrict__ out_offsets, long long n_slots, const long long* __restrict__ unit_bits,
                  const int* __restrict__ unit_strip, const long long* __restrict__ unit_len,
                  unsigned char* __restrict__ out, int* __restrict__ status) {
  extern __shared__ int lzw_smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long u = (long long)blockIdx.x * kWarpsPerCta + warp;
  if (u >= n_slots) return;
  const int s = unit_strip[u];
  if (s < 0) return;
  const long long first = slot_base(strip_offsets[s], s);
  const long long strip_bytes = out_offsets[s + 1] - out_offsets[s];
  long long dst = 0;
  for (long long v = first + lane; v < u; v += 32) dst += min(max(unit_len[v], 0LL), 1LL << 40);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) dst += __shfl_xor_sync(0xffffffffu, dst, o);
  const bool last = u + 1 == n_slots || unit_strip[u + 1] != s;
  if (dst >= strip_bytes && !last) return;
  unsigned char* out_strip = out + out_offsets[s];
  int* off = lzw_smem + warp * (kSegCodes + 1 + 32);
  long long got = 0;
  if (dst < strip_bytes)
    got = walk_unit<true>(payload + strip_offsets[s], strip_bits(strip_offsets, s), unit_bits[2 * u],
                          unit_bits[2 * u + 1], out_strip, dst, strip_bytes, off, off + kSegCodes + 1);
  if (last && status[s] == 0 && dst + got < strip_bytes) {  // the stream ended before the rows were full
    for (long long i = max(dst + got, 0LL) + lane; i < strip_bytes; i += 32) out_strip[i] = 0;
    if (lane == 0) status[s] = 1;
  }
}

// Predictor 2: every row's samples become their running sum modulo 2^(8 sizeof(T)); one warp per row, 8 samples per
// lane per step
template <typename T>
__global__ void __launch_bounds__(256) lzw_predict_kernel(T* __restrict__ stack, long long n_rows, int w) {
  const int lane = threadIdx.x & 31;
  const long long warps = (long long)gridDim.x * (blockDim.x >> 5);
  for (long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); row < n_rows; row += warps) {
    T* r = stack + row * w;
    unsigned carry = 0;
    for (int x0 = 0; x0 < w; x0 += 256) {
      const int x = x0 + lane * 8;
      unsigned v[8];
      unsigned sum = 0;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        v[i] = x + i < w ? (unsigned)r[x + i] : 0u;
        sum += v[i];
        v[i] = sum;
      }
      unsigned incl = sum;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const unsigned t = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += t;
      }
      const unsigned before = carry + incl - sum;
#pragma unroll
      for (int i = 0; i < 8; ++i)
        if (x + i < w) r[x + i] = (T)(before + v[i]);
      carry += __shfl_sync(0xffffffffu, incl, 31);
    }
  }
}

long long lzw_slots(long long payload_bytes, int n_strips) { return (8 * payload_bytes) / kUnitBits + n_strips + 1; }

size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }

}  // namespace

// workspace bytes of tmc_tiff_lzw_decode for a payload of payload_bytes holding n_strips strips
TMC_API long tmc_tiff_lzw_workspace_bytes(long payload_bytes, int n_strips) {
  if (payload_bytes < 0 || n_strips < 0) return -1;
  const long long slots = lzw_slots(payload_bytes, n_strips);
  return (long)(align256(slots * 16) + align256(slots * 8) + align256(slots * 4));
}

// LZW strips -> (n_rows, w) samples of sample_bytes (1 or 2) bytes; see include/tmc_b200.h
TMC_API int tmc_tiff_lzw_decode(const void* payload, long payload_bytes, const long long* strip_offsets,
                                const long long* out_offsets, int n_strips, long n_rows, int w, int sample_bytes,
                                int predictor, void* out, void* workspace, long workspace_bytes, int* status,
                                cudaStream_t stream) {
  TMC_CHECK_ARG(payload && strip_offsets && out_offsets && out && workspace && status, "tiff_lzw_decode: null pointer");
  TMC_CHECK_ARG(payload_bytes >= kPadBytes, "tiff_lzw_decode: payload of %ld bytes", payload_bytes);
  TMC_CHECK_ARG(n_strips >= 1 && n_rows >= 1 && w >= 1, "tiff_lzw_decode: %d strips of a (%ld, %d) stack", n_strips,
                n_rows, w);
  TMC_CHECK_ARG(sample_bytes == 1 || sample_bytes == 2, "tiff_lzw_decode: sample_bytes must be 1 or 2, got %d",
                sample_bytes);
  TMC_CHECK_ARG(predictor == 1 || predictor == 2, "tiff_lzw_decode: predictor must be 1 or 2, got %d", predictor);
  TMC_CHECK_ARG(!(reinterpret_cast<uintptr_t>(out) & (sample_bytes - 1)), "tiff_lzw_decode: out is not aligned");
  const long need = tmc_tiff_lzw_workspace_bytes(payload_bytes, n_strips);
  TMC_CHECK_ARG(workspace_bytes >= need, "tiff_lzw_decode: workspace of %ld bytes, need %ld", workspace_bytes, need);
  const long long slots = lzw_slots(payload_bytes, n_strips);
  const long long out_bytes = (long long)n_rows * w * sample_bytes;
  unsigned char* ws = static_cast<unsigned char*>(workspace);
  long long* unit_bits = reinterpret_cast<long long*>(ws);
  long long* unit_len = reinterpret_cast<long long*>(ws + align256(slots * 16));
  int* unit_strip = reinterpret_cast<int*>(ws + align256(slots * 16) + align256(slots * 8));
  const unsigned char* pl = static_cast<const unsigned char*>(payload);
  unsigned char* dst = static_cast<unsigned char*>(out);

  // only the slots a strip's scan writes hold units; the rest read as empty (-1)
  TMC_CUDA(cudaMemsetAsync(unit_strip, 0xff, (size_t)slots * sizeof(int), stream));
  TMC_TIMED("lzw_scan_kernel", stream, lzw_scan_kernel<<<n_strips, kScanThreads, 0, stream>>>(
      pl, payload_bytes, strip_offsets, out_offsets, out_bytes, n_strips, unit_bits, unit_strip, status, dst));
  TMC_CHECK_LAUNCH("tmc_tiff_lzw_decode");
  const size_t smem = sizeof(int) * (size_t)kWarpsPerCta * (kSegCodes + 1 + 32);
  const long long ctas = (slots + kWarpsPerCta - 1) / kWarpsPerCta;
  TMC_CHECK_ARG(ctas < (1LL << 31), "tiff_lzw_decode: payload too large");
  TMC_TIMED("lzw_lengths_kernel", stream, lzw_lengths_kernel<<<(unsigned)ctas, 32 * kWarpsPerCta, smem, stream>>>(
      pl, strip_offsets, slots, unit_bits, unit_strip, unit_len));
  TMC_CHECK_LAUNCH("tmc_tiff_lzw_decode");
  TMC_TIMED("lzw_decode_kernel", stream, lzw_decode_kernel<<<(unsigned)ctas, 32 * kWarpsPerCta, smem, stream>>>(
      pl, strip_offsets, out_offsets, slots, unit_bits, unit_strip, unit_len, dst, status));
  TMC_CHECK_LAUNCH("tmc_tiff_lzw_decode");
  if (predictor == 2) {
    int sms = 148;
    int dev = 0;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const long long want = (n_rows + 7) / 8;
    const int blocks = (int)(want < 8LL * sms ? want : 8LL * sms);
    if (sample_bytes == 1)
      TMC_TIMED("lzw_predict_kernel<u8>", stream, lzw_predict_kernel<unsigned char><<<blocks, 256, 0, stream>>>(
          dst, n_rows, w));
    else
      TMC_TIMED("lzw_predict_kernel<u16>", stream, lzw_predict_kernel<unsigned short><<<blocks, 256, 0, stream>>>(
          reinterpret_cast<unsigned short*>(dst), n_rows, w));
    TMC_CHECK_LAUNCH("tmc_tiff_lzw_decode");
  }
  return TMC_OK;
}

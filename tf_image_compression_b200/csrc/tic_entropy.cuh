// GPU entropy stage (SURVEY.md §8f rank 4): the per-image static-model range coder of encode.py:171-202 /
// decode.py:182-208 on the device, bit-exact with the host coder (librangecoder.so) because both compile the same
// arithmetic (include/tic_rc_core.h).  A stream (one image's symbols, patch-major then h, w, c: encode.py:171-182) is a
// serial recurrence, so the unit of parallelism is the independently coded piece: a whole stream of at most
// TIC_RC_SEGMENT_SYMBOLS symbols, or one segment of a longer one (the container format of tic_rc_core.h: one image of
// BASELINE config 2 is 24 segments, a batch of 64 is 1536).  One warp per piece, lane 0 runs the coder (the other lanes
// load the table and sum the container header), several warps per SM sub-partition so the schedulers interleave the
// dependent chains.  With the binary alphabet of every shipped config (quan_scale = 2) and the power-of-two table total
// the reference uses (resolution = 4096, encode.py:91) a symbol costs one shift, one multiply, two selects and an
// occasional byte store on the critical path.  Segments are coded into worst-case slots of a scratch buffer and a second
// kernel packs header + bodies into the caller's slot.  Symbols stay in HBM after the encoder's last layer and only the
// compressed bytes cross PCIe (0.25 sym/px -> ~0.03 B/px instead of 0.25 B/px for model_0).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/tic_rc_core.h"

namespace tic {

constexpr int kEntropyMaxSymbols = 256;

struct DevSink {
  uint8_t* p;
  long long cap, pos, len;
  int overflow;
  __device__ __forceinline__ void put(uint8_t b) {
    if (pos >= cap) {
      overflow = 1;
      return;
    }
    p[pos++] = b;
    if (b) len = pos;
  }
};

// Stored bytes through 16-byte loads, the block after the current one already in flight; zeros past the end.
struct DevSource {
  const uint4* p;     // 16-byte aligned
  long long nbytes;   // stored length
  long long blk;      // index of the block in `cur`
  uint4 cur, nxt;
  uint32_t off;       // byte offset inside cur
  __device__ __forceinline__ uint4 load(long long b) const {
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    const long long first = b * 16;
    if (first < nbytes) {
      v = __ldg(p + b);
      const long long left = nbytes - first;
      if (left < 16) {  // clear the bytes past the stored length (the slot behind them is not the stream's)
        uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const long long lo = 4 * i;
          if (left <= lo) w[i] = 0u;
          else if (left < lo + 4) w[i] &= (1u << (8 * (int)(left - lo))) - 1u;
        }
        v = make_uint4(w[0], w[1], w[2], w[3]);
      }
    }
    return v;
  }
  // any byte alignment: the loads start at the 16-byte block that holds the first byte (always inside the caller's
  // 16-byte aligned slot) and the bytes in front of it are skipped
  __device__ __forceinline__ void init(const uint8_t* base, long long n) {
    const uint32_t mis = (uint32_t)(reinterpret_cast<uintptr_t>(base) & 15);
    p = reinterpret_cast<const uint4*>(base - mis);
    nbytes = n + mis;
    blk = 0;
    off = mis;
    cur = load(0);
    nxt = load(1);
  }
  __device__ __forceinline__ uint32_t get() {
    if (off == 16) {
      cur = nxt;
      ++blk;
      nxt = load(blk + 1);
      off = 0;
    }
    const uint32_t w = off < 8 ? (off < 4 ? cur.x : cur.y) : (off < 12 ? cur.z : cur.w);
    const uint32_t b = (w >> (8 * (off & 3))) & 0xFFu;
    ++off;
    return b;
  }
};

// Worst-case slot of one segment in the scratch buffer (16-byte aligned)
constexpr long long kEntropySegSlot = ((2LL * TIC_RC_SEGMENT_SYMBOLS + (TIC_RC_SEGMENT_SYMBOLS >> 6) + 16) + 15) & ~15LL;

// status codes written to *status (first error wins): 1 = symbol outside the table / of zero probability,
// 2 = output slot too small
//
// One block (= one warp) per piece: piece = stream * npiece + j covers symbols [j * piece_len, min(stream_len, (j+1) * piece_len))
// of its stream and is written to out + piece * out_stride, its stored length to out_bytes[piece].
// Plain streams: npiece = 1, piece_len = stream_len, out = the caller's slots.  Segmented: out = the scratch slots.
__global__ void __launch_bounds__(32) rc_encode_kernel(const uint8_t* __restrict__ sym, long long stream_len, long long piece_len, int npiece,
                                                       const uint32_t* __restrict__ cum, int n_cum, uint8_t* __restrict__ out,
                                                       long long out_stride, long long* __restrict__ out_bytes, unsigned int* status) {
  __shared__ uint32_t s_cum[kEntropyMaxSymbols + 1];
  for (int i = threadIdx.x; i < n_cum; i += 32) s_cum[i] = cum[i];
  __syncwarp();
  if (threadIdx.x != 0) return;
  const long long piece = blockIdx.x;
  const long long stream = piece / npiece, j = piece - stream * npiece;
  const long long first = j * piece_len;
  const long long n = stream_len - first < piece_len ? stream_len - first : piece_len;
  const uint8_t* s = sym + stream * stream_len + first;
  DevSink sink{out + piece * out_stride, out_stride, 0, 0, 0};
  tic_rc_enc_state st;
  tic_rc_enc_init(&st);
  const uint32_t total = s_cum[n_cum - 1];
  const bool p2 = (total & (total - 1)) == 0;
  const int k = 31 - __clz(total);
  const int nsym = n_cum - 1;
  int bad = 0;
  long long done = 0;
  // 16 symbols per load when the piece starts 16-byte aligned; the next block is requested before this one is coded
  if ((reinterpret_cast<uintptr_t>(s) & 15) == 0 && nsym == 2 && p2 && s_cum[1] != 0 && s_cum[1] != total) {
    const uint32_t c1 = s_cum[1];
    const uint4* s16 = reinterpret_cast<const uint4*>(s);
    const long long nblk = n >> 4;
    uint4 nxt = nblk ? __ldg(s16) : make_uint4(0u, 0u, 0u, 0u);
    // The symbol loop is deliberately NOT unrolled: what counts is the dependent chain of a symbol (shift, multiply,
    // selects, compare) and an instruction footprint that stays inside the instruction cache (the fully unrolled
    // 16-symbol body was 66 KB of SASS and ran at ~95 cycles per symbol).
    for (long long b = 0; b < nblk; ++b) {
      uint4 cur = nxt;
      if (b + 1 < nblk) nxt = __ldg(s16 + b + 1);
      // symbols other than 0 / 1 are an error (checked once per block, outside the critical path)
      if ((cur.x | cur.y | cur.z | cur.w) & 0xFEFEFEFEu) {
        bad = 1;
        break;
      }
#pragma unroll 1
      for (int i = 0; i < 4; ++i) {
        uint32_t word = cur.x;
        cur.x = cur.y;
        cur.y = cur.z;
        cur.z = cur.w;
#pragma unroll 1
        for (int jj = 0; jj < 4; ++jj) {
          tic_rc_enc_bit(&st, sink, word & 1u, k, c1);
          word >>= 8;
        }
      }
    }
    done = nblk << 4;
  }
  for (long long i = done; i < n && !bad; ++i) {
    const int v = s[i];
    if (v >= nsym) {
      bad = 1;
      break;
    }
    const uint32_t lo = s_cum[v], hi = s_cum[v + 1];
    if (hi == lo) {
      bad = 1;
      break;
    }
    const uint32_t r = p2 ? st.range >> k : st.range / total;
    tic_rc_enc_step(&st, sink, r, lo, hi);
  }
  if (!bad) tic_rc_enc_finish(&st, sink);
  out_bytes[piece] = bad ? 0 : sink.len;
  if (bad) atomicCAS(status, 0u, 1u);
  else if (sink.overflow) atomicCAS(status, 0u, 2u);
}

// Byte offset of body j in a segmented stream's container [ nseg x uint32 | body 0 | body 1 | ... ]: the header plus the
// stored lengths of the bodies before j (lens = the stream's nseg segment lengths).  j = nseg gives the stored length of
// the whole stream.  Called once by every thread of a 256-thread block; all of them get the value.
__device__ __forceinline__ long long rc_container_offset(const long long* __restrict__ lens, int nseg, int j) {
  __shared__ long long s_part[8];
  long long before = 0;
  for (int i = threadIdx.x; i < j; i += 256) before += lens[i];
  for (int o = 16; o > 0; o >>= 1) before += __shfl_down_sync(0xffffffffu, before, o);
  if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = before;
  __syncthreads();
  before = 0;
#pragma unroll
  for (int w = 0; w < 8; ++w) before += s_part[w];
  return 4LL * nseg + before;
}

// Segmented call, second step: block stream * nseg + j writes header entry j (little-endian uint32 byte count) and copies
// body j behind the bodies before it:  out slot = [ nseg x uint32 | body 0 | body 1 | ... ].
__global__ void __launch_bounds__(256) rc_pack_kernel(const uint8_t* __restrict__ seg, const long long* __restrict__ seg_bytes, int nseg,
                                                      uint8_t* __restrict__ out, long long out_stride, long long* __restrict__ out_bytes,
                                                      unsigned int* status) {
  const long long stream = blockIdx.x / nseg;
  const int j = (int)(blockIdx.x - stream * nseg);
  const long long* lens = seg_bytes + stream * nseg;
  const long long len = lens[j];
  const long long at = rc_container_offset(lens, nseg, j);
  uint8_t* slot = out + stream * out_stride;
  if (at + len > out_stride) {
    if (threadIdx.x == 0) {
      atomicCAS(status, 0u, 2u);
      if (j == nseg - 1) out_bytes[stream] = 0;
    }
    return;
  }
  const uint8_t* src = seg + (stream * nseg + j) * kEntropySegSlot;
  for (long long i = threadIdx.x; i < len; i += 256) slot[at + i] = src[i];
  if (threadIdx.x == 0) {
    const uint32_t v = (uint32_t)len;
    slot[4 * j] = (uint8_t)v;
    slot[4 * j + 1] = (uint8_t)(v >> 8);
    slot[4 * j + 2] = (uint8_t)(v >> 16);
    slot[4 * j + 3] = (uint8_t)(v >> 24);
    if (j == nseg - 1) out_bytes[stream] = at + len;
  }
}

// Segmented call without an output slot: block `stream` writes the stored length rc_pack_kernel would give the stream
// (out_bytes of tic_entropy_encode) from its segment lengths; no body is copied.
__global__ void __launch_bounds__(256) rc_stored_length_kernel(const long long* __restrict__ seg_bytes, int nseg,
                                                               long long* __restrict__ out_bytes) {
  const long long v = rc_container_offset(seg_bytes + (long long)blockIdx.x * nseg, nseg, nseg);
  if (threadIdx.x == 0) out_bytes[blockIdx.x] = v;
}

// One block (= one warp) per piece, as in rc_encode_kernel.  nseg = 0: plain streams.  nseg > 0: the slot starts with
// nseg uint32 byte counts; piece j starts behind the header and the bodies before it (any byte alignment).
__global__ void __launch_bounds__(32) rc_decode_kernel(const uint8_t* __restrict__ in, long long in_stride, const long long* __restrict__ in_bytes,
                                                       const uint32_t* __restrict__ cum, int n_cum, uint8_t* __restrict__ sym,
                                                       long long stream_len, int nseg) {
  __shared__ uint32_t s_cum[kEntropyMaxSymbols + 1];
  for (int i = threadIdx.x; i < n_cum; i += 32) s_cum[i] = cum[i];
  const int npiece = nseg > 0 ? nseg : 1;
  const long long piece = blockIdx.x;
  const long long stream = piece / npiece, j = piece - stream * npiece;
  const uint8_t* slot = in + stream * in_stride;
  long long stored = in_bytes[stream];
  stored = stored < 0 ? 0 : (stored < in_stride ? stored : in_stride);
  const uint8_t* body = slot;
  long long body_len = stored;
  long long first = 0, n = stream_len;
  if (nseg > 0) {
    // header entries past the stored bytes read as zero (the host decoder reads zeros past the end of its source too)
    const long long max_len = tic_rc_plain_bound(TIC_RC_SEGMENT_SYMBOLS);
    auto entry = [&](long long i) -> long long {
      long long v = 0;
      for (int b = 0; b < 4; ++b)
        if (4 * i + b < stored) v |= (long long)slot[4 * i + b] << (8 * b);
      return v < max_len ? v : max_len;
    };
    long long before = 0;
    for (long long i = threadIdx.x; i < j; i += 32) before += entry(i);
    for (int o = 16; o > 0; o >>= 1) before += __shfl_down_sync(0xffffffffu, before, o);
    before = __shfl_sync(0xffffffffu, before, 0);
    const long long at = 4LL * nseg + before;
    long long len = entry(j);
    if (at >= stored) len = 0;
    else if (at + len > stored) len = stored - at;
    body = slot + (at < stored ? at : 0);
    body_len = len;
    first = j * (long long)TIC_RC_SEGMENT_SYMBOLS;
    n = stream_len - first < TIC_RC_SEGMENT_SYMBOLS ? stream_len - first : TIC_RC_SEGMENT_SYMBOLS;
  }
  __syncwarp();
  if (threadIdx.x != 0) return;
  DevSource src;
  src.init(body, body_len);
  uint8_t* o = sym + stream * stream_len + first;
  tic_rc_dec_state st;
  tic_rc_dec_init(&st);
  tic_rc_dec_prime(&st, src);
  const uint32_t total = s_cum[n_cum - 1];
  const bool p2 = (total & (total - 1)) == 0;
  const int k = 31 - __clz(total);
  long long done = 0;
  if ((reinterpret_cast<uintptr_t>(o) & 15) == 0 && n_cum == 3 && p2 && s_cum[1] != 0 && s_cum[1] != total) {
    const uint32_t c1 = s_cum[1];
    uint4* o16 = reinterpret_cast<uint4*>(o);
    uint32_t range = st.range, code = st.code;
    for (long long b = 0; b < (n >> 4); ++b) {
      uint4 o4 = make_uint4(0u, 0u, 0u, 0u);
#pragma unroll 1
      for (int i = 0; i < 4; ++i) {
        uint32_t word = 0u;
#pragma unroll 1
        for (int jj = 0; jj < 4; ++jj) {
          const uint32_t r = range >> k;
          const uint32_t t = r * c1;
          const uint32_t m = 0u - (uint32_t)(code >= t);
          word |= (m & 1u) << (8 * jj);
          code -= t & m;
          range = (t & ~m) | (((r << k) - t) & m);
          while (range < TIC_RC_TOP) {
            code = (code << 8) | src.get();
            range <<= 8;
          }
        }
        o4.x = o4.y;
        o4.y = o4.z;
        o4.z = o4.w;
        o4.w = word;
      }
      o16[b] = o4;
    }
    st.range = range;
    st.code = code;
    done = (n >> 4) << 4;
  }
  for (long long i = done; i < n; ++i) {
    const uint32_t r = p2 ? st.range >> k : st.range / total;
    const uint32_t v = tic_rc_dec_target(&st, r, total);
    // last entry with cum[s] <= v (upper_bound semantics: skips zero-width symbols): binary search over the shared table
    int lo = 0, hi = n_cum - 1;  // invariant: cum[lo] <= v < cum[hi]
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (s_cum[mid] <= v) lo = mid;
      else hi = mid;
    }
    o[i] = (uint8_t)lo;
    tic_rc_dec_step(&st, src, r, s_cum[lo], s_cum[lo + 1]);
  }
}

}  // namespace tic

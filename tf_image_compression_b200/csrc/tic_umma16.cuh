// tcgen05 / TMEM / TMA implicit-GEMM kernels, fp16-pair operands (compute mode TIC_COMPUTE_TENSOR_F16X3):
// the 3x3 conv (stride 1 and 2) and the stride-2 transposed conv of the codec
// (basic_block/basic_block.py:27-71) with fp32-class accuracy on the fp16 tensor pipe.
//
// Why fp16 pairs (measured, profiles/r1b_umma_f16_probe.log): one tcgen05.mma with M = 128 and a 32-byte
// K slice costs 85..113 cycles for N <= 128 whatever its kind, so the cost of a layer is its INSTRUCTION
// count.  kind::f16 covers 16 channels per instruction (kind::tf32: 8) and fp16 has the same 11-bit
// significand as tf32, so the error-compensated three-product scheme keeps its accuracy at half the
// instructions:   x = hi + lo' / 2048,  hi = rn_f16(x),  lo' = rn_f16((x - hi) * 2048)
//   D_main += A_hi * W_hi            D_lo += A_hi * W_lo' + A_lo' * W_hi          out = D_main + D_lo / 2048
// The first two products share their A operand, so they are ONE instruction with N = 2 * cout over the
// stacked weight tile [W_hi ; W_lo'] writing the adjacent accumulator pair (D_main | D_lo).
//
// Activations live in HBM pre-split: two fp16 planes (hi, lo') of the NHWC tensor, 4 bytes per element like
// fp32.  The producing epilogue splits once per element; consumers TMA the planes straight into
// MMA-ready swizzled tiles (no converter warps, no shared-memory round trip).
//
// Operand staging ("one box, nine taps", probe F2): per K-block ONE TMA box per plane covers the whole
// halo (stride 1: 10 columns x (rows + 2); the box dims are ordered (C, W, N, H)).  A filter tap is a
// descriptor start offset of (kh * box_columns + kw) rows — not a multiple of the swizzle atom, which is
// fine because the swizzle XOR is a function of the absolute shared-memory address — and the 8-pixel row
// groups sit box_columns rows apart (descriptor SBO).  Stride 2 uses a 5-D map ((w parity, C), W/2,
// h parity, N, H/2); the transposed conv walks INPUT pixels and feeds four sub-pixel phase accumulators.
// Weights ([W_hi ; W_lo'] per tap, pre-swizzled) are loaded ONCE per CTA and stay resident; layers whose
// weights do not fit run as output-channel slices.
//
// TMEM: per tile `nsplit` (D_main | D_lo) pairs — the tensor core truncates when it adds into the fp32
// accumulator (tests/probe/umma_accum_probe.cu), so the K steps rotate over nsplit accumulators that the
// epilogue sums with round-to-nearest adds — and two tile buffers so the epilogue of tile i overlaps the
// MMAs of tile i+1.
// Warp roles (384 threads): 0 TMA producer, 1 MMA issuer (elect.sync: a plain `if (lane == 0)` region makes
// ptxas wrap every UTCHMMA in an ELECT / BRA.U.ANY loop), 2 TMEM allocator, 4-11 epilogue (two warps per TMEM
// lane quadrant, alternating 16-column chunks).
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>

#include <string>

#include "tic_common.cuh"
#include "tic_launch.cuh"
#include "tic_ptx.cuh"
#include "tic_simt.cuh"

namespace tic {

// U16_DECONV: one (D_main | D_lo) pair per output phase, one MMA pair per filter tap (9 per K step).
// U16_DECONV_PH ("phase-stacked", cout <= 32): N = (phase, channel); the taps that read the same input pixel
// ("view": a / a-1 x b / b-1) are stacked along N with zero rows for the phases a view does not reach:
// 4 MMA pairs per K step instead of 9, and it is what makes the 3-channel last layer a tensor-core layer.
// U16_DECONV_RGB: phase-stacked with cpad = 4 (the 3-channel last layer); its own instantiation so that its
// epilogue (denormalise, clip, round, scatter into the stitched image) is not compiled next to the others.
enum U16Mode : int { U16_S1 = 0, U16_S2 = 1, U16_DECONV = 2, U16_DECONV_PH = 3, U16_DECONV_RGB = 4 };
__host__ __device__ constexpr bool u16_is_ph(int mode) { return mode == U16_DECONV_PH || mode == U16_DECONV_RGB; }

constexpr int kU16MaxSlots = 8;

struct U16Params {
  int mode;
  int n;                 // patches
  int Ht, Wt;            // tile-space map (S1/S2: output map, DECONV: input map)
  int bn, bh;            // patches per tile (1 | 2), map rows per tile per patch (16 | 8)
  int tiles_x, tiles_y;
  FastDiv tx_d, ty_d;    // / tiles_x, / tiles_y
  long long num_tiles;
  int KB;                // K-blocks (input-channel chunks of kc)
  int kc;                // channels per K-block
  int ksteps;            // MMAs (K = 16) per tap per K-block
  int npad;              // output channels of this launch rounded up to 16 (MMA N = npad or 2 * npad); PH: 4 * cpad rounded up
  int cpad;              // PH: channels per phase column block (4 | 16 | 32)
  int oc0;               // first output channel of this launch (slice)
  int nsplit;            // conv: accumulator pairs the K steps rotate over; deconv: 1
  int nbuf;              // TMEM tile buffers (1 | 2 | 4): how far the MMAs run ahead of the epilogue
  int nbshift;           // log2(nbuf)
  uint32_t acc_cols;     // TMEM columns per tile buffer
  uint32_t a_layout;     // descriptor layout code of the A rows (2 = SW128, 4 = SW64, 6 = SW32)
  uint32_t w_layout;     // ... of the weight rows
  uint32_t sbo;          // A: bytes between 8-row groups
  uint32_t w_sbo;        // W: 8 * weight row bytes
  uint32_t a_off[9];     // per tap (kh * 3 + kw): start offset inside a plane slot
  uint32_t box_bytes;    // one TMA box
  uint32_t box_stride;   // box_bytes rounded up to 1024 (second parity box of a stride-2 slot)
  int nbox;              // boxes per plane (stride 2 with 64-channel K-blocks: one per w parity)
  uint32_t slot_bytes;
  int S;                 // plane slots in the ring
  uint32_t tap_bytes;    // [W_hi ; W_lo'] of one tap of one K-block
  uint32_t w_bytes;      // KB * 9 * tap_bytes
  const uint8_t* wimg;
  int pair;              // 1: CTA-pair kernel (cta_group::2, M = 256)
  int staged;            // 1: coalesced epilogue through a per-warp shared-memory stage (u16_epilogue_tile_staged)
  uint32_t wA_bytes;     // pair: per-CTA bytes of its half of the stacked weight tiles (all taps, K-blocks)
  uint32_t wB_bytes;     // pair: per-CTA bytes of its half of W_hi for the A_lo' x W_hi product
  long long in_lo_off;   // elements between the hi and lo' planes of the input (unused by the kernel: second tensor map)
  int dbg;               // measurement aid (env TIC_DBG, pair kernel): 1 = no MMA issue, 2 = no TMA loads, 4 = no epilogue work
};

__host__ __device__ inline uint32_t u16_swz(uint32_t off, uint32_t rowbytes) {
  const uint32_t mask = rowbytes >= 128 ? 7u : rowbytes == 64 ? 3u : 1u;
  return off ^ (((off >> 7) & mask) << 4);
}
__host__ __device__ inline uint32_t u16_layout_code(uint32_t rowbytes) { return rowbytes >= 128 ? 2u : rowbytes == 64 ? 4u : 6u; }

// CTA-pair weight image = the exact per-CTA shared-memory layout, per rank r of the pair:
//   region A [kb][tap][rows nn]   : r = 0 -> W_hi rows, r = 1 -> W_lo' rows      (stacked product, N = 2 nn over the pair)
//   region B [kb][tap][rows nn/2] : W_hi rows r * nn/2 ...                         (A_lo' x W_hi product, N = nn over the pair)
// nn = npad (conv / tap-based deconv) or neff (phase-stacked deconv, row = phase * cpad + oc, tap = view).
__global__ void u16_build_weights_pair_kernel(const float* __restrict__ w, int cin, int cout, int oc0, int cs, int nn, int cpad,
                                              int ph_mode, int kc, int KB, uint32_t regA, uint32_t regB, uint8_t* __restrict__ img) {
  const int T = ph_mode ? 4 : 9;
  const uint32_t wrow = (uint32_t)kc * 2u;
  const long long perA = (long long)KB * T * nn * kc, perB = perA / 2;
  const long long total = 2 * (perA + perB);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int rank = (int)(i / (perA + perB));
    long long j = i - (long long)rank * (perA + perB);
    const bool inB = j >= perA;
    if (inB) j -= perA;
    const int rows = inB ? nn / 2 : nn;
    const int k = (int)(j % kc);
    const int rr = (int)((j / kc) % rows);
    const int t = (int)(j / ((long long)kc * rows));
    const int kb = t / T, tap = t % T;
    const int row = inB ? rank * (nn / 2) + rr : rr;  // logical output row (channel or (phase, channel))
    const bool want_lo = !inB && rank == 1;
    int kh, kw, oc;
    bool live = true;
    if (ph_mode) {
      const int dy = tap >> 1, dx = tap & 1, ph = row / cpad;
      oc = row % cpad;
      const int py = ph >> 1, px = ph & 1;
      kh = py ? (dy ? 1 : -1) : (dy ? 0 : 2);
      kw = px ? (dx ? 1 : -1) : (dx ? 0 : 2);
      live = ph < 4 && kh >= 0 && kw >= 0;
    } else {
      kh = tap / 3;
      kw = tap % 3;
      oc = row;
    }
    const int ic = kb * kc + k;
    float v = 0.f;
    if (live && oc < cs && ic < cin) v = w[((size_t)(kh * 3 + kw) * cin + ic) * cout + oc0 + oc];
    __half hi, lo;
    split16(v, hi, lo);
    const uint32_t off = (uint32_t)t * (uint32_t)rows * wrow + (uint32_t)rr * wrow + (uint32_t)k * 2u;
    uint8_t* base = img + (size_t)rank * (regA + regB) + (inB ? regA : 0u);
    *reinterpret_cast<__half*>(base + u16_swz(off, wrow)) = want_lo ? lo : hi;
  }
}

// fp32 NHWC -> fp16 pair planes (caller-provided f32 activations: tic_run_layers)
__global__ void u16_split_f32_kernel(const float* __restrict__ src, __half* __restrict__ hi, __half* __restrict__ lo, long long count,
                                     unsigned int* oflow) {
  bool bad = false;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (long long)gridDim.x * blockDim.x) {
    __half h, l;
    split16(src[i], h, l);
    bad |= ovf_hit1(h);
    hi[i] = h;
    lo[i] = l;
  }
  if (bad) ovf_raise(oflow);
}
// u8 symbols -> inverse-sigmoid LUT (model_0/model.py:153) -> fp16 pair planes.  The table (q <= 256 entries) is split
// once per block into shared memory; a thread takes 16 symbols per pass (one 16-byte load, two 32-byte stores per plane)
// when the pointers allow it (the scalar version moved 50 MB in and 200 MB out at 2 TB/s: byte loads, 2-byte stores).
__global__ void u16_split_symlut_kernel(const uint8_t* __restrict__ sym, const float* __restrict__ lut, int q, __half* __restrict__ hi,
                                        __half* __restrict__ lo, long long count, unsigned int* oflow) {
  __shared__ uint32_t s_pair[256];   // (hi, lo') of every table entry
  bool bad = false;
  for (int i = threadIdx.x; i < 256; i += blockDim.x) {
    __half h = __float2half_rn(0.f), l = h;
    if (i < q) {
      split16(__ldg(lut + i), h, l);
      bad |= ovf_hit1(h);   // (a table entry outside the fp16 range: reported whether or not a symbol uses it)
    }
    s_pair[i] = (uint32_t)__half_as_ushort(h) | ((uint32_t)__half_as_ushort(l) << 16);
  }
  __syncthreads();
  const bool vec = ((reinterpret_cast<uintptr_t>(sym) | reinterpret_cast<uintptr_t>(hi) | reinterpret_cast<uintptr_t>(lo)) & 15) == 0;
  const long long nvec = vec ? count >> 4 : 0;
  for (long long v = (long long)blockIdx.x * blockDim.x + threadIdx.x; v < nvec; v += (long long)gridDim.x * blockDim.x) {
    const uint4 w = __ldg(reinterpret_cast<const uint4*>(sym) + v);
    const uint32_t ws[4] = {w.x, w.y, w.z, w.w};
    uint32_t oh[8], ol[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const uint32_t word = ws[k >> 1] >> (16 * (k & 1));
      const uint32_t a = s_pair[word & 0xffu], b = s_pair[(word >> 8) & 0xffu];
      oh[k] = __byte_perm(a, b, 0x5410);   // (hi_a, hi_b)
      ol[k] = __byte_perm(a, b, 0x7632);   // (lo_a, lo_b)
    }
    uint4* ph = reinterpret_cast<uint4*>(hi) + 2 * v;
    uint4* pl = reinterpret_cast<uint4*>(lo) + 2 * v;
    ph[0] = make_uint4(oh[0], oh[1], oh[2], oh[3]);
    ph[1] = make_uint4(oh[4], oh[5], oh[6], oh[7]);
    pl[0] = make_uint4(ol[0], ol[1], ol[2], ol[3]);
    pl[1] = make_uint4(ol[4], ol[5], ol[6], ol[7]);
  }
  for (long long i = (nvec << 4) + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (long long)gridDim.x * blockDim.x) {
    const uint32_t pr = s_pair[sym[i]];
    reinterpret_cast<unsigned short*>(hi)[i] = (unsigned short)(pr & 0xffffu);
    reinterpret_cast<unsigned short*>(lo)[i] = (unsigned short)(pr >> 16);
  }
  if (bad) ovf_raise(oflow);
}

struct U16SmemBars {
  uint64_t w_full;
  uint64_t full[kU16MaxSlots], empty[kU16MaxSlots];
  uint64_t acc_full[4], acc_empty[4];
  uint32_t tmem_base;
};

__device__ __forceinline__ uint64_t u16_desc(uint32_t lo32, uint32_t hi32) {
  uint64_t d;
  asm("mov.b64 %0, {%1, %2};" : "=l"(d) : "r"(lo32), "r"(hi32));
  return d;
}

// Epilogue of one tile for one epilogue warp: TMEM lane = tile row = pixel (n, yt, xt); the warp takes
// every other 16-column chunk (`half`).  Sums the split accumulators (round-to-nearest), rescales the lo'
// accumulator, adds bias, activation, residual, and stores pair planes | f32 | symbols (+ histogram).
// 16 accumulator columns of one pixel: sum the split accumulators (round-to-nearest), rescale the lo' part
template <int MODE>
__device__ __forceinline__ void u16_load_chunk(float (&v)[16], const uint32_t tbuf, const int NPAD, const int nsplit,
                                               const int ph, const int c, const int cpad) {
  constexpr bool kDeconv = MODE == U16_DECONV || u16_is_ph(MODE);
  if (kDeconv || nsplit == 1) {
    float u[16];
    const uint32_t t0 = tbuf + (u16_is_ph(MODE) ? (uint32_t)(ph * cpad) : (uint32_t)ph * 2u * NPAD) + c;
    ptx::tmem_ld16_nowait(t0 + NPAD, u);
    ptx::tmem_ld16_nowait(t0, v);
    ptx::tmem_ld_wait();
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __fmaf_rn(u[i], 1.0f / 2048.0f, v[i]);
  } else {
    // lo' accumulators first (small), then the main accumulators, round-to-nearest adds
    float lo[16];
    ptx::tmem_ld16_nowait(tbuf + NPAD + c, lo);
    ptx::tmem_ld16_nowait(tbuf + c, v);
    ptx::tmem_ld_wait();
    for (int j = 1; j < nsplit; ++j) {
      float u[16], w[16];
      ptx::tmem_ld16_nowait(tbuf + (uint32_t)j * 2u * NPAD + NPAD + c, u);
      ptx::tmem_ld16_nowait(tbuf + (uint32_t)j * 2u * NPAD + c, w);
      ptx::tmem_ld_wait();
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        lo[i] = __fadd_rn(lo[i], u[i]);
        v[i] = __fadd_rn(v[i], w[i]);
      }
    }
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __fmaf_rn(lo[i], 1.0f / 2048.0f, v[i]);
  }
}

// two values -> packed (hi, hi) and (lo', lo') half2 words; same arithmetic as split16
__device__ __forceinline__ void split16x2(float v0, float v1, uint32_t& hp, uint32_t& lp, __half2& omax) {
  const __half2 h = __floats2half2_rn(v0, v1);
  ovf_track(omax, h);
  const float2 hf = __half22float2(h);
  const __half2 l = __floats2half2_rn(__fmul_rn(__fsub_rn(v0, hf.x), 2048.0f), __fmul_rn(__fsub_rn(v1, hf.y), 2048.0f));
  hp = *reinterpret_cast<const uint32_t*>(&h);
  lp = *reinterpret_cast<const uint32_t*>(&l);
}
__device__ __forceinline__ void split16x2(float v0, float v1, uint32_t& hp, uint32_t& lp) {
  const __half2 h = __floats2half2_rn(v0, v1);
  const float2 hf = __half22float2(h);
  const __half2 l = __floats2half2_rn(__fmul_rn(__fsub_rn(v0, hf.x), 2048.0f), __fmul_rn(__fsub_rn(v1, hf.y), 2048.0f));
  hp = *reinterpret_cast<const uint32_t*>(&h);
  lp = *reinterpret_cast<const uint32_t*>(&l);
}

// Epilogue of one tile for one epilogue warp: TMEM lane = tile row = pixel (n, yt, xt); the warp takes
// every other 16-column chunk (`half`).  Adds bias, activation, residual, and stores pair planes | f32 |
// symbols (+ histogram) | the denormalised, clipped, rounded image (3-channel last layer).
template <int MODE, int NP = 2>   // NP = epilogue warps per TMEM lane quadrant: `half` in [0, NP) picks every NP-th chunk
__device__ __forceinline__ void u16_epilogue_tile(const LayerArgs& a, const int NPAD, const int oc0, const int nsplit,
                                                  const uint32_t tbuf, const int n, const int yt, const int xt, const bool valid,
                                                  const int half, const float* s_bias, unsigned* s_hist, int& h_ones,
                                                  int& h_valid, __half2& omax, const int cpad = 0) {
  constexpr bool kDeconv = MODE == U16_DECONV || u16_is_ph(MODE);
#ifdef TIC_DEBUG_SKIP_EPILOGUE  // measurement aid: time the kernels without their epilogue work
  return;
#endif
  if (MODE == U16_DECONV_RGB) {
    // 3-channel last layer: the 16 columns are (phase, channel) of the 2x2 output pixels of this input pixel;
    // the two warps of a lane quadrant take the even / the odd output row
    float v[16], u[16];
    ptx::tmem_ld16_nowait(tbuf + NPAD, u);
    ptx::tmem_ld16_nowait(tbuf, v);
    ptx::tmem_ld_wait();
    if (!valid) return;
    if (a.out_mode == IO_DENORM_U8 || a.out_mode == IO_DENORM_F32) {
      // patch -> image geometry once per pixel pair (utils.concat_patches, utils/utils.py:136-167: crop to [H, W])
      const Geo& g = a.geo;
      unsigned img, gy, gx;
      geo_decode(g, (unsigned)(g.n0 + n), img, gy, gx);
      const int Y = g.oy + (int)gy * g.P + 2 * yt + half, X = g.ox + (int)gx * g.P + 2 * xt;
      if (Y >= g.H) return;
      const long long off = (((long long)img * g.H + Y) * g.W + X) * 3;
      if (a.out_mode == IO_DENORM_U8 && X + 1 < g.W && !((reinterpret_cast<uintptr_t>(a.out) + off) & 1)) {
        // both pixels inside the image and 2-byte aligned (X is even: any even W, and an even base address): three 2-byte stores instead of six bytes
        uint32_t q[6];
#pragma unroll
        for (int px = 0; px < 2; ++px)
#pragma unroll
          for (int c = 0; c < 3; ++c) {
            const float m = half ? v[8 + px * 4 + c] : v[px * 4 + c];
            const float l = half ? u[8 + px * 4 + c] : u[px * 4 + c];
            float y = apply_act(__fadd_rn(__fmaf_rn(l, 1.0f / 2048.0f, m), s_bias[c]), a.act);
            y = tic_denorm_clip(y, a.mean[c], a.stdv[c]);
            q[px * 3 + c] = (uint32_t)(int)rintf(y);
          }
        unsigned short* o2 = reinterpret_cast<unsigned short*>(reinterpret_cast<uint8_t*>(a.out) + off);
        o2[0] = (unsigned short)(q[0] | (q[1] << 8));
        o2[1] = (unsigned short)(q[2] | (q[3] << 8));
        o2[2] = (unsigned short)(q[4] | (q[5] << 8));
        return;
      }
#pragma unroll
      for (int px = 0; px < 2; ++px) {
        if (X + px >= g.W) break;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          const int col = (half * 2 + px) * 4 + c;
          // select with constant indices (v[] stays in registers): half is warp-uniform
          const float m = half ? v[8 + px * 4 + c] : v[px * 4 + c];
          const float l = half ? u[8 + px * 4 + c] : u[px * 4 + c];
          (void)col;
          float y = apply_act(__fadd_rn(__fmaf_rn(l, 1.0f / 2048.0f, m), s_bias[c]), a.act);
          y = tic_denorm_clip(y, a.mean[c], a.stdv[c]);
          if (a.out_mode == IO_DENORM_F32)
            reinterpret_cast<float*>(a.out)[off + px * 3 + c] = y;
          else
            reinterpret_cast<uint8_t*>(a.out)[off + px * 3 + c] = (uint8_t)(int)rintf(y);
        }
      }
      return;
    }
    if (half != 0) return;
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = apply_act(__fadd_rn(__fmaf_rn(u[i], 1.0f / 2048.0f, v[i]), s_bias[i & 3]), a.act);
#pragma unroll
    for (int ph = 0; ph < 4; ++ph) store_pixel<4>(a, n, 2 * yt + (ph >> 1), 2 * xt + (ph & 1), oc0, v + 4 * ph, s_hist, h_ones, h_valid);
    return;
  }
  const int phases = kDeconv ? 4 : 1;
  const int cend = u16_is_ph(MODE) ? cpad : NPAD;
  if (a.out_mode == IO_ACT16 && (a.cout & 15) == 0) {
    // ---- fast path: pair-plane output, every chunk holds 16 real channels --------------------------------
    const float floor_v = a.act ? 0.0f : -INFINITY;
    const long long pix0 = ((long long)n * a.hout + (kDeconv ? 2 * yt : yt)) * a.wout + (kDeconv ? 2 * xt : xt);
    __half* const obase = reinterpret_cast<__half*>(a.out) + pix0 * a.cout + oc0;
    const __half* const rbase = a.res ? reinterpret_cast<const __half*>(a.res) + pix0 * a.cout + oc0 : nullptr;
    // bias + activation (+ residual) + split + the four 16-byte stores of one 16-channel chunk
    auto finish = [&](float (&v)[16], const int c, const int poff) {
      const float4* bp = reinterpret_cast<const float4*>(s_bias + c);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float4 b = bp[i];
        v[4 * i] = fmaxf(__fadd_rn(v[4 * i], b.x), floor_v);
        v[4 * i + 1] = fmaxf(__fadd_rn(v[4 * i + 1], b.y), floor_v);
        v[4 * i + 2] = fmaxf(__fadd_rn(v[4 * i + 2], b.z), floor_v);
        v[4 * i + 3] = fmaxf(__fadd_rn(v[4 * i + 3], b.w), floor_v);
      }
      if (rbase) {
        const uint4* rh = reinterpret_cast<const uint4*>(rbase + poff + c);
        const uint4* rl = reinterpret_cast<const uint4*>(rbase + a.res_lo_off + poff + c);
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          const uint4 qh = __ldg(rh + j), ql = __ldg(rl + j);
          const __half2* h2 = reinterpret_cast<const __half2*>(&qh);
          const __half2* l2 = reinterpret_cast<const __half2*>(&ql);
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float2 hf = __half22float2(h2[e]), lf = __half22float2(l2[e]);
            v[8 * j + 2 * e] = __fadd_rn(__fmaf_rn(lf.x, 1.0f / 2048.0f, hf.x), v[8 * j + 2 * e]);
            v[8 * j + 2 * e + 1] = __fadd_rn(__fmaf_rn(lf.y, 1.0f / 2048.0f, hf.y), v[8 * j + 2 * e + 1]);
          }
        }
      }
      uint32_t hp[8], lp[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) split16x2(v[2 * i], v[2 * i + 1], hp[i], lp[i], omax);
      uint4* oh = reinterpret_cast<uint4*>(obase + poff + c);
      uint4* ol = reinterpret_cast<uint4*>(obase + a.out_lo_off + poff + c);
      oh[0] = make_uint4(hp[0], hp[1], hp[2], hp[3]);
      oh[1] = make_uint4(hp[4], hp[5], hp[6], hp[7]);
      ol[0] = make_uint4(lp[0], lp[1], lp[2], lp[3]);
      ol[1] = make_uint4(lp[4], lp[5], lp[6], lp[7]);
    };
    // units (phase, 16-channel chunk) alternate between the two warps of a lane quadrant; a warp works on two
    // of its units at once (all four TMEM loads first, one wait, two independent instruction streams)
    const int nch = cend >> 4, U = phases * nch;
    auto unit_t = [&](int u, int& c, int& poff) -> uint32_t {
      const int ph = u / nch;
      c = (u - ph * nch) << 4;
      poff = kDeconv ? ((ph >> 1) * a.wout + (ph & 1)) * a.cout : 0;
      return tbuf + (u16_is_ph(MODE) ? (uint32_t)(ph * cpad) : (uint32_t)ph * 2u * NPAD) + c;
    };
    if (kDeconv || nsplit == 1) {
      for (int u = half; u < U; u += 2 * NP) {
        int cA, pA, cB = 0, pB = 0;
        const uint32_t tA = unit_t(u, cA, pA);
        const bool hasB = u + NP < U;
        float va[16], la[16];
        if (hasB) {
          const uint32_t tB = unit_t(u + NP, cB, pB);
          float vb[16], lb[16];
          ptx::tmem_ld16_nowait(tA + NPAD, la);
          ptx::tmem_ld16_nowait(tA, va);
          ptx::tmem_ld16_nowait(tB + NPAD, lb);
          ptx::tmem_ld16_nowait(tB, vb);
          ptx::tmem_ld_wait();
          if (valid) {
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              va[i] = __fmaf_rn(la[i], 1.0f / 2048.0f, va[i]);
              vb[i] = __fmaf_rn(lb[i], 1.0f / 2048.0f, vb[i]);
            }
            finish(va, cA, pA);
            finish(vb, cB, pB);
          }
        } else {
          ptx::tmem_ld16_nowait(tA + NPAD, la);
          ptx::tmem_ld16_nowait(tA, va);
          ptx::tmem_ld_wait();
          if (valid) {
#pragma unroll
            for (int i = 0; i < 16; ++i) va[i] = __fmaf_rn(la[i], 1.0f / 2048.0f, va[i]);
            finish(va, cA, pA);
          }
        }
      }
    } else {
      for (int c = half * 16; c < cend; c += 16 * NP) {
        float v[16];
        u16_load_chunk<MODE>(v, tbuf, NPAD, nsplit, 0, c, cpad);
        if (valid) finish(v, c, 0);
      }
    }
    return;
  }
  for (int ph = 0; ph < phases; ++ph) {
    const int y = kDeconv ? 2 * yt + (ph >> 1) : yt;
    const int x = kDeconv ? 2 * xt + (ph & 1) : xt;
    for (int c = half * 16; c < cend; c += 16 * NP) {
      float v[16];
      u16_load_chunk<MODE>(v, tbuf, NPAD, nsplit, ph, c, cpad);
      const int cl = c;          // channel inside the slice
      const int oc = oc0 + cl;   // channel of the layer
      if (valid && oc < a.cout) {
#pragma unroll
        for (int i = 0; i < 16; ++i) v[i] = apply_act(__fadd_rn(v[i], s_bias[cl + i]), a.act);
        const long long pix = ((long long)n * a.hout + y) * a.wout + x;
        if (a.res) {
          if (a.res16) {
            const __half* rh = reinterpret_cast<const __half*>(a.res) + pix * a.cout + oc;
            const __half* rl = rh + a.res_lo_off;
#pragma unroll
            for (int i = 0; i < 16; i += 8) {
              if (oc + i < a.cout) {
                const uint4 qh = __ldg(reinterpret_cast<const uint4*>(rh + i));
                const uint4 ql = __ldg(reinterpret_cast<const uint4*>(rl + i));
                const __half* ph8 = reinterpret_cast<const __half*>(&qh);
                const __half* pl8 = reinterpret_cast<const __half*>(&ql);
#pragma unroll
                for (int e = 0; e < 8; ++e) v[i + e] = __fadd_rn(join16(ph8[e], pl8[e]), v[i + e]);
              }
            }
          } else {
            const float* rp = a.res + pix * a.cout + oc;
#pragma unroll
            for (int i = 0; i < 16; i += 4) {
              if (oc + i < a.cout) {
                const float4 r = __ldg(reinterpret_cast<const float4*>(rp + i));
                v[i] = __fadd_rn(r.x, v[i]);
                v[i + 1] = __fadd_rn(r.y, v[i + 1]);
                v[i + 2] = __fadd_rn(r.z, v[i + 2]);
                v[i + 3] = __fadd_rn(r.w, v[i + 3]);
              }
            }
          }
        }
        if (a.out_mode == IO_ACT16) {
          __half* oh = reinterpret_cast<__half*>(a.out) + pix * a.cout + oc;
          __half* ol = oh + a.out_lo_off;
#pragma unroll
          for (int i = 0; i < 16; i += 8) {
            if (oc + i < a.cout) {
              uint4 qh, ql;
              __half* ph8 = reinterpret_cast<__half*>(&qh);
              __half* pl8 = reinterpret_cast<__half*>(&ql);
#pragma unroll
              for (int e = 0; e < 8; ++e) split16(v[i + e], ph8[e], pl8[e]);
#pragma unroll
              for (int e = 0; e < 8; e += 2) ovf_track(omax, __halves2half2(ph8[e], ph8[e + 1]));
              *reinterpret_cast<uint4*>(oh + i) = qh;
              *reinterpret_cast<uint4*>(ol + i) = ql;
            }
          }
        } else {
          store_pixel<16>(a, n, y, x, oc, v, s_hist, h_ones, h_valid);
        }
      }
    }
  }
}

// ---- staged epilogue: coalesced pair-plane stores ---------------------------------------------------------
// A lane's pixel row is `cend * 2` bytes per plane, so direct stores are 16 bytes per lane at a stride of a
// row: 32 transactions per instruction (measured: the deconv epilogue was store-transaction-bound at ~5.6 k
// cycles per tile).  Here a warp owns ALL channels of its 32 pixels for every other tile (its own TMEM
// buffer), stages one plane of them in 4 KB of shared memory (16-byte chunks XOR-swizzled against bank
// conflicts) and writes it back with consecutive lanes on consecutive 16-byte chunks: a warp's 8-pixel rows
// are contiguous in the NHWC tensor, so every store instruction covers whole 512-byte runs.
constexpr uint32_t kU16StagePerWarp = 4096;
constexpr uint32_t kU16StageBytes = 8 * kU16StagePerWarp;

__host__ __device__ inline bool u16_staged_ok(const LayerArgs& a, int mode, int nbuf, int cend, bool slices_ok = false, bool allow64 = false) {
  if (nbuf < 2 || a.out_mode != IO_ACT16 || (a.cout & 15) != 0) return false;
  if (mode == U16_DECONV) return false;                       // tap-based 64-channel deconv: one TMEM buffer
  // 64-channel conv layers: 32 pixels x 128 B is exactly a warp's 4 KB stage (measured: encode_2 0.47 -> 0.38 ms, the
  // residual layers 0.21 -> 0.19 ms, the plain 8x8x64 layers 0.145 -> 0.14 ms, same output)
  if (!(cend == 16 || cend == 32 || (cend == 64 && (mode == U16_S1 || mode == U16_S2) && allow64))) return false;
  if (cend != a.cout && !slices_ok) return false;             // output-channel slices: the row is not owned by one launch
  return true;
}

__device__ __forceinline__ void sts128(uint32_t addr, uint32_t x, uint32_t y, uint32_t z, uint32_t w) {
  asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(x), "r"(y), "r"(z), "r"(w) : "memory");
}
__device__ __forceinline__ uint32_t lds32(uint32_t addr) {
  uint32_t v;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ uint4 lds128(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr) : "memory");
  return v;
}

// CEND = channels of this launch per pixel (16 | 32 | 64): all stage index arithmetic is compile-time.
template <int MODE, int CEND>
__device__ __forceinline__ void u16_epilogue_tile_staged_t(const LayerArgs& a, const int NPAD, const int oc0, const int nsplit,
                                                           const uint32_t tbuf, const int n, const int yt, const int xt,
                                                           const bool valid, const float* s_bias, const uint32_t stage,
                                                           const int lane, const int cpad, uint64_t* rel_bar,
                                                           const int rel_kind, __half2& omax) {
  constexpr bool kPh = u16_is_ph(MODE);
  constexpr int M = CEND >> 3;                       // 16-byte chunks per pixel and plane: 2 | 4 | 8
  constexpr int MSH = M == 2 ? 1 : (M == 4 ? 2 : 3);
  constexpr int FSH = 3 - MSH;                       // swizzle: chunk ^= (pixel >> FSH) & (M - 1)
  constexpr int NCI = CEND / 16;
  constexpr int NPX = kPh ? 2 : 1;
  constexpr int NPIX = kPh ? 64 : 32;                // output pixels per warp and pass
  const float floor_v = a.act ? 0.0f : -INFINITY;
  const long long pix0 = ((long long)n * a.hout + (kPh ? 2 * yt : yt)) * a.wout + (kPh ? 2 * xt : xt);
  // offset of this lane's (first) output pixel inside a plane in 16-byte units; -1 = invalid pixel (odd tail patch)
  const int my_off16 = valid ? (int)(((pix0 * a.cout + oc0) * 2) >> 4) : -1;
  const int row16 = (a.cout * 2) >> 4;               // one pixel row in 16-byte units
  uint4* const ohi = reinterpret_cast<uint4*>(a.out);
  uint4* const olo = reinterpret_cast<uint4*>(reinterpret_cast<__half*>(a.out) + a.out_lo_off);
  const __half* const rbase = a.res ? reinterpret_cast<const __half*>(a.res) + pix0 * a.cout + oc0 : nullptr;
#pragma unroll 1
  for (int py = 0; py < (kPh ? 2 : 1); ++py) {
    uint32_t lp[NPX][NCI][8];                        // lo' words kept while the hi plane goes through the stage
#pragma unroll
    for (int px = 0; px < NPX; ++px) {
      const int ph = py * 2 + px;
      const int spix = kPh ? ((lane >> 3) * 16 + 2 * (lane & 7) + px) : lane;   // pixel slot in the stage
      const uint32_t sp = stage + (uint32_t)spix * (M * 16);
      const int sw = (spix >> FSH) & (M - 1);
      // all TMEM reads of this pixel first (one wait for its NCI chunks), then the math
      float vv[NCI][16];
      if (kPh || MODE == U16_DECONV || nsplit == 1) {
        float uu[NCI][16];
#pragma unroll
        for (int ci = 0; ci < NCI; ++ci) {
          const uint32_t t0 = tbuf + (kPh ? (uint32_t)(ph * cpad) : (uint32_t)ph * 2u * NPAD) + ci * 16;
          ptx::tmem_ld16_nowait(t0 + NPAD, uu[ci]);
          ptx::tmem_ld16_nowait(t0, vv[ci]);
        }
        ptx::tmem_ld_wait();
#pragma unroll
        for (int ci = 0; ci < NCI; ++ci)
#pragma unroll
          for (int i = 0; i < 16; ++i) vv[ci][i] = __fmaf_rn(uu[ci][i], 1.0f / 2048.0f, vv[ci][i]);
      } else {
#pragma unroll
        for (int ci = 0; ci < NCI; ++ci) u16_load_chunk<MODE>(vv[ci], tbuf, NPAD, nsplit, ph, ci * 16, cpad);
      }
#pragma unroll
      for (int ci = 0; ci < NCI; ++ci) {
        const int c = ci * 16;
        float(&v)[16] = vv[ci];
        if (px == NPX - 1 && ci == 0 && py == (kPh ? 1 : 0)) {
          // last TMEM read of this tile: hand the accumulator buffer back before the remaining math and stores, so the
          // MMAs of the tile after next overlap them (with two buffers the hand-over latency was serialised: decode_1
          // ran at epilogue + MMA time per tile)
          ptx::tc_fence_before();
          __syncwarp();
          if (lane == 0) {
            if (rel_kind == 2)
              ptx::mbar_arrive_leader(rel_bar);
            else
              ptx::mbar_arrive(rel_bar);
          }
        }
        const float4* bp = reinterpret_cast<const float4*>(s_bias + c);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float4 b = bp[i];
          v[4 * i] = fmaxf(__fadd_rn(v[4 * i], b.x), floor_v);
          v[4 * i + 1] = fmaxf(__fadd_rn(v[4 * i + 1], b.y), floor_v);
          v[4 * i + 2] = fmaxf(__fadd_rn(v[4 * i + 2], b.z), floor_v);
          v[4 * i + 3] = fmaxf(__fadd_rn(v[4 * i + 3], b.w), floor_v);
        }
        if (!kPh && rbase && valid) {
          const uint4* rh = reinterpret_cast<const uint4*>(rbase + c);
          const uint4* rl = reinterpret_cast<const uint4*>(rbase + a.res_lo_off + c);
#pragma unroll
          for (int j = 0; j < 2; ++j) {
            const uint4 qh = __ldg(rh + j), ql = __ldg(rl + j);
            const __half2* h2 = reinterpret_cast<const __half2*>(&qh);
            const __half2* l2 = reinterpret_cast<const __half2*>(&ql);
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float2 hf = __half22float2(h2[e]), lf = __half22float2(l2[e]);
              v[8 * j + 2 * e] = __fadd_rn(__fmaf_rn(lf.x, 1.0f / 2048.0f, hf.x), v[8 * j + 2 * e]);
              v[8 * j + 2 * e + 1] = __fadd_rn(__fmaf_rn(lf.y, 1.0f / 2048.0f, hf.y), v[8 * j + 2 * e + 1]);
            }
          }
        }
        uint32_t hp[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) split16x2(v[2 * i], v[2 * i + 1], hp[i], lp[px][ci][i], omax);
        sts128(sp + (uint32_t)(((2 * ci) ^ sw) << 4), hp[0], hp[1], hp[2], hp[3]);
        sts128(sp + (uint32_t)(((2 * ci + 1) ^ sw) << 4), hp[4], hp[5], hp[6], hp[7]);
      }
    }
    // ---- write back one plane: chunk q of the stage -> its pixel's row in global memory ------------------
    const int row_off16 = kPh ? py * a.wout * row16 : 0;
    auto flush = [&](uint4* plane) {
      __syncwarp();
#pragma unroll
      for (int j = 0; j < NPIX * M / 32; ++j) {
        const int q = lane + 32 * j;
        const int sp_ix = q >> MSH, cq = q & (M - 1);
        const int owner = kPh ? ((sp_ix >> 4) * 8 + ((sp_ix & 15) >> 1)) : sp_ix;
        const int base = __shfl_sync(0xffffffffu, my_off16, owner);
        const int sw = (sp_ix >> FSH) & (M - 1);
        const uint4 val = lds128(stage + (uint32_t)((sp_ix * M + (cq ^ sw)) << 4));
        if (base >= 0 && !(TIC_DBG_BITS(a.dbg) & 8)) plane[(long long)base + row_off16 + (kPh ? (sp_ix & 1) * row16 : 0) + cq] = val;
      }
      __syncwarp();
    };
    flush(ohi);
#pragma unroll
    for (int px = 0; px < NPX; ++px) {
      const int spix = kPh ? ((lane >> 3) * 16 + 2 * (lane & 7) + px) : lane;
      const uint32_t sp = stage + (uint32_t)spix * (M * 16);
      const int sw = (spix >> FSH) & (M - 1);
#pragma unroll
      for (int ci = 0; ci < NCI; ++ci) {
        sts128(sp + (uint32_t)(((2 * ci) ^ sw) << 4), lp[px][ci][0], lp[px][ci][1], lp[px][ci][2], lp[px][ci][3]);
        sts128(sp + (uint32_t)(((2 * ci + 1) ^ sw) << 4), lp[px][ci][4], lp[px][ci][5], lp[px][ci][6], lp[px][ci][7]);
      }
    }
    flush(olo);
  }
}

template <int MODE>
__device__ __forceinline__ void u16_epilogue_tile_staged(const LayerArgs& a, const int NPAD, const int oc0, const int nsplit,
                                                         const uint32_t tbuf, const int n, const int yt, const int xt,
                                                         const bool valid, const float* s_bias, uint8_t* stage, const int lane,
                                                         const int cpad, uint64_t* rel_bar, const int rel_kind, __half2& omax) {
  // rel_bar: the tile buffer's `acc_empty` barrier, arrived on (rel_kind 1: this CTA's, 2: the pair leader's) by lane 0
  // right after the tile's last TMEM read
  if (MODE == U16_DECONV_RGB) return;
  const int cend = u16_is_ph(MODE) ? cpad : NPAD;
  const uint32_t st = ptx::smem_u32(stage);
  if (cend == 32)
    u16_epilogue_tile_staged_t<MODE, 32>(a, NPAD, oc0, nsplit, tbuf, n, yt, xt, valid, s_bias, st, lane, cpad, rel_bar, rel_kind, omax);
  else if (cend == 16)
    u16_epilogue_tile_staged_t<MODE, 16>(a, NPAD, oc0, nsplit, tbuf, n, yt, xt, valid, s_bias, st, lane, cpad, rel_bar, rel_kind, omax);
  else if (cend == 64 && !u16_is_ph(MODE) && MODE != U16_DECONV)   // 32 pixels x 128 B = the warp's 4 KB stage
    u16_epilogue_tile_staged_t<(u16_is_ph(MODE) || MODE == U16_DECONV) ? U16_S1 : MODE, 64>(a, NPAD, oc0, nsplit, tbuf, n, yt, xt, valid, s_bias, st, lane,
                                                                                          cpad, rel_bar, rel_kind, omax);
}

// KS = MMAs (K = 16) per tap and K-block, compile-time: with a run-time bound the unrolled body carries four
// predicated instruction groups per tap, and the issuing warp's instruction stream — not the tensor pipe — is what
// bounds the layers with small N (TIC_DBG=6: 105 cycles per MMA in decode_0 against 58 in the rate probe).
template <int MODE, int KS>
__device__ __forceinline__ void u16_issue_plane_t(const U16Params& p, uint32_t abase, uint32_t wbase, uint32_t dplane,
                                                  uint32_t pairw, uint32_t idesc, uint32_t a_hi32, uint32_t w_hi32,
                                                  uint32_t tapw, uint32_t smask, uint32_t& sp, uint32_t& fresh_left,
                                                  bool fresh_kb) {
#pragma unroll
  for (int tap = 0; tap < (u16_is_ph(MODE) ? 4 : 9); ++tap) {  // PH: tap = view
    const uint32_t ad = abase + (p.a_off[tap] >> 4);
    const uint32_t bd = wbase + (uint32_t)tap * tapw;
#pragma unroll
    for (int ks = 0; ks < KS; ++ks) {
      uint32_t d, accumulate;
      if (u16_is_ph(MODE)) {
        d = dplane;
        accumulate = (fresh_kb && tap == 0 && ks == 0) ? 0u : 1u;
      } else if (MODE == U16_DECONV) {
        const int kh = tap / 3, kw = tap - kh * 3;
        const uint32_t ph = (uint32_t)((kh == 1) * 2 + (kw == 1));
        d = dplane + ph * pairw;
        const bool first_tap = (tap == 0 || tap == 1 || tap == 3 || tap == 4);
        accumulate = (fresh_kb && first_tap && ks == 0) ? 0u : 1u;
      } else {
        d = dplane + sp * pairw;
        sp = (sp + 1u) & smask;
        accumulate = fresh_left ? 0u : 1u;
        fresh_left = fresh_left ? fresh_left - 1u : 0u;
      }
      ptx::mma2_f16_ss(d, u16_desc(ad + 2u * ks, a_hi32), u16_desc(bd + 2u * ks, w_hi32), idesc, accumulate);
    }
  }
}

template <int MODE>
__device__ __forceinline__ void u16_issue_plane(const U16Params& p, uint32_t abase, uint32_t wbase, uint32_t dplane,
                                                uint32_t pairw, uint32_t idesc, uint32_t a_hi32, uint32_t w_hi32,
                                                uint32_t tapw, int ksteps, uint32_t smask, uint32_t& sp, uint32_t& fresh_left,
                                                bool fresh_kb) {
  if (ksteps == 2)  // 32-channel K-blocks
    u16_issue_plane_t<MODE, 2>(p, abase, wbase, dplane, pairw, idesc, a_hi32, w_hi32, tapw, smask, sp, fresh_left, fresh_kb);
  else if (ksteps == 4)  // 64-channel K-blocks
    u16_issue_plane_t<MODE, 4>(p, abase, wbase, dplane, pairw, idesc, a_hi32, w_hi32, tapw, smask, sp, fresh_left, fresh_kb);
  else
    u16_issue_plane_t<MODE, 1>(p, abase, wbase, dplane, pairw, idesc, a_hi32, w_hi32, tapw, smask, sp, fresh_left, fresh_kb);
}

// ---- CTA-pair variant (cta_group::2) ------------------------------------------------------------------
// Measured (tests/probe/umma_2cta_probe.cu): an M = 256 MMA over a CTA pair costs 58 / 60 / 64 / 128 cycles
// for N = 32 / 64 / 128 / 256 — less than the single-CTA M = 128 instruction (89 / 97 / 113 / 171) for twice
// the rows.  Two CTAs of a cluster each own one 128-pixel tile: own TMA loads into own shared memory, own
// TMEM, own epilogue; the leader's elected lane issues every MMA for both.  Each CTA keeps HALF of every
// weight tile (leader W_hi, peer W_lo' for the stacked product; a half of W_hi each for A_lo' x W_hi).
// Barriers: `full` lives in the leader and counts the bytes of both CTAs' boxes; `empty` and `acc_full` are
// committed to both CTAs (multicast); `acc_empty` lives in the leader and collects both epilogues.
// PPS = planes per ring slot (compile-time: the issuing warp's instruction stream bounds the layers with small N, and
// any run-time structure in it — loops, branches, calls — measured 5-25 % slower on those layers).
// EW = epilogue warps (8 | 16): four per TMEM lane quadrant for the quantiser layer, whose per-element sigmoid makes the
// epilogue the tile time (see u16_launch_pair_pps for what was measured on the other layers).  The staged epilogue (a warp
// group per TMEM buffer) and the 3-channel image epilogue need eight.
template <int MODE, int PPS, int EW>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(128 + 32 * EW, 1)
u16_pair_kernel(const __grid_constant__ CUtensorMap tm_hi, const __grid_constant__ CUtensorMap tm_lo, const U16Params p,
                const LayerArgs a) {
  const int NPAD = p.npad;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* s_wA = smem;                                            // this CTA's half of the stacked weight tiles
  uint8_t* s_wB = smem + ((p.wA_bytes + 1023u) & ~1023u);          // this CTA's half of W_hi
  uint8_t* s_a = s_wB + ((p.wB_bytes + 1023u) & ~1023u);           // S plane slots
  uint8_t* s_stage = s_a + (size_t)p.S * p.slot_bytes;             // 8 x 4 KB epilogue stages (if p.staged)
  U16SmemBars* bars = reinterpret_cast<U16SmemBars*>(s_stage + (p.staged ? kU16StageBytes : 0u));
  __shared__ unsigned s_hist[256];
  __shared__ __align__(16) float s_bias[128];

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t rank = ptx::cluster_ctarank();
  const bool leader = rank == 0;

  if (tid < 128) s_bias[tid] = (tid < NPAD && p.oc0 + tid < a.cout) ? a.bias[p.oc0 + tid] : 0.f;
  if (tid == 0) {
    ptx::mbar_init(&bars->w_full, leader ? 2 : 1);  // leader: own bytes + the peer's "my weights landed"
    for (int i = 0; i < p.S; ++i) {
      ptx::mbar_init(&bars->full[i], 1);
      ptx::mbar_init(&bars->empty[i], 1);
    }
    for (int i = 0; i < 4; ++i) {
      ptx::mbar_init(&bars->acc_full[i], 1);
      ptx::mbar_init(&bars->acc_empty[i], p.staged ? 8 : 2 * EW);  // epilogue warps of both CTAs (leader's copy is the live one)
    }
    ptx::fence_barrier_init();
  }
  if (warp == 2) {
    ptx::tmem_alloc2(&bars->tmem_base, 512);
    ptx::tmem_relinquish2();
  }
  for (int i = tid; i < 256; i += 128 + 32 * EW) s_hist[i] = 0;
  ptx::tc_fence_before();
  __syncthreads();
  ptx::cluster_sync();  // the peer's barriers exist before anything remote touches them
  ptx::tc_fence_after();
  const uint32_t tmem_base = bars->tmem_base;
  const long long npairs = gridDim.x >> 1, pair0 = blockIdx.x >> 1;
  const long long num_pairs = (p.num_tiles + 1) >> 1;
  const uint32_t SR = (uint32_t)p.S / (uint32_t)PPS;   // ring slots

  if (warp == 0) {
    // ===== TMA producer (both CTAs): own weight halves once, then per tile and K-block the two planes =====
    if (ptx::elect_one()) {
      ptx::prefetch_tmap(&tm_hi);
      ptx::prefetch_tmap(&tm_lo);
      const uint8_t* src = p.wimg + (size_t)rank * (((p.wA_bytes + 1023u) & ~1023u) + ((p.wB_bytes + 1023u) & ~1023u));
      ptx::mbar_expect_tx(&bars->w_full, p.wA_bytes + p.wB_bytes);
      for (uint32_t off = 0; off < p.wA_bytes; off += 16384u)
        ptx::bulk_load(s_wA + off, src + off, min(16384u, p.wA_bytes - off), &bars->w_full);
      const uint8_t* srcB = src + ((p.wA_bytes + 1023u) & ~1023u);
      for (uint32_t off = 0; off < p.wB_bytes; off += 16384u)
        ptx::bulk_load(s_wB + off, srcB + off, min(16384u, p.wB_bytes - off), &bars->w_full);
    }
    __syncwarp();
    if (!leader) {
      ptx::mbar_wait(&bars->w_full, 0);
      if (ptx::elect_one()) ptx::mbar_arrive_leader(&bars->w_full);
      __syncwarp();
    }
    uint32_t s = 0, sph = 1;  // ring slot and the parity to wait for on its `empty` barrier
    for (long long tp = pair0; tp < num_pairs; tp += npairs) {
      long long tt = 2 * tp + rank;
      uint32_t tq, tx, ty, tn;
      fast_divmod((uint32_t)tt, p.tx_d, tq, tx);
      fast_divmod(tq, p.ty_d, tn, ty);
      const int n0 = (int)tn * p.bn;
      const int x0 = (int)tx * 8, y0 = (int)ty * p.bh;
      // one ring slot = the hi AND the lo' box of a K-block (one barrier round trip per K-block, not per plane: the
      // fixed cost of a wait / commit pair in the single issuing warp is ~350 cycles, TIC_DBG=7)
      // one ring slot = PPS planes of a K-block: the hi AND the lo' box when four plane buffers fit (one barrier round
      // trip per K-block, not per plane: the fixed cost of a wait / commit pair in the single issuing warp is ~350
      // cycles, TIC_DBG=7), else one plane
      for (int kb = 0; kb < p.KB; ++kb) {
#pragma unroll
        for (int pl0 = 0; pl0 < 2; pl0 += PPS) {
          ptx::mbar_wait(&bars->empty[s], sph);
          if (TIC_DBG_BITS(p.dbg) & 2) {
            if (leader && ptx::elect_one()) ptx::mbar_arrive(&bars->full[s]);
          } else if (ptx::elect_one()) {
            if (leader) ptx::mbar_expect_tx(&bars->full[s], (uint32_t)PPS * 2u * p.box_bytes * (uint32_t)p.nbox);
#pragma unroll
            for (int q = 0; q < PPS; ++q) {
              const CUtensorMap* tm = (pl0 + q) ? &tm_lo : &tm_hi;
              uint8_t* dst = s_a + (size_t)((uint32_t)PPS * s + (uint32_t)q) * p.slot_bytes;
              if (MODE == U16_S2) {
                ptx::tma2_load_5d(dst, tm, &bars->full[s], kb * p.kc, x0, 0, n0, y0);
                if (p.nbox == 2) ptx::tma2_load_5d(dst + p.box_stride, tm, &bars->full[s], a.cin + kb * p.kc, x0, 0, n0, y0);
              } else {
                ptx::tma2_load_4d(dst, tm, &bars->full[s], kb * p.kc, x0 - 1, n0, y0 - 1);
              }
            }
          }
          __syncwarp();
          if (++s == SR) {
            s = 0;
            sph ^= 1u;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer (leader CTA only) =====
    if (leader) {
      const uint32_t idesc_st = ptx::make_idesc_f16(256, 2 * NPAD);
      const uint32_t idesc_lo = ptx::make_idesc_f16(256, NPAD);
      const uint32_t a_hi32 = (p.sbo >> 4) | (1u << 14) | (p.a_layout << 29);
      const uint32_t w_hi32 = (p.w_sbo >> 4) | (1u << 14) | (p.w_layout << 29);
      constexpr uint32_t T = u16_is_ph(MODE) ? 4u : 9u;
      const uint32_t tapA = (uint32_t)NPAD * (uint32_t)p.kc * 2u, tapB = tapA >> 1;
      const uint32_t pairw = 2u * (uint32_t)NPAD, smask = (uint32_t)p.nsplit - 1u;
      const int ksteps = p.ksteps;
      ptx::mbar_wait(&bars->w_full, 0);
      uint32_t ti = 0, s = 0, sph = 0;
      for (long long tp = pair0; tp < num_pairs; tp += npairs, ++ti) {
        const uint32_t b = ti & ((uint32_t)p.nbuf - 1u);
        const uint32_t use = ti >> p.nbshift;
        ptx::mbar_wait(&bars->acc_empty[b], (use & 1) ^ 1);
        ptx::tc_fence_after();
        const uint32_t dbase = tmem_base + b * p.acc_cols;
        for (int kb = 0; kb < p.KB; ++kb) {
#pragma unroll
          for (int pl0 = 0; pl0 < 2; pl0 += PPS) {
            ptx::mbar_wait(&bars->full[s], sph);
            ptx::tc_fence_after();
            if (!(TIC_DBG_BITS(p.dbg) & 1) && ptx::elect_one()) {
#pragma unroll
              for (int q = 0; q < PPS; ++q) {
                const int plane = pl0 + q;
                const uint32_t abase =
                    (ptx::smem_u32(s_a + (size_t)((uint32_t)PPS * s + (uint32_t)q) * p.slot_bytes) >> 4) | (1u << 16);
                const uint32_t wbase = plane ? (ptx::smem_u32(s_wB + (size_t)kb * T * tapB) >> 4) | (1u << 16)
                                             : (ptx::smem_u32(s_wA + (size_t)kb * T * tapA) >> 4) | (1u << 16);
                uint32_t sp = 0, fresh_left = (plane == 0 && kb == 0) ? (uint32_t)p.nsplit : 0u;
                u16_issue_plane<MODE>(p, abase, wbase, dbase + (plane ? (uint32_t)NPAD : 0u), pairw, plane ? idesc_lo : idesc_st,
                                      a_hi32, w_hi32, (plane ? tapB : tapA) >> 4, ksteps, smask, sp, fresh_left,
                                      plane == 0 && kb == 0);
              }
            }
            __syncwarp();
            if (ptx::elect_one()) ptx::tc_commit2(&bars->empty[s]);
            __syncwarp();
            if (++s == SR) {
              s = 0;
              sph ^= 1u;
            }
          }
        }
        if (ptx::elect_one()) ptx::tc_commit2(&bars->acc_full[b]);
        __syncwarp();
      }
    }
  } else if (warp >= 4) {
    // ===== epilogue (both CTAs, own tile, own TMEM) =====
    const int q4 = warp & 3;
    const int half = (warp - 4) >> 2;
    const int m = q4 * 32 + lane;
    const int grp = m >> 3, xx = m & 7;
    const int hh = grp / p.bn, nb = grp % p.bn;
    int h_ones = 0, h_valid = 0;
    __half2 omax = __floats2half2_rn(0.f, 0.f);
    uint32_t ti = 0;
    for (long long tp = pair0; tp < num_pairs; tp += npairs, ++ti) {
      if (EW == 8 && p.staged && (int)(ti & 1u) != half) continue;  // staged: a warp group owns every other tile (= one TMEM buffer)
      const uint32_t b = ti & ((uint32_t)p.nbuf - 1u);
      const uint32_t use = ti >> p.nbshift;
      ptx::mbar_wait(&bars->acc_full[b], use & 1);
      ptx::tc_fence_after();
      long long tt = 2 * tp + rank;
      uint32_t tq, tx, ty, tn;
      fast_divmod((uint32_t)tt, p.tx_d, tq, tx);
      fast_divmod(tq, p.ty_d, tn, ty);
      const int n = (int)tn * p.bn + nb;
      const int yt = (int)ty * p.bh + hh, xt = (int)tx * 8 + xx;
      const bool valid = n < p.n;
      const uint32_t tbuf = tmem_base + ((uint32_t)(q4 * 32) << 16) + b * p.acc_cols;
      if (TIC_DBG_BITS(p.dbg) & 4) {
      } else if (EW == 8 && p.staged) {
        u16_epilogue_tile_staged<MODE>(a, NPAD, p.oc0, p.nsplit, tbuf, n, yt, xt, valid, s_bias,
                                       s_stage + (size_t)(warp - 4) * kU16StagePerWarp, lane, p.cpad, &bars->acc_empty[b], 2, omax);
        continue;  // the staged epilogue released the buffer itself
      } else
        u16_epilogue_tile<MODE, EW / 4>(a, NPAD, p.oc0, p.nsplit, tbuf, n, yt, xt, valid, half, s_bias, s_hist, h_ones, h_valid, omax, p.cpad);
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive_leader(&bars->acc_empty[b]);
    }
    if (ovf_hit(omax)) ovf_raise(a.oflow);
    if (a.out_mode == IO_QUANT_U8 || a.out_mode == IO_QUANT_F32) {
      if (a.q == 2) {
        h_ones = __reduce_add_sync(0xffffffffu, h_ones);
        h_valid = __reduce_add_sync(0xffffffffu, h_valid);
        if (lane == 0) {
          if (h_ones) atomicAdd(&s_hist[1], (unsigned)h_ones);
          if (h_valid - h_ones) atomicAdd(&s_hist[0], (unsigned)(h_valid - h_ones));
        }
      }
      asm volatile("bar.sync 1, %0;" ::"n"(32 * EW) : "memory");
      for (int i = tid - 128; i < a.q; i += 32 * EW)
        if (s_hist[i]) atomicAdd(&a.hist[i], (unsigned long long)s_hist[i]);
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  ptx::cluster_sync();  // neither CTA may leave (or free TMEM) while the pair still has MMAs / remote arrives in flight
  if (warp == 2) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc2(tmem_base, 512);
  }
}

// ---- host side -------------------------------------------------------------------------------
inline int u16_mode_of(int kind, int stride) { return kind == 1 ? U16_DECONV : (stride == 2 ? U16_S2 : U16_S1); }

// Which layers the fp16-pair tensor path takes (input must already be pair planes).
inline bool u16_supported(const LayerArgs& a, int kind, int stride) {
  if (a.in_mode != IO_ACT16) return false;
  if (!(a.cin == 16 || a.cin == 32 || (a.cin % 64 == 0 && a.cin <= 512))) return false;
  const int mode = u16_mode_of(kind, stride);
  const bool last3 = mode == U16_DECONV && a.cout <= 4;  // 3-channel last layer: phase-stacked deconv, N = 16
  if (a.cout < 16 && !last3) return false;
  if (last3 && a.out_mode == IO_ACT16) return false;
  const int Ht = mode == U16_DECONV ? a.hin : a.hout, Wt = mode == U16_DECONV ? a.win : a.wout;
  if (Wt % 8 != 0) return false;
  if (!(Ht == 8 || Ht % 16 == 0)) return false;
  if (mode == U16_S2 && (a.hin != 2 * a.hout || a.win != 2 * a.wout)) return false;
  if ((a.out_mode == IO_ACT16 || a.res16) && (a.cout % 8) != 0) return false;
  if ((a.out_mode == IO_ACT || (a.res && !a.res16)) && (a.cout % 4) != 0) return false;
  if ((a.out_mode == IO_DENORM_F32 || a.out_mode == IO_DENORM_U8) && !last3) return false;
  return true;
}

template <int MODE, int PPS, int EW>
inline cudaError_t u16_launch_pair_ew(cudaStream_t stream, const CUtensorMap& th, const CUtensorMap& tl, const U16Params& p,
                                      const LayerArgs& a, int grid, size_t smem) {
  // __cluster_dims__(2, 1, 1): grid is even
  return launch_dyn(u16_pair_kernel<MODE, PPS, EW>, grid, 128 + 32 * EW, smem, stream, th, tl, p, a);
}
template <int MODE, int PPS>
inline cudaError_t u16_launch_pair_pps(cudaStream_t stream, const CUtensorMap& th, const CUtensorMap& tl, const U16Params& p,
                                       const LayerArgs& a, int grid, size_t smem) {
  // sixteen epilogue warps only for the quantiser layer (sigmoid + symbol + histogram per element: encode_4 0.23 -> 0.17 ms).
  // Measured on every other un-staged layer: slower (8x8x64 convs 0.14 -> 0.18 ms, encode_2 0.43 -> 0.59, decode_3 0.41 ->
  // 0.44): the 96-register cap of 640 threads and the extra warps cost the issuing warp more than the epilogue gains.
  if (MODE == U16_S1 && !p.staged && (a.out_mode == IO_QUANT_U8 || a.out_mode == IO_QUANT_F32))
    return u16_launch_pair_ew<MODE, PPS, MODE == U16_S1 ? 16 : 8>(stream, th, tl, p, a, grid, smem);
  return u16_launch_pair_ew<MODE, PPS, 8>(stream, th, tl, p, a, grid, smem);
}
template <int MODE>
inline cudaError_t u16_launch_pair_t(cudaStream_t stream, const CUtensorMap& th, const CUtensorMap& tl, const U16Params& p,
                                     const LayerArgs& a, int grid, size_t smem) {
  // both planes of a K-block share a ring slot when four plane buffers fit
  return p.S >= 4 ? u16_launch_pair_pps<MODE, 2>(stream, th, tl, p, a, grid, smem)
                  : u16_launch_pair_pps<MODE, 1>(stream, th, tl, p, a, grid, smem);
}

struct U16Plan {
  int cs;      // output channels per slice
  int variant; // u16_plan's variant bits
  U16Params p;
  size_t smem;
};

// Geometry + shared-memory plan for one slice width; returns false if it does not fit.
// variant: bit 0 = 32-channel K-blocks (half-size operand slots), bit 1 = no staged epilogue (its 32 KB go to the ring)
inline bool u16_plan(const LayerArgs& a, int kind, int stride, int cs, U16Plan* out, int variant = 0) {
  U16Params p{};
  p.pair = 1;
  p.mode = u16_mode_of(kind, stride);
  p.n = a.n;
  p.Ht = p.mode == U16_DECONV ? a.hin : a.hout;
  p.Wt = p.mode == U16_DECONV ? a.win : a.wout;
  p.bn = p.Ht == 8 ? 2 : 1;
  p.bh = p.Ht == 8 ? 8 : 16;
  p.tiles_x = p.Wt / 8;
  p.tiles_y = p.Ht / p.bh;
  p.num_tiles = (long long)p.tiles_x * p.tiles_y * ((a.n + p.bn - 1) / p.bn);
  if (p.num_tiles >= (1LL << 31) - 65536) return false;  // FastDiv range (and the 32-bit tile counters)
  p.tx_d = make_fastdiv((uint32_t)p.tiles_x);
  p.ty_d = make_fastdiv((uint32_t)p.tiles_y);
  p.kc = std::min(a.cin, (variant & 1) ? 32 : 64);
  p.KB = a.cin / p.kc;
  p.ksteps = p.kc / 16;
  p.npad = (cs + 15) / 16 * 16;
  if (p.mode == U16_DECONV && cs <= 32) {
    p.mode = U16_DECONV_PH;
    p.cpad = cs <= 4 ? 4 : (cs + 15) / 16 * 16;
    p.npad = (4 * p.cpad + 15) / 16 * 16;  // N = (phase, channel)
  }
  const uint32_t wrow = (uint32_t)p.kc * 2u;
  uint32_t arow = wrow;
  int box_rows, bw;
  if (p.mode == U16_S1) {
    bw = 10;
    box_rows = bw * p.bn * (p.bh + 2);
    for (int kh = 0; kh < 3; ++kh)
      for (int kw = 0; kw < 3; ++kw) p.a_off[kh * 3 + kw] = (uint32_t)((kh * p.bn) * bw + kw) * arow;
    p.sbo = (uint32_t)bw * arow;
    p.nbox = 1;
  } else if (p.mode == U16_DECONV_PH) {
    bw = 9;
    box_rows = bw * p.bn * (p.bh + 1);
    // view (dy, dx) reads input row a - 1 + dy, column b - 1 + dx; box row 0 / column 0 = a-1 / b-1
    for (int v = 0; v < 4; ++v) p.a_off[v] = (uint32_t)(((v >> 1) * p.bn) * bw + (v & 1)) * arow;
    p.sbo = (uint32_t)bw * arow;
    p.nbox = 1;
  } else if (p.mode == U16_DECONV) {
    bw = 9;
    box_rows = bw * p.bn * (p.bh + 1);
    // tap (kh, kw) reads input row a - (kh == 2), column b - (kw == 2); box row 0 / column 0 = a-1 / b-1
    for (int kh = 0; kh < 3; ++kh)
      for (int kw = 0; kw < 3; ++kw) {
        const int dy = kh == 2 ? 0 : 1, dx = kw == 2 ? 0 : 1;
        p.a_off[kh * 3 + kw] = (uint32_t)((dy * p.bn) * bw + dx) * arow;
      }
    p.sbo = (uint32_t)bw * arow;
    p.nbox = 1;
  } else {
    bw = 9;
    const bool both = 2u * wrow <= 128u && p.KB == 1;  // a row holds both w parities of one W/2 position
    arow = both ? 2u * wrow : wrow;
    p.nbox = both ? 1 : 2;
    box_rows = bw * 2 * p.bn * (p.bh + 1);
    // input (2 oy + kh, 2 ox + kw): kh -> (h parity, h2 shift) = (0,0) (1,0) (0,1); same for kw
    for (int kh = 0; kh < 3; ++kh)
      for (int kw = 0; kw < 3; ++kw) {
        uint32_t rows = (uint32_t)((kh == 1 ? bw : 0) + (kh == 2 ? 2 * p.bn * bw : 0) + (kw == 2 ? 1 : 0));
        uint32_t off = rows * arow;
        if (kw == 1) off += both ? wrow : 0u;
        p.a_off[kh * 3 + kw] = off;  // second-parity box offset added below (needs box_stride)
      }
    p.sbo = (uint32_t)(2 * bw) * arow;
  }
  p.a_layout = u16_layout_code(arow);
  p.w_layout = u16_layout_code(wrow);
  p.w_sbo = 8u * wrow;
  p.box_bytes = (uint32_t)box_rows * arow;
  p.box_stride = (p.box_bytes + 1023u) & ~1023u;
  if (p.mode == U16_S2 && p.nbox == 2)
    for (int kh = 0; kh < 3; ++kh) p.a_off[kh * 3 + 1] += p.box_stride;
  p.slot_bytes = p.box_stride * (uint32_t)p.nbox;
  p.tap_bytes = 2u * (uint32_t)p.npad * wrow;
  p.w_bytes = (uint32_t)p.KB * (p.mode == U16_DECONV_PH ? 4u : 9u) * p.tap_bytes;
  // each CTA of the pair keeps half of every stacked tile plus half of W_hi
  p.wA_bytes = p.w_bytes / 2;
  p.wB_bytes = p.w_bytes / 4;
  p.w_bytes = ((p.wA_bytes + 1023u) & ~1023u) + ((p.wB_bytes + 1023u) & ~1023u);
  // TMEM: conv nsplit pairs x 2 buffers; deconv 4 phase pairs
  const int accw = 2 * p.npad;  // one (D_main | D_lo) accumulator pair
  if (p.mode == U16_DECONV_PH) {
    p.nsplit = 1;
    p.acc_cols = (uint32_t)accw;
    p.nbuf = accw * 4 <= 512 ? 4 : 2;
  } else if (p.mode == U16_DECONV) {
    p.nsplit = 1;
    p.acc_cols = 4u * accw;
    if (p.acc_cols > 512) return false;
    p.nbuf = p.acc_cols * 2 <= 512 ? 2 : 1;
  } else {
    if (accw > 512) return false;
    p.nbuf = accw * 2 <= 512 ? 2 : 1;
    // the tensor core truncates when adding into the accumulator: keep <= ~18 accumulation steps per
    // accumulator (what a 32-channel layer has unsplit), power of two, as TMEM allows
    const int steps = p.KB * 9 * p.ksteps;
    const int cap = (512 / p.nbuf) / accw;
    p.nsplit = 1;
    while (p.nsplit * 2 <= cap && p.nsplit < 4 && steps > 18 * p.nsplit) p.nsplit *= 2;
    p.acc_cols = (uint32_t)(p.nsplit * accw);
    if (p.acc_cols * 4 <= 512) p.nbuf = 4;
  }
  // Four tile buffers wherever TMEM holds them: the accumulator hand-over (tcgen05.commit -> epilogue wake-up -> cross-CTA
  // arrive -> issuer wake-up) is ~1400 cycles; with two buffers that alone is ~700 cycles per tile (TIC_DBG=7 skeleton:
  // 0.96 of decode_0's 1.95 ms).
  p.nbshift = p.nbuf == 4 ? 2 : (p.nbuf == 2 ? 1 : 0);
  p.dbg = tic_env_int("TIC_DBG", 0);  // -DTIC_ABLATE builds only
  if (2 * p.npad > 256) return false;  // MMA N limit for the stacked product
  // (phase-stacked output-channel slices keep the staged epilogue: a slice owns 64 contiguous bytes of every pixel row)
  p.staged = u16_staged_ok(a, p.mode, p.nbuf, p.mode == U16_DECONV_PH ? p.cpad : p.npad, p.mode == U16_DECONV_PH, true) ? 1 : 0;
  if (variant & 2) p.staged = 0;
  const size_t budget = 227 * 1024 - 2048 /* static histogram + bias */ - 1024 /* alignment slack */ - sizeof(U16SmemBars) - 256;
  const size_t wres = ((p.w_bytes + 1023u) & ~1023u) + (p.staged ? kU16StageBytes : 0u);
  if (wres + 2 * (size_t)p.slot_bytes > budget) return false;
  p.S = (int)std::min<size_t>(kU16MaxSlots, (budget - wres) / p.slot_bytes);
  if (p.S >= 4) p.S &= ~1;  // the pair kernel's ring slots hold both planes when four plane buffers fit
  out->cs = cs;
  out->variant = variant;
  out->p = p;
  out->smem = wres + (size_t)p.S * p.slot_bytes + sizeof(U16SmemBars) + 1024;
  return true;
}

// The CTA-pair weight image of output channels [oc0, oc0 + cs) of a layer for plan p (u16_build_weights_pair_kernel).
inline tic_status u16_pair_image(cudaStream_t stream, OperandImage& img, const float* w_dev, const LayerArgs& a, const U16Params& p,
                                 int oc0, int cs) {
  const uint32_t regA = (p.wA_bytes + 1023u) & ~1023u, regB = (p.wB_bytes + 1023u) & ~1023u;
  const int ph_mode = p.mode == U16_DECONV_PH;
  bool build;
  if (img.ensure(image_key(w_dev, a.cin, a.cout, oc0, cs, p.npad, p.cpad, ph_mode, p.kc, p.KB, regA, regB), 2 * (size_t)p.w_bytes,
                 &build) != TIC_OK)
    return TIC_ERR_NOMEM;
  if (build) {
    u16_build_weights_pair_kernel<<<64, 256, 0, stream>>>(w_dev, a.cin, a.cout, oc0, cs, p.npad, p.cpad, ph_mode, p.kc, p.KB, regA,
                                                          regB, img.buf.as<uint8_t>());
    if (cudaGetLastError() != cudaSuccess) return TIC_ERR_CUDA;
  }
  return TIC_OK;
}

inline tic_status launch_u16(const LaunchCtx& c, const LayerArgs& a, int kind, int stride, const float* w_dev, OperandImage* slices) {
  if (c.num_sms < 2) return c.fail("the fp16-pair tensor kernels need CTA pairs", TIC_ERR_UNSUPPORTED);
  // widest output-channel slice whose weights stay resident
  U16Plan plan{};
  int cs = std::min(a.cout, 128);
  // Transposed convs with 64 or more output channels run as phase-stacked 32-channel slices WITH the staged epilogue:
  // decode_3 (64 -> 64 on 8 x 8 maps) 0.42 ms tap-based (one TMEM buffer, epilogue-bound on 16-byte strided stores), 0.37 ms
  // as slices with the direct epilogue, 0.28 ms as slices with the staged one; the input (small) is read once per slice.
  if (kind == 1 && a.cout >= 64 && a.cout % 32 == 0) cs = std::min(cs, 32);
  cs =  (cs + 15) / 16 * 16;
  bool ok = false;
  // A stride-2 conv with 64 input channels whose full-width plan does not fit (two 83 KB parity boxes per plane next to
  // 110 KB of weights) is tried with 32-channel K-blocks before its output channels are sliced: the slices each re-read
  // the input (encode_3: 2 x 0.145 ms at 6.2 TB/s).
  const bool small_kc = kind == 0 && stride == 2 && a.cin == 64;
  for (; cs >= 16; cs -= 16) {
    const int csl = std::min(cs, a.cout);
    ok = u16_plan(a, kind, stride, csl, &plan);
    if (!ok && small_kc) ok = u16_plan(a, kind, stride, csl, &plan, 1) || u16_plan(a, kind, stride, csl, &plan, 3);
    if (ok) break;
  }
  if (!ok) return c.fail("layer does not fit the fp16-pair tensor path", TIC_ERR_UNSUPPORTED);
  cs = plan.cs;

  // tensor maps over the two planes of the input activation [n, hin, win, cin] fp16
  CUtensorMap tm[2];
  const U16Params& p0 = plan.p;
  const CUtensorMapSwizzle sw = p0.a_layout == 2 ? CU_TENSOR_MAP_SWIZZLE_128B
                                : p0.a_layout == 4 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B;
  const cuuint32_t box[4] = {(cuuint32_t)(p0.mode == U16_S2 && p0.nbox == 1 ? 2 * p0.kc : p0.kc), (cuuint32_t)(p0.mode == U16_S1 ? 10 : 9),
                             (cuuint32_t)p0.bn, (cuuint32_t)(p0.bh + (p0.mode == U16_S1 ? 2 : 1))};
  for (int pl = 0; pl < 2; ++pl)
    if (tic_status s = tmap_act(&tm[pl], reinterpret_cast<const __half*>(a.in) + (pl ? a.in_lo_off : 0), true, a, p0.mode == U16_S2, box,
                                sw, c.err))
      return s;

  int si = 0;
  for (int oc0 = 0; oc0 < a.cout; oc0 += cs, ++si) {
    if (si >= 16) return c.fail("too many output-channel slices", TIC_ERR_UNSUPPORTED);
    const int csl = std::min(cs, a.cout - oc0);
    U16Plan pl{};
    if (!u16_plan(a, kind, stride, csl, &pl, plan.variant)) return c.fail("slice plan failed", TIC_ERR_UNSUPPORTED);
    U16Params p = pl.p;
    p.oc0 = oc0;
    if (tic_status s = u16_pair_image(c.stream, slices[si], w_dev, a, p, oc0, csl))
      return c.fail(s == TIC_ERR_NOMEM ? "cudaMalloc for weight images failed" : "weight image kernel failed", s);
    p.wimg = slices[si].img();
    const int grid = 2 * (int)std::min<long long>((p.num_tiles + 1) / 2, c.num_sms / 2);
    cudaError_t e;
    if (p.mode == U16_S1)
      e = u16_launch_pair_t<U16_S1>(c.stream, tm[0], tm[1], p, a, grid, pl.smem);
    else if (p.mode == U16_S2)
      e = u16_launch_pair_t<U16_S2>(c.stream, tm[0], tm[1], p, a, grid, pl.smem);
    else if (p.mode == U16_DECONV_PH && p.cpad == 4)
      e = u16_launch_pair_t<U16_DECONV_RGB>(c.stream, tm[0], tm[1], p, a, grid, pl.smem);
    else if (p.mode == U16_DECONV_PH)
      e = u16_launch_pair_t<U16_DECONV_PH>(c.stream, tm[0], tm[1], p, a, grid, pl.smem);
    else
      e = u16_launch_pair_t<U16_DECONV>(c.stream, tm[0], tm[1], p, a, grid, pl.smem);
    if (e != cudaSuccess) return c.fail(std::string("fp16-pair tensor launch failed: ") + cudaGetErrorString(e), TIC_ERR_CUDA);
    ++*c.launches;
  }
  return TIC_OK;
}

}  // namespace tic

// tcgen05 / TMEM / TMA implicit-GEMM kernels for the 3x3 conv (stride 1 and 2) and the stride-2
// transposed conv of the codec (basic_block/basic_block.py:27-71) — compute modes
// TIC_COMPUTE_TENSOR_3XTF32 (error-compensated, default tensor mode) and TIC_COMPUTE_TENSOR_TF32.
//
// GEMM view (per filter tap): D[128 pixels, Cout] += A[128 pixels, 32 channels] * W[Cout, 32 channels]^T
//   * A: NHWC fp32 activations, staged by TMA (SWIZZLE_128B) as K-major tiles: one 128-byte row per
//     pixel, 8-pixel groups of 1024 B.  A tile is 8 columns x 16 (row, patch) pairs.  The tensor map
//     orders the dims (C, W, N, H) so the box rows come out (h, n, x)-major: a filter-row shift (kh) is
//     then a 1024-byte-aligned start offset of the SAME shared-memory box and only the three filter
//     columns (kw) need separate loads — 3 box loads instead of 9 per K-block.  Out-of-range
//     coordinates are zero-filled by TMA = TF "SAME" padding.  Stride 2 uses a 5-D map
//     ((w parity, C), W/2, h parity, N, H/2) and a group stride (SBO) of 2048 B; the transposed conv
//     walks INPUT pixels and feeds four sub-pixel phase accumulators (taps 4+2+2+1, no zero insertion).
//   * W: per (K-block, filter column) group, pre-swizzled hi / lo images, bulk-copied to shared memory.
//   * D: fp32 accumulators in TMEM, up to 8 tiles (512 columns) live per CTA so a weight group is
//     loaded once per 8 tiles.
//   * 3xTF32: the tensor core TRUNCATES fp32 operands to tf32 (measured: tests/probe/umma_probe.cu); a
//     truncating split is biased (measured 2e-5 relative error after 9 layers), so converter warps
//     rewrite each tile as hi = rn_tf32(x) in place and lo = rn_tf32(x - hi) beside it (weights are
//     pre-split the same way); D += A_lo*W_hi + A_hi*W_lo + A_hi*W_hi, small terms first.
// Warp roles (384 threads): 0 A-tile TMA producer, 1 weight producer, 2 MMA issuer (one thread),
// 3 TMEM allocator, 4-7 lo-converters, 8-11 epilogue (TMEM -> registers -> bias/act/residual/quantise -> global).
#pragma once
#include <cuda.h>

#include <string>

#include "tic_common.cuh"
#include "tic_launch.cuh"
#include "tic_ptx.cuh"
#include "tic_simt.cuh"

namespace tic {

enum UmmaMode : int { UMMA_S1 = 0, UMMA_S2 = 1, UMMA_DECONV = 2 };

constexpr int kUmmaThreads = 384;
constexpr int kMaxStages = 4;
constexpr int kMaxTiles = 8;

struct UmmaParams {
  int mode;
  int n;                   // patches
  int Ht, Wt;              // tile-space map (S1/S2: output map, DECONV: input map)
  int bn, bh;              // patches per tile (1 | 2), map rows per tile per patch (16 | 8)
  int tiles_x, tiles_y;
  long long num_tiles;
  int T;                   // tiles per super-tile (accumulator slots)
  long long num_super;
  int KB;                  // input-channel blocks of 32
  int cin;
  int gw;                  // weight groups per K-block (S1/S2: 3 filter columns, DECONV: 2)
  int npad;                // MMA N (cout rounded up to 16)
  int phases;              // output sub-pixel phases per tile (DECONV: 4, else 1)
  int nacc;                // TMEM accumulators per tile (see accumulator split below)
  int split_lo;            // lo-term products (A_lo*W_hi, A_hi*W_lo) go to their own accumulator
  int split_kw;            // S1/S2: one hi*hi accumulator per filter column
  uint32_t box_bytes;      // one TMA box (raw tile); the lo tile has the same size
  uint32_t sbo;
  uint32_t a_off[3];
  uint32_t tap_bytes;      // bytes of one tap image pair (hi + lo): 2 * npad * 128
  int S, WB;               // A stages, weight buffers
  uint32_t wbuf_bytes;
  int three_pass;
  const uint8_t* wimg;     // weight images, groups consecutive
  int oc0;                 // first output channel of this launch (layers with cout > 64 run in 64-channel slices)
};

// Tap order inside a weight group.  S1/S2 group (kb, kw): kh = 0,1,2.  DECONV group (kb, 0) = input
// column b-1: W22, W02, W12; group (kb, 1) = input column b: W20, W21, W00, W01, W10, W11.
__host__ __device__ inline int group_ntaps(int mode, int kwi) { return mode == UMMA_DECONV ? (kwi == 0 ? 3 : 6) : 3; }
__host__ __device__ inline int group_tap_offset(int mode, int kb, int kwi) {
  return mode == UMMA_DECONV ? kb * 9 + (kwi == 0 ? 0 : 3) : (kb * 3 + kwi) * 3;
}
__host__ __device__ inline int group_tap_index(int mode, int kwi, int j) {  // -> kh*3+kw of the TF kernel
  if (mode != UMMA_DECONV) return j * 3 + kwi;
  const int t0[3] = {8, 2, 5};
  const int t1[6] = {6, 7, 0, 1, 3, 4};
  return kwi == 0 ? t0[j] : t1[j];
}

// device [9][cin][cout] fp32 -> grouped, swizzled hi/lo operand images
__global__ void umma_build_weights_kernel(const float* __restrict__ w, int cin, int cout, int oc0, int npad, int mode, int KB,
                                          int gw, uint8_t* __restrict__ img) {
  const int total_taps = KB * 9;
  const long long total = (long long)total_taps * npad * 32;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int k = (int)(i % 32);
    int oc = (int)((i / 32) % npad);
    int tp = (int)(i / (32LL * npad));  // position in the grouped tap sequence
    int kb = tp / 9, r = tp % 9;
    int kwi, j;
    if (mode == UMMA_DECONV) {
      kwi = r < 3 ? 0 : 1;
      j = r < 3 ? r : r - 3;
    } else {
      kwi = r / 3;
      j = r % 3;
    }
    int tap = group_tap_index(mode, kwi, j);
    int ic = kb * 32 + k;
    float v = (oc0 + oc < cout && ic < cin) ? w[((size_t)tap * cin + ic) * cout + oc0 + oc] : 0.f;
    // round-to-nearest split (unbiased): hi = rn_tf32(v), lo = rn_tf32(v - hi).  The single-pass mode
    // reads the hi image too (rounded weights, truncated activations).
    float hi = ptx::rn_tf32(v);
    float lo = ptx::rn_tf32(v - hi);
    uint8_t* base = img + (size_t)tp * (2u * npad * 128u);
    *reinterpret_cast<float*>(base + ptx::sw128_offset(oc, k)) = hi;
    *reinterpret_cast<float*>(base + npad * 128u + ptx::sw128_offset(oc, k)) = lo;
  }
}

struct UmmaSmemBars {
  uint64_t a_full[kMaxStages], a_conv[kMaxStages], a_empty[kMaxStages];
  uint64_t w_full[2], w_empty[2];
  uint64_t acc_full[kMaxTiles], acc_empty[kMaxTiles];
  uint32_t tmem_base;
};

// 4 K-steps (4 x 8 channels = one 128-byte swizzle row) of one A-tile x W-tile product into one
// accumulator.  Descriptors are handled as (lo32, hi32) pairs: a K-step of 32 bytes is +2 in the low
// word (start address >> 4); everything else is loop-invariant — the single issuing thread must not
// spend more than a few instructions per MMA or it, not the tensor core, bounds the kernel.
__device__ __forceinline__ void umma_k4(uint32_t d_tmem, uint32_t a_lo32, uint32_t a_hi32, uint32_t b_lo32, uint32_t b_hi32,
                                        uint32_t idesc, uint32_t accumulate_first) {
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    uint64_t ad, bd;
    asm("mov.b64 %0, {%1, %2};" : "=l"(ad) : "r"(a_lo32 + 2 * k), "r"(a_hi32));
    asm("mov.b64 %0, {%1, %2};" : "=l"(bd) : "r"(b_lo32 + 2 * k), "r"(b_hi32));
    ptx::mma_tf32_ss(d_tmem, ad, bd, idesc, k == 0 ? accumulate_first : 1u);
  }
}

// One filter tap of one tile: 3xTF32 = A_lo*W_hi and A_hi*W_lo into the lo accumulator, A_hi*W_hi into
// the main accumulator (small terms first); single pass = A*W_hi only.  `first` = the accumulators have
// not been written in this super-tile yet (the first MMA overwrites instead of accumulating).
template <bool THREE_PASS>
__device__ __forceinline__ void umma_tap(uint32_t d_main, uint32_t d_lo, uint32_t a_hi_desc, uint32_t a_lo_desc,
                                         uint32_t a_hi32, uint32_t w_hi_desc, uint32_t w_lo_desc, uint32_t w_hi32,
                                         uint32_t idesc, bool first) {
  if (THREE_PASS) {
    umma_k4(d_lo, a_lo_desc, a_hi32, w_hi_desc, w_hi32, idesc, first ? 0u : 1u);
    umma_k4(d_lo, a_hi_desc, a_hi32, w_lo_desc, w_hi32, idesc, 1u);
    umma_k4(d_main, a_hi_desc, a_hi32, w_hi_desc, w_hi32, idesc, (first && d_main != d_lo) ? 0u : 1u);
  } else {
    umma_k4(d_main, a_hi_desc, a_hi32, w_hi_desc, w_hi32, idesc, first ? 0u : 1u);
  }
}

template <int MODE, bool THREE_PASS>
__global__ void __launch_bounds__(kUmmaThreads, 1)
umma_conv_kernel(const __grid_constant__ CUtensorMap tmap, const UmmaParams p, const LayerArgs a) {
  const int NPAD = p.npad;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  // carve: [WB weight buffers][S x (raw, lo) stages][barriers]; dynamic smem base is 1024-aligned by the
  // launch (we still round up defensively)
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* s_w = smem;
  uint8_t* s_a = smem + (size_t)p.WB * p.wbuf_bytes;
  UmmaSmemBars* bars = reinterpret_cast<UmmaSmemBars*>(s_a + (size_t)p.S * 2 * p.box_bytes);
  __shared__ unsigned s_hist[256];

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int groups = p.KB * p.gw;

  if (tid == 0) {
    for (int i = 0; i < p.S; ++i) {
      ptx::mbar_init(&bars->a_full[i], 1);
      ptx::mbar_init(&bars->a_conv[i], 4);
      ptx::mbar_init(&bars->a_empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      ptx::mbar_init(&bars->w_full[i], 1);
      ptx::mbar_init(&bars->w_empty[i], 1);
    }
    for (int i = 0; i < kMaxTiles; ++i) {
      ptx::mbar_init(&bars->acc_full[i], 1);
      ptx::mbar_init(&bars->acc_empty[i], 4);
    }
    ptx::fence_barrier_init();
  }
  if (warp == 3) {
    ptx::tmem_alloc(&bars->tmem_base, 512);
    ptx::tmem_relinquish();
  }
  hist_begin(s_hist);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = bars->tmem_base;

  if (warp == 0) {
    // ===== A-tile TMA producer =====
    if (lane == 0) {
      ptx::prefetch_tmap(&tmap);
      uint32_t it = 0;
      for (long long st = blockIdx.x; st < p.num_super; st += gridDim.x) {
        const long long tile0 = st * p.T;
        const int tcount = (int)min((long long)p.T, p.num_tiles - tile0);
        for (int g = 0; g < groups; ++g) {
          const int kb = g / p.gw, kwi = g % p.gw;
          for (int t = 0; t < tcount; ++t, ++it) {
            const int s = it % p.S;
            const uint32_t use = it / p.S;
            ptx::mbar_wait(&bars->a_empty[s], (use & 1) ^ 1);
            long long tile = tile0 + t;
            const int tx = (int)(tile % p.tiles_x);
            tile /= p.tiles_x;
            const int ty = (int)(tile % p.tiles_y);
            const int n0 = (int)(tile / p.tiles_y) * p.bn;
            const int x0 = tx * 8, y0 = ty * p.bh;
            uint8_t* dst = s_a + (size_t)s * 2 * p.box_bytes;
            ptx::mbar_expect_tx(&bars->a_full[s], p.box_bytes);
            if (MODE == UMMA_S1)
              ptx::tma_load_4d(dst, &tmap, &bars->a_full[s], kb * 32, x0 + kwi - 1, n0, y0 - 1);
            else if (MODE == UMMA_DECONV)
              ptx::tma_load_4d(dst, &tmap, &bars->a_full[s], kb * 32, x0 - 1 + kwi, n0, y0 - 1);
            else
              ptx::tma_load_5d(dst, &tmap, &bars->a_full[s], (kwi & 1) * p.cin + kb * 32, x0 + (kwi >> 1), 0, n0, y0);
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===== weight-group producer =====
    if (lane == 0) {
      uint32_t it = 0;
      for (long long st = blockIdx.x; st < p.num_super; st += gridDim.x) {
        for (int g = 0; g < groups; ++g, ++it) {
          const int kb = g / p.gw, kwi = g % p.gw;
          const int wb = it % p.WB;
          const uint32_t use = it / p.WB;
          ptx::mbar_wait(&bars->w_empty[wb], (use & 1) ^ 1);
          const uint32_t bytes = (uint32_t)group_ntaps(p.mode, kwi) * p.tap_bytes;
          ptx::mbar_expect_tx(&bars->w_full[wb], bytes);
          ptx::bulk_load(s_w + (size_t)wb * p.wbuf_bytes, p.wimg + (size_t)group_tap_offset(p.mode, kb, kwi) * p.tap_bytes, bytes,
                         &bars->w_full[wb]);
        }
      }
    }
  } else if (warp == 2) {
    // ===== MMA issuer (single thread) =====
    if (lane == 0) {
      const uint32_t idesc = ptx::make_idesc_tf32(128, NPAD);
      // descriptor words: lo = (addr >> 4) | LBO(1) << 16 ; hi = SBO >> 4 | version 1 << 14 | SWIZZLE_128B 2 << 29
      const uint32_t a_hi32 = (p.sbo >> 4) | (1u << 14) | (2u << 29);
      const uint32_t w_hi32 = (1024u >> 4) | (1u << 14) | (2u << 29);
      const uint32_t tapw = p.tap_bytes >> 4, lo_img = (uint32_t)(NPAD * 128) >> 4, boxw = p.box_bytes >> 4;
      const uint32_t aoff0 = p.a_off[0] >> 4, aoff1 = p.a_off[1] >> 4, aoff2 = p.a_off[2] >> 4;
      const uint32_t ncol = (uint32_t)NPAD, nacc = (uint32_t)p.nacc;
      uint32_t ait = 0, wit = 0, sti = 0;
      for (long long st = blockIdx.x; st < p.num_super; st += gridDim.x, ++sti) {
        const long long tile0 = st * p.T;
        const int tcount = (int)min((long long)p.T, p.num_tiles - tile0);
        for (int g = 0; g < groups; ++g, ++wit) {
          const int kb = g / p.gw, kwi = g % p.gw;
          const int wb = wit % p.WB;
          ptx::mbar_wait(&bars->w_full[wb], (wit / p.WB) & 1);
          const uint32_t wd = ((ptx::smem_u32(s_w + (size_t)wb * p.wbuf_bytes) >> 4) & 0x3FFF) | (1u << 16);
          for (int t = 0; t < tcount; ++t, ++ait) {
            const int s = ait % p.S;
            ptx::mbar_wait(THREE_PASS ? &bars->a_conv[s] : &bars->a_full[s], (ait / p.S) & 1);
            if (g == 0) ptx::mbar_wait(&bars->acc_empty[t], (sti & 1) ^ 1);
            ptx::tc_fence_after();
            const uint32_t ah = ((ptx::smem_u32(s_a + (size_t)s * 2 * p.box_bytes) >> 4) & 0x3FFF) | (1u << 16);
            const uint32_t al = ah + boxw;
            const uint32_t d0 = tmem_base + (uint32_t)t * nacc * ncol;
            if (MODE != UMMA_DECONV) {
              // accumulators: [0..2] hi*hi per filter column (or [0] if !split_kw), [nacc-1] lo terms
              const uint32_t d_main = d0 + (p.split_kw ? (uint32_t)kwi : 0u) * ncol;
              const uint32_t d_lo = THREE_PASS ? d0 + (nacc - 1) * ncol : d_main;
              const bool first_main = p.split_kw ? (kb == 0) : (g == 0);
              const bool first_lo = (g == 0);
              // kh = 0: may open both accumulators
              if (THREE_PASS) {
                umma_k4(d_lo, al + aoff0, a_hi32, wd, w_hi32, idesc, first_lo ? 0u : 1u);
                umma_k4(d_lo, ah + aoff0, a_hi32, wd + lo_img, w_hi32, idesc, 1u);
              }
              umma_k4(d_main, ah + aoff0, a_hi32, wd, w_hi32, idesc, first_main ? 0u : 1u);
              umma_tap<THREE_PASS>(d_main, d_lo, ah + aoff1, al + aoff1, a_hi32, wd + tapw, wd + tapw + lo_img, w_hi32, idesc, false);
              umma_tap<THREE_PASS>(d_main, d_lo, ah + aoff2, al + aoff2, a_hi32, wd + 2 * tapw, wd + 2 * tapw + lo_img, w_hi32, idesc, false);
            } else {
              // accumulators: [ph] hi*hi per output phase, [4+ph] lo terms (if split_lo)
              const uint32_t lo_sh = (THREE_PASS && p.split_lo) ? 4u * ncol : 0u;
              const bool f = (kb == 0);
#define TIC_DTAP(J, AOFF, PH, FIRST)                                                                             \
  umma_tap<THREE_PASS>(d0 + (PH) * ncol, d0 + (PH) * ncol + lo_sh, ah + (AOFF), al + (AOFF), a_hi32, wd + (J) * tapw, \
                       wd + (J) * tapw + lo_img, w_hi32, idesc, (FIRST))
              if (kwi == 0) {  // input column b-1: W22 (row a-1) -> ee ; W02 (row a) -> ee ; W12 (row a) -> oe
                TIC_DTAP(0, aoff0, 0u, f);
                TIC_DTAP(1, aoff1, 0u, false);
                TIC_DTAP(2, aoff1, 2u, f);
              } else {         // input column b: W20, W21 (row a-1) -> ee, eo ; W00, W01, W10, W11 (row a) -> ee, eo, oe, oo
                TIC_DTAP(0, aoff0, 0u, false);
                TIC_DTAP(1, aoff0, 1u, f);
                TIC_DTAP(2, aoff1, 0u, false);
                TIC_DTAP(3, aoff1, 1u, false);
                TIC_DTAP(4, aoff1, 2u, false);
                TIC_DTAP(5, aoff1, 3u, f);
              }
#undef TIC_DTAP
            }
            ptx::tc_commit(&bars->a_empty[s]);
            if (g == groups - 1) ptx::tc_commit(&bars->acc_full[t]);
          }
          ptx::tc_commit(&bars->w_empty[wb]);
        }
      }
    }
  } else if (warp >= 4 && warp < 8) {
    // ===== hi/lo converters: hi = rn_tf32(x) (in place), lo = rn_tf32(x - hi); layout unchanged =====
    if (THREE_PASS) {
      const int ctid = tid - 128;
      const uint32_t nvec = p.box_bytes / 16;
      uint32_t it = 0;
      for (long long st = blockIdx.x; st < p.num_super; st += gridDim.x) {
        const long long tile0 = st * p.T;
        const int tcount = (int)min((long long)p.T, p.num_tiles - tile0);
        const int steps = groups * tcount;
        for (int i = 0; i < steps; ++i, ++it) {
          const int s = it % p.S;
          ptx::mbar_wait(&bars->a_full[s], (it / p.S) & 1);
          float4* src = reinterpret_cast<float4*>(s_a + (size_t)s * 2 * p.box_bytes);
          float4* dst = reinterpret_cast<float4*>(s_a + (size_t)s * 2 * p.box_bytes + p.box_bytes);
          for (uint32_t v = ctid; v < nvec; v += 128) {
            const float4 x = src[v];
            float4 h, l;
            h.x = ptx::rn_tf32(x.x); l.x = ptx::rn_tf32(x.x - h.x);
            h.y = ptx::rn_tf32(x.y); l.y = ptx::rn_tf32(x.y - h.y);
            h.z = ptx::rn_tf32(x.z); l.z = ptx::rn_tf32(x.z - h.z);
            h.w = ptx::rn_tf32(x.w); l.w = ptx::rn_tf32(x.w - h.w);
            src[v] = h;  // hi in place: already tf32, so the tensor core's truncation is exact
            dst[v] = l;
          }
          ptx::fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive(&bars->a_conv[s]);
        }
      }
    }
  } else if (warp >= 8) {
    // ===== epilogue: TMEM -> registers -> bias / activation / residual / quantise / denormalise -> global =====
    const int q4 = warp & 3;            // TMEM lane quadrant this warp may access
    const int m = q4 * 32 + lane;       // tile row = pixel
    const int grp = m >> 3, xx = m & 7;
    const int hh = grp / p.bn, nb = grp % p.bn;
    int h_ones = 0, h_valid = 0;
    uint32_t sti = 0;
    for (long long st = blockIdx.x; st < p.num_super; st += gridDim.x, ++sti) {
      const long long tile0 = st * p.T;
      const int tcount = (int)min((long long)p.T, p.num_tiles - tile0);
      for (int t = 0; t < tcount; ++t) {
        ptx::mbar_wait(&bars->acc_full[t], sti & 1);
        ptx::tc_fence_after();
        long long tile = tile0 + t;
        const int tx = (int)(tile % p.tiles_x);
        tile /= p.tiles_x;
        const int ty = (int)(tile % p.tiles_y);
        const int n = (int)(tile / p.tiles_y) * p.bn + nb;
        const int yt = ty * p.bh + hh, xt = tx * 8 + xx;
        const bool valid = n < p.n;
        for (int ph = 0; ph < p.phases; ++ph) {
          const int y = MODE == UMMA_DECONV ? 2 * yt + (ph >> 1) : yt;
          const int x = MODE == UMMA_DECONV ? 2 * xt + (ph & 1) : xt;
          for (int c = 0; c < NPAD; c += 16) {
            float v[16];
            const uint32_t tbase = tmem_base + ((uint32_t)(q4 * 32) << 16) + (uint32_t)(t * p.nacc) * NPAD + c;
            if (MODE == UMMA_DECONV) {
              if (p.split_lo && THREE_PASS) {
                float u[16];
                ptx::tmem_ld16(tbase + (uint32_t)(4 + ph) * NPAD, v);
                ptx::tmem_ld16(tbase + (uint32_t)ph * NPAD, u);
#pragma unroll
                for (int i = 0; i < 16; ++i) v[i] = __fadd_rn(v[i], u[i]);
              } else {
                ptx::tmem_ld16(tbase + (uint32_t)ph * NPAD, v);
              }
            } else {
              // lo accumulator first, then the hi*hi accumulators, fp32 round-to-nearest adds
              const int nsum = THREE_PASS ? p.nacc : (p.split_kw ? 3 : 1);
              ptx::tmem_ld16(tbase + (uint32_t)(THREE_PASS ? p.nacc - 1 : 0) * NPAD, v);
              for (int q = 0; q < nsum - 1; ++q) {
                float u[16];
                ptx::tmem_ld16(tbase + (uint32_t)(THREE_PASS ? q : q + 1) * NPAD, u);
#pragma unroll
                for (int i = 0; i < 16; ++i) v[i] = __fadd_rn(v[i], u[i]);
              }
            }
            const int oc = p.oc0 + c;
            if (valid && oc < a.cout) {
#pragma unroll
              for (int i = 0; i < 16; ++i) {
                const float b = (oc + i < a.cout) ? __ldg(a.bias + oc + i) : 0.f;
                v[i] = apply_act(__fadd_rn(v[i], b), a.act);
              }
              if (a.res) {
                const float* rp = a.res + (((long long)n * a.hout + y) * a.wout + x) * a.cout + oc;
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
              store_pixel<16>(a, n, y, x, oc, v, s_hist, h_ones, h_valid);
            }
          }
        }
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(&bars->acc_empty[t]);
      }
    }
    // symbol histogram (quantising layers): reduce the 4 epilogue warps through shared memory
    if (a.out_mode == IO_QUANT_U8 || a.out_mode == IO_QUANT_F32) {
      if (a.q == 2) {
        h_ones = __reduce_add_sync(0xffffffffu, h_ones);
        h_valid = __reduce_add_sync(0xffffffffu, h_valid);
        if (lane == 0) {
          if (h_ones) atomicAdd(&s_hist[1], (unsigned)h_ones);
          if (h_valid - h_ones) atomicAdd(&s_hist[0], (unsigned)(h_valid - h_ones));
        }
      }
      asm volatile("bar.sync 1, 128;" ::: "memory");  // the four epilogue warps only
      for (int i = tid - 256; i < a.q; i += 128)
        if (s_hist[i]) atomicAdd(&a.hist[i], (unsigned long long)s_hist[i]);
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 3) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, 512);
  }
}

// ---- host side -------------------------------------------------------------------------------
inline int umma_mode_of(int kind, int stride) { return kind == 1 ? UMMA_DECONV : (stride == 2 ? UMMA_S2 : UMMA_S1); }

// Which layers the tensor path takes; everything else (first layer with 3 input channels, fused u8
// prologues, odd map sizes) runs on the fp32 CUDA-core kernels.
inline bool umma_supported(const LayerArgs& a, int kind, int stride) {
  if (a.in_mode != IO_ACT) return false;
  if (a.cin % 32 != 0 || a.cin > 256) return false;
  const int npad = (a.cout + 15) / 16 * 16;
  const int mode = umma_mode_of(kind, stride);
  if (npad > 256) return false;
  if (a.cout < 16) return false;  // 3-channel output layers are bandwidth-bound: CUDA-core kernel
  const int Ht = mode == UMMA_DECONV ? a.hin : a.hout, Wt = mode == UMMA_DECONV ? a.win : a.wout;
  if (Wt % 8 != 0) return false;
  if (!(Ht == 8 || Ht % 16 == 0)) return false;
  if (mode == UMMA_S2 && (a.hin != 2 * a.hout || a.win != 2 * a.wout)) return false;
  if (a.out_mode == IO_ACT && (a.cout % 4) != 0) return false;
  if (a.res && (a.cout % 4) != 0) return false;
  return true;
}

inline tic_status launch_umma_slice(const LaunchCtx& c, const LayerArgs& a, int kind, int stride, const float* w_dev,
                                    OperandImage& img, int oc0, int cs, bool three_pass) {
  UmmaParams p{};
  p.mode = umma_mode_of(kind, stride);
  p.n = a.n;
  p.Ht = p.mode == UMMA_DECONV ? a.hin : a.hout;
  p.Wt = p.mode == UMMA_DECONV ? a.win : a.wout;
  p.bn = p.Ht == 8 ? 2 : 1;
  p.bh = p.Ht == 8 ? 8 : 16;
  p.tiles_x = p.Wt / 8;
  p.tiles_y = p.Ht / p.bh;
  p.num_tiles = (long long)p.tiles_x * p.tiles_y * ((a.n + p.bn - 1) / p.bn);
  p.KB = a.cin / 32;
  p.cin = a.cin;
  p.gw = p.mode == UMMA_DECONV ? 2 : 3;
  p.npad = (cs + 15) / 16 * 16;
  p.oc0 = oc0;
  p.phases = p.mode == UMMA_DECONV ? 4 : 1;
  // accumulator split (accuracy) vs tiles per weight-group load (L2 traffic): keep at least 2 tiles
  if (p.mode == UMMA_DECONV) {
    p.split_kw = 0;
    p.split_lo = (three_pass && 512 / (p.npad * 8) >= 2) ? 1 : 0;
    p.nacc = p.split_lo ? 8 : 4;
  } else {
    p.split_kw = (512 / (p.npad * (three_pass ? 4 : 3)) >= 2) ? 1 : 0;
    p.split_lo = three_pass ? 1 : 0;
    p.nacc = (p.split_kw ? 3 : 1) + p.split_lo;
  }
  p.T = std::min(kMaxTiles, 512 / (p.npad * p.nacc));
  if (p.T < 1) return c.fail("accumulators do not fit TMEM", TIC_ERR_UNSUPPORTED);
  p.num_super = (p.num_tiles + p.T - 1) / p.T;
  p.three_pass = three_pass ? 1 : 0;
  p.tap_bytes = 2u * p.npad * 128u;
  int box_rows;
  if (p.mode == UMMA_S1) {
    box_rows = 8 * p.bn * (p.bh + 2);
    p.sbo = 1024;
    p.a_off[0] = 0;
    p.a_off[1] = p.bn * 1024;
    p.a_off[2] = 2 * p.bn * 1024;
  } else if (p.mode == UMMA_DECONV) {
    box_rows = 8 * p.bn * (p.bh + 1);
    p.sbo = 1024;
    p.a_off[0] = 0;               // input row a-1
    p.a_off[1] = p.bn * 1024;     // input row a
    p.a_off[2] = 0;
  } else {
    box_rows = 8 * 2 * p.bn * (p.bh + 1);
    p.sbo = 2048;
    p.a_off[0] = 0;
    p.a_off[1] = 1024;
    p.a_off[2] = 2 * p.bn * 1024;
  }
  p.box_bytes = (uint32_t)box_rows * 128u;
  p.wbuf_bytes = (uint32_t)(p.mode == UMMA_DECONV ? 6 : 3) * p.tap_bytes;
  // shared-memory budget: weight buffers + stages + barriers (+ 1 KB alignment slack)
  const size_t budget = 227 * 1024 - 2048;
  const size_t stage = 2 * (size_t)p.box_bytes;
  p.WB = 2;
  p.S = (int)std::min<size_t>(kMaxStages, (budget - 2 * (size_t)p.wbuf_bytes) / stage);
  if (budget < 2 * (size_t)p.wbuf_bytes || p.S < 2) {
    p.WB = 1;
    if (budget < p.wbuf_bytes) return c.fail("weight group does not fit shared memory", TIC_ERR_UNSUPPORTED);
    p.S = (int)std::min<size_t>(kMaxStages, (budget - p.wbuf_bytes) / stage);
  }
  if (p.S < 1) return c.fail("A stages do not fit shared memory", TIC_ERR_UNSUPPORTED);
  const size_t smem = (size_t)p.WB * p.wbuf_bytes + (size_t)p.S * stage + sizeof(UmmaSmemBars) + 1024;

  // weight images (once per layer and mode)
  bool build;
  if (img.ensure(image_key(w_dev, a.cin, a.cout, oc0, p.npad, p.mode, p.KB, p.gw), (size_t)p.KB * 9 * p.tap_bytes, &build) != TIC_OK)
    return c.fail("cudaMalloc for weight images failed", TIC_ERR_NOMEM);
  if (build) {
    umma_build_weights_kernel<<<64, 256, 0, c.stream>>>(w_dev, a.cin, a.cout, oc0, p.npad, p.mode, p.KB, p.gw, img.buf.as<uint8_t>());
    if (cudaGetLastError() != cudaSuccess) return c.fail("weight image kernel failed", TIC_ERR_CUDA);
  }
  p.wimg = img.img();

  // tensor map over the input activation [n, hin, win, cin] fp32
  CUtensorMap tm;
  const cuuint32_t box[4] = {32, 8, (cuuint32_t)p.bn, (cuuint32_t)(p.bh + (p.mode == UMMA_S1 ? 2 : 1))};
  if (tic_status s = tmap_act(&tm, a.in, false, a, p.mode == UMMA_S2, box, CU_TENSOR_MAP_SWIZZLE_128B, c.err)) return s;

  const int grid = (int)std::min<long long>(p.num_super, c.num_sms);
  auto kernel = p.mode == UMMA_S1 ? (three_pass ? umma_conv_kernel<UMMA_S1, true> : umma_conv_kernel<UMMA_S1, false>)
                : p.mode == UMMA_S2 ? (three_pass ? umma_conv_kernel<UMMA_S2, true> : umma_conv_kernel<UMMA_S2, false>)
                                    : (three_pass ? umma_conv_kernel<UMMA_DECONV, true> : umma_conv_kernel<UMMA_DECONV, false>);
  const cudaError_t e = launch_dyn(kernel, grid, kUmmaThreads, smem, c.stream, tm, p, a);
  if (e != cudaSuccess) return c.fail(std::string("tensor-path launch failed: ") + cudaGetErrorString(e), TIC_ERR_CUDA);
  return TIC_OK;
}

// A layer with more than 64 output channels runs as 64-channel slices (same A tiles, disjoint weight
// rows and output channels): N = 64 keeps four split accumulators x two tiles inside the 512 TMEM columns.
inline tic_status launch_umma(const LaunchCtx& c, const LayerArgs& a, int kind, int stride, const float* w_dev, OperandImage* slices,
                              bool three_pass) {
  int si = 0;
  for (int oc0 = 0; oc0 < a.cout; oc0 += 64, ++si) {
    const int cs = std::min(64, a.cout - oc0);
    if (tic_status s = launch_umma_slice(c, a, kind, stride, w_dev, slices[si], oc0, cs, three_pass)) return s;
    ++*c.launches;
  }
  return TIC_OK;
}

}  // namespace tic

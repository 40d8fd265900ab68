// First layer of the encoder / post-filter on the tensor pipe: 3x3 conv over 3 input channels (K = 27,
// padded to 32), stride 1 or 2, with the reference's input pipeline fused into the operand build:
//   utils.crop_image_input_patches (utils/utils.py:96-133: reflect pad, row-major patch grid)  -> index arithmetic
//   (x - mean) / std                (model_0/model.py:44)                                       -> 3 x 256 table (u8) | true division (f32)
//   basic_block.my_conv2d           (basic_block/basic_block.py:27-47)                          -> tcgen05.mma kind::f16, fp16 pairs
// With 3 input channels there is nothing for TMA to tile (a pixel is 3 bytes), so four builder warps
// write the im2col tile themselves: one thread per output pixel gathers its 27 normalised inputs, splits
// them into (hi, lo') fp16 pairs and stores one 64-byte row per plane in the SWIZZLE_64B K-major layout the
// MMA descriptors read.  Per 128-pixel tile: 2 K-steps x (A_hi x [W_hi ; W_lo'] + A_lo' x W_hi) = 4 MMAs.
// Warp roles (544 threads): 0-7 builders (two groups of 128 threads on alternating tiles: the gather is
// latency-bound, all 27 loads of a pixel are issued before any is used), 8-15 epilogue (shared with
// tic_umma16.cuh), 16 MMA issuer + TMEM.
#pragma once
#include "tic_launch.cuh"
#include "tic_umma16.cuh"

namespace tic {

constexpr int kF16Threads = 544;
constexpr int kF16Stages = 4;
constexpr uint32_t kF16StageBytes = 16384;  // hi plane 128 x 64 B | lo' plane 128 x 64 B

struct F16Params {
  int n;                 // patches
  int P;                 // input patch edge
  int stride, pad;       // TF SAME: stride 2 on even maps pads (0, 1); stride 1 pads (1, 1)
  int bn, bh;
  int tiles_x, tiles_y;
  FastDiv tx_d, ty_d, txy_d;  // / tiles_x, / tiles_y, / (tiles_x * tiles_y)
  long long num_tiles;
  int npad;
  int nbuf;              // TMEM tile buffers (power of two, <= 4)
  const uint8_t* wimg;   // [W_hi npad rows ; W_lo' npad rows] x 64 B, SW64
  int use_tma;           // stride-2 kernel: raw u8 windows arrive by TMA (image geometry allows it, f16_first_tma_ok)
  int dbg;               // measurement aid (env TIC_DBG, stride-2 kernel): 1 = no MMA issue, 2 = builders only arrive, 4 = no epilogue work
};

struct F16SmemBars {
  uint64_t full[kF16Stages], empty[kF16Stages];
  uint64_t acc_full[4], acc_empty[4];
  uint32_t tmem_base;
};

// device [9][3][cout] fp32 -> [hi rows npad | lo' rows npad][32] fp16, k = tap * 3 + c, swizzled 64-byte rows
__global__ void f16_build_weights_kernel(const float* __restrict__ w, int cout, int npad, uint8_t* __restrict__ img) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < npad * 32; i += gridDim.x * blockDim.x) {
    const int k = i & 31, oc = i >> 5;
    const float v = (k < 27 && oc < cout) ? w[k * cout + oc] : 0.f;
    __half hi, lo;
    split16(v, hi, lo);
    *reinterpret_cast<__half*>(img + u16_swz((uint32_t)oc * 64u + k * 2, 64)) = hi;
    *reinterpret_cast<__half*>(img + u16_swz((uint32_t)(npad + oc) * 64u + k * 2, 64)) = lo;
  }
}

__device__ __forceinline__ uint32_t pack_half2(__half a, __half b) {
  return (uint32_t)__half_as_ushort(a) | ((uint32_t)__half_as_ushort(b) << 16);
}

template <int S>
__global__ void __launch_bounds__(kF16Threads, 1) f16_first_kernel(const F16Params p, const LayerArgs a) {
  const int NPAD = p.npad;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* s_a = smem;                                        // kF16Stages stages
  uint8_t* s_w = smem + kF16Stages * kF16StageBytes;          // 2 * npad * 64 B
  uint8_t* s_stage = s_w + 2 * 64 * 64;                       // 8 x 4 KB epilogue stages
  F16SmemBars* bars = reinterpret_cast<F16SmemBars*>(s_stage + kU16StageBytes);
  const bool staged = u16_staged_ok(a, U16_S1, p.nbuf, p.npad);
  __shared__ unsigned s_hist[256];
  __shared__ __align__(16) float s_bias[128];
  __shared__ float s_lut[3 * 256];

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  if (tid < 128) s_bias[tid] = (tid < NPAD && tid < a.cout) ? a.bias[tid] : 0.f;
  for (int i = tid; i < 256; i += kF16Threads) s_hist[i] = 0;
  if (a.in_mode == IO_U8_NORM)
    for (int i = tid; i < 3 * 256; i += kF16Threads) s_lut[i] = a.lut[i];
  for (int i = tid; i < 2 * NPAD * 4; i += kF16Threads)  // weight image, 16-byte chunks
    reinterpret_cast<uint4*>(s_w)[i] = __ldg(reinterpret_cast<const uint4*>(p.wimg) + i);
  if (tid == 0) {
    for (int i = 0; i < kF16Stages; ++i) {
      ptx::mbar_init(&bars->full[i], 4);
      ptx::mbar_init(&bars->empty[i], 1);
    }
    for (int i = 0; i < 4; ++i) {
      ptx::mbar_init(&bars->acc_full[i], 1);
      ptx::mbar_init(&bars->acc_empty[i], staged ? 4 : 8);
    }
    ptx::fence_barrier_init();
  }
  if (warp == 16) {
    ptx::tmem_alloc(&bars->tmem_base, 512);
    ptx::tmem_relinquish();
  }
  ptx::fence_proxy_async_smem();
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = bars->tmem_base;
  const uint32_t pairw = 2u * (uint32_t)NPAD;
  const uint32_t bmask = (uint32_t)p.nbuf - 1u;
  int nbshift = 0;
  while ((1 << nbshift) < p.nbuf) ++nbshift;

  if (warp < 8) {
    // ===== builders: one thread per tile row (output pixel); group g takes tiles it = g, g + 2, ... =====
    const int group = warp >> 2;
    const int m = tid & 127;
    const int grp = m >> 3, xx = m & 7;
    const int hh = grp / p.bn, nb = grp % p.bn;
    const uint32_t sw = (uint32_t)((m >> 1) & 3);
    const Geo g = a.geo;
    uint32_t it = (uint32_t)group;
    for (long long tile = blockIdx.x + (long long)group * gridDim.x; tile < p.num_tiles; tile += 2LL * gridDim.x, it += 2) {
      uint32_t tq, tx, ty, tn;
      fast_divmod((uint32_t)tile, p.tx_d, tq, tx);
      fast_divmod(tq, p.ty_d, tn, ty);
      const int n = (int)tn * p.bn + nb;
      const int oy = (int)ty * p.bh + hh, ox = (int)tx * 8 + xx;
      // patch -> image geometry (utils/utils.py:96-133); reflect only ever fires on padded image borders
      const bool nok = n < p.n;
      unsigned img, gy, gx;
      geo_decode(g, (unsigned)(g.n0 + (nok ? n : 0)), img, gy, gx);
      const int Y0 = g.oy + (int)gy * g.P, X0 = g.ox + (int)gx * g.P;
      const long long img_off = (long long)img * g.H * g.W;
      long long off[9];
      bool ok[9];
#pragma unroll
      for (int kh = 0; kh < 3; ++kh) {
        const int iy = oy * S + kh - p.pad;
        const bool yok = nok && iy >= 0 && iy < p.P;
        const long long row = img_off + (long long)reflect_index(Y0 + (yok ? iy : 0), g.H) * g.W;
#pragma unroll
        for (int kw = 0; kw < 3; ++kw) {
          const int ix = ox * S + kw - p.pad;
          const bool xok = ix >= 0 && ix < p.P;
          ok[kh * 3 + kw] = yok && xok;
          off[kh * 3 + kw] = (row + reflect_index(X0 + (xok ? ix : 0), g.W)) * 3;
        }
      }
      float v[27];
      if (a.in_mode == IO_U8_NORM) {
        // all 27 byte loads first (independent, always in bounds), then the table look-ups
        unsigned b[27];
#pragma unroll
        for (int t = 0; t < 9; ++t) {
          const uint8_t* q = reinterpret_cast<const uint8_t*>(a.in) + off[t];
          b[3 * t] = q[0];
          b[3 * t + 1] = q[1];
          b[3 * t + 2] = q[2];
        }
#pragma unroll
        for (int t = 0; t < 9; ++t) {
          v[3 * t] = ok[t] ? s_lut[b[3 * t]] : 0.f;
          v[3 * t + 1] = ok[t] ? s_lut[256 + b[3 * t + 1]] : 0.f;
          v[3 * t + 2] = ok[t] ? s_lut[512 + b[3 * t + 2]] : 0.f;
        }
      } else {
        float b[27];
#pragma unroll
        for (int t = 0; t < 9; ++t) {
          const float* q = reinterpret_cast<const float*>(a.in) + off[t];
          b[3 * t] = q[0];
          b[3 * t + 1] = q[1];
          b[3 * t + 2] = q[2];
        }
#pragma unroll
        for (int t = 0; t < 9; ++t) {
          v[3 * t] = ok[t] ? tic_normalize(b[3 * t], a.mean[0], a.stdv[0]) : 0.f;
          v[3 * t + 1] = ok[t] ? tic_normalize(b[3 * t + 1], a.mean[1], a.stdv[1]) : 0.f;
          v[3 * t + 2] = ok[t] ? tic_normalize(b[3 * t + 2], a.mean[2], a.stdv[2]) : 0.f;
        }
      }
      uint32_t hp[16], lp[16];
#pragma unroll
      for (int k = 0; k < 32; k += 2) {
        __half h0 = __float2half_rn(0.f), l0 = h0, h1 = h0, l1 = h0;
        if (k < 27) split16(v[k], h0, l0);
        if (k + 1 < 27) split16(v[k + 1], h1, l1);
        hp[k >> 1] = pack_half2(h0, h1);
        lp[k >> 1] = pack_half2(l0, l1);
      }
      const int s = it % kF16Stages;
      ptx::mbar_wait(&bars->empty[s], ((it / kF16Stages) & 1) ^ 1);
      uint8_t* rowh = s_a + (size_t)s * kF16StageBytes + (uint32_t)m * 64u;
      uint8_t* rowl = rowh + 8192;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const uint32_t c = ((uint32_t)j ^ sw) << 4;
        *reinterpret_cast<uint4*>(rowh + c) = make_uint4(hp[4 * j], hp[4 * j + 1], hp[4 * j + 2], hp[4 * j + 3]);
        *reinterpret_cast<uint4*>(rowl + c) = make_uint4(lp[4 * j], lp[4 * j + 1], lp[4 * j + 2], lp[4 * j + 3]);
      }
      ptx::fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&bars->full[s]);
    }
  } else if (warp == 16) {
    // ===== MMA issuer =====
    const uint32_t idesc_st = ptx::make_idesc_f16(128, 2 * NPAD);
    const uint32_t idesc_lo = ptx::make_idesc_f16(128, NPAD);
    const uint32_t hi32 = (512u >> 4) | (1u << 14) | (4u << 29);  // SBO 512 B, SWIZZLE_64B
    const uint32_t wbase = (ptx::smem_u32(s_w) >> 4) | (1u << 16);
    uint32_t it = 0;
    for (long long tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++it) {
      const int s = it % kF16Stages;
      const uint32_t b = it & bmask;
      ptx::mbar_wait(&bars->acc_empty[b], ((it >> nbshift) & 1) ^ 1);
      ptx::mbar_wait(&bars->full[s], (it / kF16Stages) & 1);
      ptx::tc_fence_after();
      if (ptx::elect_one()) {
        const uint32_t ah = (ptx::smem_u32(s_a + (size_t)s * kF16StageBytes) >> 4) | (1u << 16);
        const uint32_t al = ah + (8192u >> 4);
        const uint32_t d = tmem_base + b * pairw;
#pragma unroll
        for (int ks = 0; ks < 2; ++ks) {
          ptx::mma_f16_ss(d, u16_desc(ah + 2u * ks, hi32), u16_desc(wbase + 2u * ks, hi32), idesc_st, ks ? 1u : 0u);
          ptx::mma_f16_ss(d + (uint32_t)NPAD, u16_desc(al + 2u * ks, hi32), u16_desc(wbase + 2u * ks, hi32), idesc_lo, 1u);
        }
      }
      __syncwarp();
      if (ptx::elect_one()) {
        ptx::tc_commit(&bars->empty[s]);
        ptx::tc_commit(&bars->acc_full[b]);
      }
      __syncwarp();
    }
  } else {
    // ===== epilogue (warps 8-15) =====
    const int q4 = warp & 3;
    const int half = (warp - 8) >> 2;
    const int m = q4 * 32 + lane;
    const int grp = m >> 3, xx = m & 7;
    const int hh = grp / p.bn, nb = grp % p.bn;
    int h_ones = 0, h_valid = 0;
    __half2 omax = __floats2half2_rn(0.f, 0.f);
    uint32_t it = 0;
    for (long long tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++it) {
      if (staged && (int)(it & 1u) != half) continue;  // staged: a warp group owns every other tile
      const uint32_t b = it & bmask;
      ptx::mbar_wait(&bars->acc_full[b], (it >> nbshift) & 1);
      ptx::tc_fence_after();
      uint32_t tq, tx, ty, tn;
      fast_divmod((uint32_t)tile, p.tx_d, tq, tx);
      fast_divmod(tq, p.ty_d, tn, ty);
      const int n = (int)tn * p.bn + nb;
      const uint32_t tbuf = tmem_base + ((uint32_t)(q4 * 32) << 16) + b * pairw;
      if (staged) {
        u16_epilogue_tile_staged<U16_S1>(a, NPAD, 0, 1, tbuf, n, (int)ty * p.bh + hh, (int)tx * 8 + xx, n < p.n, s_bias,
                                         s_stage + (size_t)(warp - 8) * kU16StagePerWarp, lane, 0, &bars->acc_empty[b], 1, omax);
        continue;  // the staged epilogue released the buffer itself
      } else
        u16_epilogue_tile<U16_S1>(a, NPAD, 0, 1, tbuf, n, (int)ty * p.bh + hh, (int)tx * 8 + xx, n < p.n, half, s_bias, s_hist, h_ones,
                                  h_valid, omax);
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&bars->acc_empty[b]);
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
      asm volatile("bar.sync 1, 256;" ::: "memory");
      for (int i = tid - 256; i < a.q; i += 256)
        if (s_hist[i]) atomicAdd(&a.hist[i], (unsigned long long)s_hist[i]);
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 16) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, 512);
  }
}

// ---- stride 2: no im2col at all ---------------------------------------------------------------------
// The builders write the normalised, split INPUT tile once per pixel as RGB0 quads (8 bytes per pixel and
// plane, row pitch kW2Pitch).  With stride 2 consecutive output pixels start 16 bytes apart, which is
// exactly the row pitch of an un-swizzled K-major core matrix, so the A operand of filter row kh is a
// descriptor over the input tile itself: start = pixel (2 oy0 + kh, 2 ox0), LBO (next 8 K elements) = 16
// bytes = the next two pixels, SBO (next 8 output pixels = next output row) = two input rows.  A K-step
// reads 4 pixels x 4 channels; the weight tile is zero for the 4th pixel and the 4th channel.
constexpr int kW2Cols = 18;                       // input pixels per staged row: 2 * 8 + 1 halo + 1 over-read
constexpr uint32_t kW2Pitch = kW2Cols * 8;        // 144 bytes
constexpr int kW2Rows = 33;                       // 2 * 16 + 1
constexpr uint32_t kW2Plane = 4864;               // >= 33 * 144, multiple of 128
constexpr uint32_t kW2Stage = 2 * kW2Plane + 512; // hi | lo', 1024-aligned below
constexpr int kW2Stages = 4;
constexpr int kW2Threads = 576;                   // warps 0-7 builders, 8-15 epilogue, 16 MMA + TMEM, 17 raw-window TMA
// TMA-fed builders (u8 images whose patch grid needs no reflect padding and whose row pitch is a multiple of 16
// bytes): warp 17 fetches the raw 33-row x 54-byte window of a tile as a 33 x 64-byte box (3-D map over
// [B, H, W * 3] bytes; rows below the image come back as zeros), kRawStages tiles ahead.  A builder thread then owns
// 4 consecutive pixels of a row = three aligned words of shared memory: no per-thread image addressing, no global
// load latency held in registers (the gather path kept 27 raw values of three tiles live), 165 busy threads.
constexpr int kRawStages = 6;
constexpr uint32_t kRawRow = 64;
constexpr uint32_t kRawStage = 2176;              // 33 * 64 = 2112, padded to a multiple of 128

// device [9][3][cout] fp32 -> per kh: [k group (2)][row (2 npad: hi, lo')][8 halves], k = px * 4 + c
__global__ void f16_build_weights_s2_kernel(const float* __restrict__ w, int cout, int npad, uint8_t* __restrict__ img) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < 3 * npad * 16; i += gridDim.x * blockDim.x) {
    const int k = i & 15, oc = (i >> 4) % npad, kh = i / (16 * npad);
    const int px = k >> 2, c = k & 3;
    const float v = (px < 3 && c < 3 && oc < cout) ? w[((kh * 3 + px) * 3 + c) * cout + oc] : 0.f;
    __half hi, lo;
    split16(v, hi, lo);
    uint8_t* base = img + (size_t)kh * (64u * npad) + (size_t)(k >> 3) * (32u * npad) + (k & 7) * 2;
    *reinterpret_cast<__half*>(base + (size_t)oc * 16) = hi;
    *reinterpret_cast<__half*>(base + (size_t)(npad + oc) * 16) = lo;
  }
}

struct W2SmemBars {
  uint64_t full[8], empty[8];        // kW2Stages (general kernel) | kT2Stages (TMA-fed kernel) in use
  uint64_t acc_full[4], acc_empty[4];
  uint64_t raw_full[kRawStages], raw_empty[kRawStages];
  uint32_t tmem_base;
};

__global__ void __launch_bounds__(kW2Threads, 1)
f16_first_s2_kernel(const __grid_constant__ CUtensorMap tm_img, const F16Params p, const LayerArgs a) {
  const int NPAD = p.npad;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* s_a = smem;                                  // kW2Stages stages of kW2Stage bytes
  uint8_t* s_w = smem + kW2Stages * 10240;              // 192 * npad bytes
  uint8_t* s_stage = s_w + 192 * 64;                    // 8 x 4 KB epilogue stages
  uint8_t* s_rawwin = s_stage + kU16StageBytes;         // kRawStages raw windows (TMA destination, 128-byte aligned)
  W2SmemBars* bars = reinterpret_cast<W2SmemBars*>(s_rawwin + kRawStages * kRawStage);
  const bool staged = u16_staged_ok(a, U16_S1, p.nbuf, p.npad);
  __shared__ unsigned s_hist[256];
  __shared__ __align__(16) float s_bias[128];
  __shared__ uint32_t s_plut[3 * 256];  // u8 -> (hi | lo' << 16) of the normalised value: no split in the hot loop

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  if (tid < 128) s_bias[tid] = (tid < NPAD && tid < a.cout) ? a.bias[tid] : 0.f;
  for (int i = tid; i < 256; i += kW2Threads) s_hist[i] = 0;
  if (a.in_mode == IO_U8_NORM)
    for (int i = tid; i < 3 * 256; i += kW2Threads) {
      __half hi, lo;
      split16(a.lut[i], hi, lo);
      s_plut[i] = pack_half2(hi, lo);
    }
  for (int i = tid; i < 12 * NPAD; i += kW2Threads)  // weight image, 16-byte chunks
    reinterpret_cast<uint4*>(s_w)[i] = __ldg(reinterpret_cast<const uint4*>(p.wimg) + i);
  if (tid == 0) {
    for (int i = 0; i < kW2Stages; ++i) {
      ptx::mbar_init(&bars->full[i], 8);
      ptx::mbar_init(&bars->empty[i], 1);
    }
    for (int i = 0; i < 4; ++i) {
      ptx::mbar_init(&bars->acc_full[i], 1);
      ptx::mbar_init(&bars->acc_empty[i], staged ? 4 : 8);
    }
    for (int i = 0; i < kRawStages; ++i) {
      ptx::mbar_init(&bars->raw_full[i], 1);
      ptx::mbar_init(&bars->raw_empty[i], 8);
    }
    ptx::fence_barrier_init();
  }
  if (warp == 16) {
    ptx::tmem_alloc(&bars->tmem_base, 512);
    ptx::tmem_relinquish();
  }
  ptx::fence_proxy_async_smem();
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = bars->tmem_base;
  const uint32_t pairw = 2u * (uint32_t)NPAD;
  const uint32_t bmask = (uint32_t)p.nbuf - 1u;
  int nbshift = 0;
  while ((1 << nbshift) < p.nbuf) ++nbshift;

  if (warp < 8 && p.use_tma) {
    // ===== builders, TMA-fed: thread = (row, quad of 4 pixels); 33 x 5 = 165 threads; quad 4 holds pixels 16, 17 =====
    const int ry = tid / 5, qx = tid - ry * 5;
    const bool live = ry < kW2Rows;
    const uint32_t my_raw = (uint32_t)ry * kRawRow + (uint32_t)qx * 12u;
    const uint32_t my_dst = (uint32_t)(ry * kW2Cols + 4 * qx) * 8u;
    const int npx = qx == 4 ? 2 : 4;   // pixels of this quad inside the 18-column window
    uint32_t it = 0, r = 0, rph = 0;
    for (long long tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++it) {
      // window origin inside the patch: SAME padding (0, 1) = zeros at row / column P
      unsigned n, rt, ty, tx;
      fast_divmod((unsigned)tile, p.txy_d, n, rt);
      fast_divmod(rt, p.tx_d, ty, tx);
      const int iy = 32 * (int)ty + ry, ix = 16 * (int)tx + 4 * qx;
      ptx::mbar_wait(&bars->raw_full[r], rph);
      uint32_t w0 = 0, w1 = 0, w2 = 0;
      if (live) {
        const uint32_t* rp = reinterpret_cast<const uint32_t*>(s_rawwin + (size_t)r * kRawStage + my_raw);
        w0 = rp[0];
        w1 = rp[1];
        w2 = rp[2];
      }
      uint2 vh[4], vl[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        // pixel j = bytes 3j .. 3j+2 of the 12
        const uint32_t b0 = j == 0 ? (w0 & 0xffu) : j == 1 ? (w0 >> 24) : j == 2 ? ((w1 >> 16) & 0xffu) : ((w2 >> 8) & 0xffu);
        const uint32_t b1 = j == 0 ? ((w0 >> 8) & 0xffu) : j == 1 ? (w1 & 0xffu) : j == 2 ? (w1 >> 24) : ((w2 >> 16) & 0xffu);
        const uint32_t b2 = j == 0 ? ((w0 >> 16) & 0xffu) : j == 1 ? ((w1 >> 8) & 0xffu) : j == 2 ? (w2 & 0xffu) : (w2 >> 24);
        const bool okj = live && iy < p.P && ix + j < p.P;
        const uint32_t x0 = okj ? s_plut[b0] : 0u;
        const uint32_t x1 = okj ? s_plut[256 + b1] : 0u;
        const uint32_t x2 = okj ? s_plut[512 + b2] : 0u;
        vh[j] = make_uint2(__byte_perm(x0, x1, 0x5410), x2 & 0xffffu);
        vl[j] = make_uint2(__byte_perm(x0, x1, 0x7632), x2 >> 16);
      }
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&bars->raw_empty[r]);   // the window's words are in registers (used above)
      if (++r == kRawStages) {
        r = 0;
        rph ^= 1u;
      }
      const int s = it % kW2Stages;
      ptx::mbar_wait(&bars->empty[s], ((it / kW2Stages) & 1) ^ 1);
      if (live) {
        uint8_t* st = s_a + (size_t)s * 10240 + my_dst;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          if (j < npx) {
            *reinterpret_cast<uint2*>(st + j * 8) = vh[j];
            *reinterpret_cast<uint2*>(st + kW2Plane + j * 8) = vl[j];
          }
        }
      }
      ptx::fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&bars->full[s]);
    }
  } else if (warp == 17) {
    // ===== raw-window producer: one 33 x 64-byte box per tile, kRawStages tiles ahead of the builders =====
    if (p.use_tma) {
      const Geo g = a.geo;
      if (ptx::elect_one()) ptx::prefetch_tmap(&tm_img);
      __syncwarp();
      uint32_t r = 0, rph = 1;
      for (long long tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
        ptx::mbar_wait(&bars->raw_empty[r], rph);
        if (ptx::elect_one()) {
          unsigned n, rt, ty, tx, img, gy, gx;
          fast_divmod((unsigned)tile, p.txy_d, n, rt);
          fast_divmod(rt, p.tx_d, ty, tx);
          geo_decode(g, (unsigned)g.n0 + n, img, gy, gx);
          const int Yb = (int)gy * g.P + 32 * (int)ty, Xb = (int)gx * g.P + 16 * (int)tx;
          ptx::mbar_expect_tx(&bars->raw_full[r], kW2Rows * kRawRow);
          ptx::tma_load_3d(s_rawwin + (size_t)r * kRawStage, &tm_img, &bars->raw_full[r], Xb * 3, Yb, (int)img);
        }
        __syncwarp();
        if (++r == kRawStages) {
          r = 0;
          rph ^= 1u;
        }
      }
    }
  } else if (warp < 8) {
    // ===== builders: 198 threads stage the 33 x 18 input pixels of a tile, 3 consecutive pixels (9 bytes)
    // per thread.  The gather is latency-bound, so the raw bytes of tile i+1 are requested before tile i is
    // converted; tiles whose window lies inside the image skip the reflect arithmetic. =====
    const Geo g = a.geo;
    const bool u8in = a.in_mode == IO_U8_NORM;
    const int ry = tid / 6, cx0 = (tid - ry * 6) * 3;
    const bool rowt = ry < kW2Rows;
    const unsigned thread_off = (unsigned)(ry * g.W + cx0) * 3u;
    auto request = [&](unsigned tile, uint32_t (&raw)[9], unsigned& okm) {
      // warp-uniform part: tile -> patch -> image window
      unsigned n, rt, ty, tx, img, gy, gx;
      fast_divmod(tile, p.txy_d, n, rt);
      fast_divmod(rt, p.tx_d, ty, tx);
      geo_decode(g, (unsigned)g.n0 + n, img, gy, gx);
      const int iy0 = 32 * (int)ty, ix0 = 16 * (int)tx;                               // patch-local window origin
      const int Yb = g.oy + (int)gy * g.P + iy0, Xb = g.ox + (int)gx * g.P + ix0;     // image window origin
      const long long img_off = (long long)img * g.H * g.W;
      const int iy = iy0 + ry, ix = ix0 + cx0;
      okm = 0;
#pragma unroll
      for (int i = 0; i < 9; ++i) raw[i] = 0u;
      if (!rowt || iy >= p.P) return;
#pragma unroll
      for (int j = 0; j < 3; ++j) okm |= (ix + j < p.P ? 1u : 0u) << j;
      if (Yb + kW2Rows <= g.H && Xb + kW2Cols <= g.W) {
        // the whole window lies inside the image: 9 consecutive bytes / floats at a per-thread constant offset
        const long long base = (img_off + (long long)Yb * g.W + Xb) * 3;
        if (u8in) {
          const uint8_t* q = reinterpret_cast<const uint8_t*>(a.in) + base + thread_off;
#pragma unroll
          for (int i = 0; i < 9; ++i) raw[i] = q[i];
        } else {
          const uint32_t* q = reinterpret_cast<const uint32_t*>(a.in) + base + thread_off;
#pragma unroll
          for (int i = 0; i < 9; ++i) raw[i] = q[i];
        }
      } else {
        const long long row = img_off + (long long)reflect_index(Yb + ry, g.H) * g.W;
#pragma unroll
        for (int j = 0; j < 3; ++j) {
          if (!((okm >> j) & 1u)) continue;
          const long long off = (row + reflect_index(Xb + cx0 + j, g.W)) * 3;
          if (u8in) {
            const uint8_t* q = reinterpret_cast<const uint8_t*>(a.in) + off;
            raw[3 * j] = q[0];
            raw[3 * j + 1] = q[1];
            raw[3 * j + 2] = q[2];
          } else {
            const uint32_t* q = reinterpret_cast<const uint32_t*>(a.in) + off;
            raw[3 * j] = q[0];
            raw[3 * j + 1] = q[1];
            raw[3 * j + 2] = q[2];
          }
        }
      }
    };
    // raw input of two tiles in flight per thread; the request for tile i+2 is issued before tile i is
    // converted (measured: distance 1 = 1.03 ms, distance 2 = 0.84 ms per 4096 patches, deeper does not help)
    uint32_t raw[9], raw_b[9];
    unsigned okm = 0, okm_b = 0;
    if ((long long)blockIdx.x < p.num_tiles) request(blockIdx.x, raw, okm);
    if ((long long)blockIdx.x + gridDim.x < p.num_tiles) request(blockIdx.x + gridDim.x, raw_b, okm_b);
    uint32_t it = 0;
    if (TIC_DBG_BITS(p.dbg) & 2) {
      for (long long tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++it) {
        const int s = it % kW2Stages;
        ptx::mbar_wait(&bars->empty[s], ((it / kW2Stages) & 1) ^ 1);
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(&bars->full[s]);
      }
    } else
    for (long long tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++it) {
      uint32_t raw_n[9];
      unsigned okm_n = 0;
      const long long nxt = tile + 2LL * gridDim.x;
      if (nxt < p.num_tiles) request((unsigned)nxt, raw_n, okm_n);
      uint2 vh[3], vl[3];
      if (u8in) {
#pragma unroll
        for (int j = 0; j < 3; ++j) {
          const bool okj = (okm >> j) & 1u;
          const uint32_t w0 = okj ? s_plut[raw[3 * j]] : 0u;
          const uint32_t w1 = okj ? s_plut[256 + raw[3 * j + 1]] : 0u;
          const uint32_t w2 = okj ? s_plut[512 + raw[3 * j + 2]] : 0u;
          vh[j] = make_uint2(__byte_perm(w0, w1, 0x5410), w2 & 0xffffu);
          vl[j] = make_uint2(__byte_perm(w0, w1, 0x7632), w2 >> 16);
        }
      } else {
#pragma unroll
        for (int j = 0; j < 3; ++j) {
          float f0 = 0.f, f1 = 0.f, f2 = 0.f;
          if ((okm >> j) & 1u) {
            f0 = tic_normalize(__uint_as_float(raw[3 * j]), a.mean[0], a.stdv[0]);
            f1 = tic_normalize(__uint_as_float(raw[3 * j + 1]), a.mean[1], a.stdv[1]);
            f2 = tic_normalize(__uint_as_float(raw[3 * j + 2]), a.mean[2], a.stdv[2]);
          }
          split16x2(f0, f1, vh[j].x, vl[j].x);
          split16x2(f2, 0.f, vh[j].y, vl[j].y);
        }
      }
      const int s = it % kW2Stages;
      ptx::mbar_wait(&bars->empty[s], ((it / kW2Stages) & 1) ^ 1);
      if (rowt) {
        uint8_t* st = s_a + (size_t)s * 10240 + (uint32_t)(ry * kW2Cols + cx0) * 8u;
#pragma unroll
        for (int j = 0; j < 3; ++j) {
          *reinterpret_cast<uint2*>(st + j * 8) = vh[j];
          *reinterpret_cast<uint2*>(st + kW2Plane + j * 8) = vl[j];
        }
      }
      ptx::fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&bars->full[s]);
#pragma unroll
      for (int i = 0; i < 9; ++i) {
        raw[i] = raw_b[i];
        raw_b[i] = raw_n[i];
      }
      okm = okm_b;
      okm_b = okm_n;
    }
  } else if (warp == 16) {
    // ===== MMA issuer: per tile 3 filter rows x (A_hi x [W_hi ; W_lo'] , A_lo' x W_hi) =====
    const uint32_t idesc_st = ptx::make_idesc_f16(128, 2 * NPAD);
    const uint32_t idesc_lo = ptx::make_idesc_f16(128, NPAD);
    // un-swizzled K-major: lo word = addr >> 4 | LBO >> 4 << 16 ; hi word = SBO >> 4 | version 1 << 14 | layout 0
    const uint32_t a_hi32 = ((2u * kW2Pitch) >> 4) | (1u << 14);
    const uint32_t w_hi32 = (128u >> 4) | (1u << 14);
    const uint32_t a_lbo = (16u >> 4) << 16, w_lbo = ((32u * (uint32_t)NPAD) >> 4) << 16;
    const uint32_t wbase = (ptx::smem_u32(s_w) >> 4) | w_lbo;
    uint32_t it = 0;
    for (long long tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++it) {
      const int s = it % kW2Stages;
      const uint32_t b = it & bmask;
      ptx::mbar_wait(&bars->acc_empty[b], ((it >> nbshift) & 1) ^ 1);
      ptx::mbar_wait(&bars->full[s], (it / kW2Stages) & 1);
      ptx::tc_fence_after();
      if (!(TIC_DBG_BITS(p.dbg) & 1) && ptx::elect_one()) {
        const uint32_t ah = (ptx::smem_u32(s_a + (size_t)s * 10240) >> 4) | a_lbo;
        const uint32_t al = ah + (kW2Plane >> 4);
        const uint32_t d = tmem_base + b * pairw;
#pragma unroll
        for (int kh = 0; kh < 3; ++kh) {
          const uint32_t wd = wbase + (uint32_t)kh * ((64u * (uint32_t)NPAD) >> 4);
          ptx::mma_f16_ss(d, u16_desc(ah + (uint32_t)kh * (kW2Pitch >> 4), a_hi32), u16_desc(wd, w_hi32), idesc_st, kh ? 1u : 0u);
          ptx::mma_f16_ss(d + (uint32_t)NPAD, u16_desc(al + (uint32_t)kh * (kW2Pitch >> 4), a_hi32), u16_desc(wd, w_hi32), idesc_lo, 1u);
        }
      }
      __syncwarp();
      if (ptx::elect_one()) {
        ptx::tc_commit(&bars->empty[s]);
        ptx::tc_commit(&bars->acc_full[b]);
      }
      __syncwarp();
    }
  } else {
    // ===== epilogue (warps 8-15) =====
    const int q4 = warp & 3;
    const int half = (warp - 8) >> 2;
    const int m = q4 * 32 + lane;
    const int hh = m >> 3, xx = m & 7;
    int h_ones = 0, h_valid = 0;
    __half2 omax = __floats2half2_rn(0.f, 0.f);
    uint32_t it = 0;
    for (long long tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++it) {
      if (staged && (int)(it & 1u) != half) continue;  // staged: a warp group owns every other tile
      const uint32_t b = it & bmask;
      ptx::mbar_wait(&bars->acc_full[b], (it >> nbshift) & 1);
      ptx::tc_fence_after();
      uint32_t tq, tx, ty, tn;
      fast_divmod((uint32_t)tile, p.tx_d, tq, tx);
      fast_divmod(tq, p.ty_d, tn, ty);
      const int n = (int)tn;
      const uint32_t tbuf = tmem_base + ((uint32_t)(q4 * 32) << 16) + b * pairw;
      if (TIC_DBG_BITS(p.dbg) & 4) {
      } else if (staged) {
        u16_epilogue_tile_staged<U16_S1>(a, NPAD, 0, 1, tbuf, n, (int)ty * 16 + hh, (int)tx * 8 + xx, true, s_bias,
                                         s_stage + (size_t)(warp - 8) * kU16StagePerWarp, lane, 0, &bars->acc_empty[b], 1, omax);
        continue;  // the staged epilogue released the buffer itself
      } else
        u16_epilogue_tile<U16_S1>(a, NPAD, 0, 1, tbuf, n, (int)ty * 16 + hh, (int)tx * 8 + xx, true, half, s_bias, s_hist, h_ones, h_valid, omax);
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&bars->acc_empty[b]);
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
      asm volatile("bar.sync 1, 256;" ::: "memory");
      for (int i = tid - 256; i < a.q; i += 256)
        if (s_hist[i]) atomicAdd(&a.hist[i], (unsigned long long)s_hist[i]);
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 16) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, 512);
  }
}

// ---- stride 2, TMA-fed, pair-plane output: the hot configuration of every codec variant ---------------------
// Same operands and MMAs as f16_first_s2_kernel, but sized for thread-level parallelism in the epilogue: its fixed
// per-tile chain (accumulator wait, TMEM load, stage, two flushes) cost 570 cycles per 128-pixel tile at two warps per
// scheduler (epilogue alone, no stores: 1.70 ms against 0.93 ms for the same number of elements in decode_1's 4x
// larger tiles).  Warps: 0-5 builders (165 live threads), 6 MMA + TMEM, 7 raw-window TMA, 8-23 epilogue = four groups
// of four warps, group g owns TMEM buffer g = tiles it % 4 == g.  An epilogue warp stages BOTH planes of its 32
// pixels (8 KB, no lo' words held in registers: <= 80 registers per thread at 768 threads) and flushes them in one pass.
constexpr int kT2Builders = 6, kT2MmaWarp = 6, kT2TmaWarp = 7, kT2EpiWarp0 = 8, kT2EpiWarps = 16;
constexpr int kT2Threads = 32 * (kT2EpiWarp0 + kT2EpiWarps);
constexpr uint32_t kT2StagePerWarp = 4096;        // hi plane | lo' plane of 32 pixels x 32 channels
constexpr uint32_t kT2LoOff = 2048;
// f32 images (rmbe post-filter, submit/2/rmbe/rmbe.py:15-111): the raw window is 33 rows x 18 pixels x 12 bytes, fetched
// as a 33 x 224-byte box (56 floats); a builder thread owns 4 pixels = three aligned 16-byte words and normalises with
// the reference's true division (model.py:44) before the fp16 split.
constexpr uint32_t kRawRowF32 = 224;
constexpr uint32_t kRawStageF32 = 7424;            // 33 * 224 = 7392, padded to a multiple of 128
constexpr int kRawStagesF32 = 4;
constexpr int kT2Stages = 6;                       // operand stages = raw-window stages = builder warps (warp w owns slot w)

// The stage of a warp is the TMA-store image of its 32 pixels = rows [y0, y0 + 4) x columns [x0, x0 + 8) of the tile:
// [4][8][CEND] halves per plane, 16-byte chunks XOR-swizzled exactly like CU_TENSOR_MAP_SWIZZLE_64B (CEND = 32) /
// _32B (CEND = 16) of the output tensor maps (chunk ^= (pixel >> FSH) & (M - 1): the pattern is a function of the
// shared-memory address bits, the stage is 1024-byte aligned).  One lane ships both planes with two
// cp.async.bulk.tensor stores (UTMASTG): no shared-memory read-back, no per-lane global stores.
template <int CEND>
__device__ __forceinline__ void f16_t2_epilogue_tile(const LayerArgs& a, const CUtensorMap* tm_ohi, const CUtensorMap* tm_olo,
                                                     const uint32_t tbuf, const int NPAD, const int n, const int y0, const int x0,
                                                     const float* s_bias, const uint32_t stage, const int lane,
                                                     uint64_t* rel_bar, __half2& omax, const bool rel_leader = false,
                                                     const bool store = true) {
  constexpr int M = CEND >> 3;                       // 16-byte chunks per pixel and plane
  constexpr int MSH = M == 2 ? 1 : 2;
  constexpr int FSH = 3 - MSH;                       // swizzle: chunk ^= (pixel >> FSH) & (M - 1)
  constexpr int NCI = CEND / 16;
  const float floor_v = a.act ? 0.0f : -INFINITY;
  const uint32_t sp = stage + (uint32_t)lane * (M * 16);
  const int sw = (lane >> FSH) & (M - 1);
  // the stores of this warp's previous tile have read the stage (they had a whole tile period for it)
  if (lane == 0) ptx::bulk_wait_group_read<0>();
  __syncwarp();
#pragma unroll
  for (int ci = 0; ci < NCI; ++ci) {
    float v[16], u[16];
    ptx::tmem_ld16_nowait(tbuf + NPAD + ci * 16, u);
    ptx::tmem_ld16_nowait(tbuf + ci * 16, v);
    ptx::tmem_ld_wait();
    if (ci == NCI - 1) {  // last TMEM read of the tile: hand the buffer back
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (rel_leader)
          ptx::mbar_arrive_leader(rel_bar);   // CTA-pair kernels: the barrier lives in the leader CTA
        else
          ptx::mbar_arrive(rel_bar);
      }
    }
    const float4* bp = reinterpret_cast<const float4*>(s_bias + ci * 16);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float4 b = bp[i];
      v[4 * i] = fmaxf(__fadd_rn(__fmaf_rn(u[4 * i], 1.0f / 2048.0f, v[4 * i]), b.x), floor_v);
      v[4 * i + 1] = fmaxf(__fadd_rn(__fmaf_rn(u[4 * i + 1], 1.0f / 2048.0f, v[4 * i + 1]), b.y), floor_v);
      v[4 * i + 2] = fmaxf(__fadd_rn(__fmaf_rn(u[4 * i + 2], 1.0f / 2048.0f, v[4 * i + 2]), b.z), floor_v);
      v[4 * i + 3] = fmaxf(__fadd_rn(__fmaf_rn(u[4 * i + 3], 1.0f / 2048.0f, v[4 * i + 3]), b.w), floor_v);
    }
    uint32_t hp[8], lp[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) split16x2(v[2 * i], v[2 * i + 1], hp[i], lp[i], omax);
    sts128(sp + (uint32_t)(((2 * ci) ^ sw) << 4), hp[0], hp[1], hp[2], hp[3]);
    sts128(sp + (uint32_t)(((2 * ci + 1) ^ sw) << 4), hp[4], hp[5], hp[6], hp[7]);
    sts128(sp + kT2LoOff + (uint32_t)(((2 * ci) ^ sw) << 4), lp[0], lp[1], lp[2], lp[3]);
    sts128(sp + kT2LoOff + (uint32_t)(((2 * ci + 1) ^ sw) << 4), lp[4], lp[5], lp[6], lp[7]);
  }
  ptx::fence_proxy_async_smem();  // generic-proxy stage writes -> visible to the TMA store
  __syncwarp();
  if (lane == 0 && store && !(TIC_DBG_BITS(a.dbg) & 8)) {
    ptx::tma_store_4d_s(tm_ohi, stage, 0, x0, y0, n);
    ptx::tma_store_4d_s(tm_olo, stage + kT2LoOff, 0, x0, y0, n);
    ptx::bulk_commit_group();
  }
}

// (x - mean) / std for a launch-constant std without the division routine (~15 instructions, 12 per builder thread
// and tile: it bounded the f32 first layer of rmbe at 3.4 ms per 5696 tiles): q0 = y * RN(1 / std), one residual
// correction q = q0 + r * (y - std * q0) with the residual exact in an FMA (Markstein) — the correctly rounded quotient
// for these operand ranges; any last-ulp disagreement with the division is 4x below the fp16-pair format's own 2^-22.
__device__ __forceinline__ float f16_norm_fast(float x, float mean, float stdv, float rstd) {
  const float y = __fsub_rn(x, mean);
  const float q0 = __fmul_rn(y, rstd);
  return __fmaf_rn(__fmaf_rn(-stdv, q0, y), rstd, q0);
}

template <bool F32>
__global__ void __launch_bounds__(kT2Threads, 1)
f16_first_s2_tma_kernel(const __grid_constant__ CUtensorMap tm_img, const __grid_constant__ CUtensorMap tm_ohi,
                        const __grid_constant__ CUtensorMap tm_olo, const F16Params p, const LayerArgs a) {
  constexpr uint32_t RAW_ROW = F32 ? kRawRowF32 : kRawRow, RAW_STAGE = F32 ? kRawStageF32 : kRawStage;
  constexpr uint32_t RAW_STAGES = kT2Stages;
  const int NPAD = p.npad;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* s_a = smem;                                  // kW2Stages stages
  uint8_t* s_w = smem + kT2Stages * 10240;              // 192 * npad bytes
  uint8_t* s_stage = s_w + 192 * 64;                    // 16 x 8 KB epilogue stages (hi | lo')
  uint8_t* s_rawwin = s_stage + kT2EpiWarps * kT2StagePerWarp;
  W2SmemBars* bars = reinterpret_cast<W2SmemBars*>(s_rawwin + RAW_STAGES * RAW_STAGE);
  __shared__ __align__(16) float s_bias[128];
  // u8 -> (hi | lo' << 16) of the normalised value, kLutRep interleaved copies: lane l reads copy l % kLutRep, so two lanes
  // only share a bank when they are the same copy AND their bytes agree modulo 32 / kLutRep (the byte-indexed look-ups
  // were 60 % of this kernel's shared-load wavefronts as bank conflicts, profiles/r1g_summary_f16x3.md)
  constexpr int kLutRep = 8;
  __shared__ uint32_t s_plut[3 * 256 * kLutRep];

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  if (tid < 128) s_bias[tid] = (tid < NPAD && tid < a.cout) ? a.bias[tid] : 0.f;
  if (!F32)
    for (int i = tid; i < 3 * 256 * kLutRep; i += kT2Threads) {
      __half hi, lo;
      split16(a.lut[i / kLutRep], hi, lo);
      s_plut[i] = pack_half2(hi, lo);
    }
  for (int i = tid; i < 12 * NPAD; i += kT2Threads)
    reinterpret_cast<uint4*>(s_w)[i] = __ldg(reinterpret_cast<const uint4*>(p.wimg) + i);
  if (tid == 0) {
    for (int i = 0; i < kT2Stages; ++i) {
      ptx::mbar_init(&bars->full[i], 1);
      ptx::mbar_init(&bars->empty[i], 1);
    }
    for (int i = 0; i < 4; ++i) {
      ptx::mbar_init(&bars->acc_full[i], 1);
      ptx::mbar_init(&bars->acc_empty[i], 4);
    }
    for (int i = 0; i < (int)RAW_STAGES; ++i) {
      ptx::mbar_init(&bars->raw_full[i], 1);
      ptx::mbar_init(&bars->raw_empty[i], 1);
    }
    ptx::fence_barrier_init();
  }
  if (warp == kT2MmaWarp) {
    ptx::tmem_alloc(&bars->tmem_base, 512);
    ptx::tmem_relinquish();
  }
  ptx::fence_proxy_async_smem();
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = bars->tmem_base;
  const uint32_t pairw = 2u * (uint32_t)NPAD;

  if (warp < kT2Builders) {
    // ===== builders: warp w builds the tiles it == w (mod 6) ALONE, into slot w: six tiles are in flight, and the 165
    // (row, quad of 4 pixels) items of a tile are six independent passes per lane, so the shared-memory latencies of
    // one pass hide under the next (six warps in lock-step on one tile ran at 12 cycles per instruction) =====
    const float rstd0 = __frcp_rn(a.stdv[0]), rstd1 = __frcp_rn(a.stdv[1]), rstd2 = __frcp_rn(a.stdv[2]);
    const uint32_t* const plut0 = s_plut + (lane & (kLutRep - 1));
    const uint32_t* const plut1 = plut0 + 256 * kLutRep;
    const uint32_t* const plut2 = plut1 + 256 * kLutRep;
    const uint32_t slot = (uint32_t)warp;
    const uint8_t* rawb = s_rawwin + (size_t)slot * RAW_STAGE;
    uint8_t* stb = s_a + (size_t)slot * 10240;
    uint32_t ph = 0;
    if (TIC_DBG_BITS(p.dbg) & 2) {  // measurement aid: consume the raw windows, publish empty stages
      for (long long tile = blockIdx.x + (long long)warp * gridDim.x; tile < p.num_tiles; tile += 6LL * gridDim.x, ph ^= 1u) {
        ptx::mbar_wait(&bars->raw_full[slot], ph);
        ptx::mbar_wait(&bars->empty[slot], ph ^ 1u);
        __syncwarp();
        if (lane == 0) {
          ptx::mbar_arrive(&bars->raw_empty[slot]);
          ptx::mbar_arrive(&bars->full[slot]);
        }
      }
    } else
    for (long long tile = blockIdx.x + (long long)warp * gridDim.x; tile < p.num_tiles; tile += 6LL * gridDim.x, ph ^= 1u) {
      unsigned n, rt, ty, tx;
      fast_divmod((unsigned)tile, p.txy_d, n, rt);
      fast_divmod(rt, p.tx_d, ty, tx);
      ptx::mbar_wait(&bars->raw_full[slot], ph);
      ptx::mbar_wait(&bars->empty[slot], ph ^ 1u);
#pragma unroll
      for (int pass = 0; pass < 6; ++pass) {
        const int item = pass * 32 + lane;
        if (item < kW2Rows * 5) {
          const int ry = item / 5, qx = item - ry * 5;
          const int iy = 32 * (int)ty + ry, ix = 16 * (int)tx + 4 * qx;
          const uint8_t* rp8 = rawb + (uint32_t)ry * RAW_ROW + (uint32_t)qx * (F32 ? 48u : 12u);
          uint2 vh[4], vl[4];
          if (F32) {
            const float4* rp = reinterpret_cast<const float4*>(rp8);
            const float4 q0 = rp[0], q1 = rp[1], q2 = rp[2];
            const float f[12] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w, q2.x, q2.y, q2.z, q2.w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const bool okj = iy < p.P && ix + j < p.P;
              const float f0 = okj ? f16_norm_fast(f[3 * j], a.mean[0], a.stdv[0], rstd0) : 0.f;
              const float f1 = okj ? f16_norm_fast(f[3 * j + 1], a.mean[1], a.stdv[1], rstd1) : 0.f;
              const float f2 = okj ? f16_norm_fast(f[3 * j + 2], a.mean[2], a.stdv[2], rstd2) : 0.f;
              split16x2(f0, f1, vh[j].x, vl[j].x);
              split16x2(f2, 0.f, vh[j].y, vl[j].y);
            }
          } else {
            const uint32_t* rp = reinterpret_cast<const uint32_t*>(rp8);
            const uint32_t w0 = rp[0], w1 = rp[1], w2 = rp[2];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const uint32_t b0 = j == 0 ? (w0 & 0xffu) : j == 1 ? (w0 >> 24) : j == 2 ? ((w1 >> 16) & 0xffu) : ((w2 >> 8) & 0xffu);
              const uint32_t b1 = j == 0 ? ((w0 >> 8) & 0xffu) : j == 1 ? (w1 & 0xffu) : j == 2 ? (w1 >> 24) : ((w2 >> 16) & 0xffu);
              const uint32_t b2 = j == 0 ? ((w0 >> 16) & 0xffu) : j == 1 ? ((w1 >> 8) & 0xffu) : j == 2 ? (w2 & 0xffu) : (w2 >> 24);
              const bool okj = iy < p.P && ix + j < p.P;
              const uint32_t x0 = okj ? plut0[b0 * kLutRep] : 0u;
              const uint32_t x1 = okj ? plut1[b1 * kLutRep] : 0u;
              const uint32_t x2 = okj ? plut2[b2 * kLutRep] : 0u;
              vh[j] = make_uint2(__byte_perm(x0, x1, 0x5410), x2 & 0xffffu);
              vl[j] = make_uint2(__byte_perm(x0, x1, 0x7632), x2 >> 16);
            }
          }
          uint8_t* st = stb + (uint32_t)(ry * kW2Cols + 4 * qx) * 8u;
          const int npx = qx == 4 ? 2 : 4;
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            if (j < npx) {
              *reinterpret_cast<uint2*>(st + j * 8) = vh[j];
              *reinterpret_cast<uint2*>(st + kW2Plane + j * 8) = vl[j];
            }
          }
        }
      }
      ptx::fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        ptx::mbar_arrive(&bars->raw_empty[slot]);
        ptx::mbar_arrive(&bars->full[slot]);
      }
    }
  } else if (warp == kT2TmaWarp) {
    // ===== raw-window producer =====
    const Geo g = a.geo;
    if (ptx::elect_one()) ptx::prefetch_tmap(&tm_img);
    __syncwarp();
    uint32_t r = 0, rph = 1;
    for (long long tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
      ptx::mbar_wait(&bars->raw_empty[r], rph);
      if (ptx::elect_one()) {
        unsigned n, rt, ty, tx, img, gy, gx;
        fast_divmod((unsigned)tile, p.txy_d, n, rt);
        fast_divmod(rt, p.tx_d, ty, tx);
        geo_decode(g, (unsigned)g.n0 + n, img, gy, gx);
        const int Yb = g.oy + (int)gy * g.P + 32 * (int)ty, Xb = g.ox + (int)gx * g.P + 16 * (int)tx;
        ptx::mbar_expect_tx(&bars->raw_full[r], kW2Rows * RAW_ROW);
        ptx::tma_load_3d(s_rawwin + (size_t)r * RAW_STAGE, &tm_img, &bars->raw_full[r], Xb * 3, Yb, (int)img);
      }
      __syncwarp();
      if (++r == RAW_STAGES) {
        r = 0;
        rph ^= 1u;
      }
    }
  } else if (warp == kT2MmaWarp) {
    // ===== MMA issuer: per tile 3 filter rows x (A_hi x [W_hi ; W_lo'] , A_lo' x W_hi); TMEM buffer = tile & 3 =====
    const uint32_t idesc_st = ptx::make_idesc_f16(128, 2 * NPAD);
    const uint32_t idesc_lo = ptx::make_idesc_f16(128, NPAD);
    const uint32_t a_hi32 = ((2u * kW2Pitch) >> 4) | (1u << 14);
    const uint32_t w_hi32 = (128u >> 4) | (1u << 14);
    const uint32_t a_lbo = (16u >> 4) << 16, w_lbo = ((32u * (uint32_t)NPAD) >> 4) << 16;
    const uint32_t wbase = (ptx::smem_u32(s_w) >> 4) | w_lbo;
    uint32_t it = 0, s = 0, sph = 0;
    for (long long tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++it) {
      const uint32_t b = it & 3u;
      ptx::mbar_wait(&bars->acc_empty[b], ((it >> 2) & 1) ^ 1);
      ptx::mbar_wait(&bars->full[s], sph);
      ptx::tc_fence_after();
      if (!(TIC_DBG_BITS(p.dbg) & 1) && ptx::elect_one()) {
        const uint32_t ah = (ptx::smem_u32(s_a + (size_t)s * 10240) >> 4) | a_lbo;
        const uint32_t al = ah + (kW2Plane >> 4);
        const uint32_t d = tmem_base + b * pairw;
#pragma unroll
        for (int kh = 0; kh < 3; ++kh) {
          const uint32_t wd = wbase + (uint32_t)kh * ((64u * (uint32_t)NPAD) >> 4);
          ptx::mma_f16_ss(d, u16_desc(ah + (uint32_t)kh * (kW2Pitch >> 4), a_hi32), u16_desc(wd, w_hi32), idesc_st, kh ? 1u : 0u);
          ptx::mma_f16_ss(d + (uint32_t)NPAD, u16_desc(al + (uint32_t)kh * (kW2Pitch >> 4), a_hi32), u16_desc(wd, w_hi32), idesc_lo, 1u);
        }
      }
      __syncwarp();
      if (ptx::elect_one()) {
        ptx::tc_commit(&bars->empty[s]);
        ptx::tc_commit(&bars->acc_full[b]);
      }
      __syncwarp();
      if (++s == kT2Stages) {
        s = 0;
        sph ^= 1u;
      }
    }
  } else {
    // ===== epilogue: group g = TMEM buffer g = tiles it % 4 == g =====
    const int ew = warp - kT2EpiWarp0;
    const int q4 = warp & 3, group = ew >> 2;
    const uint32_t stage = ptx::smem_u32(s_stage + (size_t)ew * kT2StagePerWarp);
    const uint32_t tbuf = tmem_base + ((uint32_t)(q4 * 32) << 16) + (uint32_t)group * pairw;
    if (lane == 0) {
      ptx::prefetch_tmap(&tm_ohi);
      ptx::prefetch_tmap(&tm_olo);
    }
    uint32_t use = 0;
    __half2 omax = __floats2half2_rn(0.f, 0.f);
    for (long long tile = blockIdx.x + (long long)group * gridDim.x; tile < p.num_tiles; tile += 4LL * gridDim.x, ++use) {
      ptx::mbar_wait(&bars->acc_full[group], use & 1);
      ptx::tc_fence_after();
      uint32_t tq, tx, ty, tn;
      fast_divmod((uint32_t)tile, p.tx_d, tq, tx);
      fast_divmod(tq, p.ty_d, tn, ty);
      if (TIC_DBG_BITS(p.dbg) & 4) {
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(&bars->acc_empty[group]);
      } else if (NPAD == 32)
        f16_t2_epilogue_tile<32>(a, &tm_ohi, &tm_olo, tbuf, NPAD, (int)tn, (int)ty * 16 + 4 * q4, (int)tx * 8, s_bias, stage, lane,
                                 &bars->acc_empty[group], omax);
      else
        f16_t2_epilogue_tile<16>(a, &tm_ohi, &tm_olo, tbuf, NPAD, (int)tn, (int)ty * 16 + 4 * q4, (int)tx * 8, s_bias, stage, lane,
                                 &bars->acc_empty[group], omax);
    }
    if (lane == 0) ptx::bulk_wait_group<0>();  // every store of this warp is complete before the CTA may exit
    if (ovf_hit(omax)) ovf_raise(a.oflow);
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == kT2MmaWarp) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, 512);
  }
}

inline bool f16_first_supported(const LayerArgs& a, int kind, int stride) {
  if (kind != 0 || a.cin != 3) return false;
  if (a.in_mode != IO_U8_NORM && a.in_mode != IO_F32_NORM) return false;
  if (a.cout % 16 != 0 || a.cout > 64) return false;
  if (a.hin != a.win) return false;
  if (stride == 2 && (a.hin != 2 * a.hout || a.win != 2 * a.wout)) return false;
  if (a.wout % 8 != 0 || !(a.hout == 8 || a.hout % 16 == 0)) return false;
  if (a.out_mode == IO_DENORM_F32 || a.out_mode == IO_DENORM_U8) return false;
  return true;
}

// The raw-window TMA path needs: u8 pixels, a patch grid that covers the image exactly (no reflect padding, no grid
// offset), and a global address / row pitch the tensor map accepts (16-byte multiples).
inline bool f16_first_tma_ok(const LayerArgs& a) {
  const Geo& g = a.geo;
  if (a.in_mode != IO_U8_NORM && a.in_mode != IO_F32_NORM) return false;
  // the patch grid lies inside the image: no reflect padding (rmbe tile grids are inside by construction)
  if (g.oy < 0 || g.ox < 0 || g.oy + g.gh * g.P > g.H || g.ox + g.gw * g.P > g.W || g.P != a.hin) return false;
  const size_t row_bytes = (size_t)g.W * 3 * (a.in_mode == IO_U8_NORM ? 1 : 4);
  if (row_bytes % 16 != 0 || (reinterpret_cast<uintptr_t>(a.in) & 15u) != 0) return false;
  if (a.hin % 32 != 0) return false;
  return true;
}

inline tic_status launch_first16(const LaunchCtx& c, const LayerArgs& a, int stride, const float* w_dev, OperandImage& img) {
  F16Params p{};
  p.n = a.n;
  p.P = a.hin;
  p.stride = stride;
  p.pad = stride == 1 ? 1 : 0;
  p.bn = a.hout == 8 ? 2 : 1;
  p.bh = a.hout == 8 ? 8 : 16;
  p.tiles_x = a.wout / 8;
  p.tiles_y = a.hout / p.bh;
  p.num_tiles = (long long)p.tiles_x * p.tiles_y * ((a.n + p.bn - 1) / p.bn);
  if (p.num_tiles >= (1LL << 31) - 65536) return c.fail("too many tiles for one launch", TIC_ERR_UNSUPPORTED);
  p.tx_d = make_fastdiv((uint32_t)p.tiles_x);
  p.ty_d = make_fastdiv((uint32_t)p.tiles_y);
  p.txy_d = make_fastdiv((uint32_t)(p.tiles_x * p.tiles_y));
  p.npad = a.cout;
  p.dbg = tic_env_int("TIC_DBG", 0);  // -DTIC_ABLATE builds only
  p.nbuf = std::min(4, 512 / (2 * p.npad));
  const bool windowed = stride == 2 && p.bn == 1;  // operands straight from the staged input tile (no im2col)
  auto builder = windowed ? f16_build_weights_s2_kernel : f16_build_weights_kernel;
  bool build;
  if (img.ensure(image_key(builder, w_dev, a.cout, p.npad), 192 * 64, &build) != TIC_OK)
    return c.fail("cudaMalloc for first-layer weight image failed", TIC_ERR_NOMEM);
  if (build) {
    if (cudaMemsetAsync(img.buf.p, 0, 192 * 64, c.stream) != cudaSuccess)
      return c.fail("cudaMemsetAsync of the first-layer weight image failed", TIC_ERR_CUDA);
    builder<<<8, 256, 0, c.stream>>>(w_dev, a.cout, p.npad, img.buf.as<uint8_t>());
    if (cudaGetLastError() != cudaSuccess) return c.fail("first-layer weight image kernel failed", TIC_ERR_CUDA);
  }
  p.wimg = img.img();
  CUtensorMap tm_img{};
  // raw u8 / f32 image windows by TMA where the geometry allows it (otherwise the builders load them)
  const bool f32in = a.in_mode == IO_F32_NORM;
  p.use_tma = windowed && f16_first_tma_ok(a) &&
              tmap_image_rows(&tm_img, a, f32in, f32in ? kRawRowF32 / 4 : kRawRow, kW2Rows, nullptr, nullptr) == TIC_OK;
  const int grid = (int)std::min<long long>(p.num_tiles, c.num_sms);
  // the TMA-fed, pair-plane-output kernel (16 epilogue warps) when the launch qualifies
  const bool t2 = windowed && p.use_tma && a.out_mode == IO_ACT16 && (a.cout == 32 || a.cout == 16) && p.nbuf == 4;
  // the general kernel's TMA builders take u8 windows of an un-shifted grid only
  if (!t2 && (a.in_mode != IO_U8_NORM || a.geo.oy != 0 || a.geo.ox != 0)) p.use_tma = 0;
  cudaError_t e;
  if (t2) {
    const size_t smem_t2 = kT2Stages * 10240 + 192 * 64 + kT2EpiWarps * kT2StagePerWarp +
                           kT2Stages * (f32in ? kRawStageF32 : kRawStage) + sizeof(W2SmemBars) + 1024;
    // output tensor maps (hi / lo' plane of the NHWC pair-plane activation)
    CUtensorMap tm_o[2];
    for (int pl = 0; pl < 2; ++pl)
      if (tic_status s = tmap_pair_out(&tm_o[pl], reinterpret_cast<__half*>(a.out) + (pl ? a.out_lo_off : 0), a.n, a.hout, a.wout, a.cout,
                                       "first-layer output", c.err))
        return s;
    e = launch_dyn(f32in ? f16_first_s2_tma_kernel<true> : f16_first_s2_tma_kernel<false>, grid, kT2Threads, smem_t2, c.stream, tm_img,
                   tm_o[0], tm_o[1], p, a);
  } else if (windowed) {
    const size_t smem_w2 = kW2Stages * 10240 + 192 * 64 + kU16StageBytes + kRawStages * kRawStage + sizeof(W2SmemBars) + 1024;
    e = launch_dyn(f16_first_s2_kernel, grid, kW2Threads, smem_w2, c.stream, tm_img, p, a);
  } else {
    const size_t smem = kF16Stages * kF16StageBytes + 2 * 64 * 64 + kU16StageBytes + sizeof(F16SmemBars) + 1024;
    e = launch_dyn(stride == 1 ? f16_first_kernel<1> : f16_first_kernel<2>, grid, kF16Threads, smem, c.stream, p, a);
  }
  if (e != cudaSuccess) return c.fail(std::string("first-layer tensor launch failed: ") + cudaGetErrorString(e), TIC_ERR_CUDA);
  ++*c.launches;
  return TIC_OK;
}

}  // namespace tic

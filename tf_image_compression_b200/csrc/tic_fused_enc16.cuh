// Back-to-back fused first two layers of the analysis transform (model_0/model.py:50-71: encode_0 3 -> 32 stride 2 relu on
// the normalised u8 patch, encode_1 32 -> 32 stride 2 relu) as ONE kernel.  Unfused, the 64 x 64 x 32 tensor between them
// (6.4 GB per 12 288 patches as fp16 pair planes) is written by the first-layer kernel and read back by the next:
// 12.9 GB of the encoder's 16.6 GB of HBM traffic, and encode_1 sits on the HBM roofline because of it.  Here it lives
// in shared memory only:
//
//   TMA (raw u8 window of the image) -> builders (normalise, fp16 split, RGB0 quads: the operand window of tic_first16.cuh)
//   -> MMA1 (no-im2col windowed operands, four 16 x 8 sub-tiles) -> TMEM -> epilogue 1: bias, relu, fp16 split, written as
//   the swizzled K-major stride-2 operand tile of the next layer -> MMA2 (nine taps) -> TMEM -> epilogue 2: bias, relu,
//   fp16 split -> pair-plane output.
//
// A CTA pair (cta_group::2, M = 256) walks two patches in lock-step; a step is one encode_1 output tile (16 x 8) = a
// 32 x 16 region of the intermediate map.  The stride-2 SAME conv reads intermediate rows 2y .. 2y + 2: one halo row BELOW
// and one halo column RIGHT of the region.  They are not recomputed: tiles are walked bottom-to-top, right-to-left, and
// the first row / first column of every tile is kept in small shared-memory caches for the tile above / to the left
// (zeros at the patch border = the conv's zero padding), so MMA1 does exactly the work of the unfused layer.
//
// Warps (768 threads, 80 registers): 0 raw-window TMA, 1 MMA issuer (leader CTA), 2 TMEM allocator, 4-19 epilogue
// (four per TMEM lane quadrant: one first-layer sub-tile each, and an eight-channel share of epilogue 2 one tile
// behind), 20-23 builders (four: with the integer operand they are never late, and two warps fewer leave the epilogue warps
// 80 instead of 72 registers: 1.77 -> 1.70 ms; three builders: 1.77).  TMEM: 4 x 64 columns for MMA1's sub-tiles, two buffers of 64 columns for MMA2.
// Waiting: one warp of a group polls an mbarrier and releases the others through a named barrier, and a group's
// arrivals are gathered by a named barrier into one mbarrier arrival per CTA — a warp parked in `mbarrier.try_wait`
// is woken by every mbarrier event of the CTA and re-polls (7 instructions): with every warp polling and arriving for
// itself 42 % of the kernel's executed instructions were polls (profiles/r2b).
#pragma once
#include "tic_first16.cuh"
#include "tic_fused16.cuh"
#include "tic_launch.cuh"

namespace tic {

constexpr int kFEThreads = 768;
constexpr int kFEBuilderWarp0 = 20, kFEBuilders = 4;
constexpr int kFEOpCols = 34;                                   // input pixels per operand row: 2 * 16 + 1 halo + 1 over-read
constexpr uint32_t kFEOpPitch = kFEOpCols * 8;                  // 272 bytes (RGB0 fp16 quads)
constexpr int kFEOpRows = 65;                                   // 2 * 32 + 1
constexpr uint32_t kFEOpPlane = 17920;                          // >= 65 * 272 = 17680, multiple of 256
constexpr uint32_t kFERawRow = 112;                             // bytes per raw-window row (34 px * 3 = 102, padded to 16)
constexpr uint32_t kFERawStage = 7424;                          // >= 65 * 112 = 7280, multiple of 128
constexpr int kFERawStages = 2;
constexpr uint32_t kFERegionPlane = 39936;                      // >= 17 * 2 * 9 * 128 = 39168, multiple of 1024
constexpr uint32_t kFEStagePerWarp = 4096;                      // epilogue 2: hi | lo' plane of 32 pixels x 32 channels (TMA-store image)

struct FusedEncParams {
  int n;                    // patches
  int P;                    // patch edge (input of encode_0)
  int tiles_x, tiles_y;     // encode_1 output tiles per patch (16 rows x 8 columns)
  int tiles_pp;
  long long pairs_total;
  const uint8_t* w1img;     // first-layer operand image, per CTA rank (f16_build_weights_s2_pair_kernel)
  uint32_t w1_off, w2_off, w2B_off, op_off, raw_off, region_off, rowc_off, colc_off, stage_off, bars_off;
  uint32_t smem_bytes;
  float bias1[32];          // encode_0's bias as launch constants (constant-bank operands: no shared-memory loads in phase A)
  int moff[3];              // m_c = round(mean_c): the builders' exact integer operand is x - m_c (FusedEncNorm)
};

struct FusedEncBars {
  uint64_t w_full;
  uint64_t raw_full[kFERawStages], raw_empty[kFERawStages];
  uint64_t op_full, op_empty;
  uint64_t acc1_full, acc1_empty;
  uint64_t reg_full, reg_empty;
  uint64_t acc2_full[2], acc2_empty[2];
  uint32_t tmem_base;
};

__device__ __forceinline__ uint32_t fused_swz128(uint32_t addr) { return addr ^ (((addr >> 7) & 7u) << 4); }

// The first layer reads u8 pixels, and (x - mean) / std of an integer is not needed as an fp16 PAIR: with m_c = round(mean_c)
// the operand A = x - m_c is an integer of magnitude <= 255, EXACT in one fp16, and
//     sum_c ((x_c - mean_c) / std_c) * W_c  =  sum_c (x_c - m_c) * (W_c / std_c)  +  1 * sum_c (m_c - mean_c) * (W_c / std_c).
// The RGB0 quad's spare fourth channel carries the 1 (0 outside the patch, like the pixel itself: the conv's zero padding
// stays exact at the patch border), W' = W / std and the correction row are split into (hi, lo') as before, and the A_lo' x
// W_hi product of the pair scheme disappears: MMA1 is 12 instead of 24 instructions per step, the builders write one plane.
struct FusedEncNorm {
  float mean[3], stdv[3];
  int m[3];
};

// device [9][3][32] fp32 -> per CTA rank r of the pair, per filter row kh:
//   [k group (2)][32 rows][8 halves]: r = 0 -> W'_hi rows, r = 1 -> W'_lo' rows   (stacked product, N = 64 over the pair)
// k = px * 4 + c (RGB1 quads of 4 consecutive input pixels; the 4th pixel has zero weights).  Per rank: 3 x 1024 B.
__global__ void f16_build_weights_s2_pair_kernel(const float* __restrict__ w, int cout, uint8_t* __restrict__ img, const FusedEncNorm nm) {
  const int per_rank = 3 * 2 * 32 * 8;  // halves
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < 2 * per_rank; i += gridDim.x * blockDim.x) {
    const int rank = i / per_rank;
    const int j = i - rank * per_rank;
    const int e = j & 7, row = (j >> 3) & 31, kg = (j >> 8) & 1, kh = j >> 9;
    const int k = kg * 8 + e, px = k >> 2, c = k & 3;
    const int oc = row;
    float v = 0.f;
    if (px < 3 && oc < cout) {
      const float* wt = w + (size_t)((kh * 3 + px) * 3) * cout + oc;   // [c][oc] of this tap
      if (c < 3) {
        v = __fdiv_rn(wt[c * cout], nm.stdv[c]);
      } else {
        for (int cc = 0; cc < 3; ++cc) v = __fmaf_rn(__fsub_rn((float)nm.m[cc], nm.mean[cc]), __fdiv_rn(wt[cc * cout], nm.stdv[cc]), v);
      }
    }
    __half hi, lo;
    split16(v, hi, lo);
    uint8_t* base = img + (size_t)rank * 4608 + kh * 1024;
    *reinterpret_cast<__half*>(base + (size_t)kg * 512 + (size_t)row * 16 + e * 2) = rank == 1 ? lo : hi;
  }
}

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kFEThreads, 1)
fused_enc_kernel(const __grid_constant__ CUtensorMap tm_img, const __grid_constant__ CUtensorMap tm_ohi,
                 const __grid_constant__ CUtensorMap tm_olo, const LayerArgs a1, const U16Params p2, const LayerArgs a2,
                 const FusedEncParams fp) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* s_w1 = smem + fp.w1_off;            // 4608 B: this rank's first-layer operand image
  uint8_t* s_w2A = smem + fp.w2_off;
  uint8_t* s_w2B = smem + fp.w2B_off;
  uint8_t* s_op = smem + fp.op_off;            // the input window as exact fp16 integers (x - m_c, 1): RGB1 quads, one plane
  uint8_t* s_rawwin = smem + fp.raw_off;
  uint8_t* s_region = smem + fp.region_off;    // hi plane | lo' plane of the 33 x 17 intermediate region (stride-2 box layout)
  uint8_t* s_rowc = smem + fp.rowc_off;        // [parity][chunk: hi 0-3, lo' 4-7][tiles_x * 16 px][16 B]
  uint8_t* s_colc = smem + fp.colc_off;        // [parity][chunk][32 px][16 B]
  uint8_t* s_stage = smem + fp.stage_off;      // 4 x 4 KB: epilogue 2's TMA-store images (one per TMEM lane quadrant)
  FusedEncBars* bars = reinterpret_cast<FusedEncBars*>(smem + fp.bars_off);
  __shared__ __align__(16) float s_bias2[32];

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t rank = ptx::cluster_ctarank();
  const bool leader = rank == 0;

  if (tid < 32) s_bias2[tid] = tid < a2.cout ? a2.bias[tid] : 0.f;
  for (int i = tid; i < 4608 / 16; i += kFEThreads)
    reinterpret_cast<uint4*>(s_w1)[i] = __ldg(reinterpret_cast<const uint4*>(fp.w1img + (size_t)rank * 4608) + i);
  if (tid == 0) {
    ptx::mbar_init(&bars->w_full, leader ? 2 : 1);
    for (int i = 0; i < kFERawStages; ++i) {
      ptx::mbar_init(&bars->raw_full[i], 1);
      ptx::mbar_init(&bars->raw_empty[i], 1);
    }
    // arrivals of a warp group are gathered with a named barrier first: one mbarrier arrival per CTA (every mbarrier event
    // wakes every warp parked in a try_wait of this CTA, and sixteen warps arriving one by one kept the others polling)
    ptx::mbar_init(&bars->op_full, 2);
    ptx::mbar_init(&bars->op_empty, 1);
    ptx::mbar_init(&bars->acc1_full, 1);
    ptx::mbar_init(&bars->acc1_empty, 2);
    ptx::mbar_init(&bars->reg_full, 2);
    ptx::mbar_init(&bars->reg_empty, 1);
    for (int i = 0; i < 2; ++i) {
      ptx::mbar_init(&bars->acc2_full[i], 1);
      ptx::mbar_init(&bars->acc2_empty[i], 2 * 4);
    }
    ptx::fence_barrier_init();
  }
  if (warp == 2) {
    ptx::tmem_alloc2(&bars->tmem_base, 512);
    ptx::tmem_relinquish2();
  }
  ptx::fence_proxy_async_smem();
  ptx::tc_fence_before();
  __syncthreads();
  ptx::cluster_sync();
  ptx::tc_fence_after();
  const uint32_t tmem_base = bars->tmem_base;
  const long long npairs = gridDim.x >> 1, pair0 = blockIdx.x >> 1;
  const int NPAD2 = p2.npad;   // 32
  long long my_pairs = fp.pairs_total > pair0 ? (fp.pairs_total - pair0 + npairs - 1) / npairs : 0;
  const long long nsteps = my_pairs * fp.tiles_pp;
  // step -> tile: tiles are walked bottom-to-top, right-to-left inside a patch
  auto tile_of = [&](int t, int& ty, int& tx) {
    const int r = fp.tiles_pp - 1 - t;
    ty = r / fp.tiles_x;
    tx = r - ty * fp.tiles_x;
  };

  if (warp == 0) {
    // ===== raw-window producer (both CTAs): encode_1's weight halves once, then one 65 x 112-byte box per tile =====
    const Geo g = a1.geo;
    if (ptx::elect_one()) {
      ptx::prefetch_tmap(&tm_img);
      const uint32_t w2A = (p2.wA_bytes + 1023u) & ~1023u, w2B = (p2.wB_bytes + 1023u) & ~1023u;
      const uint8_t* src2 = p2.wimg + (size_t)rank * (w2A + w2B);
      ptx::mbar_expect_tx(&bars->w_full, p2.wA_bytes + p2.wB_bytes);
      for (uint32_t off = 0; off < p2.wA_bytes; off += 16384u) ptx::bulk_load(s_w2A + off, src2 + off, min(16384u, p2.wA_bytes - off), &bars->w_full);
      ptx::bulk_load(s_w2B, src2 + w2A, p2.wB_bytes, &bars->w_full);
    }
    __syncwarp();
    if (!leader) {
      ptx::mbar_wait(&bars->w_full, 0);
      if (ptx::elect_one()) ptx::mbar_arrive_leader(&bars->w_full);
      __syncwarp();
    }
    long long step = 0;
    for (long long pp = pair0; pp < fp.pairs_total; pp += npairs) {
      const long long n0 = 2 * pp + rank;
      unsigned img = 0, gy = 0, gx = 0;
      if (n0 < fp.n) geo_decode(g, (unsigned)(g.n0 + n0), img, gy, gx);
      for (int t = 0; t < fp.tiles_pp; ++t, ++step) {
        int ty, tx;
        tile_of(t, ty, tx);
        const uint32_t r = (uint32_t)(step % kFERawStages);
        ptx::mbar_wait(&bars->raw_empty[r], (uint32_t)((step / kFERawStages) & 1) ^ 1u);
        if (ptx::elect_one()) {
          // a patch beyond the batch (odd tail): fetch image 0's window, epilogue 2 stores nothing
          const int Yb = g.oy + (int)gy * g.P + 64 * ty, Xb = g.ox + (int)gx * g.P + 32 * tx;
          ptx::mbar_expect_tx(&bars->raw_full[r], kFEOpRows * kFERawRow);
          ptx::tma_load_3d(s_rawwin + (size_t)r * kFERawStage, &tm_img, &bars->raw_full[r], Xb * 3, Yb, (int)img);
        }
        __syncwarp();
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer (leader): MMA1 of tile i + 1 is issued before MMA2 of tile i =====
    if (leader && nsteps > 0) {
      // first layer: un-swizzled K-major operands straight over the input window (tic_first16.cuh), M = 256 over the pair
      const uint32_t idesc1_st = ptx::make_idesc_f16(256, 64);
      const uint32_t a1_hi32 = ((2u * kFEOpPitch) >> 4) | (1u << 14);
      const uint32_t w1_hi32 = (128u >> 4) | (1u << 14);
      const uint32_t a1_lbo = (16u >> 4) << 16;
      const uint32_t w1A_d = (ptx::smem_u32(s_w1) >> 4) | (((32u * 16u) >> 4) << 16);           // k-group stride: 32 rows x 16 B
      const uint32_t op_d = (ptx::smem_u32(s_op) >> 4) | a1_lbo;
      // second layer: the stride-2 pair kernel's operand geometry over the region buffer
      const uint32_t idesc2_st = ptx::make_idesc_f16(256, 2 * NPAD2), idesc2_lo = ptx::make_idesc_f16(256, NPAD2);
      const uint32_t a2_hi32 = (p2.sbo >> 4) | (1u << 14) | (p2.a_layout << 29);
      const uint32_t w2_hi32 = (p2.w_sbo >> 4) | (1u << 14) | (p2.w_layout << 29);
      const uint32_t tap2A = (uint32_t)NPAD2 * (uint32_t)p2.kc * 2u, tap2B = tap2A >> 1;
      const uint32_t w2A_d = (ptx::smem_u32(s_w2A) >> 4) | (1u << 16), w2B_d = (ptx::smem_u32(s_w2B) >> 4) | (1u << 16);
      const uint32_t reg_d = (ptx::smem_u32(s_region) >> 4) | (1u << 16);
      ptx::mbar_wait(&bars->w_full, 0);
      [[maybe_unused]] long long pw0 = 0, pw1 = 0, pw2 = 0, pw3 = 0;
      [[maybe_unused]] const long long pt0 = TIC_PROF_NOW();
      auto mma1 = [&](long long step) {
        TIC_PROF_WAIT(pw0, ptx::mbar_wait(&bars->acc1_empty, (uint32_t)(step & 1) ^ 1u));
        TIC_PROF_WAIT(pw1, ptx::mbar_wait(&bars->op_full, (uint32_t)(step & 1)));
        ptx::tc_fence_after();
        if (!(TIC_DBG_BITS(p2.dbg) & 16) && ptx::elect_one()) {
#pragma unroll
          for (int sub = 0; sub < 4; ++sub) {
            const uint32_t aoff = ((uint32_t)((sub >> 1) * 32) * kFEOpPitch + (uint32_t)((sub & 1) * 16) * 8u) >> 4;
            const uint32_t ah = op_d + aoff;
            const uint32_t d = tmem_base + (uint32_t)sub * 64u;   // columns 0-31: A x W'_hi, 32-63: A x W'_lo' (A is exact)
#pragma unroll
            for (int kh = 0; kh < 3; ++kh)
              ptx::mma2_f16_ss(d, u16_desc(ah + (uint32_t)kh * (kFEOpPitch >> 4), a1_hi32), u16_desc(w1A_d + (uint32_t)kh * (1024u >> 4), w1_hi32),
                               idesc1_st, kh ? 1u : 0u);
          }
        }
        __syncwarp();
        if (ptx::elect_one()) {
          ptx::tc_commit2(&bars->op_empty);
          ptx::tc_commit2(&bars->acc1_full);
        }
        __syncwarp();
      };
      mma1(0);
      for (long long step = 0; step < nsteps; ++step) {
        if (step + 1 < nsteps) mma1(step + 1);
        const uint32_t b = (uint32_t)(step & 1);
        TIC_PROF_WAIT(pw2, ptx::mbar_wait(&bars->acc2_empty[b], (uint32_t)((step >> 1) & 1) ^ 1u));
        TIC_PROF_WAIT(pw3, ptx::mbar_wait(&bars->reg_full, (uint32_t)(step & 1)));
        ptx::tc_fence_after();
        if (!(TIC_DBG_BITS(p2.dbg) & 1) && ptx::elect_one()) {
          const uint32_t d = tmem_base + 256u + b * 64u;
          uint32_t sp = 0, fresh = 1;
          u16_issue_plane_t<U16_S2, 2>(p2, reg_d, w2A_d, d, 2u * NPAD2, idesc2_st, a2_hi32, w2_hi32, tap2A >> 4, 0u, sp, fresh, true);
          fresh = 0;
          u16_issue_plane_t<U16_S2, 2>(p2, reg_d + (kFERegionPlane >> 4), w2B_d, d + (uint32_t)NPAD2, 2u * NPAD2, idesc2_lo, a2_hi32,
                                       w2_hi32, tap2B >> 4, 0u, sp, fresh, false);
        }
        __syncwarp();
        if (ptx::elect_one()) {
          ptx::tc_commit2(&bars->reg_empty);
          ptx::tc_commit2(&bars->acc2_full[b]);
        }
        __syncwarp();
      }
      TIC_PROF_ADD(0, pw0);
      TIC_PROF_ADD(1, pw1);
      TIC_PROF_ADD(2, pw2);
      TIC_PROF_ADD(3, pw3);
      TIC_PROF_ADD(4, TIC_PROF_NOW() - pt0);
      TIC_PROF_ADD(5, nsteps);
    }
  } else if (warp >= kFEBuilderWarp0) {
    // ===== builders: raw u8 window -> the exact integer operand (x - m_c, 1) as RGB1 fp16 quads of the 65 x 34 window =====
    // The kernel sits on the shared-memory data pipe (ncu: LSU + tensor-core wavefronts = 92 % of its cycles before this
    // layout), so the builders are written for wavefronts: an item is (row, PAIR of pixels) — 65 x 17 = 1105 items,
    // consecutive lanes take consecutive pairs.  Six raw bytes come from two aligned words (consecutive lanes: consecutive
    // words); a byte b becomes the fp16 integer 1024 + b by byte permutation (0x6400 | b) and x - m_c by one exact half2
    // subtraction (FusedEncNorm: no normalisation, no split, no table); the two quads go out as one 16-byte store at
    // item * 16 — consecutive lanes, consecutive chunks.
    const int bl = (warp - kFEBuilderWarp0) * 32 + lane;
    const __half2 c_rg = __floats2half2_rn(1024.0f + (float)fp.moff[0], 1024.0f + (float)fp.moff[1]);
    const __half2 c_b1 = __floats2half2_rn(1024.0f + (float)fp.moff[2], 0.0f);
    long long step = 0;
    [[maybe_unused]] long long pw0 = 0, pw1 = 0;
    [[maybe_unused]] const long long pt0 = TIC_PROF_NOW();
    auto as_h2 = [](const uint32_t x) { return *reinterpret_cast<const __half2*>(&x); };
    auto as_u32 = [](const __half2 x) { return *reinterpret_cast<const uint32_t*>(&x); };
    auto build = [&](const int item, const uint32_t w0, const uint32_t w1, const int ty, const int tx) {
      const int ry = item / 17, pp = item - ry * 17;
      const uint32_t sh = (uint32_t)(pp & 1) * 16u;           // byte offset 6 * pp is 0 or 2 (mod 4)
      const uint32_t p0 = __funnelshift_r(w0, w1, sh);        // R0 G0 B0 R1
      const uint32_t p1 = __byte_perm(p0, w1 >> sh, 0x5543);  // R1 G1 B1 .
      const bool row_ok = 64 * ty + ry < fp.P;
      const int ix = 32 * tx + 2 * pp;
      const bool ok0 = row_ok && ix < fp.P, ok1 = row_ok && ix + 1 < fp.P;
      // (1024 + R, 1024 + G) and (1024 + B, 1.0): bytes (b, 0x64, b', 0x64) and (b, 0x64, 0x00, 0x3C)
      uint32_t q0 = as_u32(__hsub2(as_h2(__byte_perm(p0, 0x64646464u, 0x4140)), c_rg));
      uint32_t q1 = as_u32(__hsub2(as_h2(__byte_perm(p0, 0x3C000064u, 0x7542)), c_b1));
      uint32_t q2 = as_u32(__hsub2(as_h2(__byte_perm(p1, 0x64646464u, 0x4140)), c_rg));
      uint32_t q3 = as_u32(__hsub2(as_h2(__byte_perm(p1, 0x3C000064u, 0x7542)), c_b1));
      if (!ok0) q0 = q1 = 0u;   // outside the patch: the conv's zero padding (pixel and its constant 1)
      if (!ok1) q2 = q3 = 0u;
      sts128(ptx::smem_u32(s_op) + (uint32_t)item * 16u, q0, q1, q2, q3);   // row pitch 272 B = 17 pairs x 16 B
    };
    constexpr int kItems = kFEOpRows * 17, kLanes = kFEBuilders * 32;
    for (long long pp = pair0; pp < fp.pairs_total; pp += npairs) {
      for (int t = 0; t < fp.tiles_pp; ++t, ++step) {
        int ty, tx;
        tile_of(t, ty, tx);
        const uint32_t r = (uint32_t)(step % kFERawStages);
        // one warp polls the mbarriers, the others park in the named barrier (no issue slots spent on waiting)
        if (warp == kFEBuilderWarp0) {
          TIC_PROF_WAIT(pw0, ptx::mbar_wait(&bars->raw_full[r], (uint32_t)((step / kFERawStages) & 1)));
          TIC_PROF_WAIT(pw1, ptx::mbar_wait(&bars->op_empty, (uint32_t)(step & 1) ^ 1u));   // MMA1 of the previous tile has read the operand buffer
        }
        asm volatile("bar.sync 8, %0;" ::"n"(kFEBuilders * 32) : "memory");
        const uint32_t rawb = ptx::smem_u32(s_rawwin + (size_t)r * kFERawStage);
        if (!(TIC_DBG_BITS(p2.dbg) & 8)) {
          // two independent items per pass: their shared-memory round trips overlap
#pragma unroll 1
          for (int item = bl; item < kItems; item += 2 * kLanes) {
            const int itemB = item + kLanes;
            const bool hasB = itemB < kItems;
            const int ryA = item / 17, ppA = item - ryA * 17;
            const int ryB = hasB ? itemB / 17 : ryA, ppB = hasB ? itemB - ryB * 17 : ppA;
            const uint32_t adA = rawb + (uint32_t)ryA * kFERawRow + ((uint32_t)(6 * ppA) & ~3u);
            const uint32_t adB = rawb + (uint32_t)ryB * kFERawRow + ((uint32_t)(6 * ppB) & ~3u);
            const uint32_t a0 = lds32(adA), a1w = lds32(adA + 4u), b0 = lds32(adB), b1w = lds32(adB + 4u);
            build(item, a0, a1w, ty, tx);
            if (hasB) build(itemB, b0, b1w, ty, tx);
          }
        }
        ptx::fence_proxy_async_smem();
        // the warp with the longest item list gathers the others and arrives once
        if (warp == kFEBuilderWarp0) {
          asm volatile("bar.sync 9, %0;" ::"n"(kFEBuilders * 32) : "memory");
          if (lane == 0) {
            ptx::mbar_arrive(&bars->raw_empty[r]);
            ptx::mbar_arrive_leader(&bars->op_full);
          }
        } else {
          asm volatile("bar.arrive 9, %0;" ::"n"(kFEBuilders * 32) : "memory");
        }
      }
    }
    if (warp == kFEBuilderWarp0) {
      TIC_PROF_ADD(8, pw0);
      TIC_PROF_ADD(9, pw1);
      TIC_PROF_ADD(10, TIC_PROF_NOW() - pt0);
    }
  } else if (warp >= 4 && warp < kFEBuilderWarp0) {
    // ===== epilogue warps.  Per tile: A  first-layer accumulators -> registers, bias, relu, fp16 split (overlaps the
    // previous tile's MMA2);  B  halo + region writes, "region full";  C  epilogue 2 of the previous tile. =====
    const int q4 = warp & 3, sub = (warp - 4) >> 2;     // TMEM lane quadrant; first-layer sub-tile of this warp
    const int m = q4 * 32 + lane, hh = m >> 3, xx = m & 7;
    const int e = tid - 128;                            // 0 .. 511 among the epilogue threads
    const uint32_t reg_hi = ptx::smem_u32(s_region), reg_lo = reg_hi + kFERegionPlane;
    const uint32_t rowc = ptx::smem_u32(s_rowc), colc = ptx::smem_u32(s_colc);
    const uint32_t rowc_par = (uint32_t)fp.tiles_x * 16u * 128u;
    const int rowc_px = fp.tiles_x * 16;   // pixels of one cached row (chunk-major caches: [chunk 8][pixel][16 B])
    const uint32_t tq = tmem_base + ((uint32_t)(q4 * 32) << 16);
    const uint32_t tbuf1 = tq + (uint32_t)sub * 64u;
    const float floor1 = a1.act ? 0.0f : -INFINITY;
    const int R = (sub >> 1) * 16 + hh, C = (sub & 1) * 8 + xx;   // region coordinates of this lane's intermediate pixel
    // byte offset of intermediate pixel (r, c) inside a region plane: the stride-2 box layout [h2][h parity][w2][w parity][32 ch]
    auto cell = [](int r, int c) { return (uint32_t)((((r >> 1) * 2 + (r & 1)) * 9 + (c >> 1)) * 128 + (c & 1) * 64); };
    const uint32_t pix = cell(R, C);
    __half2 omax = __floats2half2_rn(0.f, 0.f);
    [[maybe_unused]] long long pw0 = 0, pw1 = 0, pw2 = 0, pw3 = 0, pw4 = 0, pw5 = 0, pw6 = 0, pw7 = 0, pw8 = 0;
    [[maybe_unused]] const long long pt0 = TIC_PROF_NOW();
    // epilogue 2, one tile behind, shared by all sixteen warps (on the four warps of sub-tile 0 alone it took 2400 cycles
    // of a 6100-cycle step and everything else waited for them): the four warps of a TMEM lane quadrant take eight of
    // encode_1's 32 channels each — one 16-byte chunk per pixel and plane of the quadrant's TMA-store image
    // (tic_first16.cuh: 32 pixels x 64 B, 64-byte swizzle) — and the warp of sub-tile 0 stores both planes.
    const uint32_t stage2 = ptx::smem_u32(s_stage + (size_t)q4 * kFEStagePerWarp);
    const uint32_t stage_px = stage2 + (uint32_t)lane * 64u + (uint32_t)((sub ^ ((lane >> 1) & 3)) << 4);
    const float floor2 = a2.act ? 0.0f : -INFINITY;
    auto epilogue2 = [&](long long estep, long long en, int ety, int etx) {
      const uint32_t b = (uint32_t)(estep & 1);
      // (already complete: phase B of this step waited for the same MMA2; a first-try success, no polling)
      TIC_PROF_WAIT(pw2, ptx::mbar_wait(&bars->acc2_full[b], (uint32_t)((estep >> 1) & 1)));
      ptx::tc_fence_after();
      if (!(TIC_DBG_BITS(p2.dbg) & 2)) {
        float v[8], u[8];
        const uint32_t tb = tq + 256u + b * 64u + (uint32_t)(sub * 8);
        ptx::tmem_ld8_nowait(tb + (uint32_t)NPAD2, u);
        ptx::tmem_ld8_nowait(tb, v);
        ptx::tmem_ld_wait();
        ptx::tc_fence_before();
        const float4 b0 = *reinterpret_cast<const float4*>(s_bias2 + sub * 8), b1 = *reinterpret_cast<const float4*>(s_bias2 + sub * 8 + 4);
        v[0] = fmaxf(__fadd_rn(__fmaf_rn(u[0], 1.0f / 2048.0f, v[0]), b0.x), floor2);
        v[1] = fmaxf(__fadd_rn(__fmaf_rn(u[1], 1.0f / 2048.0f, v[1]), b0.y), floor2);
        v[2] = fmaxf(__fadd_rn(__fmaf_rn(u[2], 1.0f / 2048.0f, v[2]), b0.z), floor2);
        v[3] = fmaxf(__fadd_rn(__fmaf_rn(u[3], 1.0f / 2048.0f, v[3]), b0.w), floor2);
        v[4] = fmaxf(__fadd_rn(__fmaf_rn(u[4], 1.0f / 2048.0f, v[4]), b1.x), floor2);
        v[5] = fmaxf(__fadd_rn(__fmaf_rn(u[5], 1.0f / 2048.0f, v[5]), b1.y), floor2);
        v[6] = fmaxf(__fadd_rn(__fmaf_rn(u[6], 1.0f / 2048.0f, v[6]), b1.z), floor2);
        v[7] = fmaxf(__fadd_rn(__fmaf_rn(u[7], 1.0f / 2048.0f, v[7]), b1.w), floor2);
        uint32_t h4[4], l4[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) split16x2(v[2 * i], v[2 * i + 1], h4[i], l4[i], omax);
        sts128(stage_px, h4[0], h4[1], h4[2], h4[3]);
        sts128(stage_px + kT2LoOff, l4[0], l4[1], l4[2], l4[3]);
        ptx::fence_proxy_async_smem();   // generic-proxy stage writes -> visible to the TMA store
      } else {
        ptx::tc_fence_before();
      }
      // quadrant barrier 10 + q4: the warp of sub-tile 0 gathers the other three, hands the accumulators back and stores
      if (sub == 0) {
        asm volatile("bar.sync %0, 128;" ::"r"(10 + q4) : "memory");
        if (lane == 0) {
          ptx::mbar_arrive_leader(&bars->acc2_empty[b]);
          if (en < fp.n && !(TIC_DBG_BITS(p2.dbg) & 2)) {
            ptx::tma_store_4d_s(&tm_ohi, stage2, 0, etx * 8, ety * 16 + 4 * q4, (int)en);
            ptx::tma_store_4d_s(&tm_olo, stage2 + kT2LoOff, 0, etx * 8, ety * 16 + 4 * q4, (int)en);
            ptx::bulk_commit_group();
          }
        }
      } else {
        asm volatile("bar.arrive %0, 128;" ::"r"(10 + q4) : "memory");
      }
    };
    long long step = 0, pn = 0;
    int pty = 0, ptx_ = 0;
    for (long long pp = pair0; pp < fp.pairs_total; pp += npairs) {
      for (int t = 0; t < fp.tiles_pp; ++t, ++step) {
        int ty, tx;
        tile_of(t, ty, tx);
        // caches: this tile READS the row cache the tile below wrote (parity (ty + 1) & 1) and the column cache of the tile
        // to the right (parity (tx + 1) & 1), and WRITES parities ty & 1 / tx & 1
        const uint32_t rowc_rd = rowc + (uint32_t)((ty + 1) & 1) * rowc_par, rowc_wr = rowc + (uint32_t)(ty & 1) * rowc_par;
        const uint32_t colc_rd = colc + (uint32_t)((tx + 1) & 1) * 4096u, colc_wr = colc + (uint32_t)(tx & 1) * 4096u;
        const bool has_below = ty + 1 < fp.tiles_y, has_right = tx + 1 < fp.tiles_x;
        // ---- phase A ----
        // one warp polls, the rest parks in a named barrier (every polling warp costs issue slots)
        if (warp == 8) TIC_PROF_WAIT(pw0, ptx::mbar_wait(&bars->acc1_full, (uint32_t)(step & 1)));
        TIC_PROF_WAIT(pw5, asm volatile("bar.sync 3, 512;" ::: "memory"));
        [[maybe_unused]] const long long pta = TIC_PROF_NOW();
        ptx::tc_fence_after();
        uint32_t hp[2][8], lp[2][8];
#pragma unroll
        for (int ci = 0; ci < 2; ++ci) {
          float v[16], u[16];
          ptx::tmem_ld16_nowait(tbuf1 + (uint32_t)(32 + ci * 16), u);
          ptx::tmem_ld16_nowait(tbuf1 + (uint32_t)(ci * 16), v);
          ptx::tmem_ld_wait();
          if (ci == 1) {   // last TMEM read: one warp gathers the group and arrives once
            ptx::tc_fence_before();
            if (warp == 4) {
              TIC_PROF_WAIT(pw6, asm volatile("bar.sync 6, 512;" ::: "memory"));
              if (lane == 0) ptx::mbar_arrive_leader(&bars->acc1_empty);
            } else {
              asm volatile("bar.arrive 6, 512;" ::: "memory");
            }
          }
#pragma unroll
          for (int i = 0; i < 16; ++i)
            v[i] = fmaxf(__fadd_rn(__fmaf_rn(u[i], 1.0f / 2048.0f, v[i]), fp.bias1[ci * 16 + i]), floor1);
#pragma unroll
          for (int i = 0; i < 8; ++i) split16x2(v[2 * i], v[2 * i + 1], hp[ci][i], lp[ci][i], omax);
        }
        // ---- phase B ----
        pw7 += TIC_PROF_NOW() - pta;   // phase A
        if (warp == 8) TIC_PROF_WAIT(pw1, ptx::mbar_wait(&bars->reg_empty, (uint32_t)(step & 1) ^ 1u));
        if (sub == 0 && lane == 0) ptx::bulk_wait_group_read<0>();   // this quadrant's previous TMA store has read the stage
        // region free; the previous tile's cache writes are visible; the stage may be rewritten in phase C
        TIC_PROF_WAIT(pw4, asm volatile("bar.sync 2, 512;" ::: "memory"));
        [[maybe_unused]] const long long ptb = TIC_PROF_NOW();
        // halo: row 32 (17 pixels, corner last) and column 16 (32 pixels) of the region, 8 chunks of 16 B each
        if (e < 49 * 8 && !(TIC_DBG_BITS(p2.dbg) & 4)) {
          // consecutive lanes take consecutive halo pixels of one chunk: the caches are chunk-major ([chunk][pixel][16 B])
          const int ch = e / 49, hx = e - ch * 49;        // ch 0..3: hi plane, 4..7: lo' plane
          uint4 val = make_uint4(0u, 0u, 0u, 0u);
          uint32_t dst;
          if (hx < 17) {                                  // region row 32, column hx (corner hx = 16: the tile below-right)
            if (has_below && (hx < 16 || has_right)) val = lds128(rowc_rd + (uint32_t)((ch * rowc_px + tx * 16 + hx) * 16));
            dst = cell(32, hx);
          } else {                                        // region column 16, row hx - 17
            if (has_right) val = lds128(colc_rd + (uint32_t)((ch * 32 + hx - 17) * 16));
            dst = cell(hx - 17, 16);
          }
          const uint32_t addr = (ch < 4 ? reg_hi : reg_lo) + dst + (uint32_t)(ch & 3) * 16u;
          sts128(fused_swz128(addr), val.x, val.y, val.z, val.w);
        }
#pragma unroll
        for (int ci = 0; ci < ((TIC_DBG_BITS(p2.dbg) & 4) ? 0 : 2); ++ci) {
          const uint32_t ah = reg_hi + pix + (uint32_t)ci * 32u, al = reg_lo + pix + (uint32_t)ci * 32u;
          sts128(fused_swz128(ah), hp[ci][0], hp[ci][1], hp[ci][2], hp[ci][3]);
          sts128(fused_swz128(ah + 16u), hp[ci][4], hp[ci][5], hp[ci][6], hp[ci][7]);
          sts128(fused_swz128(al), lp[ci][0], lp[ci][1], lp[ci][2], lp[ci][3]);
          sts128(fused_swz128(al + 16u), lp[ci][4], lp[ci][5], lp[ci][6], lp[ci][7]);
          if (R == 0) {    // first row of the region: halo row of the tile above (corner of the tile above-left)
            const uint32_t c0 = rowc_wr + (uint32_t)((2 * ci * rowc_px + tx * 16 + C) * 16), cs = (uint32_t)rowc_px * 16u;
            sts128(c0, hp[ci][0], hp[ci][1], hp[ci][2], hp[ci][3]);
            sts128(c0 + cs, hp[ci][4], hp[ci][5], hp[ci][6], hp[ci][7]);
            sts128(c0 + 4u * cs, lp[ci][0], lp[ci][1], lp[ci][2], lp[ci][3]);
            sts128(c0 + 5u * cs, lp[ci][4], lp[ci][5], lp[ci][6], lp[ci][7]);
          }
          if (C == 0) {    // first column: halo column of the tile to the left
            const uint32_t c0 = colc_wr + (uint32_t)((2 * ci * 32 + R) * 16);
            sts128(c0, hp[ci][0], hp[ci][1], hp[ci][2], hp[ci][3]);
            sts128(c0 + 512u, hp[ci][4], hp[ci][5], hp[ci][6], hp[ci][7]);
            sts128(c0 + 2048u, lp[ci][0], lp[ci][1], lp[ci][2], lp[ci][3]);
            sts128(c0 + 2560u, lp[ci][4], lp[ci][5], lp[ci][6], lp[ci][7]);
          }
        }
        ptx::fence_proxy_async_smem();
        pw8 += TIC_PROF_NOW() - ptb;   // phase B
        if (warp == 8) {
          TIC_PROF_WAIT(pw6, asm volatile("bar.sync 7, 512;" ::: "memory"));
          if (lane == 0) ptx::mbar_arrive_leader(&bars->reg_full);
        } else {
          asm volatile("bar.arrive 7, 512;" ::: "memory");
        }
        // ---- phase C: epilogue 2 of the previous tile ----
        if (step > 0) TIC_PROF_WAIT(pw3, epilogue2(step - 1, pn, pty, ptx_));
        pn = 2 * pp + rank;
        pty = ty;
        ptx_ = tx;
      }
    }
    if (step > 0) {
      if (sub == 0 && lane == 0) ptx::bulk_wait_group_read<0>();
      asm volatile("bar.sync 2, 512;" ::: "memory");
      epilogue2(step - 1, pn, pty, ptx_);
    }
    if (sub == 0 && lane == 0) ptx::bulk_wait_group<0>();   // every TMA store of this warp is complete before the CTA may exit
    if (ovf_hit(omax)) ovf_raise(a1.oflow);
    if (warp == 4 || warp == 8) {   // an epilogue-2 warp and a plain one
      [[maybe_unused]] const int base = warp == 4 ? 16 : 24;
      TIC_PROF_ADD(base + 0, pw0);
      TIC_PROF_ADD(base + 1, pw1);
      TIC_PROF_ADD(base + 2, pw2);
      TIC_PROF_ADD(base + 3, pw3);
      TIC_PROF_ADD(base + 4, pw4);
      TIC_PROF_ADD(base + 5, TIC_PROF_NOW() - pt0);
      TIC_PROF_ADD(base + 16, pw5);
      TIC_PROF_ADD(base + 17, pw6);
      TIC_PROF_ADD(base + 18, pw7);
      TIC_PROF_ADD(base + 19, pw8);
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  ptx::cluster_sync();
  if (warp == 2) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc2(tmem_base, 512);
  }
}

// The builders' operand is the exact integer x - m_c with m_c = round(mean_c): it must stay inside the exact fp16 integer
// range the weight image was laid out for.
inline bool fused_enc_mean_ok(float mean) {
  const long m = lrintf(mean);
  return m >= -768 && m <= 1023;
}

// Which layer pairs take the fused kernel: the u8 image through conv 3 -> 32 stride 2 (TMA-fed windowed first layer)
// followed by conv 32 -> 32 stride 2 into pair planes.  Other channel means take the first-layer + u16 kernels.
inline bool fused_enc_supported(const LayerArgs& a1, int kind1, int stride1, const LayerArgs& a2, int kind2, int stride2) {
  if (kind1 != 0 || kind2 != 0 || stride1 != 2 || stride2 != 2) return false;
  if (a1.in_mode != IO_U8_NORM || a1.cin != 3 || a1.cout != 32 || a2.cin != 32 || a2.cout != 32) return false;
  for (int c = 0; c < 3; ++c)
    if (!fused_enc_mean_ok(a1.mean[c])) return false;
  if (a1.res || a2.res || a2.out_mode != IO_ACT16) return false;
  if (a1.hin != a1.win || a1.hin % 64 != 0 || a1.hin / 32 > kFusedMaxTilesX) return false;
  if (a1.hout * 2 != a1.hin || a2.hin != a1.hout || a2.hout * 2 != a2.hin || a2.wout * 2 != a2.win) return false;
  return f16_first_tma_ok(a1);
}

// img[0]: the first layer's operand image with the normalisation folded in (f16_build_weights_s2_pair_kernel), img[1]: the
// second layer's
inline tic_status launch_fused_enc(const LaunchCtx& c, const LayerArgs& a1, const LayerArgs& a2, const float* w1_dev, const float* w2_dev,
                                   const float* bias1_host, OperandImage* img) {
  if (c.num_sms < 2) return c.fail("the fused encoder kernel needs CTA pairs", TIC_ERR_UNSUPPORTED);
  U16Plan pl2{};
  if (!u16_plan(a2, 0, 2, a2.cout, &pl2)) return c.fail("fused encoder plan failed", TIC_ERR_UNSUPPORTED);
  U16Params p2 = pl2.p;
  if (p2.mode != U16_S2 || p2.nbox != 1 || p2.ksteps != 2 || p2.KB != 1 || p2.bn != 1 || p2.npad != 32 || p2.nsplit != 1)
    return c.fail("fused encoder: unexpected layer plan", TIC_ERR_UNSUPPORTED);
  FusedEncNorm nm{};
  for (int ch = 0; ch < 3; ++ch) {
    nm.mean[ch] = a1.mean[ch];
    nm.stdv[ch] = a1.stdv[ch];
    nm.m[ch] = (int)lrintf(a1.mean[ch]);
    if (!fused_enc_mean_ok(a1.mean[ch])) return c.fail("fused encoder: channel mean outside the exact fp16 integer range", TIC_ERR_UNSUPPORTED);
  }
  bool build;  // (tic_set_norm after the first launch changes nm: the image is rebuilt)
  if (img[0].ensure(image_key(w1_dev, a1.cout, nm), 2 * 4608, &build) != TIC_OK)
    return c.fail("cudaMalloc for the fused first-layer weight image failed", TIC_ERR_NOMEM);
  if (build) {
    f16_build_weights_s2_pair_kernel<<<8, 256, 0, c.stream>>>(w1_dev, a1.cout, img[0].buf.as<uint8_t>(), nm);
    if (cudaGetLastError() != cudaSuccess) return c.fail("fused first-layer weight image kernel failed", TIC_ERR_CUDA);
  }
  if (tic_status s = u16_pair_image(c.stream, img[1], w2_dev, a2, p2, 0, a2.cout)) return c.fail("fused encoder: weight images failed", s);
  p2.wimg = img[1].img();
  p2.dbg = tic_env_int("TIC_DBG", 0);  // -DTIC_ABLATE builds only: 1 no MMA2, 16 no MMA1, 2 no epilogue 2, 4 no region writes, 8 no builders

  FusedEncParams fp{};
  fp.n = a1.n;
  fp.P = a1.hin;
  fp.tiles_x = a2.wout / 8;
  fp.tiles_y = a2.hout / 16;
  fp.tiles_pp = fp.tiles_x * fp.tiles_y;
  fp.pairs_total = ((long long)a1.n + 1) / 2;
  fp.w1img = img[0].img();
  for (int ch = 0; ch < 3; ++ch) fp.moff[ch] = nm.m[ch];
  for (int i = 0; i < 32; ++i) fp.bias1[i] = i < a1.cout ? bias1_host[i] : 0.f;
  auto up = [](uint32_t v) { return (v + 1023u) & ~1023u; };
  uint32_t off = 0;
  fp.w1_off = off;
  off += up(4608);
  fp.w2_off = off;
  off += up(p2.wA_bytes);
  fp.w2B_off = off;
  off += up(p2.wB_bytes);
  fp.op_off = off;
  off += up(kFEOpPlane);
  fp.raw_off = off;
  off += up(kFERawStages * kFERawStage);
  fp.region_off = off;
  off += 2u * kFERegionPlane;
  fp.rowc_off = off;
  off += 2u * (uint32_t)fp.tiles_x * 16u * 128u;
  fp.colc_off = off;
  off += 2u * 32u * 128u;
  fp.stage_off = off;
  off += 4u * kFEStagePerWarp;
  fp.bars_off = off;
  off += (uint32_t)sizeof(FusedEncBars);
  fp.smem_bytes = off + 1024u;
  if (fp.smem_bytes + 1024u /* static: bias, alignment */ > 227u * 1024u)
    return c.fail("fused encoder: shared memory plan does not fit", TIC_ERR_UNSUPPORTED);

  // raw image windows: box 65 rows x 112 bytes; encode_1's output planes
  CUtensorMap tm_img, tm_o[2];
  if (tic_status s = tmap_image_rows(&tm_img, a1, false, kFERawRow, kFEOpRows, "image windows", c.err)) return s;
  for (int pl = 0; pl < 2; ++pl)
    if (tic_status s = tmap_pair_out(&tm_o[pl], reinterpret_cast<__half*>(a2.out) + (pl ? a2.out_lo_off : 0), a2.n, a2.hout, a2.wout,
                                     a2.cout, "fused encoder output", c.err))
      return s;
  const int grid = 2 * (int)std::min<long long>(fp.pairs_total, c.num_sms / 2);
  const cudaError_t e = launch_dyn(fused_enc_kernel, grid, kFEThreads, fp.smem_bytes, c.stream, tm_img, tm_o[0], tm_o[1], a1, p2, a2, fp);
  if (e != cudaSuccess) return c.fail(std::string("fused encoder launch failed: ") + cudaGetErrorString(e), TIC_ERR_CUDA);
  ++*c.launches;
  return TIC_OK;
}

}  // namespace tic

// Back-to-back fused transposed convolutions: the last two layers of the synthesis transform
// (model_0/model.py:224-246: decode_1 32 -> 32 relu, decode_0 32 -> 3 identity + denormalise + clip; the same pair ends
// base_model/input_256) as ONE kernel.  Unfused, the 64 x 64 x 32 tensor between them (512 KB per 128 x 128 patch as
// fp16 pair planes, 6.4 GB per 12 288 patches) is written by one kernel and read back by the next: 12.9 GB of the
// decoder's 15 GB of HBM traffic.  Here it lives in shared memory only:
//
//   TMA (input boxes of decode_1) -> MMA1 (phase-stacked, N = 256 | 128) -> TMEM -> epilogue 1: bias, relu, fp16 split,
//   written as the swizzled K-major operand tile of the next layer -> MMA2 (phase-stacked RGB, four 16 x 8 sub-tiles) ->
//   TMEM -> epilogue 2: bias, denormalise, clip, round, u8 pixels scattered into the stitched image.
//
// A CTA pair (cta_group::2, M = 256) walks two patches in lock-step, tile by tile (16 x 8 input pixels of decode_1 =
// 32 x 16 intermediate pixels = four decode_0 tiles), row-major inside the patch.  decode_0 reads intermediate pixel
// (a - 1 + dy, b - 1 + dx): one halo row above and one halo column left of the 32 x 16 region.  They are not recomputed:
// the last row of every tile of the tile-row above, the last column of the tile to the left and the corner pixel are
// kept in small shared-memory caches (zeros at the patch border = the transposed conv's out-of-range input), so MMA1
// does exactly the work of the unfused layer.
//
// Shared memory per CTA (model_0: 195 KB): weight halves of both layers, a two-slot input ring, ONE region buffer
// (33 x 17 pixels x 64 B x two planes = 72 KB) and the halo caches (two parities each: a tile reads the cache its
// neighbour wrote while it writes the other one).  TMEM: 256 columns for MMA1's accumulators, two buffers of 128
// columns for the four sub-tiles of MMA2.  Warps (640 threads, <= 102 registers): 0 TMA producer, 1 MMA issuer (leader
// CTA), 2 TMEM allocator, 4-19 epilogue (four per TMEM lane quadrant; each does its share of BOTH epilogues, see the
// role code).  The issuer runs MMA1 of tile i + 1 ahead of MMA2 of tile i, and epilogue 1 converts the accumulators
// while the previous MMA2 still runs, so only the region writes sit between two MMA2s.
#pragma once
#include "tic_launch.cuh"
#include "tic_umma16.cuh"

namespace tic {

constexpr int kFusedEpiWarps = 16;                       // every epilogue warp does epilogue 1 AND epilogue 2 work
constexpr int kFusedThreads = 32 * (4 + kFusedEpiWarps);  // 640
constexpr int kFusedRegionCols = 17, kFusedRegionRows = 33;
constexpr uint32_t kFusedRegionPitch = kFusedRegionCols * 64;                 // bytes per region row and plane (32 ch fp16)
constexpr uint32_t kFusedRegionPlane = 36864;                                   // >= 33 * 17 * 64 = 35904, multiple of 1024
// The lo' plane starts one pixel (64 B) past a 128-byte line: a warp's 32 pixels of one output phase all have the same
// pixel parity, so a 16-byte store per lane into ONE plane touches only four of the eight 16-byte bank groups (2-way
// conflict, ncu: x2.4 the ideal wavefronts and the kernel sits on the shared-memory data pipe).  With the planes half a
// line apart, half the lanes store their hi chunk while the other half store their lo' chunk: eight bank groups.
constexpr uint32_t kFusedRegionLoOff = kFusedRegionPlane + 64;
constexpr int kFusedMaxTilesX = 8;

struct FusedDecParams {
  int n;                    // patches
  int tiles_x, tiles_y;     // decode_1 tiles per patch (16 rows x 8 columns of its input map)
  int tiles_pp;             // tiles_x * tiles_y
  long long pairs_total;    // ceil(n / 2)
  uint32_t w1_off, w1B_off, w2_off, w2B_off, in_off, region_off, rowc_off, colc_off, corner_off, bars_off;
  uint32_t smem_bytes;
  float bias1[32];          // decode_1's bias as launch constants (constant-bank operands: no shared-memory loads in phase A)
  float bias2[4];           // decode_0's
};

struct FusedDecBars {
  uint64_t w_full;
  uint64_t in_full[2], in_empty[2];
  uint64_t acc1_full, acc1_empty;
  uint64_t reg_full, reg_empty;
  uint64_t acc2_full[2], acc2_empty[2];
  uint32_t tmem_base;
};

__device__ __forceinline__ uint32_t fused_swz64(uint32_t addr) { return addr ^ (((addr >> 7) & 3u) << 4); }

// decode_0's epilogue for one lane of a 16 x 8 sub-tile: the 16 accumulator columns are (output phase (py, px), channel) of
// the 2 x 2 image pixels of this lane's region pixel (yt, xt).  Bias, denormalise, clip (model_0/model.py:250-259), round
// (decode.py:249), both output rows from ONE pair of TMEM loads and one patch -> image decode (the shared epilogue of
// tic_umma16.cuh takes a row per call: twice the loads, twelve selects).
__device__ __forceinline__ void fused_rgb_epilogue(const LayerArgs& a, const uint32_t tbuf, const int NPAD, const int n, const int yt,
                                                   const int xt, const bool valid, const float* bias3) {
  float v[16], u[16];
  ptx::tmem_ld16_nowait(tbuf + NPAD, u);
  ptx::tmem_ld16_nowait(tbuf, v);
  ptx::tmem_ld_wait();
  if (!valid) return;
  const Geo& g = a.geo;
  unsigned img, gy, gx;
  geo_decode(g, (unsigned)(g.n0 + n), img, gy, gx);   // utils.concat_patches, utils/utils.py:136-167: crop to [H, W]
  const int Y0 = g.oy + (int)gy * g.P + 2 * yt, X = g.ox + (int)gx * g.P + 2 * xt;
#pragma unroll
  for (int half = 0; half < 2; ++half) {
    const int Y = Y0 + half;
    if (Y >= g.H) break;
    const long long off = (((long long)img * g.H + Y) * g.W + X) * 3;
    float y[6];
#pragma unroll
    for (int px = 0; px < 2; ++px)
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const int col = (half * 2 + px) * 4 + c;
        const float t = apply_act(__fadd_rn(__fmaf_rn(u[col], 1.0f / 2048.0f, v[col]), bias3[c]), a.act);
        y[px * 3 + c] = tic_denorm_clip(t, a.mean[c], a.stdv[c]);
      }
    if (a.out_mode == IO_DENORM_U8 && X + 1 < g.W && !((reinterpret_cast<uintptr_t>(a.out) + off) & 1)) {
      // both pixels inside the image and 2-byte aligned (X is even: any even W, and an even base address): three 2-byte stores
      uint32_t q[6];
#pragma unroll
      for (int i = 0; i < 6; ++i) q[i] = (uint32_t)(int)rintf(y[i]);
      unsigned short* o2 = reinterpret_cast<unsigned short*>(reinterpret_cast<uint8_t*>(a.out) + off);
      o2[0] = (unsigned short)(q[0] | (q[1] << 8));
      o2[1] = (unsigned short)(q[2] | (q[3] << 8));
      o2[2] = (unsigned short)(q[4] | (q[5] << 8));
    } else {
#pragma unroll
      for (int px = 0; px < 2; ++px) {
        if (X + px >= g.W) break;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          if (a.out_mode == IO_DENORM_F32)
            reinterpret_cast<float*>(a.out)[off + px * 3 + c] = y[px * 3 + c];
          else
            reinterpret_cast<uint8_t*>(a.out)[off + px * 3 + c] = (uint8_t)(int)rintf(y[px * 3 + c]);
        }
      }
    }
  }
}

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kFusedThreads, 1)
fused_dec_kernel(const __grid_constant__ CUtensorMap tm_hi, const __grid_constant__ CUtensorMap tm_lo, const U16Params p1,
                 const LayerArgs a1, const U16Params p2, const LayerArgs a2, const FusedDecParams fp) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* s_w1A = smem + fp.w1_off;
  uint8_t* s_w1B = smem + fp.w1B_off;
  uint8_t* s_w2A = smem + fp.w2_off;
  uint8_t* s_w2B = smem + fp.w2B_off;
  uint8_t* s_in = smem + fp.in_off;            // 2 ring slots x (hi box | lo box)
  uint8_t* s_region = smem + fp.region_off;    // hi plane | lo plane
  uint8_t* s_rowc = smem + fp.rowc_off;        // [parity][chunk: hi 0-3, lo' 4-7][tiles_x * 16 px][16 B]
  uint8_t* s_colc = smem + fp.colc_off;        // [parity][chunk][32 px][16 B]
  FusedDecBars* bars = reinterpret_cast<FusedDecBars*>(smem + fp.bars_off);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t rank = ptx::cluster_ctarank();
  const bool leader = rank == 0;

  if (tid == 0) {
    ptx::mbar_init(&bars->w_full, leader ? 2 : 1);
    for (int i = 0; i < 2; ++i) {
      ptx::mbar_init(&bars->in_full[i], 1);
      ptx::mbar_init(&bars->in_empty[i], 1);
      ptx::mbar_init(&bars->acc2_full[i], 1);
      ptx::mbar_init(&bars->acc2_empty[i], 2 * kFusedEpiWarps);
    }
    ptx::mbar_init(&bars->acc1_full, 1);
    ptx::mbar_init(&bars->acc1_empty, 2 * kFusedEpiWarps);
    ptx::mbar_init(&bars->reg_full, 2 * kFusedEpiWarps);
    ptx::mbar_init(&bars->reg_empty, 1);
    ptx::fence_barrier_init();
  }
  if (warp == 2) {
    ptx::tmem_alloc2(&bars->tmem_base, 512);
    ptx::tmem_relinquish2();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::cluster_sync();
  ptx::tc_fence_after();
  const uint32_t tmem_base = bars->tmem_base;
  const long long npairs = gridDim.x >> 1, pair0 = blockIdx.x >> 1;
  const uint32_t slot_bytes = 2u * p1.slot_bytes;   // hi + lo box of one tile
  const int NPAD1 = p1.npad, NPAD2 = p2.npad;       // 128, 16
  // steps of this pair: patches pair0, pair0 + npairs, ... x tiles_pp tiles
  long long my_pairs = fp.pairs_total > pair0 ? (fp.pairs_total - pair0 + npairs - 1) / npairs : 0;
  const long long nsteps = my_pairs * fp.tiles_pp;

  if (warp == 0) {
    // ===== TMA producer (both CTAs): own weight halves, then the two input boxes of every tile =====
    if (ptx::elect_one()) {
      ptx::prefetch_tmap(&tm_hi);
      ptx::prefetch_tmap(&tm_lo);
      const uint32_t w1A = (p1.wA_bytes + 1023u) & ~1023u, w1B = (p1.wB_bytes + 1023u) & ~1023u;
      const uint32_t w2A = (p2.wA_bytes + 1023u) & ~1023u, w2B = (p2.wB_bytes + 1023u) & ~1023u;
      const uint8_t* src1 = p1.wimg + (size_t)rank * (w1A + w1B);
      const uint8_t* src2 = p2.wimg + (size_t)rank * (w2A + w2B);
      ptx::mbar_expect_tx(&bars->w_full, p1.wA_bytes + p1.wB_bytes + p2.wA_bytes + p2.wB_bytes);
      for (uint32_t off = 0; off < p1.wA_bytes; off += 16384u) ptx::bulk_load(s_w1A + off, src1 + off, min(16384u, p1.wA_bytes - off), &bars->w_full);
      for (uint32_t off = 0; off < p1.wB_bytes; off += 16384u) ptx::bulk_load(s_w1B + off, src1 + w1A + off, min(16384u, p1.wB_bytes - off), &bars->w_full);
      ptx::bulk_load(s_w2A, src2, p2.wA_bytes, &bars->w_full);
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
      const int n0 = (int)(2 * pp + rank);          // this CTA's patch (beyond n: TMA returns zeros, epilogue 2 stores nothing)
      for (int t = 0; t < fp.tiles_pp; ++t, ++step) {
        const int ty = t / fp.tiles_x, tx = t - ty * fp.tiles_x;
        const uint32_t s = (uint32_t)(step & 1);
        ptx::mbar_wait(&bars->in_empty[s], (uint32_t)((step >> 1) & 1) ^ 1u);
        if (ptx::elect_one()) {
          if (leader) ptx::mbar_expect_tx(&bars->in_full[s], 4u * p1.box_bytes);   // two boxes from each CTA
          uint8_t* dst = s_in + (size_t)s * slot_bytes;
          ptx::tma2_load_4d(dst, &tm_hi, &bars->in_full[s], 0, tx * 8 - 1, n0, ty * 16 - 1);
          ptx::tma2_load_4d(dst + p1.slot_bytes, &tm_lo, &bars->in_full[s], 0, tx * 8 - 1, n0, ty * 16 - 1);
        }
        __syncwarp();
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer (leader): MMA1 of tile i + 1 is issued before MMA2 of tile i =====
    if (leader && nsteps > 0) {
      const uint32_t idesc1_st = ptx::make_idesc_f16(256, 2 * NPAD1), idesc1_lo = ptx::make_idesc_f16(256, NPAD1);
      const uint32_t idesc2_st = ptx::make_idesc_f16(256, 2 * NPAD2), idesc2_lo = ptx::make_idesc_f16(256, NPAD2);
      const uint32_t a1_hi32 = (p1.sbo >> 4) | (1u << 14) | (p1.a_layout << 29);
      const uint32_t w1_hi32 = (p1.w_sbo >> 4) | (1u << 14) | (p1.w_layout << 29);
      const uint32_t a2_hi32 = (p2.sbo >> 4) | (1u << 14) | (p2.a_layout << 29);      // p2.sbo = region pitch (host)
      const uint32_t w2_hi32 = (p2.w_sbo >> 4) | (1u << 14) | (p2.w_layout << 29);
      const uint32_t tap1A = (uint32_t)NPAD1 * (uint32_t)p1.kc * 2u, tap1B = tap1A >> 1;
      const uint32_t tap2A = (uint32_t)NPAD2 * (uint32_t)p2.kc * 2u, tap2B = tap2A >> 1;
      const uint32_t w1A_d = (ptx::smem_u32(s_w1A) >> 4) | (1u << 16), w1B_d = (ptx::smem_u32(s_w1B) >> 4) | (1u << 16);
      const uint32_t w2A_d = (ptx::smem_u32(s_w2A) >> 4) | (1u << 16), w2B_d = (ptx::smem_u32(s_w2B) >> 4) | (1u << 16);
      const uint32_t reg_d = (ptx::smem_u32(s_region) >> 4) | (1u << 16);
      ptx::mbar_wait(&bars->w_full, 0);
      [[maybe_unused]] long long pw0 = 0, pw1 = 0, pw2 = 0, pw3 = 0;
      [[maybe_unused]] const long long pt0 = TIC_PROF_NOW();
      auto mma1 = [&](long long step) {
        const uint32_t s = (uint32_t)(step & 1);
        TIC_PROF_WAIT(pw0, ptx::mbar_wait(&bars->acc1_empty, (uint32_t)(step & 1) ^ 1u));
        TIC_PROF_WAIT(pw1, ptx::mbar_wait(&bars->in_full[s], (uint32_t)((step >> 1) & 1)));
        ptx::tc_fence_after();
        if (!(TIC_DBG_BITS(p1.dbg) & 16) && ptx::elect_one()) {
          const uint32_t ah = (ptx::smem_u32(s_in + (size_t)s * slot_bytes) >> 4) | (1u << 16);
          const uint32_t al = ah + (p1.slot_bytes >> 4);
          uint32_t sp = 0, fresh = 0;
          u16_issue_plane_t<U16_DECONV_PH, 2>(p1, ah, w1A_d, tmem_base, 2u * NPAD1, idesc1_st, a1_hi32, w1_hi32, tap1A >> 4, 0u, sp,
                                              fresh, true);
          u16_issue_plane_t<U16_DECONV_PH, 2>(p1, al, w1B_d, tmem_base + (uint32_t)NPAD1, 2u * NPAD1, idesc1_lo, a1_hi32, w1_hi32,
                                              tap1B >> 4, 0u, sp, fresh, false);
        }
        __syncwarp();
        if (ptx::elect_one()) {
          ptx::tc_commit2(&bars->in_empty[s]);
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
        if (!(TIC_DBG_BITS(p1.dbg) & 1) && ptx::elect_one()) {
          const uint32_t dbase = tmem_base + 256u + b * 128u;
#pragma unroll
          for (int sub = 0; sub < 4; ++sub) {
            const uint32_t aoff = (uint32_t)(((sub >> 1) * 16) * kFusedRegionCols + (sub & 1) * 8) * 64u;
            const uint32_t ah = reg_d + (aoff >> 4), al = ah + (kFusedRegionLoOff >> 4);
            const uint32_t d = dbase + (uint32_t)sub * 32u;
            uint32_t sp = 0, fresh = 0;
            u16_issue_plane_t<U16_DECONV_RGB, 2>(p2, ah, w2A_d, d, 2u * NPAD2, idesc2_st, a2_hi32, w2_hi32, tap2A >> 4, 0u, sp, fresh,
                                                 true);
            u16_issue_plane_t<U16_DECONV_RGB, 2>(p2, al, w2B_d, d + (uint32_t)NPAD2, 2u * NPAD2, idesc2_lo, a2_hi32, w2_hi32,
                                                 tap2B >> 4, 0u, sp, fresh, false);
          }
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
  } else if (warp >= 4) {
    // ===== epilogue warps.  Per tile, in this order:
    //   A  epilogue 1, first half (overlaps the previous tile's MMA2): decode_1's accumulators -> registers, bias, relu,
    //      fp16 split; the TMEM buffer goes straight back to the issuer
    //   B  epilogue 1, second half (the only work between two MMA2s): halo + region writes, then "region full"
    //   C  epilogue 2 of the PREVIOUS tile (overlaps MMA1 / MMA2 of the next ones; its accumulators are double-buffered):
    //      decode_0's accumulators -> bias, denormalise, clip, round -> the stitched image
    // Measured (tools/fused_ablate.py): epilogue 2 on four dedicated warps alone took 2.5 ms per 12 288 patches (~900 cycles
    // per 32-pixel call, latency-bound), so its 32 calls per tile are spread over all sixteen warps.
    // warp = (TMEM lane quadrant, output phase (py, px)): 32 input pixels x one phase x 32 channels = two 16-column units
    const int q4 = warp & 3, py = ((warp - 4) >> 2) & 1, px = (warp - 4) >> 3;
    const int e2_j = (warp - 4) >> 2;                   // epilogue 2: this warp takes sub-tile e2_j of its lane quadrant
    const int ph = py * 2 + px;
    const int m = q4 * 32 + lane, hh = m >> 3, xx = m & 7;
    const int e = tid - 128;                            // 0 .. 511 among the epilogue-1 threads
    const uint32_t reg_hi = ptx::smem_u32(s_region), reg_lo = reg_hi + kFusedRegionLoOff;
    const uint32_t rowc = ptx::smem_u32(s_rowc), colc = ptx::smem_u32(s_colc);
    const uint32_t rowc_par = (uint32_t)fp.tiles_x * 16u * 128u;   // bytes of one parity of the row cache
    const int rowc_px = fp.tiles_x * 16;                            // pixels of one cached row (chunk-major: [chunk 8][pixel][16 B])
    const uint32_t tbuf = tmem_base + ((uint32_t)(q4 * 32) << 16);
    const float floor_v = a1.act ? 0.0f : -INFINITY;
    const int R = 2 * hh + py, C = 2 * xx + px;         // region coordinates of this lane's output pixel
    const uint32_t pix = (uint32_t)((R + 1) * kFusedRegionCols + (C + 1)) * 64u;
    __half2 omax = __floats2half2_rn(0.f, 0.f);
    // epilogue 2 of tile `estep` (patch en, tile ety / etx): one of the four sub-tiles of this quadrant, both output rows
    [[maybe_unused]] long long pw0 = 0, pw1 = 0, pw2 = 0, pw3 = 0, pw4 = 0;
    [[maybe_unused]] const long long pt0 = TIC_PROF_NOW();
    auto epilogue2 = [&](long long estep, int en, int ety, int etx) {
      const uint32_t b = (uint32_t)(estep & 1);
      TIC_PROF_WAIT(pw2, ptx::mbar_wait(&bars->acc2_full[b], (uint32_t)((estep >> 1) & 1)));
      ptx::tc_fence_after();
      const uint32_t tb = tmem_base + ((uint32_t)(q4 * 32) << 16) + 256u + b * 128u;
      if (!(TIC_DBG_BITS(p1.dbg) & 2)) {
        const int sub = e2_j;   // this warp's sub-tile of the 32 x 16 region
        fused_rgb_epilogue(a2, tb + (uint32_t)sub * 32u, NPAD2, en, ety * 32 + (sub >> 1) * 16 + hh, etx * 16 + (sub & 1) * 8 + xx, en < fp.n,
                           fp.bias2);
      }
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive_leader(&bars->acc2_empty[b]);
    };
    long long step = 0;
    int pn = 0, pty = 0, ptx_ = 0;                      // the previous tile (epilogue 2 runs one tile behind)
    for (long long pp = pair0; pp < fp.pairs_total; pp += npairs) {
      for (int t = 0; t < fp.tiles_pp; ++t, ++step) {
        const int ty = t / fp.tiles_x, tx = t - ty * fp.tiles_x;
        // caches: this tile READS the row cache of parity (ty - 1) & 1 and the column cache of parity (tx - 1) & 1 and
        // WRITES parities ty & 1 / tx & 1: no hazard inside a step
        const uint32_t rowc_rd = rowc + (uint32_t)((ty + 1) & 1) * rowc_par, rowc_wr = rowc + (uint32_t)(ty & 1) * rowc_par;
        const uint32_t colc_rd = colc + (uint32_t)((tx + 1) & 1) * 4096u, colc_wr = colc + (uint32_t)(tx & 1) * 4096u;
        // ---- phase A (overlaps the previous tile's MMA2): accumulators -> registers, math, fp16 split; the TMEM buffer
        // goes back to the issuer at once, so MMA1 of the next tile queues behind the running MMA2 ----
        TIC_PROF_WAIT(pw0, ptx::mbar_wait(&bars->acc1_full, (uint32_t)(step & 1)));
        ptx::tc_fence_after();
        uint32_t hp[2][8], lp[2][8];
#pragma unroll
        for (int ci = 0; ci < 2; ++ci) {
          float v[16], u[16];
          ptx::tmem_ld16_nowait(tbuf + (uint32_t)(NPAD1 + ph * 32 + ci * 16), u);
          ptx::tmem_ld16_nowait(tbuf + (uint32_t)(ph * 32 + ci * 16), v);
          ptx::tmem_ld_wait();
          if (ci == 1) {   // last TMEM read of this tile
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive_leader(&bars->acc1_empty);
          }
#pragma unroll
          for (int i = 0; i < 16; ++i)
            v[i] = fmaxf(__fadd_rn(__fmaf_rn(u[i], 1.0f / 2048.0f, v[i]), fp.bias1[ci * 16 + i]), floor_v);
#pragma unroll
          for (int i = 0; i < 8; ++i) split16x2(v[2 * i], v[2 * i + 1], hp[ci][i], lp[ci][i], omax);
        }
        // ---- phase B (the only part between two MMA2s): the previous tile's MMA2 has finished reading the region ----
        TIC_PROF_WAIT(pw1, ptx::mbar_wait(&bars->reg_empty, (uint32_t)(step & 1) ^ 1u));
        TIC_PROF_WAIT(pw4, asm volatile("bar.sync 2, 512;" ::: "memory"));   // the previous tile's cache writes are visible to every epilogue-1 thread
        // halo: row -1 (17 pixels, corner first) and column -1 (32 pixels) of the region, 8 chunks of 16 B each
        if (e < 49 * 8 && !(TIC_DBG_BITS(p1.dbg) & 4)) {
          // consecutive lanes take consecutive halo pixels of one chunk: the caches are chunk-major ([chunk][pixel][16 B]),
          // so their reads here and the row-cache writes below touch consecutive 16-byte units (pixel-major, the eight
          // lanes that own a cached row wrote at a 128-byte stride: 8x the wavefronts)
          const int ch = e / 49, hp_ix = e - ch * 49;     // ch 0..3: hi plane, 4..7: lo' plane
          uint4 val = make_uint4(0u, 0u, 0u, 0u);
          uint32_t dst_pix;
          if (hp_ix < 17) {                               // region row -1, column hp_ix - 1 (corner: the tile above-left)
            if (ty > 0 && (hp_ix > 0 || tx > 0)) val = lds128(rowc_rd + (uint32_t)((ch * rowc_px + tx * 16 + hp_ix - 1) * 16));
            dst_pix = (uint32_t)hp_ix;
          } else {                                        // region column -1, row hp_ix - 17
            if (tx > 0) val = lds128(colc_rd + (uint32_t)((ch * 32 + hp_ix - 17) * 16));
            dst_pix = (uint32_t)((hp_ix - 17 + 1) * kFusedRegionCols);
          }
          const uint32_t addr = (ch < 4 ? reg_hi : reg_lo) + dst_pix * 64u + (uint32_t)(ch & 3) * 16u;
          sts128(fused_swz64(addr), val.x, val.y, val.z, val.w);
        }
#pragma unroll
        for (int ci = 0; ci < ((TIC_DBG_BITS(p1.dbg) & 4) ? 0 : 2); ++ci) {
          const uint32_t ah = reg_hi + pix + (uint32_t)ci * 32u, al = reg_lo + pix + (uint32_t)ci * 32u;
          {
            // lanes xx < 4 store hi then lo', lanes xx >= 4 lo' then hi (kFusedRegionLoOff): eight bank groups per quarter-warp
            const bool lo_first = (xx & 4) != 0;
            const uint32_t a0 = lo_first ? al : ah, a1 = lo_first ? ah : al;
            sts128(fused_swz64(a0), lo_first ? lp[ci][0] : hp[ci][0], lo_first ? lp[ci][1] : hp[ci][1], lo_first ? lp[ci][2] : hp[ci][2],
                   lo_first ? lp[ci][3] : hp[ci][3]);
            sts128(fused_swz64(a1), lo_first ? hp[ci][0] : lp[ci][0], lo_first ? hp[ci][1] : lp[ci][1], lo_first ? hp[ci][2] : lp[ci][2],
                   lo_first ? hp[ci][3] : lp[ci][3]);
            sts128(fused_swz64(a0 + 16u), lo_first ? lp[ci][4] : hp[ci][4], lo_first ? lp[ci][5] : hp[ci][5], lo_first ? lp[ci][6] : hp[ci][6],
                   lo_first ? lp[ci][7] : hp[ci][7]);
            sts128(fused_swz64(a1 + 16u), lo_first ? hp[ci][4] : lp[ci][4], lo_first ? hp[ci][5] : lp[ci][5], lo_first ? hp[ci][6] : lp[ci][6],
                   lo_first ? hp[ci][7] : lp[ci][7]);
          }
          if (R == 31) {   // last row of the region: halo row of the tile below (corner of the tile below-right)
            const uint32_t c0 = rowc_wr + (uint32_t)((2 * ci * rowc_px + tx * 16 + C) * 16), cs = (uint32_t)rowc_px * 16u;
            sts128(c0, hp[ci][0], hp[ci][1], hp[ci][2], hp[ci][3]);
            sts128(c0 + cs, hp[ci][4], hp[ci][5], hp[ci][6], hp[ci][7]);
            sts128(c0 + 4u * cs, lp[ci][0], lp[ci][1], lp[ci][2], lp[ci][3]);
            sts128(c0 + 5u * cs, lp[ci][4], lp[ci][5], lp[ci][6], lp[ci][7]);
          }
          if (C == 15) {   // last column: halo column of the tile to the right
            const uint32_t c0 = colc_wr + (uint32_t)((2 * ci * 32 + R) * 16);
            sts128(c0, hp[ci][0], hp[ci][1], hp[ci][2], hp[ci][3]);
            sts128(c0 + 512u, hp[ci][4], hp[ci][5], hp[ci][6], hp[ci][7]);
            sts128(c0 + 2048u, lp[ci][0], lp[ci][1], lp[ci][2], lp[ci][3]);
            sts128(c0 + 2560u, lp[ci][4], lp[ci][5], lp[ci][6], lp[ci][7]);
          }
        }
        ptx::fence_proxy_async_smem();   // generic-proxy region writes -> visible to the tensor core's operand reads
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive_leader(&bars->reg_full);
        // ---- phase C: epilogue 2 of the previous tile ----
        if (step > 0) TIC_PROF_WAIT(pw3, epilogue2(step - 1, pn, pty, ptx_));
        pn = (int)(2 * pp + rank);
        pty = ty;
        ptx_ = tx;
      }
    }
    if (step > 0) epilogue2(step - 1, pn, pty, ptx_);
    if (ovf_hit(omax)) ovf_raise(a1.oflow);
    if (warp == 4 || warp == 8) {
      [[maybe_unused]] const int base = warp == 4 ? 16 : 24;
      TIC_PROF_ADD(base + 0, pw0);
      TIC_PROF_ADD(base + 1, pw1);
      TIC_PROF_ADD(base + 2, pw2);
      TIC_PROF_ADD(base + 3, pw3);
      TIC_PROF_ADD(base + 4, pw4);
      TIC_PROF_ADD(base + 5, TIC_PROF_NOW() - pt0);
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

// Which layer pairs take the fused kernel: transposed conv 32 -> 32 (pair planes in) followed by transposed conv 32 -> 3
// into the denormalised image, on maps the 16 x 8 tiling covers.
inline bool fused_dec_supported(const LayerArgs& a1, int kind1, const LayerArgs& a2, int kind2) {
  if (kind1 != 1 || kind2 != 1) return false;
  if (a1.in_mode != IO_ACT16 || a1.cin != 32 || a1.cout != 32 || a2.cin != 32 || a2.cout != 3) return false;
  if (a1.res || a2.res) return false;
  if (a2.out_mode != IO_DENORM_U8 && a2.out_mode != IO_DENORM_F32) return false;
  if (a1.hin % 16 != 0 || a1.win % 8 != 0 || a1.win / 8 > kFusedMaxTilesX) return false;
  if (a2.hin != 2 * a1.hin || a2.win != 2 * a1.win) return false;
  return true;
}

// img[0], img[1]: the operand images of the two layers
inline tic_status launch_fused_dec(const LaunchCtx& c, const LayerArgs& a1, const LayerArgs& a2, const float* w1_dev, const float* w2_dev,
                                   const float* bias1_host, const float* bias2_host, OperandImage* img) {
  if (c.num_sms < 2) return c.fail("the fused decoder kernel needs CTA pairs", TIC_ERR_UNSUPPORTED);
  U16Plan pl1{}, pl2{};
  if (!u16_plan(a1, 1, 2, a1.cout, &pl1) || !u16_plan(a2, 1, 2, a2.cout, &pl2)) return c.fail("fused decoder plan failed", TIC_ERR_UNSUPPORTED);
  U16Params p1 = pl1.p, p2 = pl2.p;
  if (p1.mode != U16_DECONV_PH || p1.cpad != 32 || p2.mode != U16_DECONV_PH || p2.cpad != 4 || p1.ksteps != 2 || p2.ksteps != 2)
    return c.fail("fused decoder: unexpected layer plan", TIC_ERR_UNSUPPORTED);
  // layer 2 reads its operand from the region buffer: pitch 17 pixels, views (dy, dx) = rows / columns -1 + dy / dx
  for (int v = 0; v < 4; ++v) p2.a_off[v] = (uint32_t)(((v >> 1) * kFusedRegionCols + (v & 1)) * 64);
  p2.sbo = kFusedRegionPitch;
  tic_status s = u16_pair_image(c.stream, img[0], w1_dev, a1, p1, 0, a1.cout);
  if (s == TIC_OK) s = u16_pair_image(c.stream, img[1], w2_dev, a2, p2, 0, a2.cout);
  if (s != TIC_OK) return c.fail("fused decoder: weight images failed", s);
  p1.wimg = img[0].img();
  p2.wimg = img[1].img();
  p1.dbg = tic_env_int("TIC_DBG", 0);  // -DTIC_ABLATE builds only: 1 no MMA2, 16 no MMA1, 2 no epilogue 2, 4 no region writes

  FusedDecParams fp{};
  fp.n = a1.n;
  fp.tiles_x = a1.win / 8;
  fp.tiles_y = a1.hin / 16;
  fp.tiles_pp = fp.tiles_x * fp.tiles_y;
  fp.pairs_total = ((long long)a1.n + 1) / 2;
  for (int i = 0; i < 32; ++i) fp.bias1[i] = i < a1.cout ? bias1_host[i] : 0.f;
  for (int i = 0; i < 4; ++i) fp.bias2[i] = i < a2.cout ? bias2_host[i] : 0.f;
  auto up = [](uint32_t v) { return (v + 1023u) & ~1023u; };
  uint32_t off = 0;
  fp.w1_off = off;
  off += up(p1.wA_bytes);
  fp.w1B_off = off;
  off += up(p1.wB_bytes);
  fp.w2_off = off;
  off += up(p2.wA_bytes);
  fp.w2B_off = off;
  off += up(p2.wB_bytes);
  fp.in_off = off;
  off += 2u * 2u * p1.slot_bytes;
  fp.region_off = off;
  off += 2u * kFusedRegionPlane;
  fp.rowc_off = off;
  off += 2u * (uint32_t)fp.tiles_x * 16u * 128u;   // two parities
  fp.colc_off = off;
  off += 2u * 32u * 128u;
  fp.corner_off = off;                             // (unused: the corner is read from the row cache)
  off += 256u;
  fp.bars_off = off;
  off += (uint32_t)sizeof(FusedDecBars);
  fp.smem_bytes = off + 1024u;
  if (fp.smem_bytes > 227u * 1024u - 1024u) return c.fail("fused decoder: shared memory plan does not fit", TIC_ERR_UNSUPPORTED);

  CUtensorMap tm[2];
  for (int pl = 0; pl < 2; ++pl)
    if (tic_status st = tmap_act(&tm[pl], reinterpret_cast<const __half*>(a1.in) + (pl ? a1.in_lo_off : 0), true, a1, false,
                                 {(cuuint32_t)p1.kc, 9, 1, 17}, CU_TENSOR_MAP_SWIZZLE_64B, c.err))
      return st;
  const int grid = 2 * (int)std::min<long long>(fp.pairs_total, c.num_sms / 2);
  const cudaError_t e = launch_dyn(fused_dec_kernel, grid, kFusedThreads, fp.smem_bytes, c.stream, tm[0], tm[1], p1, a1, p2, a2, fp);
  if (e != cudaSuccess) return c.fail(std::string("fused decoder launch failed: ") + cudaGetErrorString(e), TIC_ERR_CUDA);
  ++*c.launches;
  return TIC_OK;
}

}  // namespace tic

// Shared device-side types for the codec kernels: fused-I/O geometry (crop / stitch by index
// arithmetic), per-layer launch arguments, first-layer prologue and last-layer epilogue helpers.
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>
#include "../../include/tic_math.h"

namespace tic {

// Measurement aids (the TIC_DBG stage switches and the fused kernels' wait counters) exist only in builds made with
// -DTIC_ABLATE (tools/build_ablate.sh).  The shipped library ignores every TIC_* environment variable: a stray variable
// must never change what a kernel computes.
#ifdef TIC_ABLATE
// wait-time accounting of the fused kernels' roles (cluster 0 only): cycles spent inside each barrier wait, summed over the
// kernel's steps, read back by tools/fused_waits.py through tic_debug_prof_read (not part of the shipped ABI)
__device__ unsigned long long g_tic_prof[64];
#define TIC_PROF_WAIT(acc, ...)            \
  do {                                     \
    const long long _t0 = clock64();       \
    __VA_ARGS__;                           \
    (acc) += clock64() - _t0;              \
  } while (0)
#define TIC_PROF_NOW() clock64()
#define TIC_PROF_ADD(slot, v)                                                                     \
  do {                                                                                            \
    if (blockIdx.x == 0 && (threadIdx.x & 31) == 0) atomicAdd(&g_tic_prof[slot], (unsigned long long)(v)); \
  } while (0)
inline int tic_env_int(const char* name, int dflt) {
  const char* e = getenv(name);
  return e ? atoi(e) : dflt;
}
#define TIC_DBG_BITS(x) (x)
#else
#define TIC_PROF_WAIT(acc, ...) \
  do {                          \
    __VA_ARGS__;                \
  } while (0)
#define TIC_PROF_NOW() 0LL
#define TIC_PROF_ADD(slot, v) \
  do {                        \
  } while (0)
inline int tic_env_int(const char*, int dflt) { return dflt; }
#define TIC_DBG_BITS(x) 0
#endif

// How the first layer reads its input / the last layer writes its output.
enum IoMode : int {
  IO_ACT = 0,          // f32 NHWC activation [n,h,w,c] (workspace)
  IO_U8_NORM = 1,      // in: u8 pixels through Geo, (x-mean)/std via 3x256 table         (model_0/model.py:44)
  IO_F32_NORM = 2,     // in: f32 pixels through Geo, (x-mean)/std computed                (model_0/model.py:44)
  IO_U8_SYMLUT = 3,    // in: u8 symbols [n,h,w,c] through the q-entry inverse-sigmoid LUT (model_0/model.py:153)
  IO_QUANT_U8 = 4,     // out: sigmoid*(q-1), round -> u8 symbols + histogram              (model_0/model.py:137-138)
  IO_QUANT_F32 = 5,    // out: same, stored as integer-valued f32 (what sess.run returns)
  IO_DENORM_F32 = 6,   // out: clip(y*std+mean,0,255) f32 through Geo                      (model_0/model.py:251,259)
  IO_DENORM_U8 = 7,    // out: same then np.around -> u8 through Geo                       (decode.py:249)
  IO_ACT16 = 8         // fp16 pair planes (hi, lo' = (x - hi) * 2048) of an NHWC activation (tic_umma16.cuh)
};

// Division by a launch constant.  A 32-bit `/` by a kernel parameter compiles to a ~20-instruction reciprocal
// routine (a 64-bit one to ~4x that); the tile -> (patch, row, column) -> image decode runs once per tile in every
// lane of the builder and epilogue warps, where it was a third of all issued instructions (profiles/r1e_*).
// Round-up multiplier method: exact for dividends below 2^31 (launchers check the tile / patch counts).
struct FastDiv {
  uint32_t d, mul, shr;
};
inline FastDiv make_fastdiv(uint32_t d) {
  FastDiv f{d, 0u, 0u};
  if (d > 1) {
    uint32_t lg = 0;
    while ((1ull << lg) < d) ++lg;
    const uint32_t p = 31 + lg;
    f.mul = (uint32_t)(((1ull << p) + d - 1) / d);
    f.shr = p - 32;
  }
  return f;
}
__host__ __device__ __forceinline__ uint32_t fast_div(uint32_t n, const FastDiv& f) {
#ifdef __CUDA_ARCH__
  return f.d == 1 ? n : __umulhi(n, f.mul) >> f.shr;
#else
  return f.d == 1 ? n : (uint32_t)(((uint64_t)n * f.mul) >> 32) >> f.shr;
#endif
}
__host__ __device__ __forceinline__ void fast_divmod(uint32_t n, const FastDiv& f, uint32_t& q, uint32_t& r) {
  q = fast_div(n, f);
  r = n - q * f.d;
}

// Patch <-> image geometry.  A "patch array" [n,P,P,3] is the degenerate case
// H = W = P, gh = gw = 1.  utils.crop_image_input_patches (utils/utils.py:96-133) pads
// bottom/right with np.pad(...,'reflect') and walks the patch grid row-major;
// utils.concat_patches (utils/utils.py:136-167) stitches row-major and crops to [H,W];
// rmbe tiles (submit/2/rmbe/rmbe.py:70-111) are the same grid shifted by (oy, ox).
struct Geo {
  int H, W;      // image height / width
  int gh, gw;    // patch grid per image
  int oy, ox;    // origin of the grid inside the image
  int P;         // patch edge
  long long n0;  // global index of the chunk's first patch
  FastDiv per_img_d, gw_d;  // / (gh * gw), / gw  (geo_finish)
};
inline void geo_finish(Geo& g) {
  g.per_img_d = make_fastdiv((uint32_t)(g.gh * g.gw > 0 ? g.gh * g.gw : 1));
  g.gw_d = make_fastdiv((uint32_t)(g.gw > 0 ? g.gw : 1));
}
// global patch -> (image, grid row, grid column)
__device__ __forceinline__ void geo_decode(const Geo& g, unsigned patch, unsigned& img, unsigned& gy, unsigned& gx) {
  unsigned r;
  fast_divmod(patch, g.per_img_d, img, r);
  fast_divmod(r, g.gw_d, gy, gx);
}

__device__ __forceinline__ int reflect_index(int i, int n) {
  // numpy 'reflect' (no edge repeat): period 2(n-1)
  if (i < n) return i;
  int period = 2 * (n - 1);
  if (period <= 0) return 0;
  int m = i % period;
  return m < n ? m : period - m;
}

// pixel (y,x) of global patch g -> element offset (in pixels) inside the image batch, or -1
// when outside the image and reflect == false.
__device__ __forceinline__ long long geo_pixel(const Geo& g, long long patch, int y, int x, bool reflect) {
  // 32-bit index arithmetic (host guarantees patch < 2^31); only the final offset is 64-bit
  unsigned img, gy, gx;
  geo_decode(g, (unsigned)patch, img, gy, gx);
  int Y = g.oy + (int)gy * g.P + y;
  int X = g.ox + (int)gx * g.P + x;
  if (reflect) {
    Y = reflect_index(Y, g.H);
    X = reflect_index(X, g.W);
  } else if (Y >= g.H || X >= g.W) {
    return -1;
  }
  return ((long long)img * g.H + Y) * (long long)g.W + X;
}

struct LayerArgs {
  const void* in;        // first layer: caller input (u8 / f32); else f32 activation
  void* out;             // last layer: caller output; else f32 activation
  const float* wgt;      // [9][cin][cout] fp32 (tap-major, cout contiguous)
  const float* bias;     // [cout]
  const float* res;      // residual source [n,hout,wout,cout] or nullptr
  int n;                 // patches in this chunk
  int hin, win, cin;
  int hout, wout, cout;
  int pad_t, pad_l;      // TF SAME padding before (conv)
  int TW, TH, TP;        // CTA tile: columns, rows, patches (conv: output px; deconv: input px)
  int tiles_x, tiles_y;
  int act;
  int in_mode, out_mode;
  Geo geo;               // used by the *_NORM / DENORM_* modes
  const float* lut;      // IO_U8_NORM: [3][256]; IO_U8_SYMLUT: [q]
  float mean[3], stdv[3];
  int q;
  unsigned long long* hist;  // [256] symbol counts (IO_QUANT_*)
  // IO_ACT16 tensors: `in` / `out` / `res` point at the hi plane, the lo' plane starts *_lo_off halves later
  long long in_lo_off, out_lo_off, res_lo_off;
  int res16;             // residual source is a pair-plane tensor
  unsigned int* oflow;   // sticky fp16-range flag (host-mapped): set to 1 when a pair-plane split sees |x| >= 65504
  int dbg;               // -DTIC_ABLATE builds only (env TIC_DBG bit 8: the staged epilogue skips its global stores)
};

__device__ __forceinline__ float apply_act(float v, int act) { return act ? fmaxf(v, 0.0f) : v; }

// fp16 pair representation of an fp32 value: x ~= hi + lo' / 2048 (22 significant bits; the parts do not
// overlap, so the re-join is exact in fp32).  |x| must stay below 65504 (fp16 range).
__device__ __forceinline__ void split16(float v, __half& hi, __half& lo) {
  hi = __float2half_rn(v);
  lo = __float2half_rn(__fmul_rn(__fsub_rn(v, __half2float(hi)), 2048.0f));
}
__device__ __forceinline__ float join16(__half hi, __half lo) {
  return __fmaf_rn(__half2float(lo), 1.0f / 2048.0f, __half2float(hi));
}

// fp16-range guard of the pair-plane format (include/tic.h: TIC_COMPUTE_TENSOR_F16X3 needs |activation| < 65504).
// A split of a larger value gives hi = inf; every epilogue keeps a running max of |hi| (one HMNMX2 per two
// elements) and raises the handle's sticky flag once per warp at the end of its tile loop.
__device__ __forceinline__ void ovf_track(__half2& m, const __half2 h) { m = __hmax2(m, __habs2(h)); }
__device__ __forceinline__ bool ovf_hit(const __half2 m) {
  const uint32_t w = *reinterpret_cast<const uint32_t*>(&m);
  return (w & 0x7fffu) >= 0x7c00u || ((w >> 16) & 0x7fffu) >= 0x7c00u;
}
__device__ __forceinline__ bool ovf_hit1(const __half h) { return (__half_as_ushort(h) & 0x7fffu) >= 0x7c00u; }
__device__ __forceinline__ void ovf_raise(unsigned int* flag) {
  if (flag) *reinterpret_cast<volatile unsigned int*>(flag) = 1u;
}

}  // namespace tic

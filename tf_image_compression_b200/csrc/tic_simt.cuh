// fp32 CUDA-core kernels for the 3x3 conv / stride-2 transposed conv layers of the codec
// (basic_block/basic_block.py:27-71).  This is the exact-fp32 compute mode (TIC_COMPUTE_FP32):
// fp32 FMA accumulation, register-tiled, shared-memory staged.  It is the numerical anchor
// for the tcgen05 path and serves every layer shape (Cin = 3 … 128, Cout = 3 … 128).
//
// Layouts: activations NHWC fp32; weights [tap = kh*3+kw][cin][cout] fp32 (converted once
// from the TF variable layout at tic_load_weights).
//
// Thread tile (conv): 4 output rows x 1 column x 8 output channels (32 accumulators).  A warp
// shares one 8-channel group (weight reads are shared-memory broadcasts) and spans 32
// adjacent pixels (input reads are conflict-free for stride 1).  Per input channel a thread
// issues 18-27 scalar LDS + 18 LDS.128 for 288 FFMA.
// Thread tile (deconv): 4 input rows x 1 column -> 8x2 output pixels x 4 output channels
// (64 accumulators); all nine taps of an input pixel are used exactly once (no zero-insertion):
//   out[2i+kh, 2j+kw, oc] += x[i, j, ic] * W[kh, kw, oc, ic]      (gradient of the stride-2 SAME conv)
#pragma once
#include "tic_common.cuh"

namespace tic {

constexpr int kIcc = 8;         // input channels staged per shared-memory pass
constexpr int kThreads = 256;

struct SmemPlan {
  int ih, iw, iwp;   // staged input tile rows / cols / padded row pitch (floats)
  int cstr;          // channel stride (floats)
  int pstr;          // patch stride (floats)
};

// ---- first-layer input fetch (prologue fusion) ---------------------------------------------
__device__ __forceinline__ float fetch_input(const LayerArgs& a, int n, int Y, int X, int c) {
  switch (a.in_mode) {
    case IO_ACT:
      return reinterpret_cast<const float*>(a.in)[(((long long)n * a.hin + Y) * a.win + X) * a.cin + c];
    case IO_U8_NORM: {
      long long off = geo_pixel(a.geo, a.geo.n0 + n, Y, X, true);
      unsigned v = reinterpret_cast<const uint8_t*>(a.in)[off * 3 + c];
      return __ldg(a.lut + c * 256 + v);
    }
    case IO_F32_NORM: {
      long long off = geo_pixel(a.geo, a.geo.n0 + n, Y, X, true);
      float v = reinterpret_cast<const float*>(a.in)[off * 3 + c];
      return tic_normalize(v, a.mean[c], a.stdv[c]);
    }
    case IO_ACT16: {
      const long long off = (((long long)n * a.hin + Y) * a.win + X) * a.cin + c;
      const __half* hp = reinterpret_cast<const __half*>(a.in);
      return join16(hp[off], hp[off + a.in_lo_off]);
    }
    case IO_U8_SYMLUT: {
      unsigned v = reinterpret_cast<const uint8_t*>(
          a.in)[((((long long)a.geo.n0 + n) * a.hin + Y) * a.win + X) * a.cin + c];
      return __ldg(a.lut + v);
    }
    default:
      return 0.0f;
  }
}

// Stage [TP][kIcc][ih][iw] input values (zero outside the map: TF SAME padding pads the
// *normalised* tensor with zeros) and [9][kIcc][OCB] weights.
template <int OCB>
__device__ __forceinline__ void stage_tiles(const LayerArgs& a, const SmemPlan& sp, float* s_in, float* s_w,
                                            int pg, int y_in0, int x_in0, int ic0, int oc0) {
  const int tid = threadIdx.x;
  const int npix = a.TP * sp.ih * sp.iw;
  if ((a.in_mode == IO_U8_NORM || a.in_mode == IO_F32_NORM) && a.cin == 3) {
    // first layer: one thread per staged pixel — patch/image geometry, reflect indices and the three
    // channel fetches are done once per pixel (the compute loop only reads the cin = 3 planes)
    if (ic0 == 0) {
      for (int u = tid; u < npix; u += kThreads) {
        const int ix = u % sp.iw;
        const int r = u / sp.iw;
        const int iy = r % sp.ih;
        const int pp = r / sp.ih;
        const int n = pg * a.TP + pp, Y = y_in0 + iy, X = x_in0 + ix;
        float v0 = 0.f, v1 = 0.f, v2 = 0.f;
        if (n < a.n && Y >= 0 && Y < a.hin && X >= 0 && X < a.win) {
          const long long off = geo_pixel(a.geo, a.geo.n0 + n, Y, X, true) * 3;
          if (a.in_mode == IO_U8_NORM) {
            const uint8_t* q = reinterpret_cast<const uint8_t*>(a.in) + off;
            v0 = __ldg(a.lut + q[0]);
            v1 = __ldg(a.lut + 256 + q[1]);
            v2 = __ldg(a.lut + 512 + q[2]);
          } else {
            const float* q = reinterpret_cast<const float*>(a.in) + off;
            v0 = tic_normalize(q[0], a.mean[0], a.stdv[0]);
            v1 = tic_normalize(q[1], a.mean[1], a.stdv[1]);
            v2 = tic_normalize(q[2], a.mean[2], a.stdv[2]);
          }
        }
        float* d = s_in + pp * sp.pstr + iy * sp.iwp + ix;
        d[0] = v0;
        d[sp.cstr] = v1;
        d[2 * sp.cstr] = v2;
      }
    }
  } else if (a.in_mode == IO_ACT && (a.cin & 3) == 0) {
    const float* in = reinterpret_cast<const float*>(a.in);
    for (int u = tid; u < npix * (kIcc / 4); u += kThreads) {
      int c4 = u % (kIcc / 4);
      int pix = u / (kIcc / 4);
      int ix = pix % sp.iw;
      int r = pix / sp.iw;
      int iy = r % sp.ih;
      int pp = r / sp.ih;
      int n = pg * a.TP + pp, Y = y_in0 + iy, X = x_in0 + ix, c = ic0 + c4 * 4;
      float4 val = make_float4(0.f, 0.f, 0.f, 0.f);
      if (n < a.n && Y >= 0 && Y < a.hin && X >= 0 && X < a.win && c < a.cin)
        val = __ldg(reinterpret_cast<const float4*>(in + (((long long)n * a.hin + Y) * a.win + X) * a.cin + c));
      float* d = s_in + pp * sp.pstr + (c4 * 4) * sp.cstr + iy * sp.iwp + ix;
      d[0] = val.x;
      d[sp.cstr] = val.y;
      d[2 * sp.cstr] = val.z;
      d[3 * sp.cstr] = val.w;
    }
  } else if (a.in_mode == IO_ACT16 && (a.cin & 3) == 0) {
    const __half* in = reinterpret_cast<const __half*>(a.in);
    for (int u = tid; u < npix * (kIcc / 4); u += kThreads) {
      int c4 = u % (kIcc / 4);
      int pix = u / (kIcc / 4);
      int ix = pix % sp.iw;
      int r = pix / sp.iw;
      int iy = r % sp.ih;
      int pp = r / sp.ih;
      int n = pg * a.TP + pp, Y = y_in0 + iy, X = x_in0 + ix, c = ic0 + c4 * 4;
      float4 val = make_float4(0.f, 0.f, 0.f, 0.f);
      if (n < a.n && Y >= 0 && Y < a.hin && X >= 0 && X < a.win && c < a.cin) {
        const __half* q = in + (((long long)n * a.hin + Y) * a.win + X) * a.cin + c;
        const uint2 qh = __ldg(reinterpret_cast<const uint2*>(q));
        const uint2 ql = __ldg(reinterpret_cast<const uint2*>(q + a.in_lo_off));
        const __half* h4 = reinterpret_cast<const __half*>(&qh);
        const __half* l4 = reinterpret_cast<const __half*>(&ql);
        val = make_float4(join16(h4[0], l4[0]), join16(h4[1], l4[1]), join16(h4[2], l4[2]), join16(h4[3], l4[3]));
      }
      float* d = s_in + pp * sp.pstr + (c4 * 4) * sp.cstr + iy * sp.iwp + ix;
      d[0] = val.x;
      d[sp.cstr] = val.y;
      d[2 * sp.cstr] = val.z;
      d[3 * sp.cstr] = val.w;
    }
  } else {
    for (int u = tid; u < npix * kIcc; u += kThreads) {
      int c = u % kIcc;
      int pix = u / kIcc;
      int ix = pix % sp.iw;
      int r = pix / sp.iw;
      int iy = r % sp.ih;
      int pp = r / sp.ih;
      int n = pg * a.TP + pp, Y = y_in0 + iy, X = x_in0 + ix;
      float val = 0.f;
      if (n < a.n && Y >= 0 && Y < a.hin && X >= 0 && X < a.win && ic0 + c < a.cin)
        val = fetch_input(a, n, Y, X, ic0 + c);
      s_in[pp * sp.pstr + c * sp.cstr + iy * sp.iwp + ix] = val;
    }
  }
  // weights: global [9][cin][cout] -> shared [9][kIcc][OCB]
  if ((a.cout & 3) == 0) {
    for (int u = tid; u < 9 * kIcc * (OCB / 4); u += kThreads) {
      int o4 = u % (OCB / 4);
      int r = u / (OCB / 4);
      int ic = r % kIcc;
      int tap = r / kIcc;
      float4 w = make_float4(0.f, 0.f, 0.f, 0.f);
      int oc = oc0 + o4 * 4;
      if (ic0 + ic < a.cin && oc < a.cout)
        w = __ldg(reinterpret_cast<const float4*>(a.wgt + ((long long)tap * a.cin + ic0 + ic) * a.cout + oc));
      *reinterpret_cast<float4*>(s_w + (tap * kIcc + ic) * OCB + o4 * 4) = w;
    }
  } else {
    for (int u = tid; u < 9 * kIcc * OCB; u += kThreads) {
      int o = u % OCB;
      int r = u / OCB;
      int ic = r % kIcc;
      int tap = r / kIcc;
      float w = 0.f;
      if (ic0 + ic < a.cin && oc0 + o < a.cout)
        w = __ldg(a.wgt + ((long long)tap * a.cin + ic0 + ic) * a.cout + oc0 + o);
      s_w[(tap * kIcc + ic) * OCB + o] = w;
    }
  }
}

// ---- last-layer / activation stores (epilogue fusion) --------------------------------------
// v[NV] = accumulator + bias already activated (+ residual) for channels oc .. oc+NV-1 of
// output pixel (n, y, x).  s_hist: CTA-private symbol histogram.
template <int NV>
__device__ __forceinline__ void store_pixel(const LayerArgs& a, int n, int y, int x, int oc, const float* v,
                                            unsigned* s_hist, int& ones, int& valid) {
  const long long pix = ((long long)n * a.hout + y) * a.wout + x;
  switch (a.out_mode) {
    case IO_ACT: {
      float* o = reinterpret_cast<float*>(a.out) + pix * a.cout + oc;
      if ((a.cout & 3) == 0) {
#pragma unroll
        for (int i = 0; i < NV; i += 4)
          if (oc + i < a.cout) *reinterpret_cast<float4*>(o + i) = make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]);
      } else {
#pragma unroll
        for (int i = 0; i < NV; ++i)
          if (oc + i < a.cout) o[i] = v[i];
      }
      break;
    }
    case IO_ACT16: {
      __half* oh = reinterpret_cast<__half*>(a.out) + pix * a.cout + oc;
      __half* ol = oh + a.out_lo_off;
      if ((a.cout & 3) == 0) {
#pragma unroll
        for (int i = 0; i < NV; i += 4) {
          if (oc + i < a.cout) {
            uint2 qh, ql;
            __half* h4 = reinterpret_cast<__half*>(&qh);
            __half* l4 = reinterpret_cast<__half*>(&ql);
#pragma unroll
            for (int e = 0; e < 4; ++e) split16(v[i + e], h4[e], l4[e]);
            if (ovf_hit1(h4[0]) | ovf_hit1(h4[1]) | ovf_hit1(h4[2]) | ovf_hit1(h4[3])) ovf_raise(a.oflow);
            *reinterpret_cast<uint2*>(oh + i) = qh;
            *reinterpret_cast<uint2*>(ol + i) = ql;
          }
        }
      } else {
#pragma unroll
        for (int i = 0; i < NV; ++i)
          if (oc + i < a.cout) {
            split16(v[i], oh[i], ol[i]);
            if (ovf_hit1(oh[i])) ovf_raise(a.oflow);
          }
      }
      break;
    }
    case IO_QUANT_U8:
    case IO_QUANT_F32: {
      const long long gp = (((long long)a.geo.n0 + n) * a.hout + y) * a.wout + x;
      if (a.out_mode == IO_QUANT_U8 && NV == 16 && oc + NV <= a.cout && (a.cout & 15) == 0 &&
          (reinterpret_cast<uintptr_t>(a.out) & 15) == 0) {
        // 16 symbols of one pixel are 16 consecutive bytes of a 16-byte aligned symbol tensor: one 16-byte store
        uint32_t w[4] = {0u, 0u, 0u, 0u};
#pragma unroll
        for (int i = 0; i < NV; ++i) {
          const int s = tic_quantize_symbol(v[i], a.q);
          w[i >> 2] |= (uint32_t)s << (8 * (i & 3));
          if (a.q == 2) {
            ones += s;
            ++valid;
          } else {
            atomicAdd(&s_hist[s], 1u);
          }
        }
        *reinterpret_cast<uint4*>(reinterpret_cast<uint8_t*>(a.out) + gp * a.cout + oc) = make_uint4(w[0], w[1], w[2], w[3]);
        break;
      }
#pragma unroll
      for (int i = 0; i < NV; ++i) {
        if (oc + i < a.cout) {
          int s = tic_quantize_symbol(v[i], a.q);
          if (a.out_mode == IO_QUANT_U8)
            reinterpret_cast<uint8_t*>(a.out)[gp * a.cout + oc + i] = (uint8_t)s;
          else
            reinterpret_cast<float*>(a.out)[gp * a.cout + oc + i] = (float)s;
          if (a.q == 2) {
            ones += s;
            ++valid;
          } else {
            atomicAdd(&s_hist[s], 1u);
          }
        }
      }
      break;
    }
    case IO_DENORM_F32:
    case IO_DENORM_U8: {
      long long off = geo_pixel(a.geo, a.geo.n0 + n, y, x, false);
      if (off < 0) break;
#pragma unroll
      for (int i = 0; i < NV; ++i) {
        int c = oc + i;
        if (c < a.cout && c < 3) {
          float r = tic_denorm_clip(v[i], a.mean[c], a.stdv[c]);
          if (a.out_mode == IO_DENORM_F32)
            reinterpret_cast<float*>(a.out)[off * 3 + c] = r;
          else
            reinterpret_cast<uint8_t*>(a.out)[off * 3 + c] = (uint8_t)(int)rintf(r);
        }
      }
      break;
    }
    default:
      break;
  }
}

__device__ __forceinline__ void hist_begin(unsigned* s_hist) {
  for (int i = threadIdx.x; i < 256; i += kThreads) s_hist[i] = 0;
}
// q == 2 (every shipped config): symbols were counted in registers (ones / valid); reduce over
// the warp and issue one shared atomic pair per warp.  q > 2: per-symbol shared atomics above.
__device__ __forceinline__ void hist_flush(const LayerArgs& a, unsigned* s_hist, int ones, int valid) {
  if (a.out_mode != IO_QUANT_U8 && a.out_mode != IO_QUANT_F32) return;
  if (a.q == 2) {
    ones = __reduce_add_sync(0xffffffffu, ones);
    valid = __reduce_add_sync(0xffffffffu, valid);
    if ((threadIdx.x & 31) == 0) {
      if (ones) atomicAdd(&s_hist[1], (unsigned)ones);
      if (valid - ones) atomicAdd(&s_hist[0], (unsigned)(valid - ones));
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < a.q; i += kThreads)
    if (s_hist[i]) atomicAdd(&a.hist[i], (unsigned long long)s_hist[i]);
}

// ---- 3x3 conv, stride S, TF SAME ------------------------------------------------------------
template <int OCB, int S>
__global__ void __launch_bounds__(kThreads) conv3x3_simt_kernel(const LayerArgs a, const SmemPlan sp) {
  extern __shared__ __align__(16) float smem[];
  __shared__ unsigned s_hist[256];
  constexpr int OCG = OCB / 8;
  constexpr int PG = kThreads / OCG;
  constexpr int NR = 3 * S + 3;
  float* s_w = smem;                    // [9][kIcc][OCB], 16-byte aligned
  float* s_in = smem + 9 * kIcc * OCB;  // [TP] x pstr

  const int tid = threadIdx.x;
  const int ocg = tid / PG, g = tid % PG;
  const int x = g % a.TW;
  const int t = g / a.TW;
  const int thq = a.TH >> 2;
  const int yq = t % thq, p = t / thq;
  int tile = blockIdx.x;
  const int tx = tile % a.tiles_x;
  tile /= a.tiles_x;
  const int ty = tile % a.tiles_y;
  const int pg = tile / a.tiles_y;
  const int oc0 = blockIdx.y * OCB;
  const int y_in0 = ty * a.TH * S - a.pad_t;
  const int x_in0 = tx * a.TW * S - a.pad_l;

  hist_begin(s_hist);

  float acc[4][8];
#pragma unroll
  for (int j = 0; j < 4; ++j)
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[j][i] = 0.f;

  const float* spx = s_in + p * sp.pstr + (yq * 4 * S) * sp.iwp + x * S;
  for (int ic0 = 0; ic0 < a.cin; ic0 += kIcc) {
    __syncthreads();
    stage_tiles<OCB>(a, sp, s_in, s_w, pg, y_in0, x_in0, ic0, oc0);
    __syncthreads();
    const int icn = min(kIcc, a.cin - ic0);
    for (int ic = 0; ic < icn; ++ic) {
      float v[NR][3];
      const float* q = spx + ic * sp.cstr;
#pragma unroll
      for (int r = 0; r < NR; ++r)
#pragma unroll
        for (int k = 0; k < 3; ++k) v[r][k] = q[r * sp.iwp + k];
#pragma unroll
      for (int kh = 0; kh < 3; ++kh)
#pragma unroll
        for (int kw = 0; kw < 3; ++kw) {
          const float4* wp = reinterpret_cast<const float4*>(s_w + ((kh * 3 + kw) * kIcc + ic) * OCB + ocg * 8);
          const float4 w0 = wp[0], w1 = wp[1];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float xv = v[j * S + kh][kw];
            acc[j][0] = fmaf(xv, w0.x, acc[j][0]);
            acc[j][1] = fmaf(xv, w0.y, acc[j][1]);
            acc[j][2] = fmaf(xv, w0.z, acc[j][2]);
            acc[j][3] = fmaf(xv, w0.w, acc[j][3]);
            acc[j][4] = fmaf(xv, w1.x, acc[j][4]);
            acc[j][5] = fmaf(xv, w1.y, acc[j][5]);
            acc[j][6] = fmaf(xv, w1.z, acc[j][6]);
            acc[j][7] = fmaf(xv, w1.w, acc[j][7]);
          }
        }
    }
  }

  // epilogue: + bias -> activation -> (+ residual) -> store / quantise / denormalise
  const int n = pg * a.TP + p;
  const int xo = tx * a.TW + x;
  const int oc = oc0 + ocg * 8;
  int h_ones = 0, h_valid = 0;
  float b[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) b[i] = (oc + i < a.cout) ? __ldg(a.bias + oc + i) : 0.f;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int y = ty * a.TH + yq * 4 + j;
    if (n < a.n && y < a.hout && xo < a.wout && oc < a.cout) {
      float o[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) o[i] = apply_act(__fadd_rn(acc[j][i], b[i]), a.act);
      if (a.res) {
        const long long ro = (((long long)n * a.hout + y) * a.wout + xo) * a.cout + oc;
        if (a.res16) {
          const __half* rh = reinterpret_cast<const __half*>(a.res) + ro;
#pragma unroll
          for (int i = 0; i < 8; ++i)
            if (oc + i < a.cout) o[i] = __fadd_rn(join16(rh[i], rh[i + a.res_lo_off]), o[i]);
        } else {
          const float* rp = a.res + ro;
#pragma unroll
          for (int i = 0; i < 8; ++i)
            if (oc + i < a.cout) o[i] = __fadd_rn(__ldg(rp + i), o[i]);
        }
      }
      store_pixel<8>(a, n, y, xo, oc, o, s_hist, h_ones, h_valid);
    }
  }
  hist_flush(a, s_hist, h_ones, h_valid);
}

// ---- 3x3 transposed conv, stride 2, TF SAME, output = 2x input ------------------------------
template <int OCB>
__global__ void __launch_bounds__(kThreads) deconv3x3_simt_kernel(const LayerArgs a, const SmemPlan sp) {
  extern __shared__ __align__(16) float smem[];
  __shared__ unsigned s_hist[256];
  constexpr int OCG = OCB / 4;
  constexpr int PG = kThreads / OCG;
  float* s_w = smem;                    // [9][kIcc][OCB], 16-byte aligned
  float* s_in = smem + 9 * kIcc * OCB;  // [TP] x pstr

  const int tid = threadIdx.x;
  const int ocg = tid / PG, g = tid % PG;
  const int bx = g % a.TW;
  const int t = g / a.TW;
  const int thq = a.TH >> 2;
  const int aq = t % thq, p = t / thq;
  int tile = blockIdx.x;
  const int tx = tile % a.tiles_x;
  tile /= a.tiles_x;
  const int ty = tile % a.tiles_y;
  const int pg = tile / a.tiles_y;
  const int oc0 = blockIdx.y * OCB;
  const int y_in0 = ty * a.TH - 1;  // one halo row above / column left of the tile
  const int x_in0 = tx * a.TW - 1;

  hist_begin(s_hist);

  float acc[4][4][4];  // [input row j][output position dy*2+dx][oc]
#pragma unroll
  for (int j = 0; j < 4; ++j)
#pragma unroll
    for (int q = 0; q < 4; ++q)
#pragma unroll
      for (int i = 0; i < 4; ++i) acc[j][q][i] = 0.f;

  const float* spx = s_in + p * sp.pstr + (aq * 4) * sp.iwp + bx;
  for (int ic0 = 0; ic0 < a.cin; ic0 += kIcc) {
    __syncthreads();
    stage_tiles<OCB>(a, sp, s_in, s_w, pg, y_in0, x_in0, ic0, oc0);
    __syncthreads();
    const int icn = min(kIcc, a.cin - ic0);
    for (int ic = 0; ic < icn; ++ic) {
      float v[5][2];  // rows a-1 .. a+3, cols b-1, b
      const float* q = spx + ic * sp.cstr;
#pragma unroll
      for (int r = 0; r < 5; ++r) {
        v[r][0] = q[r * sp.iwp];
        v[r][1] = q[r * sp.iwp + 1];
      }
      float4 w[9];
#pragma unroll
      for (int tp = 0; tp < 9; ++tp)
        w[tp] = *reinterpret_cast<const float4*>(s_w + (tp * kIcc + ic) * OCB + ocg * 4);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float x00 = v[j + 1][1], xm0 = v[j][1], x0m = v[j + 1][0], xmm = v[j][0];
#define TIC_FMA4(A, X, W)               \
  A[0] = fmaf(X, W.x, A[0]);            \
  A[1] = fmaf(X, W.y, A[1]);            \
  A[2] = fmaf(X, W.z, A[2]);            \
  A[3] = fmaf(X, W.w, A[3]);
        // (2a, 2b): taps (kh,kw) in {0,2}x{0,2}
        TIC_FMA4(acc[j][0], x00, w[0]) TIC_FMA4(acc[j][0], x0m, w[2]) TIC_FMA4(acc[j][0], xm0, w[6])
            TIC_FMA4(acc[j][0], xmm, w[8])
        // (2a, 2b+1): kw = 1, kh in {0,2}
        TIC_FMA4(acc[j][1], x00, w[1]) TIC_FMA4(acc[j][1], xm0, w[7])
        // (2a+1, 2b): kh = 1, kw in {0,2}
        TIC_FMA4(acc[j][2], x00, w[3]) TIC_FMA4(acc[j][2], x0m, w[5])
        // (2a+1, 2b+1): centre tap
        TIC_FMA4(acc[j][3], x00, w[4])
#undef TIC_FMA4
      }
    }
  }

  const int n = pg * a.TP + p;
  const int xi = tx * a.TW + bx;
  const int oc = oc0 + ocg * 4;
  int h_ones = 0, h_valid = 0;
  float b[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) b[i] = (oc + i < a.cout) ? __ldg(a.bias + oc + i) : 0.f;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int yi = ty * a.TH + aq * 4 + j;
    if (n < a.n && yi < a.hin && xi < a.win && oc < a.cout) {
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        float o[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) o[i] = apply_act(__fadd_rn(acc[j][q][i], b[i]), a.act);
        store_pixel<4>(a, n, 2 * yi + (q >> 1), 2 * xi + (q & 1), oc, o, s_hist, h_ones, h_valid);
      }
    }
  }
  hist_flush(a, s_hist, h_ones, h_valid);
}

// ---- small elementwise kernels --------------------------------------------------------------
// np.around -> uint8 (decode.py:249)
__global__ void round_u8_kernel(const float* __restrict__ src, uint8_t* __restrict__ dst, long long count) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (; i < count; i += stride) {
    float v = src[i];
    v = v < 0.f ? 0.f : (v > 255.f ? 255.f : v);
    dst[i] = (uint8_t)(int)rintf(v);
  }
}

// per-position symbol sums over patches (cal_encoded_distribution.py:111-128); one thread owns
// one bottleneck position, patches are walked with coalesced reads; no atomics, deterministic.
__global__ void position_sums_kernel(const uint8_t* __restrict__ sym, long long n, long long npos,
                                     unsigned long long* __restrict__ sums) {
  long long pos = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (pos >= npos) return;
  unsigned long long s = 0;
  for (long long i = 0; i < n; ++i) s += sym[i * npos + pos];
  sums[pos] += s;
}

// the same per batch of `batch` patches: sums[b][pos] = sum over the patches of batch b (the reference folds one
// sess.run batch of 64 at a time into its running mean, cal_encoded_distribution.py:111-128); grid.y = batches
__global__ void position_sums_batched_kernel(const uint8_t* __restrict__ sym, long long n, long long npos, long long batch,
                                             unsigned long long* __restrict__ sums) {
  const long long pos = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (pos >= npos) return;
  const long long b = blockIdx.y, i0 = b * batch, i1 = min(n, i0 + batch);
  unsigned long long s = 0;
  for (long long i = i0; i < i1; ++i) s += sym[i * npos + pos];
  sums[b * npos + pos] = s;
}

}  // namespace tic

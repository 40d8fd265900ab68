// C-ABI implementation (include/tic.h): handle, graph executor, chunked H2D -> compute -> D2H
// pipeline, and kernel dispatch.  No torch types, no exceptions across the boundary.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <functional>
#include <initializer_list>
#include <string>
#include <vector>

#include "../../include/tic.h"
#include "tic_launch.cuh"
#include "tic_simt.cuh"
#include "tic_umma.cuh"
#include "tic_umma16.cuh"
#include "tic_first16.cuh"
#include "tic_fused16.cuh"
#include "tic_fused_enc16.cuh"
#include "tic_entropy.cuh"
#include "tic_eval.cuh"

using namespace tic;

namespace {

std::string g_create_error;

struct Layer {
  tic_layer_desc d{};
  float* w = nullptr;     // device [9][cin][cout]
  float* b = nullptr;     // device [cout]
  std::vector<float> hb;  // host copy of the bias (the fused kernels take it as launch constants)
  // operand images, built lazily from w: TF32 slices of 64 output channels, fp16-pair output-channel slices, the fp16-pair
  // first layer (cin = 3), and this layer's and the next one's for a fused pair kernel (decoder tail or encoder head)
  OperandImage img[4 + 16 + 1 + 2];
  OperandImage* tf32() { return img; }
  OperandImage* pair16() { return img + 4; }
  OperandImage& first16() { return img[20]; }
  OperandImage* fused() { return img + 21; }
  bool loaded = false;
  void release() {  // the operand images (rebuilt from w on the next launch)
    for (OperandImage& i : img) i.release();
  }
};

struct Graph {
  std::vector<Layer> layers;
  float mean[3] = {0, 0, 0}, stdv[3] = {1, 1, 1};
  bool has_norm = false;
  float* d_normlut = nullptr;  // [3][256]
};

struct IoSpec {
  int mode = IO_ACT;
  const void* in = nullptr;
  void* out = nullptr;
  Geo geo{};
};

}  // namespace

struct tic_codec {
  int device = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  cudaStream_t s_h2d = nullptr, s_d2h = nullptr;
  cudaEvent_t ev_in[2]{}, ev_comp[2]{}, ev_out[2]{}, ev_enc[2]{}, ev_t0 = nullptr, ev_t1 = nullptr;
  Graph g[3];
  int q = 0;
  float* d_symlut = nullptr;  // [256]
  unsigned long long* d_hist = nullptr;  // [256]
  int mode = TIC_COMPUTE_FP32;
  int chunk128 = 4096;
  // workspaces
  DevBuf act[3];        // rotating chunk activations
  DevBuf stage_in[2];   // host-buffer staging sets
  DevBuf stage_out[2];
  DevBuf stage_sym[2];  // round trips: the symbols between the two graphs
  int64_t launches = 0;
  float last_ms = 0.f;
  bool profile = false;
  struct ProfRec {
    int graph, layer;
    cudaEvent_t e0, e1;
  };
  std::vector<ProfRec> prof_pending;
  std::vector<float> prof_ms[3];
  std::vector<int64_t> prof_n[3];
  int num_sms = 148;
  unsigned int* h_oflow = nullptr;  // host-mapped sticky flags: [0] a pair-plane split saw |x| >= 65504 (fp16 range),
                                    // [1] entropy stage (1: symbol outside the table / of zero width, 2: slot too small)
  unsigned int* d_oflow = nullptr;  // their device address
  uint32_t* d_cum = nullptr;        // entropy stage: the call's cumulative-frequency table [257]
  DevBuf d_seg;                     // entropy stage: worst-case slots of a segmented call's pieces
  DevBuf d_seg_bytes;               //   and their stored lengths (long long)
  DevBuf d_eval;                    // tic_evaluate_images with host buffers: per-image stored lengths, then squared errors
  cudaEvent_t ev_switch = nullptr;  // orders the old stream before the new one in tic_set_stream
  std::string err;
};

namespace {

int fail(tic_codec* h, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  if (h) h->err = buf;
  return code;
}

#define TIC_CUDA(h, expr)                                                                         \
  do {                                                                                            \
    cudaError_t e_ = (expr);                                                                      \
    if (e_ != cudaSuccess)                                                                        \
      return fail((h), TIC_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_), __FILE__, __LINE__); \
  } while (0)

// The set bufs[0, count) grows together: each buffer holds at least `need` bytes.  Work queued earlier on any stream
// may still use the memory a grown set frees, so the device is drained first.  A failed allocation returns `nomem`.
int grow(tic_codec* h, DevBuf* bufs, int count, size_t need, int nomem = TIC_ERR_CUDA) {
  if (bufs[0].bytes >= need) return TIC_OK;
  bool held = false;
  for (int i = 0; i < count; ++i) held = held || bufs[i].p;
  if (held) TIC_CUDA(h, cudaDeviceSynchronize());
  for (int i = 0; i < count; ++i) bufs[i].reset();
  for (int i = 0; i < count; ++i) {
    const cudaError_t e = cudaMalloc(&bufs[i].p, need);
    if (e != cudaSuccess) return fail(h, nomem, "cudaMalloc(%zu) failed: %s", need, cudaGetErrorString(e));
  }
  for (int i = 0; i < count; ++i) bufs[i].bytes = need;
  return TIC_OK;
}

// Device temporaries of one host-buffer call.  They are freed on every return path, after the handle's stream, where
// their copies and kernels are queued, has drained.
struct CallTemps {
  tic_codec* h;
  DevBuf buf[3];
  ~CallTemps() {
    if (buf[0].p || buf[1].p || buf[2].p) cudaStreamSynchronize(h->stream);
  }
};

const char* kOverflowMsg =
    "fp16-pair tensor mode: an activation reached the fp16 range limit (|x| >= 65504); results are invalid. "
    "Use compute mode fp32 or 3xtf32 for these weights (tic_set_compute_mode clears the flag)";

// Sticky fp16-range status: checked at the start of every hot-path call and after every call that synchronises.
int overflow_status(tic_codec* h) {
  if (h->h_oflow && *reinterpret_cast<volatile unsigned int*>(h->h_oflow)) return fail(h, TIC_ERR_UNSUPPORTED, "%s", kOverflowMsg);
  if (h->h_oflow) {
    const unsigned int es = *reinterpret_cast<volatile unsigned int*>(h->h_oflow + 1);
    if (es) {
      *reinterpret_cast<volatile unsigned int*>(h->h_oflow + 1) = 0u;  // reported once
      return fail(h, TIC_ERR_INVALID, es == 1 ? "entropy stage: symbol outside the table or of zero probability"
                                                : "entropy stage: output slot too small (use tic_entropy_bound)");
    }
  }
  return TIC_OK;
}

int pow2ceil(int v) {
  int p = 1;
  while (p < v) p <<= 1;
  return p;
}

// TF SAME: out = ceil(in / s); pad_total = max((out-1)*s + 3 - in, 0); before = total / 2
void same_pad(int in, int s, int* out, int* before) {
  *out = (in + s - 1) / s;
  int total = std::max((*out - 1) * s + 3 - in, 0);
  *before = total / 2;
}

// ---- SIMT launch planning -------------------------------------------------------------------
// Pick the row pitch so that the (up to four) row groups a warp spans land in distinct banks.
int pick_pitch(int iw, int lanes_x, int row_words /* words between a warp's row groups, per pitch unit */, int s) {
  if (lanes_x * s >= 32) return iw | 1;
  for (int c = iw; c < iw + 32; ++c)
    if ((row_words * c) % 32 == (lanes_x * s) % 32) return c;
  return iw;
}

int launch_simt(tic_codec* h, LayerArgs a, int kind, int stride) {
  SmemPlan sp{};
  int ocb, grid_y;
  if (kind == TIC_CONV) {
    ocb = a.cout >= 64 ? 64 : a.cout > 16 ? 32 : a.cout > 8 ? 16 : 8;
    const int ppc = 8192 / ocb;  // output pixels per CTA
    a.TW = std::min(32, pow2ceil(a.wout));
    a.TH = std::min(std::max(4, pow2ceil(a.hout)), ppc / a.TW);
    a.TP = ppc / (a.TW * a.TH);
    a.tiles_x = (a.wout + a.TW - 1) / a.TW;
    a.tiles_y = (a.hout + a.TH - 1) / a.TH;
    sp.ih = (a.TH - 1) * stride + 3;
    sp.iw = (a.TW - 1) * stride + 3;
    sp.iwp = pick_pitch(sp.iw, a.TW, 4 * stride, stride);
  } else {
    ocb = a.cout >= 32 ? 32 : a.cout > 8 ? 16 : a.cout > 4 ? 8 : 4;
    const int ipc = 4096 / ocb;  // input pixels per CTA
    a.TW = std::min(32, pow2ceil(a.win));
    a.TH = std::min(std::max(4, pow2ceil(a.hin)), ipc / a.TW);
    a.TP = ipc / (a.TW * a.TH);
    a.tiles_x = (a.win + a.TW - 1) / a.TW;
    a.tiles_y = (a.hin + a.TH - 1) / a.TH;
    sp.ih = a.TH + 1;
    sp.iw = a.TW + 1;
    sp.iwp = pick_pitch(sp.iw, a.TW, 4, 1);
  }
  sp.cstr = sp.ih * sp.iwp;
  sp.pstr = kIcc * sp.cstr;
  {
    // lanes of one warp may straddle patches: offset consecutive patches to fresh banks
    const int lanes_per_patch = a.TW * a.TH / 4;
    if (lanes_per_patch < 32 && a.TP > 1) {
      const int want = (lanes_per_patch * (kind == TIC_CONV ? stride : 1)) % 32;
      while (sp.pstr % 32 != want) ++sp.pstr;
    }
  }
  grid_y = (a.cout + ocb - 1) / ocb;
  const long long groups = (a.n + a.TP - 1) / a.TP;
  const long long gx = (long long)a.tiles_x * a.tiles_y * groups;
  if (gx <= 0 || gx > 0x7fffffffLL) return fail(h, TIC_ERR_INVALID, "grid too large (%lld)", gx);
  dim3 grid((unsigned)gx, (unsigned)grid_y);
  const size_t smem = ((size_t)a.TP * sp.pstr + 9 * kIcc * ocb) * sizeof(float);
  if (smem > 200 * 1024) return fail(h, TIC_ERR_UNSUPPORTED, "tile needs %zu B shared memory", smem);
  void (*kernel)(LayerArgs, SmemPlan);
  if (kind != TIC_CONV)
    kernel = ocb == 32   ? deconv3x3_simt_kernel<32>
             : ocb == 16 ? deconv3x3_simt_kernel<16>
             : ocb == 8  ? deconv3x3_simt_kernel<8>
                         : deconv3x3_simt_kernel<4>;
  else if (stride == 1)
    kernel = ocb == 64   ? conv3x3_simt_kernel<64, 1>
             : ocb == 32 ? conv3x3_simt_kernel<32, 1>
             : ocb == 16 ? conv3x3_simt_kernel<16, 1>
                         : conv3x3_simt_kernel<8, 1>;
  else
    kernel = ocb == 64   ? conv3x3_simt_kernel<64, 2>
             : ocb == 32 ? conv3x3_simt_kernel<32, 2>
             : ocb == 16 ? conv3x3_simt_kernel<16, 2>
                         : conv3x3_simt_kernel<8, 2>;
  h->launches++;
  TIC_CUDA(h, launch_dyn(kernel, grid, kThreads, smem, h->stream, a, sp));
  return TIC_OK;
}

// ---- graph executor -------------------------------------------------------------------------
struct Shape {
  int h, w, c;
};

struct LayerShape {
  int hin, win, cin, hout, wout, cout, pad_t, pad_l;
};

// Shapes of the first `limit` layers of g (all of them for limit <= 0) on an `in` input; false when a layer's cin is not
// the channel count it receives.
bool layer_shapes(const Graph& g, Shape in, int limit, std::vector<LayerShape>* sh) {
  const size_t L = limit > 0 ? std::min<size_t>((size_t)limit, g.layers.size()) : g.layers.size();
  sh->resize(L);
  Shape s = in;
  for (size_t i = 0; i < L; ++i) {
    const tic_layer_desc& d = g.layers[i].d;
    if (d.cin != s.c) return false;
    LayerShape& t = (*sh)[i];
    t.hin = s.h;
    t.win = s.w;
    t.cin = s.c;
    t.pad_t = t.pad_l = 0;
    if (d.kind == TIC_CONV) {
      same_pad(s.h, d.stride, &t.hout, &t.pad_t);
      same_pad(s.w, d.stride, &t.wout, &t.pad_l);
    } else {
      t.hout = 2 * s.h;
      t.wout = 2 * s.w;
    }
    t.cout = d.cout;
    s = Shape{t.hout, t.wout, t.cout};
  }
  return true;
}

int graph_out_shape(const Graph& g, Shape in, Shape* out, int limit = -1) {
  std::vector<LayerShape> sh;
  if (!layer_shapes(g, in, limit, &sh)) return -1;
  *out = sh.empty() ? in : Shape{sh.back().hout, sh.back().wout, sh.back().cout};
  return 0;
}

int check_graph_ready(tic_codec* h, int gi, bool need_norm) {
  Graph& g = h->g[gi];
  if (g.layers.empty()) return fail(h, TIC_ERR_STATE, "graph %d not configured (tic_set_graph)", gi);
  for (size_t i = 0; i < g.layers.size(); ++i)
    if (!g.layers[i].loaded) return fail(h, TIC_ERR_STATE, "graph %d layer %zu has no weights (tic_load_weights)", gi, i);
  if (need_norm && !g.has_norm) return fail(h, TIC_ERR_STATE, "graph %d has no normalisation (tic_set_norm)", gi);
  return TIC_OK;
}

// The fields of a layer's launch arguments that come from the layer itself: shapes, padding, activation, weights.
void set_layer(LayerArgs& a, const Layer& ly, const LayerShape& t) {
  a.hin = t.hin;
  a.win = t.win;
  a.cin = t.cin;
  a.hout = t.hout;
  a.wout = t.wout;
  a.cout = t.cout;
  a.pad_t = t.pad_t;
  a.pad_l = t.pad_l;
  a.act = ly.d.act;
  a.wgt = ly.w;
  a.bias = ly.b;
}

// Run graph gi over n patches whose first-layer input map is h0 x w0 x c0.
int run_graph(tic_codec* h, int gi, const IoSpec& io_in, const IoSpec& io_out, int n, int h0, int w0, int limit = -1) {
  Graph& g = h->g[gi];
  std::vector<LayerShape> sh;
  if (!layer_shapes(g, Shape{h0, w0, g.layers[0].d.cin}, limit, &sh))
    return fail(h, TIC_ERR_INVALID, "layer channel chain is inconsistent");
  if (n == 0) return TIC_OK;
  const int L = (int)sh.size();
  const bool pair16 = h->mode == TIC_COMPUTE_TENSOR_F16X3;  // intermediate activations are fp16 pair planes
  // pair mode: f32 / symbol inputs of a tensor-capable first layer are split into a workspace buffer first
  bool split_input = false;
  if (pair16 && (io_in.mode == IO_ACT || io_in.mode == IO_U8_SYMLUT)) {
    LayerArgs t{};
    t.n = n;
    set_layer(t, g.layers[0], sh[0]);
    t.in_mode = IO_ACT16;
    t.out_mode = L == 1 ? io_out.mode : IO_ACT16;
    split_input = u16_supported(t, g.layers[0].d.kind, g.layers[0].d.stride);
  }
  // workspaces: three rotating activation buffers
  size_t act_elems = 0;
  for (int i = 0; i + 1 < L; ++i) act_elems = std::max(act_elems, (size_t)n * sh[i].hout * sh[i].wout * sh[i].cout);
  if (split_input) act_elems = std::max(act_elems, (size_t)n * sh[0].hin * sh[0].win * sh[0].cin);
  const int rc0 = grow(h, h->act, 3, act_elems * sizeof(float), TIC_ERR_NOMEM);
  if (rc0 != TIC_OK) return rc0;

  int cur = -1;        // act[] index holding the current activation (-1: the caller's input)
  int res_buf = -1;    // act[] index of the live residual source (-1: none, or not an act[] buffer)
  const void* res_ptr = nullptr;
  long long res_lo = 0;
  if (split_input) {
    const long long per = (long long)sh[0].hin * sh[0].win * sh[0].cin;
    const long long count = (long long)n * per;
    __half* hi = h->act[0].as<__half>();
    const int blocks = (int)std::min<long long>((count + 255) / 256, (long long)h->num_sms * 8);
    if (io_in.mode == IO_ACT)
      u16_split_f32_kernel<<<blocks, 256, 0, h->stream>>>(reinterpret_cast<const float*>(io_in.in), hi, hi + count, count, h->d_oflow);
    else
      u16_split_symlut_kernel<<<blocks, 256, 0, h->stream>>>(reinterpret_cast<const uint8_t*>(io_in.in) + (long long)io_in.geo.n0 * per,
                                                             h->d_symlut, h->q, hi, hi + count, count, h->d_oflow);
    h->launches++;
    TIC_CUDA(h, cudaGetLastError());
    cur = 0;
  }
  const LaunchCtx ctx{h->stream, h->num_sms, &h->err, &h->launches};
  for (int i = 0; i < L; ++i) {
    Layer& ly = g.layers[i];
    const tic_layer_desc& d = ly.d;
    LayerArgs a{};
    a.n = n;
    set_layer(a, ly, sh[i]);
    a.q = h->q;
    a.hist = h->d_hist;
    a.oflow = h->d_oflow;
    a.dbg = tic_env_int("TIC_DBG", 0);  // -DTIC_ABLATE builds only
    for (int c = 0; c < 3; ++c) {
      a.mean[c] = g.mean[c];
      a.stdv[c] = g.stdv[c];
    }
    const long long ein = (long long)a.hin * a.win * a.cin, eout = (long long)a.hout * a.wout * a.cout;
    // ---- input
    if (cur < 0) {
      a.in_mode = io_in.mode;
      a.geo = io_in.geo;
      a.lut = (io_in.mode == IO_U8_NORM) ? g.d_normlut : (io_in.mode == IO_U8_SYMLUT ? h->d_symlut : nullptr);
      a.in = io_in.in;
    } else {
      a.in = h->act[cur].p;
      a.in_mode = pair16 ? IO_ACT16 : IO_ACT;
      a.in_lo_off = (long long)n * ein;
    }
    if (d.res_begin) {
      res_buf = cur;
      res_ptr = a.in;
      res_lo = a.in_lo_off;
    }
    // ---- output: a workspace buffer that is neither the input nor the live residual
    int ob = -1;
    if (i == L - 1) {
      a.out_mode = io_out.mode;
      a.out = io_out.out;
      // a single-layer graph shares one geo between prologue and epilogue only if both need it
      if (!(i == 0 && io_out.mode == IO_ACT)) a.geo = io_out.geo;
    } else {
      for (int b = 0; b < 3; ++b)
        if (b != cur && b != res_buf) {
          ob = b;
          break;
        }
      a.out = h->act[ob].p;
      a.out_mode = pair16 ? IO_ACT16 : IO_ACT;
      a.out_lo_off = (long long)n * eout;
    }
    if (d.res_end) {
      if (!res_ptr) return fail(h, TIC_ERR_INVALID, "res_end without res_begin at layer %d", i);
      a.res = reinterpret_cast<const float*>(res_ptr);
      a.res16 = pair16 ? 1 : 0;
      a.res_lo_off = res_lo;
    }
    int rc;
    tic_codec::ProfRec pr{gi, i, nullptr, nullptr};
    if (h->profile) {
      cudaEventCreate(&pr.e0);
      cudaEventCreate(&pr.e1);
      cudaEventRecord(pr.e0, h->stream);
    }
    // the last two transposed convs of a decoder (32 -> 32 -> 3 into the image) run as one back-to-back kernel: the
    // tensor between them never leaves shared memory (tic_fused16.cuh)
    bool fused = false;
    if (pair16 && i + 2 == L && !d.res_begin && !d.res_end && !g.layers[i + 1].d.res_begin && !g.layers[i + 1].d.res_end) {
      Layer& ly2 = g.layers[i + 1];
      LayerArgs a2 = a;
      set_layer(a2, ly2, sh[i + 1]);
      a2.res = nullptr;
      a2.in = nullptr;
      a2.in_mode = IO_ACT16;
      a2.out_mode = io_out.mode;
      a2.out = io_out.mode == IO_ACT ? nullptr : io_out.out;
      a2.geo = io_out.geo;
      if (a2.out && fused_dec_supported(a, d.kind, a2, ly2.d.kind)) {
        rc = launch_fused_dec(ctx, a, a2, ly.w, ly2.w, ly.hb.data(), ly2.hb.data(), ly.fused());
        fused = true;
      }
    }
    // ... and the first two layers of an encoder (u8 image -> 3 -> 32 -> 32, both stride 2): tic_fused_enc16.cuh
    if (!fused && pair16 && i == 0 && cur < 0 && L >= 3 && !g.layers[1].d.res_begin && !g.layers[1].d.res_end) {
      Layer& ly2 = g.layers[1];
      LayerArgs a2 = a;
      set_layer(a2, ly2, sh[1]);
      a2.res = nullptr;
      a2.in = nullptr;
      a2.in_mode = IO_ACT16;
      a2.out_mode = IO_ACT16;
      a2.out = h->act[0].p;
      a2.out_lo_off = (long long)n * a2.hout * a2.wout * a2.cout;
      if (fused_enc_supported(a, d.kind, d.stride, a2, ly2.d.kind, ly2.d.stride)) {
        rc = launch_fused_enc(ctx, a, a2, ly.w, ly2.w, ly.hb.data(), ly.fused());
        fused = true;
        ob = 0;  // the pair's output lives in act[0]
      }
    }
    if (fused) {
      ++i;  // the next layer ran inside this launch (its time is reported with this layer)
    } else if (pair16 && f16_first_supported(a, d.kind, d.stride)) {
      rc = launch_first16(ctx, a, d.stride, ly.w, ly.first16());
    } else if (pair16 && u16_supported(a, d.kind, d.stride)) {
      rc = launch_u16(ctx, a, d.kind, d.stride, ly.w, ly.pair16());
    } else if (h->mode != TIC_COMPUTE_FP32 && !pair16 && umma_supported(a, d.kind, d.stride)) {
      rc = launch_umma(ctx, a, d.kind, d.stride, ly.w, ly.tf32(), h->mode == TIC_COMPUTE_TENSOR_3XTF32);
    } else {
      rc = launch_simt(h, a, d.kind, d.stride);
    }
    if (h->profile) {
      cudaEventRecord(pr.e1, h->stream);
      h->prof_pending.push_back(pr);
    }
    if (rc != TIC_OK) return rc;
    if (d.res_end) {
      res_buf = -1;
      res_ptr = nullptr;
    }
    cur = ob;
  }
  return TIC_OK;
}

int patches_per_chunk(const tic_codec* h, int P) {
  double scale = (128.0 / P) * (128.0 / P);
  int c = (int)(h->chunk128 * scale);
  return std::max(1, c);
}

// Host-staged calls overlap H2D, kernels and D2H chunk by chunk; what does not overlap is the first chunk's H2D and
// the last chunk's kernels + D2H, so chunks are equal-sized and small: 16 of them as long as a chunk keeps >= 768
// patches of 128x128 (measured on the 64-image round trip: 8 / 12 / 16 / 24 chunks -> 12.8 / 12.9 / 13.2 / 13.1
// Gpixel/s).  A ramped schedule (chunks doubling from 384 patches to the workspace chunk and halving again:
// 2, 4, 8, 18, 18, 8, 4, 2 images) was measured SLOWER (11.3 Gpixel/s): the round trip is bound by the D2H direction
// running next to the H2D (654 MB at 50 GB/s under duplex load, tools/pcie_probe.py), and large chunks leave it idle
// at both ends.
std::vector<int64_t> host_chunk_schedule(int64_t units, int64_t cap, double patches128_per_unit) {
  cap = std::max<int64_t>(1, std::min(cap, units));
  int64_t chunks = (units + cap - 1) / cap;
  const int64_t by_size = (int64_t)((double)units * patches128_per_unit / 768.0);
  chunks = std::max<int64_t>(chunks, std::min<int64_t>(16, by_size));
  chunks = std::max<int64_t>(1, std::min<int64_t>(chunks, units));
  const int64_t upc = (units + chunks - 1) / chunks;
  std::vector<int64_t> out;
  for (int64_t u0 = 0; u0 < units; u0 += upc) out.push_back(std::min<int64_t>(upc, units - u0));
  return out;
}

// Device-buffer calls have no staging to overlap with: fewer, longer launch sequences (up to 16384 patches of 128x128
// each), equal-sized.
std::vector<int64_t> device_chunk_schedule(int64_t units, int64_t cap) {
  cap *= 4;
  const int64_t upc = (units + (units + cap - 1) / cap - 1) / ((units + cap - 1) / cap);
  std::vector<int64_t> out;
  for (int64_t u0 = 0; u0 < units; u0 += upc) out.push_back(std::min<int64_t>(upc, units - u0));
  return out;
}

std::vector<int64_t> chunk_schedule(int mem, int64_t units, int64_t cap, double patches128_per_unit) {
  return mem == TIC_MEM_DEVICE ? device_chunk_schedule(units, cap) : host_chunk_schedule(units, cap, patches128_per_unit);
}

// One output of a driven call: the caller's buffer `dst`, `unit` bytes per unit.  With host buffers it is staged in the
// pair `stage` and copied back chunk by chunk; dst == nullptr: the run still writes the staging buffer, nothing is
// copied.  An `early` output is copied once the run has marked its input consumed, the others at the end of the run.
// stage == h->stage_in: the run works in place on the input's staging buffer.
struct Output {
  void* dst;
  size_t unit;
  DevBuf* stage;
  bool early;
};

// One chunk of a driven call, as its run callback sees it.
struct Chunk {
  const void* in;        // the chunk's staging buffer, or the caller's device buffer
  void* out[2];          // the outputs, likewise (device buffers: the caller's pointers, possibly nullptr)
  int64_t off;           // index of the chunk's first unit in `in` / `out`: 0 when staged
  int64_t u0, nu;        // the chunk's first unit in the call, and its unit count
  bool last;             // the call's last chunk
  // Host buffers: marks the point on the handle's stream after which the input staging buffer may be refilled, and
  // queues the early outputs' copies from there.  Without a mark that point is the end of the run.
  std::function<int()> mark;
};

int mark_consumed(Chunk& c) { return c.mark ? c.mark() : (int)TIC_OK; }

// The chunked driver of every call that takes host or device buffers.  `units` (patches, whole images, elements) of
// `in_unit` bytes run in chunks of at most `upc`; run(Chunk&) queues one chunk's work on the handle's stream.  Device
// buffers: device_chunk_schedule over the caller's pointers.  Host buffers: host_chunk_schedule over two staging sets
// and three streams, so that the H2D of chunk i+1 (s_h2d) runs under the kernels of chunk i and the D2H of chunk i-1
// (s_d2h).
template <typename RunFn>
int drive(tic_codec* h, int mem, const void* in, size_t in_unit, std::initializer_list<Output> outs, int64_t units,
          int64_t upc, RunFn run, double patches128_per_unit = 1.0) {
  if (units <= 0) return TIC_OK;
  TIC_CUDA(h, cudaSetDevice(h->device));
  const std::vector<int64_t> sched = chunk_schedule(mem, units, upc, patches128_per_unit);
  Output o[2] = {};
  std::copy(outs.begin(), outs.end(), o);
  if (mem != TIC_MEM_DEVICE) {
    const size_t most = (size_t)*std::max_element(sched.begin(), sched.end());
    int rc = grow(h, h->stage_in, 2, most * in_unit);
    for (const Output& x : outs)
      if (rc == TIC_OK) rc = grow(h, x.stage, 2, most * x.unit);
    if (rc != TIC_OK) return rc;
  }
  if (int st = overflow_status(h)) return st;
  TIC_CUDA(h, cudaEventRecord(h->ev_t0, h->stream));
  if (mem == TIC_MEM_DEVICE) {
    int64_t u0 = 0;
    for (size_t idx = 0; idx < sched.size(); u0 += sched[idx++]) {
      Chunk c{in, {o[0].dst, o[1].dst}, u0, u0, sched[idx], idx + 1 == sched.size(), nullptr};
      if (int rc = run(c)) return rc;
    }
    TIC_CUDA(h, cudaEventRecord(h->ev_t1, h->stream));
    return TIC_OK;
  }
  bool in_place = false, copies = false;
  for (const Output& x : outs) {
    in_place = in_place || x.stage == h->stage_in;
    copies = copies || x.dst;
  }
  // the pipeline proper runs inside a lambda: ANY failure (a CUDA call, a layer launch) drains the three streams before
  // the error is returned, so no copy is still in flight into or out of the caller's buffers
  const int rc_pipe = [&]() -> int {
    cudaEvent_t consumed[2] = {};  // where chunk idx-2 was done with stage_in[b]
    int64_t u0 = 0;
    for (size_t idx = 0; idx < sched.size(); u0 += sched[idx++]) {
      const int b = (int)(idx & 1);
      const int64_t nu = sched[idx];
      if (idx >= 2) TIC_CUDA(h, cudaStreamWaitEvent(h->s_h2d, in_place ? h->ev_out[b] : consumed[b], 0));
      TIC_CUDA(h, cudaMemcpyAsync(h->stage_in[b].p, (const char*)in + (size_t)u0 * in_unit, (size_t)nu * in_unit,
                                  cudaMemcpyHostToDevice, h->s_h2d));
      TIC_CUDA(h, cudaEventRecord(h->ev_in[b], h->s_h2d));
      TIC_CUDA(h, cudaStreamWaitEvent(h->stream, h->ev_in[b], 0));
      if (idx >= 2 && copies && !in_place) TIC_CUDA(h, cudaStreamWaitEvent(h->stream, h->ev_out[b], 0));  // outputs copied
      // copies the early outputs, or the others, back once the stream has passed `ready`
      auto copy_back = [&](bool early, cudaEvent_t ready) -> int {
        for (const Output& x : outs) {
          if (!x.dst || x.early != early) continue;
          TIC_CUDA(h, cudaStreamWaitEvent(h->s_d2h, ready, 0));
          TIC_CUDA(h, cudaMemcpyAsync((char*)x.dst + (size_t)u0 * x.unit, x.stage[b].p, (size_t)nu * x.unit,
                                      cudaMemcpyDeviceToHost, h->s_d2h));
        }
        return TIC_OK;
      };
      consumed[b] = nullptr;
      Chunk c{h->stage_in[b].p, {o[0].stage ? o[0].stage[b].p : nullptr, o[1].stage ? o[1].stage[b].p : nullptr}, 0, u0, nu,
              idx + 1 == sched.size(), [&]() -> int {
                TIC_CUDA(h, cudaEventRecord(h->ev_enc[b], h->stream));
                consumed[b] = h->ev_enc[b];
                return copy_back(true, h->ev_enc[b]);
              }};
      if (int rc = run(c)) return rc;
      TIC_CUDA(h, cudaEventRecord(h->ev_comp[b], h->stream));
      if (!consumed[b]) {
        consumed[b] = h->ev_comp[b];
        if (int rc = copy_back(true, h->ev_comp[b])) return rc;
      }
      if (int rc = copy_back(false, h->ev_comp[b])) return rc;
      if (copies) TIC_CUDA(h, cudaEventRecord(h->ev_out[b], h->s_d2h));
    }
    TIC_CUDA(h, cudaEventRecord(h->ev_t1, h->stream));
    TIC_CUDA(h, cudaStreamSynchronize(h->s_d2h));
    TIC_CUDA(h, cudaStreamSynchronize(h->stream));
    return TIC_OK;
  }();
  if (rc_pipe != TIC_OK) {
    cudaStreamSynchronize(h->s_h2d);
    cudaStreamSynchronize(h->stream);
    cudaStreamSynchronize(h->s_d2h);
    return rc_pipe;
  }
  return overflow_status(h);
}

Geo patch_geo(int P, long long n0) {
  Geo g{};
  g.H = P;
  g.W = P;
  g.gh = 1;
  g.gw = 1;
  g.oy = 0;
  g.ox = 0;
  g.P = P;
  g.n0 = n0;
  geo_finish(g);
  return g;
}

Geo image_geo(int H, int W, int P, long long n0) {
  Geo g{};
  g.H = H;
  g.W = W;
  g.gh = (H + P - 1) / P;
  g.gw = (W + P - 1) / P;
  g.oy = 0;
  g.ox = 0;
  g.P = P;
  g.n0 = n0;
  geo_finish(g);
  return g;
}

// What an image call needs to know about its graphs: the symbol map of one P x P patch (hb x wb x cb) and the patches
// per H x W image.
struct ImageShapes {
  int hb, wb, cb, ppi;
};

// The checks every image call makes.  `enc` / `dec`: the call runs the encoder / the decoder graph.
int image_shapes(tic_codec* h, int H, int W, int P, bool enc, bool dec, ImageShapes* s) {
  if (enc && ((H % P != 0 && H < 2) || (W % P != 0 && W < 2)))
    return fail(h, TIC_ERR_INVALID, "reflect padding needs at least 2 pixels");
  if (enc)
    if (int rc = check_graph_ready(h, TIC_GRAPH_ENCODER, true)) return rc;
  if (dec)
    if (int rc = check_graph_ready(h, TIC_GRAPH_DECODER, true)) return rc;
  if (h->q < 2) return fail(h, TIC_ERR_STATE, "quantiser not configured (tic_set_quantizer)");
  const Graph& gd = h->g[TIC_GRAPH_DECODER];
  Shape so;
  if (enc) {
    if (h->g[TIC_GRAPH_ENCODER].layers[0].d.cin != 3) return fail(h, TIC_ERR_INVALID, "encoder must take 3 channels");
    if (int rc = tic_bottleneck_shape(h, P, &s->hb, &s->wb, &s->cb)) return rc;
    if (dec && (gd.layers[0].d.cin != s->cb || graph_out_shape(gd, Shape{s->hb, s->wb, s->cb}, &so) != 0 || so.c != 3 ||
                so.h != P || so.w != P))
      return fail(h, TIC_ERR_INVALID, "decoder graph does not map the encoder's %dx%dx%d symbols back to %dx%d RGB", s->hb, s->wb,
                  s->cb, P, P);
  } else {
    // bottleneck map size for patch size P: invert the decoder's upsampling
    int up = 1;
    for (auto& l : gd.layers)
      if (l.d.kind == TIC_DECONV) up *= 2;
    if (P % up != 0) return fail(h, TIC_ERR_INVALID, "patch size %d is not a multiple of the decoder upsampling %d", P, up);
    s->hb = s->wb = P / up;
    s->cb = gd.layers[0].d.cin;
    if (graph_out_shape(gd, Shape{s->hb, s->wb, s->cb}, &so) != 0 || so.c != 3 || so.h != P)
      return fail(h, TIC_ERR_INVALID, "decoder graph does not map %dx%d symbols to %dx%d RGB", s->hb, s->wb, P, P);
  }
  const Geo g0 = image_geo(H, W, P, 0);
  s->ppi = g0.gh * g0.gw;
  return TIC_OK;
}

// Frees a graph's weights (its layers' operand images go with the layers).
void free_layers(Graph& g) {
  for (auto& l : g.layers) {
    cudaFree(l.w);
    cudaFree(l.b);
  }
  g.layers.clear();
}

}  // namespace

// =============================================================================================
extern "C" {

const char* tic_version(void) { return "tic-b200 0.1 (sm_100a)"; }
const char* tic_create_error(void) { return g_create_error.c_str(); }

int tic_create(tic_codec** out, int device) {
  if (!out) return TIC_ERR_INVALID;
  *out = nullptr;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count <= 0) {
    g_create_error = std::string("no CUDA device: ") + cudaGetErrorString(e) +
                     " (this library has no CPU fallback)";
    return TIC_ERR_CUDA;
  }
  if (device < 0 || device >= count) {
    g_create_error = "device index out of range";
    return TIC_ERR_INVALID;
  }
  tic_codec* h = new tic_codec();
  h->device = device;
  auto bail = [&](const char* what, cudaError_t err) {
    g_create_error = std::string(what) + ": " + cudaGetErrorString(err);
    delete h;
    return TIC_ERR_CUDA;
  };
  if ((e = cudaSetDevice(device)) != cudaSuccess) return bail("cudaSetDevice", e);
  cudaDeviceProp prop;
  if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) return bail("cudaGetDeviceProperties", e);
  h->num_sms = prop.multiProcessorCount;
  if (prop.major != 10) {
    g_create_error = "this build targets sm_100a (B200); device is sm_" + std::to_string(prop.major * 10 + prop.minor);
    delete h;
    return TIC_ERR_UNSUPPORTED;
  }
  if ((e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking)) != cudaSuccess) return bail("stream", e);
  h->own_stream = true;
  if ((e = cudaStreamCreateWithFlags(&h->s_h2d, cudaStreamNonBlocking)) != cudaSuccess) return bail("stream", e);
  if ((e = cudaStreamCreateWithFlags(&h->s_d2h, cudaStreamNonBlocking)) != cudaSuccess) return bail("stream", e);
  for (int b = 0; b < 2; ++b) {
    cudaEventCreateWithFlags(&h->ev_in[b], cudaEventDisableTiming);
    cudaEventCreateWithFlags(&h->ev_comp[b], cudaEventDisableTiming);
    cudaEventCreateWithFlags(&h->ev_out[b], cudaEventDisableTiming);
    cudaEventCreateWithFlags(&h->ev_enc[b], cudaEventDisableTiming);
  }
  cudaEventCreate(&h->ev_t0);
  cudaEventCreate(&h->ev_t1);
  if ((e = cudaMalloc(&h->d_hist, 256 * sizeof(unsigned long long))) != cudaSuccess) return bail("cudaMalloc", e);
  cudaMemset(h->d_hist, 0, 256 * sizeof(unsigned long long));
  if ((e = cudaMalloc(&h->d_symlut, 256 * sizeof(float))) != cudaSuccess) return bail("cudaMalloc", e);
  cudaMemset(h->d_symlut, 0, 256 * sizeof(float));
  if ((e = cudaHostAlloc((void**)&h->h_oflow, 2 * sizeof(unsigned int), cudaHostAllocMapped | cudaHostAllocPortable)) != cudaSuccess)
    return bail("cudaHostAlloc", e);
  h->h_oflow[0] = h->h_oflow[1] = 0u;
  if ((e = cudaMalloc(&h->d_cum, (kEntropyMaxSymbols + 1) * sizeof(uint32_t))) != cudaSuccess) return bail("cudaMalloc", e);
  if ((e = cudaHostGetDevicePointer((void**)&h->d_oflow, h->h_oflow, 0)) != cudaSuccess) return bail("cudaHostGetDevicePointer", e);
  cudaEventCreateWithFlags(&h->ev_switch, cudaEventDisableTiming);
  *out = h;
  return TIC_OK;
}

void tic_destroy(tic_codec* h) {
  if (!h) return;
  cudaSetDevice(h->device);
  cudaDeviceSynchronize();
  for (Graph& g : h->g) {
    free_layers(g);
    if (g.d_normlut) cudaFree(g.d_normlut);
  }
  for (int b = 0; b < 2; ++b) {
    cudaEventDestroy(h->ev_enc[b]);
    cudaEventDestroy(h->ev_in[b]);
    cudaEventDestroy(h->ev_comp[b]);
    cudaEventDestroy(h->ev_out[b]);
  }
  cudaEventDestroy(h->ev_t0);
  cudaEventDestroy(h->ev_t1);
  if (h->d_hist) cudaFree(h->d_hist);
  if (h->d_symlut) cudaFree(h->d_symlut);
  if (h->h_oflow) cudaFreeHost(h->h_oflow);
  if (h->d_cum) cudaFree(h->d_cum);
  if (h->ev_switch) cudaEventDestroy(h->ev_switch);
  if (h->own_stream && h->stream) cudaStreamDestroy(h->stream);
  if (h->s_h2d) cudaStreamDestroy(h->s_h2d);
  if (h->s_d2h) cudaStreamDestroy(h->s_d2h);
  delete h;
}

const char* tic_last_error(const tic_codec* h) { return h ? h->err.c_str() : "null handle"; }

int tic_set_stream(tic_codec* h, void* cuda_stream) {
  if (!h) return TIC_ERR_INVALID;
  cudaStream_t next = (cudaStream_t)cuda_stream;
  if (next == h->stream) return TIC_OK;
  TIC_CUDA(h, cudaSetDevice(h->device));
  // The handle's workspaces (rotating activation buffers, weight images under construction, the histogram, the
  // staging sets) are shared by everything it launches: work queued on the old stream must finish before work on the
  // new stream may touch them.  Device-side ordering (event), no host stall — except when leaving the private
  // stream, which is destroyed.
  if (h->own_stream && h->stream) {
    cudaStreamSynchronize(h->stream);
    cudaStreamDestroy(h->stream);
  } else {
    TIC_CUDA(h, cudaEventRecord(h->ev_switch, h->stream));
    TIC_CUDA(h, cudaStreamWaitEvent(next, h->ev_switch, 0));
  }
  h->stream = next;
  h->own_stream = false;
  return TIC_OK;
}

int tic_set_compute_mode(tic_codec* h, int mode) {
  if (!h) return TIC_ERR_INVALID;
  if (mode < TIC_COMPUTE_FP32 || mode > TIC_COMPUTE_TENSOR_F16X3) return fail(h, TIC_ERR_INVALID, "unknown compute mode %d", mode);
  h->mode = mode;
  if (h->h_oflow) {
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->stream);
    *h->h_oflow = 0u;  // the fp16-range flag belongs to the previous mode's runs
  }
  return TIC_OK;
}

int tic_set_chunk_patches(tic_codec* h, int chunk) {
  if (!h || chunk <= 0) return h ? fail(h, TIC_ERR_INVALID, "chunk must be positive") : TIC_ERR_INVALID;
  h->chunk128 = chunk;
  return TIC_OK;
}

int tic_set_graph(tic_codec* h, int graph, const tic_layer_desc* layers, int n_layers) {
  if (!h) return TIC_ERR_INVALID;
  if (graph < 0 || graph > 2 || !layers || n_layers <= 0) return fail(h, TIC_ERR_INVALID, "bad graph arguments");
  TIC_CUDA(h, cudaSetDevice(h->device));
  int prev = -1;
  bool open_res = false;
  for (int i = 0; i < n_layers; ++i) {
    const tic_layer_desc& d = layers[i];
    if (d.kind != TIC_CONV && d.kind != TIC_DECONV) return fail(h, TIC_ERR_INVALID, "layer %d: bad kind", i);
    if (d.cin <= 0 || d.cout <= 0 || d.cin > 1024 || d.cout > 1024) return fail(h, TIC_ERR_INVALID, "layer %d: bad channels", i);
    if (d.kind == TIC_CONV && d.stride != 1 && d.stride != 2) return fail(h, TIC_ERR_INVALID, "layer %d: conv stride must be 1 or 2", i);
    if (d.kind == TIC_DECONV && d.stride != 2) return fail(h, TIC_ERR_INVALID, "layer %d: deconv stride must be 2", i);
    if (prev >= 0 && d.cin != prev) return fail(h, TIC_ERR_INVALID, "layer %d: cin %d != previous cout %d", i, d.cin, prev);
    if (d.res_begin) {
      if (open_res || i == 0) return fail(h, TIC_ERR_INVALID, "layer %d: bad res_begin", i);
      open_res = true;
    }
    if (d.res_end) {
      if (!open_res || d.kind != TIC_CONV || d.stride != 1) return fail(h, TIC_ERR_INVALID, "layer %d: bad res_end", i);
      open_res = false;
    }
    if (open_res && (d.kind != TIC_CONV || d.stride != 1 || d.cin != d.cout))
      return fail(h, TIC_ERR_INVALID, "layer %d: residual blocks need stride-1 convs with cin == cout", i);
    if (i == n_layers - 1 && open_res) return fail(h, TIC_ERR_INVALID, "unterminated residual block");
    prev = d.cout;
  }
  Graph& g = h->g[graph];
  free_layers(g);
  g.layers.resize(n_layers);
  for (int i = 0; i < n_layers; ++i) {
    Layer& l = g.layers[i];
    l.d = layers[i];
    TIC_CUDA(h, cudaMalloc(&l.w, (size_t)9 * l.d.cin * l.d.cout * sizeof(float)));
    TIC_CUDA(h, cudaMalloc(&l.b, (size_t)l.d.cout * sizeof(float)));
  }
  return TIC_OK;
}

int tic_load_weights(tic_codec* h, int graph, int layer, const float* kernel, const float* bias) {
  if (!h) return TIC_ERR_INVALID;
  if (graph < 0 || graph > 2 || !kernel || !bias) return fail(h, TIC_ERR_INVALID, "bad arguments");
  Graph& g = h->g[graph];
  if (layer < 0 || layer >= (int)g.layers.size()) return fail(h, TIC_ERR_INVALID, "layer index %d out of range", layer);
  TIC_CUDA(h, cudaSetDevice(h->device));
  Layer& l = g.layers[layer];
  const int cin = l.d.cin, cout = l.d.cout;
  std::vector<float> w((size_t)9 * cin * cout);
  if (l.d.kind == TIC_CONV) {
    // TF HWIO [3][3][cin][cout] is already [tap][cin][cout]
    std::memcpy(w.data(), kernel, w.size() * sizeof(float));
  } else {
    // TF conv2d_transpose filter [3][3][cout][cin] (basic_block.py:53) -> [tap][cin][cout]
    for (int t = 0; t < 9; ++t)
      for (int oc = 0; oc < cout; ++oc)
        for (int ic = 0; ic < cin; ++ic) w[((size_t)t * cin + ic) * cout + oc] = kernel[((size_t)t * cout + oc) * cin + ic];
  }
  TIC_CUDA(h, cudaStreamSynchronize(h->stream));
  TIC_CUDA(h, cudaMemcpy(l.w, w.data(), w.size() * sizeof(float), cudaMemcpyHostToDevice));
  TIC_CUDA(h, cudaMemcpy(l.b, bias, (size_t)cout * sizeof(float), cudaMemcpyHostToDevice));
  l.hb.assign(bias, bias + cout);
  l.release();
  if (layer > 0)  // the fused pair kernels keep this layer's operand image with the previous layer
    for (int k = 0; k < 2; ++k) g.layers[layer - 1].fused()[k].release();
  l.loaded = true;
  return TIC_OK;
}

int tic_set_norm(tic_codec* h, int graph, const float* mean3, const float* std3) {
  if (!h) return TIC_ERR_INVALID;
  if (graph < 0 || graph > 2 || !mean3 || !std3) return fail(h, TIC_ERR_INVALID, "bad arguments");
  TIC_CUDA(h, cudaSetDevice(h->device));
  Graph& g = h->g[graph];
  std::vector<float> lut(3 * 256);
  for (int c = 0; c < 3; ++c) {
    if (!(std3[c] != 0.0f)) return fail(h, TIC_ERR_INVALID, "std[%d] is zero", c);
    g.mean[c] = mean3[c];
    g.stdv[c] = std3[c];
    for (int v = 0; v < 256; ++v) lut[c * 256 + v] = tic_normalize((float)v, mean3[c], std3[c]);
  }
  if (!g.d_normlut) TIC_CUDA(h, cudaMalloc(&g.d_normlut, lut.size() * sizeof(float)));
  TIC_CUDA(h, cudaStreamSynchronize(h->stream));
  TIC_CUDA(h, cudaMemcpy(g.d_normlut, lut.data(), lut.size() * sizeof(float), cudaMemcpyHostToDevice));
  g.has_norm = true;
  return TIC_OK;
}

int tic_set_quantizer(tic_codec* h, int quan_scale, const float* inv_sigmoid_lut) {
  if (!h) return TIC_ERR_INVALID;
  if (quan_scale < 2 || quan_scale > 256 || !inv_sigmoid_lut)
    return fail(h, TIC_ERR_INVALID, "quan_scale must be in [2, 256] (symbols are stored as uint8)");
  TIC_CUDA(h, cudaSetDevice(h->device));
  TIC_CUDA(h, cudaStreamSynchronize(h->stream));
  TIC_CUDA(h, cudaMemcpy(h->d_symlut, inv_sigmoid_lut, (size_t)quan_scale * sizeof(float), cudaMemcpyHostToDevice));
  h->q = quan_scale;
  return TIC_OK;
}

int tic_bottleneck_shape(tic_codec* h, int P, int* hb, int* wb, int* cb) {
  if (!h) return TIC_ERR_INVALID;
  Graph& g = h->g[TIC_GRAPH_ENCODER];
  if (g.layers.empty()) return fail(h, TIC_ERR_STATE, "encoder graph not configured");
  Shape so;
  if (graph_out_shape(g, Shape{P, P, g.layers[0].d.cin}, &so) != 0) return fail(h, TIC_ERR_INVALID, "inconsistent graph");
  if (hb) *hb = so.h;
  if (wb) *wb = so.w;
  if (cb) *cb = so.c;
  return TIC_OK;
}

// ---- hot path ---------------------------------------------------------------------------------
int tic_encode_patches(tic_codec* h, const void* patches, int in_dtype, int64_t n, int P, void* symbols,
                       int out_dtype, int mem) {
  if (!h) return TIC_ERR_INVALID;
  if (n < 0 || P <= 0 || (n > 0 && (!patches || !symbols))) return fail(h, TIC_ERR_INVALID, "bad arguments");
  if (in_dtype != TIC_U8 && in_dtype != TIC_F32) return fail(h, TIC_ERR_INVALID, "bad in_dtype");
  if (out_dtype != TIC_U8 && out_dtype != TIC_F32) return fail(h, TIC_ERR_INVALID, "bad out_dtype");
  ImageShapes s;
  if (int rc = image_shapes(h, P, P, P, true, false, &s)) return rc;  // a patch is a P x P image
  const size_t in_unit = (size_t)P * P * 3 * (in_dtype == TIC_U8 ? 1 : 4);
  const size_t out_unit = (size_t)s.hb * s.wb * s.cb * (out_dtype == TIC_U8 ? 1 : 4);
  return drive(h, mem, patches, in_unit, {{symbols, out_unit, h->stage_out, false}}, n, patches_per_chunk(h, P),
               [&](Chunk& c) {
                 IoSpec i, o;
                 i.mode = in_dtype == TIC_U8 ? IO_U8_NORM : IO_F32_NORM;
                 i.in = c.in;
                 i.geo = patch_geo(P, c.off);
                 o.mode = out_dtype == TIC_U8 ? IO_QUANT_U8 : IO_QUANT_F32;
                 o.out = c.out[0];
                 o.geo = patch_geo(P, c.off);
                 return run_graph(h, TIC_GRAPH_ENCODER, i, o, (int)c.nu, P, P);
               }, (double)P * P / 16384.0);
}

int tic_encode_images(tic_codec* h, const uint8_t* images, int64_t n_images, int H, int W, int P, uint8_t* symbols,
                      int mem) {
  if (!h) return TIC_ERR_INVALID;
  if (n_images < 0 || H <= 0 || W <= 0 || P <= 0 || (n_images > 0 && (!images || !symbols)))
    return fail(h, TIC_ERR_INVALID, "bad arguments");
  ImageShapes s;
  if (int rc = image_shapes(h, H, W, P, true, false, &s)) return rc;
  const int ppi = s.ppi;
  const int64_t ipc = std::max<int64_t>(1, patches_per_chunk(h, P) / ppi);
  const size_t in_unit = (size_t)H * W * 3;
  const size_t out_unit = (size_t)ppi * s.hb * s.wb * s.cb;
  return drive(h, mem, images, in_unit, {{symbols, out_unit, h->stage_out, false}}, n_images, ipc,
               [&](Chunk& c) {
                 IoSpec i, o;
                 i.mode = IO_U8_NORM;
                 i.in = c.in;
                 i.geo = image_geo(H, W, P, c.off * ppi);
                 o.mode = IO_QUANT_U8;
                 o.out = c.out[0];
                 o.geo = i.geo;
                 return run_graph(h, TIC_GRAPH_ENCODER, i, o, (int)(c.nu * ppi), P, P);
               }, (double)ppi * P * P / 16384.0);
}

int tic_decode_patches(tic_codec* h, const uint8_t* symbols, int64_t n, int hb, int wb, float* recon, int mem) {
  if (!h) return TIC_ERR_INVALID;
  if (n < 0 || hb <= 0 || wb <= 0 || (n > 0 && (!symbols || !recon))) return fail(h, TIC_ERR_INVALID, "bad arguments");
  int rc = check_graph_ready(h, TIC_GRAPH_DECODER, true);
  if (rc != TIC_OK) return rc;
  if (h->q < 2) return fail(h, TIC_ERR_STATE, "quantiser not configured (tic_set_quantizer)");
  Graph& g = h->g[TIC_GRAPH_DECODER];
  const int cb = g.layers[0].d.cin;
  Shape so;
  if (graph_out_shape(g, Shape{hb, wb, cb}, &so) != 0) return fail(h, TIC_ERR_INVALID, "inconsistent graph");
  if (so.c != 3 || so.h != so.w) return fail(h, TIC_ERR_INVALID, "decoder must produce square RGB patches (got %dx%dx%d)", so.h, so.w, so.c);
  const int P = so.h;
  return drive(h, mem, symbols, (size_t)hb * wb * cb, {{recon, (size_t)P * P * 3 * 4, h->stage_out, false}}, n,
               patches_per_chunk(h, P),
               [&](Chunk& c) {
                 IoSpec i, o;
                 i.mode = IO_U8_SYMLUT;
                 i.in = c.in;
                 i.geo = patch_geo(P, c.off);
                 o.mode = IO_DENORM_F32;
                 o.out = c.out[0];
                 o.geo = patch_geo(P, c.off);
                 return run_graph(h, TIC_GRAPH_DECODER, i, o, (int)c.nu, hb, wb);
               }, (double)P * P / 16384.0);
}

int tic_decode_images(tic_codec* h, const uint8_t* symbols, int64_t n_images, int H, int W, int P, void* images,
                      int out_dtype, int mem) {
  if (!h) return TIC_ERR_INVALID;
  if (n_images < 0 || H <= 0 || W <= 0 || P <= 0 || (n_images > 0 && (!symbols || !images)))
    return fail(h, TIC_ERR_INVALID, "bad arguments");
  if (out_dtype != TIC_U8 && out_dtype != TIC_F32) return fail(h, TIC_ERR_INVALID, "bad out_dtype");
  ImageShapes s;
  if (int rc = image_shapes(h, H, W, P, false, true, &s)) return rc;
  const int ppi = s.ppi;
  const int64_t ipc = std::max<int64_t>(1, patches_per_chunk(h, P) / ppi);
  const size_t in_unit = (size_t)ppi * s.hb * s.wb * s.cb;
  const size_t out_unit = (size_t)H * W * 3 * (out_dtype == TIC_U8 ? 1 : 4);
  return drive(h, mem, symbols, in_unit, {{images, out_unit, h->stage_out, false}}, n_images, ipc,
               [&](Chunk& c) {
                 IoSpec i, o;
                 i.mode = IO_U8_SYMLUT;
                 i.in = c.in;
                 i.geo = image_geo(H, W, P, c.off * ppi);
                 o.mode = out_dtype == TIC_U8 ? IO_DENORM_U8 : IO_DENORM_F32;
                 o.out = c.out[0];
                 o.geo = i.geo;
                 return run_graph(h, TIC_GRAPH_DECODER, i, o, (int)(c.nu * ppi), s.hb, s.wb);
               }, (double)ppi * P * P / 16384.0);
}

int tic_roundtrip_images(tic_codec* h, const uint8_t* images, int64_t n_images, int H, int W, int P, uint8_t* symbols,
                         void* recon, int out_dtype, int mem) {
  if (!h) return TIC_ERR_INVALID;
  if (n_images < 0 || H <= 0 || W <= 0 || P <= 0 || (n_images > 0 && (!images || !recon)))
    return fail(h, TIC_ERR_INVALID, "bad arguments");
  if (out_dtype != TIC_U8 && out_dtype != TIC_F32) return fail(h, TIC_ERR_INVALID, "bad out_dtype");
  if (mem == TIC_MEM_DEVICE && !symbols && n_images > 0)
    return fail(h, TIC_ERR_INVALID, "device-resident round trips need a symbol buffer");
  ImageShapes s;
  if (int rc = image_shapes(h, H, W, P, true, true, &s)) return rc;
  const int ppi = s.ppi;
  const int64_t ipc = std::max<int64_t>(1, patches_per_chunk(h, P) / ppi);
  const size_t sym_unit = (size_t)ppi * s.hb * s.wb * s.cb;
  const size_t rec_unit = (size_t)H * W * 3 * (out_dtype == TIC_U8 ? 1 : 4);
  // Per chunk: encoder -> symbols -> decoder.  With host buffers the next chunk's images may overwrite this one's once
  // the encoder has read them, and the symbols go back while the decoder runs.
  return drive(h, mem, images, (size_t)H * W * 3, {{symbols, sym_unit, h->stage_sym, true}, {recon, rec_unit, h->stage_out, false}},
               n_images, ipc,
               [&](Chunk& c) {
                 IoSpec i, o;
                 i.mode = IO_U8_NORM;
                 i.in = c.in;
                 i.geo = image_geo(H, W, P, c.off * ppi);
                 o.mode = IO_QUANT_U8;
                 o.out = c.out[0];
                 o.geo = i.geo;
                 if (int rc = run_graph(h, TIC_GRAPH_ENCODER, i, o, (int)(c.nu * ppi), P, P)) return rc;
                 if (int rc = mark_consumed(c)) return rc;
                 IoSpec di, dout;
                 di.mode = IO_U8_SYMLUT;
                 di.in = c.out[0];
                 di.geo = i.geo;
                 dout.mode = out_dtype == TIC_U8 ? IO_DENORM_U8 : IO_DENORM_F32;
                 dout.out = c.out[1];
                 dout.geo = i.geo;
                 return run_graph(h, TIC_GRAPH_DECODER, di, dout, (int)(c.nu * ppi), s.hb, s.wb);
               }, (double)ppi * P * P / 16384.0);
}

int tic_postfilter_patches(tic_codec* h, const float* tiles, int64_t n, int P, float* out, int mem) {
  if (!h) return TIC_ERR_INVALID;
  if (n < 0 || P <= 0 || (n > 0 && (!tiles || !out))) return fail(h, TIC_ERR_INVALID, "bad arguments");
  int rc = check_graph_ready(h, TIC_GRAPH_POSTFILTER, true);
  if (rc != TIC_OK) return rc;
  Graph& g = h->g[TIC_GRAPH_POSTFILTER];
  Shape so;
  if (g.layers[0].d.cin != 3 || graph_out_shape(g, Shape{P, P, 3}, &so) != 0 || so.c != 3 || so.h != P || so.w != P)
    return fail(h, TIC_ERR_INVALID, "post-filter graph must map PxPx3 to PxPx3");
  const size_t unit = (size_t)P * P * 3 * 4;
  return drive(h, mem, tiles, unit, {{out, unit, h->stage_out, false}}, n, patches_per_chunk(h, P),
               [&](Chunk& c) {
                 IoSpec i, o;
                 i.mode = IO_F32_NORM;
                 i.in = c.in;
                 i.geo = patch_geo(P, c.off);
                 o.mode = IO_DENORM_F32;
                 o.out = c.out[0];
                 o.geo = patch_geo(P, c.off);
                 return run_graph(h, TIC_GRAPH_POSTFILTER, i, o, (int)c.nu, P, P);
               });
}

int tic_postfilter_images(tic_codec* h, float* images, int64_t n_images, int H, int W, int mem) {
  if (!h) return TIC_ERR_INVALID;
  if (n_images < 0 || H <= 0 || W <= 0 || (n_images > 0 && !images)) return fail(h, TIC_ERR_INVALID, "bad arguments");
  int rc = check_graph_ready(h, TIC_GRAPH_POSTFILTER, true);
  if (rc != TIC_OK) return rc;
  Graph& g = h->g[TIC_GRAPH_POSTFILTER];
  const int P = 128, off = 64;  // submit/2/rmbe/rmbe.py:12,16
  Shape so;
  if (g.layers[0].d.cin != 3 || graph_out_shape(g, Shape{P, P, 3}, &so) != 0 || so.c != 3 || so.h != P || so.w != P)
    return fail(h, TIC_ERR_INVALID, "post-filter graph must map 128x128x3 to 128x128x3");
  const size_t unit = (size_t)H * W * 3 * 4;
  // tiles per image of the two passes; whole images per chunk so that pass 2 reads pass-1 output
  const int t1 = (H / P) * ((W - off) / P), t2 = ((H - off) / P) * (W / P);
  const int64_t ipc = std::max<int64_t>(1, patches_per_chunk(h, P) / std::max(1, std::max(t1, t2)));
  return drive(h, mem, images, unit, {{images, unit, h->stage_in, false}}, n_images, ipc,
               [&](Chunk& c) {
                 for (int pass = 0; pass < 2; ++pass) {
                   Geo gg{};
                   gg.H = H;
                   gg.W = W;
                   gg.P = P;
                   if (pass == 0) {  // rmbe_height: rows i*128, cols 64 + j*128 (rmbe.py:70-89)
                     gg.gh = H / P;
                     gg.gw = W >= off ? (W - off) / P : 0;
                     gg.oy = 0;
                     gg.ox = off;
                   } else {          // rmbe_width: rows 64 + i*128, cols j*128 (rmbe.py:92-111)
                     gg.gh = H >= off ? (H - off) / P : 0;
                     gg.gw = W / P;
                     gg.oy = off;
                     gg.ox = 0;
                   }
                   const int tiles = gg.gh * gg.gw;
                   if (tiles <= 0) continue;
                   gg.n0 = c.off * tiles;
                   geo_finish(gg);
                   IoSpec i, o;
                   i.mode = IO_F32_NORM;
                   i.in = c.out[0];  // in place: pass 2 reads what pass 1 wrote
                   i.geo = gg;
                   o.mode = IO_DENORM_F32;
                   o.out = c.out[0];
                   o.geo = gg;
                   int r2 = run_graph(h, TIC_GRAPH_POSTFILTER, i, o, (int)(c.nu * tiles), P, P);
                   if (r2 != TIC_OK) return r2;
                 }
                 return (int)TIC_OK;
               });
}

int tic_run_layers(tic_codec* h, int graph, const float* in, int64_t n, int h0, int w0, int n_layers, float* out,
                   int mem) {
  if (!h) return TIC_ERR_INVALID;
  if (graph < 0 || graph > 2 || n < 0 || h0 <= 0 || w0 <= 0 || n_layers <= 0 || (n > 0 && (!in || !out)))
    return fail(h, TIC_ERR_INVALID, "bad arguments");
  int rc = check_graph_ready(h, graph, false);
  if (rc != TIC_OK) return rc;
  Graph& g = h->g[graph];
  if (n_layers > (int)g.layers.size()) return fail(h, TIC_ERR_INVALID, "graph has only %zu layers", g.layers.size());
  if (g.layers[n_layers - 1].d.res_begin) return fail(h, TIC_ERR_INVALID, "cannot stop inside a residual block");
  const int cin = g.layers[0].d.cin;
  Shape so;
  if (graph_out_shape(g, Shape{h0, w0, cin}, &so, n_layers) != 0) return fail(h, TIC_ERR_INVALID, "inconsistent graph");
  const size_t in_unit = (size_t)h0 * w0 * cin * 4, out_unit = (size_t)so.h * so.w * so.c * 4;
  const int64_t upc = std::max<int64_t>(1, (int64_t)h->chunk128 * 128 * 128 / ((int64_t)std::max(h0 * w0, so.h * so.w)));
  return drive(h, mem, in, in_unit, {{out, out_unit, h->stage_out, false}}, n, upc, [&](Chunk& c) {
    IoSpec i, o;
    i.mode = IO_ACT;
    i.in = (const char*)c.in + (size_t)c.off * in_unit;
    o.mode = IO_ACT;
    o.out = (char*)c.out[0] + (size_t)c.off * out_unit;
    return run_graph(h, graph, i, o, (int)c.nu, h0, w0, n_layers);
  });
}

int tic_round_u8(tic_codec* h, const float* src, uint8_t* dst, int64_t count, int mem) {
  if (!h) return TIC_ERR_INVALID;
  if (count < 0 || (count > 0 && (!src || !dst))) return fail(h, TIC_ERR_INVALID, "bad arguments");
  const int64_t upc = 1 << 26;
  return drive(h, mem, src, 4, {{dst, 1, h->stage_out, false}}, count, upc, [&](Chunk& c) {
    const float* s = (const float*)c.in + c.off;
    uint8_t* d = (uint8_t*)c.out[0] + c.off;
    int blocks = (int)std::min<int64_t>((c.nu + 255) / 256, (int64_t)h->num_sms * 16);
    round_u8_kernel<<<blocks, 256, 0, h->stream>>>(s, d, c.nu);
    h->launches++;
    TIC_CUDA(h, cudaGetLastError());
    return (int)TIC_OK;
  });
}

// ---- statistics -------------------------------------------------------------------------------
int tic_hist_reset(tic_codec* h) {
  if (!h) return TIC_ERR_INVALID;
  TIC_CUDA(h, cudaSetDevice(h->device));
  TIC_CUDA(h, cudaMemsetAsync(h->d_hist, 0, 256 * sizeof(unsigned long long), h->stream));
  return TIC_OK;
}

int tic_hist_read(tic_codec* h, uint64_t* counts, int q) {
  if (!h) return TIC_ERR_INVALID;
  if (!counts || q <= 0 || q > 256) return fail(h, TIC_ERR_INVALID, "bad arguments");
  TIC_CUDA(h, cudaSetDevice(h->device));
  TIC_CUDA(h, cudaMemcpyAsync(counts, h->d_hist, (size_t)q * sizeof(uint64_t), cudaMemcpyDeviceToHost, h->stream));
  TIC_CUDA(h, cudaStreamSynchronize(h->stream));
  return TIC_OK;
}

int tic_hist_device_ptr(tic_codec* h, void** dev_ptr) {
  if (!h || !dev_ptr) return TIC_ERR_INVALID;
  *dev_ptr = h->d_hist;
  return TIC_OK;
}

int tic_position_sums(tic_codec* h, const uint8_t* symbols, int64_t n, int64_t npos, uint64_t* sums, int mem) {
  if (!h) return TIC_ERR_INVALID;
  if (n < 0 || npos <= 0 || !sums || (n > 0 && !symbols)) return fail(h, TIC_ERR_INVALID, "bad arguments");
  TIC_CUDA(h, cudaSetDevice(h->device));
  const uint8_t* dsym = symbols;
  unsigned long long* dsum = (unsigned long long*)sums;
  CallTemps t{h};
  if (mem == TIC_MEM_HOST) {
    int rc = grow(h, &t.buf[0], 1, (size_t)std::max<int64_t>(1, n * npos));
    if (rc == TIC_OK) rc = grow(h, &t.buf[1], 1, (size_t)npos * 8);
    if (rc != TIC_OK) return rc;
    dsym = t.buf[0].as<uint8_t>();
    dsum = t.buf[1].as<unsigned long long>();
    TIC_CUDA(h, cudaMemcpyAsync(t.buf[0].p, symbols, (size_t)(n * npos), cudaMemcpyHostToDevice, h->stream));
    TIC_CUDA(h, cudaMemcpyAsync(dsum, sums, (size_t)npos * 8, cudaMemcpyHostToDevice, h->stream));
  }
  position_sums_kernel<<<(unsigned)((npos + 255) / 256), 256, 0, h->stream>>>(dsym, n, npos, dsum);
  h->launches++;
  TIC_CUDA(h, cudaGetLastError());
  if (mem == TIC_MEM_HOST) {
    TIC_CUDA(h, cudaMemcpyAsync(sums, dsum, (size_t)npos * 8, cudaMemcpyDeviceToHost, h->stream));
    TIC_CUDA(h, cudaStreamSynchronize(h->stream));
  }
  return TIC_OK;
}

int tic_position_sums_batched(tic_codec* h, const uint8_t* symbols, int64_t n, int64_t npos, int64_t batch, uint64_t* sums,
                              int mem) {
  if (!h) return TIC_ERR_INVALID;
  if (n < 0 || npos <= 0 || batch <= 0 || !sums || (n > 0 && !symbols)) return fail(h, TIC_ERR_INVALID, "bad arguments");
  const int64_t nb = (n + batch - 1) / batch;
  if (nb == 0) return TIC_OK;
  if (nb > 65535) return fail(h, TIC_ERR_INVALID, "too many batches (%lld)", (long long)nb);
  TIC_CUDA(h, cudaSetDevice(h->device));
  const uint8_t* dsym = symbols;
  unsigned long long* dsum = (unsigned long long*)sums;
  CallTemps t{h};
  if (mem == TIC_MEM_HOST) {
    int rc = grow(h, &t.buf[0], 1, (size_t)(n * npos));
    if (rc == TIC_OK) rc = grow(h, &t.buf[1], 1, (size_t)(nb * npos) * 8);
    if (rc != TIC_OK) return rc;
    dsym = t.buf[0].as<uint8_t>();
    dsum = t.buf[1].as<unsigned long long>();
    TIC_CUDA(h, cudaMemcpyAsync(t.buf[0].p, symbols, (size_t)(n * npos), cudaMemcpyHostToDevice, h->stream));
  }
  position_sums_batched_kernel<<<dim3((unsigned)((npos + 255) / 256), (unsigned)nb), 256, 0, h->stream>>>(dsym, n, npos, batch, dsum);
  h->launches++;
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess && mem == TIC_MEM_HOST)
    e = cudaMemcpyAsync(sums, dsum, (size_t)(nb * npos) * 8, cudaMemcpyDeviceToHost, h->stream);
  if (mem == TIC_MEM_HOST) cudaStreamSynchronize(h->stream);
  if (e != cudaSuccess) return fail(h, TIC_ERR_CUDA, "position sums failed: %s", cudaGetErrorString(e));
  return TIC_OK;
}

static int prof_collect(tic_codec* h) {
  for (auto& r : h->prof_pending) {
    float ms = 0.f;
    cudaEventSynchronize(r.e1);
    cudaEventElapsedTime(&ms, r.e0, r.e1);
    cudaEventDestroy(r.e0);
    cudaEventDestroy(r.e1);
    auto& v = h->prof_ms[r.graph];
    auto& c = h->prof_n[r.graph];
    if ((int)v.size() <= r.layer) {
      v.resize(r.layer + 1, 0.f);
      c.resize(r.layer + 1, 0);
    }
    v[r.layer] += ms;
    c[r.layer] += 1;
  }
  h->prof_pending.clear();
  return TIC_OK;
}

int tic_profile_enable(tic_codec* h, int on) {
  if (!h) return TIC_ERR_INVALID;
  h->profile = on != 0;
  return TIC_OK;
}

int tic_profile_reset(tic_codec* h) {
  if (!h) return TIC_ERR_INVALID;
  prof_collect(h);
  for (int g = 0; g < 3; ++g) {
    h->prof_ms[g].clear();
    h->prof_n[g].clear();
  }
  return TIC_OK;
}

int tic_profile_read(tic_codec* h, int graph, float* ms, int64_t* launches, int n_layers) {
  if (!h) return TIC_ERR_INVALID;
  if (graph < 0 || graph > 2 || !ms || !launches || n_layers <= 0) return fail(h, TIC_ERR_INVALID, "bad arguments");
  prof_collect(h);
  for (int i = 0; i < n_layers; ++i) {
    ms[i] = i < (int)h->prof_ms[graph].size() ? h->prof_ms[graph][i] : 0.f;
    launches[i] = i < (int)h->prof_n[graph].size() ? h->prof_n[graph][i] : 0;
  }
  return TIC_OK;
}

// ---- GPU entropy stage ------------------------------------------------------------------------
int64_t tic_entropy_bound(int64_t stream_len) { return (tic_rc_bound(stream_len < 0 ? 0 : stream_len) + 15) & ~(int64_t)15; }

static int entropy_table_check(tic_codec* h, const uint32_t* cum, int n_cum) {
  if (!cum || n_cum < 2 || n_cum - 1 > kEntropyMaxSymbols) return fail(h, TIC_ERR_INVALID, "entropy stage: tables of 1..256 symbols");
  if (cum[0] != 0) return fail(h, TIC_ERR_INVALID, "entropy stage: cumulative frequencies must start at 0");
  for (int i = 1; i < n_cum; ++i)
    if (cum[i] < cum[i - 1]) return fail(h, TIC_ERR_INVALID, "entropy stage: cumulative frequencies must not decrease");
  if (cum[n_cum - 1] == 0 || cum[n_cum - 1] > TIC_RC_MAX_TOTAL) return fail(h, TIC_ERR_INVALID, "entropy stage: frequency total must be in [1, 65536]");
  return TIC_OK;
}

static int entropy_table(tic_codec* h, const uint32_t* cum, int n_cum) {
  int rc = entropy_table_check(h, cum, n_cum);
  if (rc != TIC_OK) return rc;
  TIC_CUDA(h, cudaMemcpyAsync(h->d_cum, cum, (size_t)n_cum * sizeof(uint32_t), cudaMemcpyHostToDevice, h->stream));
  return TIC_OK;
}

// Scratch of `pieces` worst-case segment slots and their stored lengths.
static int ensure_seg_scratch(tic_codec* h, int64_t pieces) {
  const int rc = grow(h, &h->d_seg, 1, (size_t)(pieces * kEntropySegSlot));
  return rc != TIC_OK ? rc : grow(h, &h->d_seg_bytes, 1, (size_t)pieces * sizeof(long long));
}

int tic_entropy_encode(tic_codec* h, const uint8_t* symbols, int64_t n_streams, int64_t stream_len, const uint32_t* cum_freq,
                       int n_cum, uint8_t* out, int64_t out_stride, int64_t* out_bytes, int mem) {
  if (!h) return TIC_ERR_INVALID;
  if (n_streams < 0 || stream_len < 0 || out_stride < 0 || (n_streams > 0 && (!symbols || !out || !out_bytes)))
    return fail(h, TIC_ERR_INVALID, "bad arguments");
  if (n_streams == 0) return TIC_OK;
  if (n_streams > 0x7fffffffLL) return fail(h, TIC_ERR_INVALID, "too many streams");
  TIC_CUDA(h, cudaSetDevice(h->device));
  if (int st = overflow_status(h)) return st;
  int rc = entropy_table(h, cum_freq, n_cum);
  if (rc != TIC_OK) return rc;
  const uint8_t* dsym = symbols;
  uint8_t* dout = out;
  long long* dbytes = reinterpret_cast<long long*>(out_bytes);
  CallTemps t{h};
  if (mem == TIC_MEM_HOST) {
    rc = grow(h, &t.buf[0], 1, (size_t)std::max<int64_t>(16, n_streams * stream_len));
    if (rc == TIC_OK) rc = grow(h, &t.buf[1], 1, (size_t)std::max<int64_t>(16, n_streams * out_stride));
    if (rc == TIC_OK) rc = grow(h, &t.buf[2], 1, (size_t)n_streams * 8);
    if (rc != TIC_OK) return rc;
    TIC_CUDA(h, cudaMemcpyAsync(t.buf[0].p, symbols, (size_t)(n_streams * stream_len), cudaMemcpyHostToDevice, h->stream));
    dsym = t.buf[0].as<uint8_t>();
    dout = t.buf[1].as<uint8_t>();
    dbytes = t.buf[2].as<long long>();
  }
  const int64_t nseg = tic_rc_segments(stream_len);
  if (nseg > 0x7fffffffLL / std::max<int64_t>(1, n_streams)) return fail(h, TIC_ERR_INVALID, "too many segments");
  if (nseg > 0 && (rc = ensure_seg_scratch(h, n_streams * nseg)) != TIC_OK) return rc;
  TIC_CUDA(h, cudaEventRecord(h->ev_t0, h->stream));
  if (nseg == 0) {
    rc_encode_kernel<<<(unsigned)n_streams, 32, 0, h->stream>>>(dsym, stream_len, stream_len, 1, h->d_cum, n_cum, dout, out_stride, dbytes,
                                                                  h->d_oflow + 1);
    h->launches++;
  } else {
    rc_encode_kernel<<<(unsigned)(n_streams * nseg), 32, 0, h->stream>>>(dsym, stream_len, TIC_RC_SEGMENT_SYMBOLS, (int)nseg, h->d_cum, n_cum,
                                                                           h->d_seg.as<uint8_t>(), kEntropySegSlot,
                                                                           h->d_seg_bytes.as<long long>(), h->d_oflow + 1);
    rc_pack_kernel<<<(unsigned)(n_streams * nseg), 256, 0, h->stream>>>(h->d_seg.as<uint8_t>(), h->d_seg_bytes.as<long long>(), (int)nseg,
                                                                        dout, out_stride, dbytes, h->d_oflow + 1);
    h->launches += 2;
  }
  cudaError_t e = cudaGetLastError();
  cudaEventRecord(h->ev_t1, h->stream);
  if (mem == TIC_MEM_HOST) {
    if (e == cudaSuccess) e = cudaMemcpyAsync(out_bytes, dbytes, (size_t)n_streams * 8, cudaMemcpyDeviceToHost, h->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    // only the stored bytes of every stream come back
    for (int64_t i = 0; e == cudaSuccess && i < n_streams; ++i)
      if (out_bytes[i] > 0)
        e = cudaMemcpyAsync(out + i * out_stride, dout + i * out_stride, (size_t)out_bytes[i], cudaMemcpyDeviceToHost, h->stream);
    cudaStreamSynchronize(h->stream);
    if (e != cudaSuccess) return fail(h, TIC_ERR_CUDA, "entropy encode failed: %s", cudaGetErrorString(e));
    return overflow_status(h);
  }
  if (e != cudaSuccess) return fail(h, TIC_ERR_CUDA, "entropy encode launch failed: %s", cudaGetErrorString(e));
  return TIC_OK;
}

int tic_entropy_decode(tic_codec* h, const uint8_t* in, int64_t n_streams, int64_t in_stride, const int64_t* in_bytes,
                       const uint32_t* cum_freq, int n_cum, uint8_t* symbols, int64_t stream_len, int mem) {
  if (!h) return TIC_ERR_INVALID;
  if (n_streams < 0 || stream_len < 0 || in_stride < 0 || (n_streams > 0 && (!symbols || !in || !in_bytes)))
    return fail(h, TIC_ERR_INVALID, "bad arguments");
  if (n_streams == 0) return TIC_OK;
  if (n_streams > 0x7fffffffLL) return fail(h, TIC_ERR_INVALID, "too many streams");
  if (in_stride % 16 != 0) return fail(h, TIC_ERR_INVALID, "entropy decode: in_stride must be a multiple of 16 bytes");
  TIC_CUDA(h, cudaSetDevice(h->device));
  if (int st = overflow_status(h)) return st;
  int rc = entropy_table(h, cum_freq, n_cum);
  if (rc != TIC_OK) return rc;
  const uint8_t* din = in;
  const long long* dbytes = reinterpret_cast<const long long*>(in_bytes);
  uint8_t* dsym = symbols;
  CallTemps t{h};
  if (mem == TIC_MEM_HOST) {
    for (int64_t i = 0; i < n_streams; ++i)
      if (in_bytes[i] < 0 || in_bytes[i] > in_stride)
        return fail(h, TIC_ERR_INVALID, "entropy decode: stream %lld has %lld bytes in a %lld-byte slot", (long long)i,
                    (long long)in_bytes[i], (long long)in_stride);
    rc = grow(h, &t.buf[0], 1, (size_t)std::max<int64_t>(16, n_streams * in_stride));
    if (rc == TIC_OK) rc = grow(h, &t.buf[1], 1, (size_t)n_streams * 8);
    if (rc == TIC_OK) rc = grow(h, &t.buf[2], 1, (size_t)std::max<int64_t>(16, n_streams * stream_len));
    if (rc != TIC_OK) return rc;
    for (int64_t i = 0; i < n_streams; ++i) {
      if (in_bytes[i] > 0)
        TIC_CUDA(h, cudaMemcpyAsync(t.buf[0].as<uint8_t>() + i * in_stride, in + i * in_stride, (size_t)in_bytes[i], cudaMemcpyHostToDevice, h->stream));
    }
    TIC_CUDA(h, cudaMemcpyAsync(t.buf[1].p, in_bytes, (size_t)n_streams * 8, cudaMemcpyHostToDevice, h->stream));
    din = t.buf[0].as<uint8_t>();
    dbytes = t.buf[1].as<long long>();
    dsym = t.buf[2].as<uint8_t>();
  } else if ((reinterpret_cast<uintptr_t>(in) & 15) != 0) {
    return fail(h, TIC_ERR_INVALID, "entropy decode: the stream buffer must be 16-byte aligned");
  }
  TIC_CUDA(h, cudaEventRecord(h->ev_t0, h->stream));
  const int64_t nseg = tic_rc_segments(stream_len);
  if (nseg > 0x7fffffffLL / n_streams) return fail(h, TIC_ERR_INVALID, "too many segments");
  rc_decode_kernel<<<(unsigned)(n_streams * std::max<int64_t>(1, nseg)), 32, 0, h->stream>>>(din, in_stride, dbytes, h->d_cum, n_cum, dsym,
                                                                                                stream_len, (int)nseg);
  h->launches++;
  cudaError_t e = cudaGetLastError();
  cudaEventRecord(h->ev_t1, h->stream);
  if (mem == TIC_MEM_HOST) {
    if (e == cudaSuccess) e = cudaMemcpyAsync(symbols, dsym, (size_t)(n_streams * stream_len), cudaMemcpyDeviceToHost, h->stream);
    cudaStreamSynchronize(h->stream);
  }
  if (e != cudaSuccess) return fail(h, TIC_ERR_CUDA, "entropy decode failed: %s", cudaGetErrorString(e));
  return TIC_OK;
}

// ---- rate-distortion evaluation -----------------------------------------------------------------
int tic_evaluate_images(tic_codec* h, const uint8_t* images, int64_t n_images, int H, int W, int P, const uint32_t* cum_freq,
                        int n_cum, int64_t* code_bytes, uint64_t* sq_err, uint8_t* recon, int mem) {
  if (!h) return TIC_ERR_INVALID;
  if (n_images < 0 || H <= 0 || W <= 0 || P <= 0 || (n_images > 0 && (!images || !code_bytes || !sq_err)))
    return fail(h, TIC_ERR_INVALID, "bad arguments");
  ImageShapes s;
  if (int rc = image_shapes(h, H, W, P, true, true, &s)) return rc;
  if (int rc = entropy_table_check(h, cum_freq, n_cum)) return rc;
  if (n_images == 0) return TIC_OK;
  TIC_CUDA(h, cudaSetDevice(h->device));
  const bool host = mem != TIC_MEM_DEVICE;
  const int ppi = s.ppi;
  const int64_t cap = std::max<int64_t>(1, patches_per_chunk(h, P) / ppi);
  const double p128 = (double)ppi * P * P / 16384.0;
  const std::vector<int64_t> sched = chunk_schedule(mem, n_images, cap, p128);
  const int64_t ipc = *std::max_element(sched.begin(), sched.end());
  const size_t img_unit = (size_t)H * W * 3;
  const int64_t stream_len = (int64_t)ppi * s.hb * s.wb * s.cb;  // one image's symbols: one range-coded stream
  const int64_t nseg = tic_rc_segments(stream_len);
  const int64_t npiece = std::max<int64_t>(1, nseg);
  // A piece (one segment, or one plain stream) is a serial chain: a coder launch takes about as long as one piece, however
  // few pieces it has (one launch per 4-image chunk of config 2 made the host-buffer call 2.5x slower, DESIGN.md §4.10).
  // So the range coder runs over the symbols of several chunks at once: they accumulate in the symbol workspace until at
  // least kCoderPieces pieces are pending (config 2: all 64 images, 1536 pieces, one launch) or the last chunk is encoded.
  constexpr int64_t kCoderPieces = 2048;
  const int64_t coder_imgs = (kCoderPieces + npiece - 1) / npiece;
  const int64_t sym_cap = std::min<int64_t>(n_images, coder_imgs - 1 + ipc);
  if (sym_cap * npiece > 0x7fffffffLL) return fail(h, TIC_ERR_INVALID, "too many segments");
  int rc = grow(h, h->stage_sym, 2, (size_t)sym_cap * stream_len);
  if (rc == TIC_OK && !host && !recon) rc = grow(h, h->stage_out, 2, (size_t)ipc * img_unit);  // the reconstruction's workspace
  if (rc == TIC_OK && host) rc = grow(h, &h->d_eval, 1, (size_t)n_images * 2 * sizeof(long long));
  if (rc == TIC_OK) rc = ensure_seg_scratch(h, sym_cap * npiece);
  if (rc != TIC_OK) return rc;
  long long* d_bytes = host ? h->d_eval.as<long long>() : reinterpret_cast<long long*>(code_bytes);
  unsigned long long* d_sse = host ? reinterpret_cast<unsigned long long*>(d_bytes + n_images) : reinterpret_cast<unsigned long long*>(sq_err);
  // Per chunk, all on the handle's stream: encoder -> symbols -> decoder -> u8 reconstruction -> squared error against
  // the input still in place, then (see kCoderPieces) the range coder, stored lengths only, over the pending symbols.
  // With host buffers the next chunk's images may overwrite this one's after the squared error, and the reconstruction
  // (when asked for) goes back from then on.  Only n_images * 16 bytes of results come back.
  // The table and the zeroed squared errors go first on the stream: they overlap the first chunk's H2D.  Nothing is
  // queued for a handle that is already in error.
  if (int st = overflow_status(h)) return st;
  if ((rc = entropy_table(h, cum_freq, n_cum)) != TIC_OK) return rc;
  TIC_CUDA(h, cudaMemsetAsync(d_sse, 0, (size_t)n_images * sizeof(unsigned long long), h->stream));
  int64_t p0 = 0;  // images [p0, c.u0) are encoded and wait for the range coder
  return drive(h, mem, images, img_unit, {{recon, img_unit, h->stage_out, true}}, n_images, cap, [&](Chunk& c) {
    uint8_t* rec = (uint8_t*)c.out[0];
    int64_t rec0 = c.off;
    if (!rec) {  // device buffers, no reconstruction asked for
      rec = h->stage_out[0].as<uint8_t>();
      rec0 = 0;
    }
    uint8_t* sym = h->stage_sym[0].as<uint8_t>() + (size_t)(c.u0 - p0) * stream_len;
    IoSpec i, o;
    i.mode = IO_U8_NORM;
    i.in = c.in;
    i.geo = image_geo(H, W, P, c.off * ppi);
    o.mode = IO_QUANT_U8;
    o.out = sym;
    o.geo = image_geo(H, W, P, 0);
    if (int rc2 = run_graph(h, TIC_GRAPH_ENCODER, i, o, (int)(c.nu * ppi), P, P)) return rc2;
    IoSpec di, dout;
    di.mode = IO_U8_SYMLUT;
    di.in = sym;
    di.geo = image_geo(H, W, P, 0);
    dout.mode = IO_DENORM_U8;
    dout.out = rec;
    dout.geo = image_geo(H, W, P, rec0 * ppi);
    if (int rc2 = run_graph(h, TIC_GRAPH_DECODER, di, dout, (int)(c.nu * ppi), s.hb, s.wb)) return rc2;
    // enough blocks to keep every SM streaming (8 per SM over the chunk), at least 2048 16-byte loads each
    const int64_t nvec = (int64_t)(img_unit + 15) / 16;
    const int parts = (int)std::max<int64_t>(1, std::min<int64_t>((nvec + 2047) / 2048, (8LL * h->num_sms + c.nu - 1) / c.nu));
    sse_u8_kernel<<<(unsigned)(c.nu * parts), kSseThreads, 0, h->stream>>>((const uint8_t*)c.in + (size_t)c.off * img_unit,
                                                                           rec + (size_t)rec0 * img_unit, (long long)img_unit, parts,
                                                                           d_sse + c.u0);
    h->launches++;
    TIC_CUDA(h, cudaGetLastError());
    if (int rc2 = mark_consumed(c)) return rc2;
    const int64_t pend = c.u0 + c.nu - p0;
    if (pend >= coder_imgs || c.last) {
      // the stored length of each image's stream, exactly tic_entropy_encode's out_bytes: plain streams report it
      // directly, segmented ones through their segment lengths.  The next chunk's encoder overwrites the symbols
      // after these kernels in stream order.
      const uint8_t* s0 = h->stage_sym[0].as<uint8_t>();
      if (nseg == 0) {
        rc_encode_kernel<<<(unsigned)pend, 32, 0, h->stream>>>(s0, stream_len, stream_len, 1, h->d_cum, n_cum, h->d_seg.as<uint8_t>(),
                                                               kEntropySegSlot, d_bytes + p0, h->d_oflow + 1);
        h->launches++;
      } else {
        rc_encode_kernel<<<(unsigned)(pend * nseg), 32, 0, h->stream>>>(s0, stream_len, TIC_RC_SEGMENT_SYMBOLS, (int)nseg, h->d_cum, n_cum,
                                                                        h->d_seg.as<uint8_t>(), kEntropySegSlot,
                                                                        h->d_seg_bytes.as<long long>(), h->d_oflow + 1);
        rc_stored_length_kernel<<<(unsigned)pend, 256, 0, h->stream>>>(h->d_seg_bytes.as<long long>(), (int)nseg, d_bytes + p0);
        h->launches += 2;
      }
      TIC_CUDA(h, cudaGetLastError());
      p0 = c.u0 + c.nu;
    }
    if (c.last && host) {
      TIC_CUDA(h, cudaMemcpyAsync(code_bytes, d_bytes, (size_t)n_images * sizeof(int64_t), cudaMemcpyDeviceToHost, h->stream));
      TIC_CUDA(h, cudaMemcpyAsync(sq_err, d_sse, (size_t)n_images * sizeof(uint64_t), cudaMemcpyDeviceToHost, h->stream));
    }
    return (int)TIC_OK;
  }, p128);
}

#ifdef TIC_ABLATE
// ablation builds only (tools/fused_waits.py): the fused kernels' wait-time counters of cluster 0
extern "C" int tic_debug_prof_read(unsigned long long* out64, int reset) {
  if (cudaDeviceSynchronize() != cudaSuccess) return -1;
  if (out64 && cudaMemcpyFromSymbol(out64, g_tic_prof, sizeof(unsigned long long) * 64) != cudaSuccess) return -1;
  if (reset) {
    unsigned long long z[64] = {};
    if (cudaMemcpyToSymbol(g_tic_prof, z, sizeof(z)) != cudaSuccess) return -1;
  }
  return 0;
}
#endif

int tic_check_status(tic_codec* h) {
  if (!h) return TIC_ERR_INVALID;
  TIC_CUDA(h, cudaSetDevice(h->device));
  TIC_CUDA(h, cudaStreamSynchronize(h->stream));
  return overflow_status(h);
}

uint32_t tic_crc32c(const void* data, uint64_t n) {
  static uint32_t table[8][256];
  static const bool ready = [] {
    for (uint32_t i = 0; i < 256; ++i) {
      uint32_t c = i;
      for (int k = 0; k < 8; ++k) c = (c >> 1) ^ (0x82F63B78u & (0u - (c & 1u)));
      table[0][i] = c;
    }
    for (uint32_t i = 0; i < 256; ++i)
      for (int t = 1; t < 8; ++t) table[t][i] = (table[t - 1][i] >> 8) ^ table[0][table[t - 1][i] & 0xffu];
    return true;
  }();
  (void)ready;
  const uint8_t* p = static_cast<const uint8_t*>(data);
  uint32_t c = 0xffffffffu;
  while (n >= 8) {  // slicing-by-8
    uint32_t lo, hi;
    memcpy(&lo, p, 4);
    memcpy(&hi, p + 4, 4);
    lo ^= c;
    c = table[7][lo & 0xffu] ^ table[6][(lo >> 8) & 0xffu] ^ table[5][(lo >> 16) & 0xffu] ^ table[4][lo >> 24] ^
        table[3][hi & 0xffu] ^ table[2][(hi >> 8) & 0xffu] ^ table[1][(hi >> 16) & 0xffu] ^ table[0][hi >> 24];
    p += 8;
    n -= 8;
  }
  while (n--) c = (c >> 8) ^ table[0][(c ^ *p++) & 0xffu];
  return c ^ 0xffffffffu;
}

int64_t tic_launch_count(const tic_codec* h) { return h ? h->launches : 0; }

float tic_last_kernel_ms(const tic_codec* h) {
  if (!h) return 0.f;
  float ms = 0.f;
  if (cudaEventSynchronize(h->ev_t1) != cudaSuccess) return -1.f;
  if (cudaEventElapsedTime(&ms, h->ev_t0, h->ev_t1) != cudaSuccess) return -1.f;
  return ms;
}

}  // extern "C"

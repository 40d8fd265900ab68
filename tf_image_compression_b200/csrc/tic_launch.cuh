// Host-side plumbing the tensor-path launchers share: tensor maps of the three layouts they read and write, launches
// with dynamic shared memory, device buffers and the operand images built from a layer's weights, and how a launcher
// reports a failure.
#pragma once
#include <cuda.h>
#include <cudaTypedefs.h>
#include <cuda_runtime.h>

#include <map>
#include <mutex>
#include <string>
#include <type_traits>
#include <utility>

#include "../../include/tic.h"
#include "tic_common.cuh"

namespace tic {

// What a launcher needs from its handle: the stream, the SM count, where a failure's message goes and the handle's
// launch count (one per compute kernel; the operand-image builders are not counted).
struct LaunchCtx {
  cudaStream_t stream;
  int num_sms;
  std::string* err;
  int64_t* launches;
  tic_status fail(const std::string& what, tic_status code) const {
    if (err) *err = what;
    return code;
  }
};

// ---- tensor maps -------------------------------------------------------------------------------
inline PFN_cuTensorMapEncodeTiled_v12000 tmap_encode_fn(std::string* err) {
  static const PFN_cuTensorMapEncodeTiled_v12000 fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    const bool ok = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
                    q == cudaDriverEntryPointSuccess;
    return ok ? reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(p) : nullptr;
  }();
  if (!fn && err) *err = "cuTensorMapEncodeTiled is unavailable (driver too old?)";
  return fn;
}

inline tic_status tmap_status(CUresult r, const char* what, std::string* err) {
  if (r == CUDA_SUCCESS) return TIC_OK;
  if (err)
    *err = std::string("cuTensorMapEncodeTiled") + (what ? std::string(" (") + what + ")" : "") + " failed (" + std::to_string((int)r) + ")";
  return TIC_ERR_CUDA;
}

// A conv kernel's input: the NHWC activation of `a` at `base` (fp32, or one fp16 pair plane) as boxes
// {c, w, n, h} of the dims (C, W, N, H); with s2 the stride-2 parity view ((w parity, C), W/2, h parity, N, H/2) and
// boxes {c, w, 2, n, h}.
inline tic_status tmap_act(CUtensorMap* tm, const void* base, bool f16, const LayerArgs& a, bool s2, const cuuint32_t (&box)[4],
                           CUtensorMapSwizzle sw, std::string* err) {
  auto encode = tmap_encode_fn(err);
  if (!encode) return TIC_ERR_CUDA;
  const cuuint64_t C = a.cin, W = a.win, H = a.hin, N = a.n, e = f16 ? 2 : 4;
  const cuuint64_t dims4[4] = {C, W, N, H}, strides4[3] = {C * e, H * W * C * e, W * C * e};
  const cuuint64_t dims5[5] = {2 * C, W / 2, 2, N, H / 2}, strides5[4] = {2 * C * e, W * C * e, H * W * C * e, 2 * W * C * e};
  const cuuint32_t box5[5] = {box[0], box[1], 2, box[2], box[3]}, es[5] = {1, 1, 1, 1, 1};
  return tmap_status(encode(tm, f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, s2 ? 5 : 4,
                            const_cast<void*>(base), s2 ? dims5 : dims4, s2 ? strides5 : strides4, s2 ? box5 : box, es,
                            CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE),
                     nullptr, err);
}

// One fp16 plane of a pair-plane output [N, H, W, C] (C = 16 | 32) stored by TMA: dims (C, W, H, N), one box per
// epilogue warp of 4 rows x 8 columns.
inline tic_status tmap_pair_out(CUtensorMap* tm, void* base, int N, int H, int W, int C, const char* what, std::string* err) {
  auto encode = tmap_encode_fn(err);
  if (!encode) return TIC_ERR_CUDA;
  const cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
  const cuuint64_t strides[3] = {dims[0] * 2, dims[1] * dims[0] * 2, dims[2] * dims[1] * dims[0] * 2};
  const cuuint32_t box[4] = {(cuuint32_t)C, 8, 4, 1}, es[4] = {1, 1, 1, 1};
  return tmap_status(encode(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, base, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                            C == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE),
                     what, err);
}

// The raw rows of the images a first layer's patches come from: [B, H, W * 3] u8 or f32, B = the images the patches of
// `a` reach, boxes of `rows` rows x `row` elements.
inline tic_status tmap_image_rows(CUtensorMap* tm, const LayerArgs& a, bool f32, cuuint32_t row, cuuint32_t rows, const char* what,
                                  std::string* err) {
  auto encode = tmap_encode_fn(err);
  if (!encode) return TIC_ERR_CUDA;
  const Geo& g = a.geo;
  const long long per_img = (long long)g.gh * g.gw;
  const cuuint64_t eb = f32 ? 4 : 1;
  const cuuint64_t dims[3] = {(cuuint64_t)g.W * 3, (cuuint64_t)g.H, (cuuint64_t)((g.n0 + a.n + per_img - 1) / per_img)};
  const cuuint64_t strides[2] = {(cuuint64_t)g.W * 3 * eb, (cuuint64_t)g.H * g.W * 3 * eb};
  const cuuint32_t box[3] = {row, rows, 1}, es[3] = {1, 1, 1};
  return tmap_status(encode(tm, f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, const_cast<void*>(a.in), dims,
                            strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                            CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE),
                     what, err);
}

// ---- launches ----------------------------------------------------------------------------------
// Launches kernel<<<grid, block, smem, stream>>>(args...) and returns cudaGetLastError().  Above the default 48 KB,
// cudaFuncAttributeMaxDynamicSharedMemorySize must be raised first.  It is a per-device attribute of each kernel, so
// the sizes already set are remembered per (kernel, device), under a mutex because handles of different devices may
// launch from different threads.
template <class... P, class... A>
cudaError_t launch_dyn(void (*kernel)(P...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, const A&... args) {
  if (smem > 48 * 1024) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    static std::mutex mu;
    static std::map<std::pair<const void*, int>, size_t> have;
    std::lock_guard<std::mutex> lock(mu);
    size_t& set = have[{reinterpret_cast<const void*>(kernel), dev}];
    if (smem > set) {
      e = cudaFuncSetAttribute(reinterpret_cast<const void*>(kernel), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      if (e != cudaSuccess) return e;
      set = smem;
    }
  }
  kernel<<<grid, block, smem, stream>>>(args...);
  return cudaGetLastError();
}

// ---- device memory -----------------------------------------------------------------------------
// A device allocation with one owner: it frees the memory when reset or destroyed.
struct DevBuf {
  void* p = nullptr;
  size_t bytes = 0;
  DevBuf() = default;
  DevBuf(DevBuf&& o) noexcept : p(std::exchange(o.p, nullptr)), bytes(std::exchange(o.bytes, 0)) {}
  DevBuf& operator=(DevBuf&&) = delete;
  ~DevBuf() { cudaFree(p); }
  void reset() {
    cudaFree(p);
    p = nullptr;
    bytes = 0;
  }
  template <typename T>
  T* as() const { return static_cast<T*>(p); }
};

// The bytes of a builder kernel's arguments (all but its output): what an operand image was built from.
template <class... A>
std::string image_key(const A&... args) {
  static_assert((std::is_trivially_copyable<A>::value && ...), "operand-image keys are raw argument bytes");
  std::string k;
  (k.append(reinterpret_cast<const char*>(&args), sizeof(A)), ...);
  return k;
}

// A layer's weights laid out as one kernel's operand tiles, and the builder arguments they were made with.
struct OperandImage {
  DevBuf buf;
  std::string key;  // empty: nothing built
  const uint8_t* img() const { return buf.as<const uint8_t>(); }
  // TIC_OK with *build = false when the image holds `k`; otherwise it holds `bytes` of device memory and *build = true: the
  // caller launches the builder into it.  An image rebuilt in place is rewritten in stream order, behind the launches
  // that still read it.  TIC_ERR_NOMEM when the allocation fails.
  tic_status ensure(const std::string& k, size_t bytes, bool* build) {
    *build = false;
    if (buf.p && k == key && buf.bytes == bytes) return TIC_OK;
    key.clear();
    if (buf.bytes != bytes) {
      buf.reset();
      if (cudaMalloc(&buf.p, bytes) != cudaSuccess) {
        buf.p = nullptr;
        return TIC_ERR_NOMEM;
      }
      buf.bytes = bytes;
    }
    key = k;
    *build = true;
    return TIC_OK;
  }
  void release() {
    buf.reset();
    key.clear();
  }
};

}  // namespace tic

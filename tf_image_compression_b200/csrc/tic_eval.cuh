// Rate-distortion evaluation on the device (tic_evaluate_images): the distortion half of processing_utils/evaluate.py
// (:10-30) as exact integers.  The rate half is the entropy stage's stored length (rc_stored_length_kernel,
// tic_entropy.cuh).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace tic {

constexpr int kSseThreads = 256;

// sse[img] += sum over the img_bytes bytes of image img of (a - b)^2, for the images of `a` and `b` (both [n, img_bytes] u8,
// dense).  `parts` blocks share one image, block = img * parts + part.  Exact integer arithmetic: |a - b| per byte
// (vabsdiff4), squares summed four at a time by dp4a into a 32-bit partial of one 16-byte load (at most 16 * 255^2 =
// 1 040 400), that partial added to a 64-bit per-thread sum, then one 64-bit atomic per block.  HBM-bound: 16-byte loads
// when a and b share their alignment modulo 16 (always the case for the codec's own staging buffers), scalar loads for the
// unaligned head and tail, and for every byte otherwise.
__global__ void __launch_bounds__(kSseThreads) sse_u8_kernel(const uint8_t* __restrict__ a, const uint8_t* __restrict__ b, long long img_bytes,
                                                             int parts, unsigned long long* __restrict__ sse) {
  const long long img = blockIdx.x / parts;
  const int part = (int)(blockIdx.x - img * parts);
  const uint8_t* pa = a + img * img_bytes;
  const uint8_t* pb = b + img * img_bytes;
  const int mis = (int)(reinterpret_cast<uintptr_t>(pa) & 15);
  long long head = 0, nvec = 0;
  if (mis == (int)(reinterpret_cast<uintptr_t>(pb) & 15)) {
    head = (16 - mis) & 15;
    if (head > img_bytes) head = img_bytes;
    nvec = (img_bytes - head) >> 4;
  }
  const long long step = (long long)parts * kSseThreads;
  const long long first = (long long)part * kSseThreads + threadIdx.x;
  const uint4* va = reinterpret_cast<const uint4*>(pa + head);
  const uint4* vb = reinterpret_cast<const uint4*>(pb + head);
  unsigned long long acc = 0;
#pragma unroll 2
  for (long long v = first; v < nvec; v += step) {
    const uint4 x = __ldg(va + v), y = __ldg(vb + v);
    unsigned int d = __vabsdiffu4(x.x, y.x);
    unsigned int s = __dp4a(d, d, 0u);
    d = __vabsdiffu4(x.y, y.y);
    s = __dp4a(d, d, s);
    d = __vabsdiffu4(x.z, y.z);
    s = __dp4a(d, d, s);
    d = __vabsdiffu4(x.w, y.w);
    s = __dp4a(d, d, s);
    acc += s;
  }
  // bytes outside the 16-byte body: [0, head) and [tail0, img_bytes)
  const long long tail0 = head + 16 * nvec;
  const long long rest = head + (img_bytes - tail0);
  for (long long i = first; i < rest; i += step) {
    const long long k = i < head ? i : tail0 + (i - head);
    const int d = (int)pa[k] - (int)pb[k];
    acc += (unsigned int)(d * d);
  }
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, o);
  __shared__ unsigned long long s_part[kSseThreads / 32];
  if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long t = 0;
#pragma unroll
    for (int w = 0; w < kSseThreads / 32; ++w) t += s_part[w];
    if (t) atomicAdd(sse + img, t);
  }
}

}  // namespace tic

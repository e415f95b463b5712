// Device and host helpers shared by the kernel files.  The two numerical rules here -- torch's bilinear source index
// and the K3 sigmoid threshold -- are what the parity claims of DESIGN.md section 2 rest on, so each has exactly one
// definition.
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stddef.h>

namespace cgg {

// ATen upsample_bilinear2d (F.interpolate, align_corners=False) along one axis: source taps i0 / i1 and their weights
// l0 / l1 for output index dst, with scale = (float)in_size / (float)out_size.  src = scale (dst + 0.5) - 0.5 clamped
// at 0; a 2-D value is h0 (w0 a + w1 b) + h1 (w0 c + w1 d) in that operation order.
struct BilinearAxis { int i0, i1; float l0, l1; };
__device__ __forceinline__ BilinearAxis bilinear_src(float scale, int dst, int in_size) {
  float src = scale * ((float)dst + 0.5f) - 0.5f;
  if (src < 0.f) src = 0.f;
  BilinearAxis a;
  a.i0 = (int)src;
  if (a.i0 > in_size - 1) a.i0 = in_size - 1;
  a.i1 = a.i0 + ((a.i0 < in_size - 1) ? 1 : 0);
  a.l1 = src - (float)a.i0;
  a.l0 = 1.f - a.l1;
  return a;
}

// torch's fp32 sigmoid, IEEE expf and division (no fast math)
__device__ __forceinline__ float sigmoid_f32(float x) { return 1.0f / (1.0f + expf(-x)); }

// K3 attention-mask bit: torch's sigmoid(x) < 0.5 in fp32.  Not a sign test: it holds exactly for x <= MASKED_LOGIT_MAX
// (SURVEY.md section 7.2).  The fp32 route evaluates the sigmoid; the tcgen05 epilogue (gemm_tc.cu) compares with the
// constant.
constexpr float MASKED_LOGIT_MAX = -1.7881392e-07f;
__device__ __forceinline__ bool masked_from_logit(float x) { return sigmoid_f32(x) < 0.5f; }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

inline int round_up(int x, int m) { return (x + m - 1) / m * m; }
inline size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

}  // namespace cgg

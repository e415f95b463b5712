// Kernels of the step BEFORE the decoder-head path (SURVEY.md section 8 row f3): mmdet's MSDeformAttnPixelDecoder
// (configs/instance/coco_b48n17.py:38-70, called at open_set/models/mask2former_head.py:787) on TOKEN-MAJOR fp32
// activations (B, pixels, C) -- the layout every GEMM of the encoder wants (k contiguous) and the one in which a
// deformable-attention tap is one contiguous 128-byte read per head.
//
//   ms_deform_attn_{fwd,bwd}_kernel   mmcv MultiScaleDeformableAttention core (softmax over levels x points, bilinear taps
//                                     with zero padding, align_corners=False); HBM/L2-bound gather, no tensor cores
//   gn_*_kernel                       GroupNorm(32) of mmcv's ConvModule over (pixels x channels-of-a-group) per image,
//                                     forward (+ReLU) and backward, deterministic two-stage reductions
//   upsample_add_*_kernel             FPN top-down step: lateral + bilinear(align_corners=False) upsample of the coarser map
//   tokens_to_nchw / nchw_to_tokens   layout change at the boundary (the decoder head consumes NCHW memories)
//
// The contractions (1x1 convs, the 3x3 output conv as an implicit GEMM over 9 taps, every linear layer of the encoder) are
// calls of cgg_gemm_f32 (gemm_tf32.cu: tcgen05 kind::tf32 fed by TMA, zero-filled out-of-bounds taps; kernels_f32.cu in the
// fp32 parity mode).
#include "common.cuh"
#include "kernels.h"
#include <math.h>

namespace cgg {
namespace {

constexpr int MAX_LEVELS = 4;

struct MsdaP {
  int B, S, heads, levels, points;     // head_dim fixed at 32 (8 lanes x float4)
  int h[MAX_LEVELS], w[MAX_LEVELS], start[MAX_LEVELS];
  int pw[MAX_LEVELS], pstart[MAX_LEVELS + 1];   // 8x8-query patches per level row / first patch of the level
  int vs, os, ls;                      // forward: elements between consecutive tokens of value / offsets / logits
};

__device__ __forceinline__ float group8_sum(float v) {
  v += __shfl_xor_sync(0xffffffffu, v, 1);
  v += __shfl_xor_sync(0xffffffffu, v, 2);
  v += __shfl_xor_sync(0xffffffffu, v, 4);
  return v;
}

__device__ __forceinline__ float dot4(const float4& a, const float4& b) { return a.x * b.x + a.y * b.y + a.z * b.z + a.w * b.w; }
__device__ __forceinline__ float4 fma4(float s, const float4& a, const float4& c) {
  return make_float4(fmaf(s, a.x, c.x), fmaf(s, a.y, c.y), fmaf(s, a.z, c.z), fmaf(s, a.w, c.w));
}

// One thread = (image, query, head, 4 channels); 8 consecutive lanes share a (query, head).  A CTA is an 8x8 patch of
// queries of one level x ONE head: its 64 x levels x points x 4 taps fall into a window of a few pixels around the patch in
// each level, so most of them hit L1 (the query-major mapping of mmcv's op re-fetches every tap from L2: 17 GB per layer
// at 16 x 1024^2).
// value (B, S, heads*32); off (B, S, heads*levels*points*2) as (x, y) pixel offsets; logits (B, S, heads*levels*points).
// Reference point of query s at level-local (y, x): ((x + 0.5) / w, (y + 0.5) / h) -- the same for every level
// (valid ratios are one).  Sampling location in level l: ref + off / (w_l, h_l); pixel = loc * size - 0.5.
template <bool BWD>
__global__ void __launch_bounds__(512) ms_deform_attn_kernel(const MsdaP p, const float* __restrict__ value,
                                                             const float* __restrict__ off, const float* __restrict__ logits,
                                                             float* __restrict__ out, const float* __restrict__ dout,
                                                             float* __restrict__ dvalue, float* __restrict__ doff,
                                                             float* __restrict__ dlogits) {
  // (level geometry through static selects, blockIdx as (head, patch, image): see the forward kernel below)
  auto geom = [&](int l, int& H, int& W, int& start) {
    H = p.h[0]; W = p.w[0]; start = p.start[0];
#pragma unroll
    for (int q = 1; q < MAX_LEVELS; ++q)
      if (l == q) { H = p.h[q]; W = p.w[q]; start = p.start[q]; }
  };
  const int C = p.heads * 32;
  const int head = blockIdx.x, b = blockIdx.z;
  int pl = blockIdx.y, ql = 0, pfirst = 0, pwq = p.pw[0];
#pragma unroll
  for (int l = 1; l < MAX_LEVELS; ++l)
    if (l < p.levels && pl >= p.pstart[l]) { ql = l; pfirst = p.pstart[l]; pwq = p.pw[l]; }
  pl -= pfirst;
  int Hq, Wq, startq;
  geom(ql, Hq, Wq, startq);
  const int qi = threadIdx.x >> 3, c4 = (threadIdx.x & 7) * 4;
  const int qy = (pl / pwq) * 8 + (qi >> 3), qx = (pl % pwq) * 8 + (qi & 7);
  const bool valid = qy < Hq && qx < Wq;
  const int s = startq + (valid ? qy * Wq + qx : 0);
  const long tq = (long)b * p.S + s;
  const float ref_x = ((float)qx + 0.5f) / (float)Wq;
  const float ref_y = ((float)qy + 0.5f) / (float)Hq;
  const int LP = p.levels * p.points;                                // <= 16
  const float* lg = logits + ((long)tq * p.heads + head) * LP;
  const float* of = off + ((long)tq * p.heads + head) * LP * 2;
  float aw[16];
  float mx = -INFINITY;
#pragma unroll
  for (int i = 0; i < 16; ++i)
    if (i < LP) { aw[i] = lg[i]; mx = fmaxf(mx, aw[i]); }
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < 16; ++i)
    if (i < LP) { aw[i] = expf(aw[i] - mx); sum += aw[i]; }
  const float inv = 1.0f / sum;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
  if (BWD && valid) g = *reinterpret_cast<const float4*>(dout + (long)tq * C + head * 32 + c4);
  float daw[16];
  float dot_aw = 0.f;
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    if (i >= LP) continue;
    const int l = (i >= p.points) + (i >= 2 * p.points) + (i >= 3 * p.points);
    const float a = aw[i] * inv;
    int H, W, startl;
    geom(l, H, W, startl);
    const float loc_x = ref_x + of[2 * i] / (float)W, loc_y = ref_y + of[2 * i + 1] / (float)H;
    const float wim = loc_x * (float)W - 0.5f, him = loc_y * (float)H - 0.5f;
    float dwx = 0.f, dwy = 0.f, dsample = 0.f;
    if (valid && him > -1.f && wim > -1.f && him < (float)H && wim < (float)W) {
      const int hl = (int)floorf(him), wl = (int)floorf(wim);
      const float lh = him - (float)hl, lw = wim - (float)wl, hh = 1.f - lh, hw = 1.f - lw;
      const float* vb = value + ((long)b * p.S + startl) * C + head * 32 + c4;
      float* gb = BWD ? dvalue + ((long)b * p.S + startl) * C + head * 32 + c4 : nullptr;
      const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
      const bool t0 = hl >= 0, t1 = hl + 1 <= H - 1, l0 = wl >= 0, l1 = wl + 1 <= W - 1;
      const long o1 = ((long)hl * W + wl) * C, o2 = o1 + C, o3 = o1 + (long)W * C, o4 = o3 + C;
      const float4 v1 = (t0 && l0) ? *reinterpret_cast<const float4*>(vb + o1) : z;
      const float4 v2 = (t0 && l1) ? *reinterpret_cast<const float4*>(vb + o2) : z;
      const float4 v3 = (t1 && l0) ? *reinterpret_cast<const float4*>(vb + o3) : z;
      const float4 v4 = (t1 && l1) ? *reinterpret_cast<const float4*>(vb + o4) : z;
      const float w1 = hh * hw, w2 = hh * lw, w3 = lh * hw, w4 = lh * lw;
      if (!BWD) {
        float4 sm = make_float4(w1 * v1.x + w2 * v2.x + w3 * v3.x + w4 * v4.x, w1 * v1.y + w2 * v2.y + w3 * v3.y + w4 * v4.y,
                                w1 * v1.z + w2 * v2.z + w3 * v3.z + w4 * v4.z, w1 * v1.w + w2 * v2.w + w3 * v3.w + w4 * v4.w);
        acc = fma4(a, sm, acc);
      } else {
        const float d1 = dot4(g, v1), d2 = dot4(g, v2), d3 = dot4(g, v3), d4 = dot4(g, v4);
        dsample = w1 * d1 + w2 * d2 + w3 * d3 + w4 * d4;
        dwx = a * (-hh * d1 + hh * d2 - lh * d3 + lh * d4);        // d / d(pixel x); d pixel / d offset = 1
        dwy = a * (-hw * d1 - lw * d2 + hw * d3 + lw * d4);
        const float4 ga = make_float4(a * g.x, a * g.y, a * g.z, a * g.w);
        if (t0 && l0) atomicAdd(reinterpret_cast<float4*>(gb + o1), make_float4(w1 * ga.x, w1 * ga.y, w1 * ga.z, w1 * ga.w));
        if (t0 && l1) atomicAdd(reinterpret_cast<float4*>(gb + o2), make_float4(w2 * ga.x, w2 * ga.y, w2 * ga.z, w2 * ga.w));
        if (t1 && l0) atomicAdd(reinterpret_cast<float4*>(gb + o3), make_float4(w3 * ga.x, w3 * ga.y, w3 * ga.z, w3 * ga.w));
        if (t1 && l1) atomicAdd(reinterpret_cast<float4*>(gb + o4), make_float4(w4 * ga.x, w4 * ga.y, w4 * ga.z, w4 * ga.w));
      }
    }
    if (BWD) {
      dwx = group8_sum(dwx); dwy = group8_sum(dwy); dsample = group8_sum(dsample);
      daw[i] = dsample;
      dot_aw += a * dsample;
      if (valid && (threadIdx.x & 7) == 0) {
        float* dof = doff + ((long)tq * p.heads + head) * LP * 2;
        dof[2 * i] = dwx; dof[2 * i + 1] = dwy;
      }
    }
  }
  if (!BWD) {
    if (valid) *reinterpret_cast<float4*>(out + (long)tq * C + head * 32 + c4) = acc;
  } else if (valid && (threadIdx.x & 7) == 0) {
    float* dl = dlogits + ((long)tq * p.heads + head) * LP;
#pragma unroll
    for (int i = 0; i < 16; ++i)
      if (i < LP) dl[i] = aw[i] * inv * (daw[i] - dot_aw);
  }
}

// Forward, inference form.  Same CTA = (8x8 query patch of one level) x (one head), 512 threads, but in two phases:
//  1. lane j of a (query, head) group prepares points j and j + 8: softmax weight, the four tap offsets (elements from the
//     head's value base) and the four tap weights a * bilinear (0 for taps outside the level) -> shared memory, 8 words per
//     point.  The coordinate arithmetic is done once per point instead of once per lane.
//  2. every lane walks the group's levels*points*4 (offset, weight) pairs -- branch-free: one LDS.64, one LDG.128, four FMAs
//     per tap, so the compiler keeps many independent loads in flight (the one-phase form was latency-bound: 16 warps per
//     SM each waiting on a load -> coordinates -> four loads chain per point).
__global__ void __launch_bounds__(512, 2) ms_deform_attn_fwd_kernel(const MsdaP p, const float* __restrict__ value,
                                                                    const float* __restrict__ off, const float* __restrict__ logits,
                                                                    float* __restrict__ out) {
  __shared__ int2 taps[64][16 * 4 + 1];          // (element offset, weight bits) per (query, point, tap); rows padded: the 4 groups of a warp read different banks
  // (level geometry is picked with static selects: a kernel parameter indexed by a run-time level is an indexed
  // constant load, and those -- the ADU pipe -- were the busiest unit of the first version)
  auto geom = [&](int l, int& H, int& W, int& start) {
    H = p.h[0]; W = p.w[0]; start = p.start[0];
#pragma unroll
    for (int q = 1; q < MAX_LEVELS; ++q)
      if (l == q) { H = p.h[q]; W = p.w[q]; start = p.start[q]; }
  };
  const int C = p.heads * 32;
  const int head = blockIdx.x, b = blockIdx.z;
  int pl = blockIdx.y, ql = 0, pfirst = 0, pwq = p.pw[0];
#pragma unroll
  for (int l = 1; l < MAX_LEVELS; ++l)
    if (l < p.levels && pl >= p.pstart[l]) { ql = l; pfirst = p.pstart[l]; pwq = p.pw[l]; }
  pl -= pfirst;
  int Hq, Wq, startq;
  geom(ql, Hq, Wq, startq);
  const int qi = threadIdx.x >> 3, j = threadIdx.x & 7;
  const int qy = (pl / pwq) * 8 + (qi >> 3), qx = (pl % pwq) * 8 + (qi & 7);
  const bool valid = qy < Hq && qx < Wq;
  const int s = startq + (valid ? qy * Wq + qx : 0);
  const long tq = (long)b * p.S + s;
  const float ref_x = ((float)qx + 0.5f) / (float)Wq;
  const float ref_y = ((float)qy + 0.5f) / (float)Hq;
  const int LP = p.levels * p.points;                                // <= 16
  const float* lg = logits + (long)tq * p.ls + head * LP;
  const float2* of = reinterpret_cast<const float2*>(off + (long)tq * p.os + head * LP * 2);
  // ---- phase 1: this lane's points j and j + 8
  float e[2];
  float2 o[2];
  float mx = -INFINITY;
#pragma unroll
  for (int t = 0; t < 2; ++t) {
    const int i = j + 8 * t;
    e[t] = i < LP ? lg[i] : -INFINITY;
    o[t] = i < LP ? of[i] : make_float2(0.f, 0.f);
    mx = fmaxf(mx, e[t]);
  }
  mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
  mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
  mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 4));
  float sum = 0.f;
#pragma unroll
  for (int t = 0; t < 2; ++t) { e[t] = (j + 8 * t) < LP ? expf(e[t] - mx) : 0.f; sum += e[t]; }
  sum = group8_sum(sum);
  const float inv = 1.0f / sum;
#pragma unroll
  for (int t = 0; t < 2; ++t) {
    const int i = j + 8 * t;
    if (i >= LP) continue;
    const int l = (i >= p.points) + (i >= 2 * p.points) + (i >= 3 * p.points);
    const float a = e[t] * inv;
    int H, W, startl;
    geom(l, H, W, startl);
    const float loc_x = ref_x + o[t].x / (float)W, loc_y = ref_y + o[t].y / (float)H;
    const float wim = loc_x * (float)W - 0.5f, him = loc_y * (float)H - 0.5f;
    const bool inside = valid && him > -1.f && wim > -1.f && him < (float)H && wim < (float)W;
    const int hl = (int)floorf(him), wl = (int)floorf(wim);
    const float lh = him - (float)hl, lw = wim - (float)wl, hh = 1.f - lh, hw = 1.f - lw;
    const bool t0 = inside && hl >= 0, t1 = inside && hl + 1 <= H - 1, l0 = wl >= 0, l1 = wl + 1 <= W - 1;
    const int base = (startl + hl * W + wl) * p.vs;                 // (< 2^31 elements per image: checked by the launcher)
    int2* dst = &taps[qi][i * 4];
    dst[0] = make_int2((t0 && l0) ? base : 0, __float_as_int((t0 && l0) ? a * hh * hw : 0.f));
    dst[1] = make_int2((t0 && l1) ? base + p.vs : 0, __float_as_int((t0 && l1) ? a * hh * lw : 0.f));
    dst[2] = make_int2((t1 && l0) ? base + W * p.vs : 0, __float_as_int((t1 && l0) ? a * lh * hw : 0.f));
    dst[3] = make_int2((t1 && l1) ? base + W * p.vs + p.vs : 0, __float_as_int((t1 && l1) ? a * lh * lw : 0.f));
  }
  __syncwarp();
  // ---- phase 2
  const float* vb = value + (long)b * p.S * p.vs + head * 32 + j * 4;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  const int n = LP * 4;
#pragma unroll 8
  for (int i = 0; i < n; ++i) {
    const int2 tw = taps[qi][i];
    const float4 v = __ldg(reinterpret_cast<const float4*>(vb + tw.x));
    acc = fma4(__int_as_float(tw.y), v, acc);
  }
  if (valid) *reinterpret_cast<float4*>(out + (long)tq * C + head * 32 + j * 4) = acc;
}

// ------------------------------------------------------------------------------------------------ GroupNorm
// x (B, P, C) token-major; groups of cpg = C / G consecutive channels; statistics over P x cpg per (image, group).
// Stage 1: per (image, row chunk) channel sums -> partial[b][chunk][C][2]; stage 2 re-reduces them in a fixed order (double).
constexpr int GN_ROWS = 256;        // rows per stage-1 block

__global__ void __launch_bounds__(256) gn_partial_kernel(const float* __restrict__ x, const float* __restrict__ x2, int mode,
                                                         const float* __restrict__ mean_rstd, int G,
                                                         float* __restrict__ partial, int P, int C, int chunks) {
  // mode 0: (sum x, sum x^2);  mode 1 (backward): x = dy (already ReLU-masked), x2 = input: (sum dy, sum dy * xhat)
  __shared__ float red[2][256];
  const int b = blockIdx.y, chunk = blockIdx.x;
  const int r0 = chunk * GN_ROWS, r1 = min(P, r0 + GN_ROWS);
  const int nvec = C >> 2;                       // float4 columns per row
  const int rows_per_pass = 256 / nvec > 0 ? 256 / nvec : 1;
  for (int cv0 = 0; cv0 < nvec; cv0 += 256) {    // (C <= 1024: one pass)
    const int cv = cv0 + (threadIdx.x % (nvec < 256 ? nvec : 256));
    const int rsub = threadIdx.x / (nvec < 256 ? nvec : 256);
    float4 s1 = make_float4(0.f, 0.f, 0.f, 0.f), s2 = s1;
    float mu = 0.f, rs = 1.f;
    if (mode == 1 && cv < nvec) {
      const int g = (cv * 4) / (C / G);
      mu = mean_rstd[((long)b * G + g) * 2]; rs = mean_rstd[((long)b * G + g) * 2 + 1];
    }
    if (cv < nvec && rsub < rows_per_pass)
      for (int r = r0 + rsub; r < r1; r += rows_per_pass) {
        const float4 v = *reinterpret_cast<const float4*>(x + ((long)b * P + r) * C + cv * 4);
        if (mode == 0) {
          s1.x += v.x; s1.y += v.y; s1.z += v.z; s1.w += v.w;
          s2.x = fmaf(v.x, v.x, s2.x); s2.y = fmaf(v.y, v.y, s2.y); s2.z = fmaf(v.z, v.z, s2.z); s2.w = fmaf(v.w, v.w, s2.w);
        } else {
          const float4 u = *reinterpret_cast<const float4*>(x2 + ((long)b * P + r) * C + cv * 4);
          s1.x += v.x; s1.y += v.y; s1.z += v.z; s1.w += v.w;
          s2.x = fmaf(v.x, (u.x - mu) * rs, s2.x); s2.y = fmaf(v.y, (u.y - mu) * rs, s2.y);
          s2.z = fmaf(v.z, (u.z - mu) * rs, s2.z); s2.w = fmaf(v.w, (u.w - mu) * rs, s2.w);
        }
      }
    // fold the row sub-groups (fixed order) through shared memory, one float4 component at a time
    const float a1[4] = {s1.x, s1.y, s1.z, s1.w}, a2[4] = {s2.x, s2.y, s2.z, s2.w};
    for (int comp = 0; comp < 4; ++comp) {
      red[0][threadIdx.x] = a1[comp]; red[1][threadIdx.x] = a2[comp];
      __syncthreads();
      if (rsub == 0 && cv < nvec) {
        float t1 = 0.f, t2 = 0.f;
        const int stride = nvec < 256 ? nvec : 256;
        for (int q = 0; q < rows_per_pass; ++q) { t1 += red[0][threadIdx.x + q * stride]; t2 += red[1][threadIdx.x + q * stride]; }
        float* o = partial + (((long)b * chunks + chunk) * C + cv * 4 + comp) * 2;
        o[0] = t1; o[1] = t2;
      }
      __syncthreads();
    }
  }
}

// mean / rstd per (image, group) from the stage-1 channel sums: one warp per group, lanes stride over the row chunks,
// fixed-order tree over the lanes (deterministic), double accumulation
__global__ void gn_finish_kernel(const float* __restrict__ partial, float* __restrict__ mean_rstd, int P, int C, int G, int chunks,
                                 float eps) {
  const int b = blockIdx.x, lane = threadIdx.x & 31;
  const int cpg = C / G;
  for (int g = threadIdx.x >> 5; g < G; g += blockDim.x >> 5) {
    double s1 = 0.0, s2 = 0.0;
    for (int ch = lane; ch < chunks; ch += 32)
      for (int c = g * cpg; c < (g + 1) * cpg; ++c) {
        const float* o = partial + (((long)b * chunks + ch) * C + c) * 2;
        s1 += (double)o[0]; s2 += (double)o[1];
      }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      s1 += __shfl_xor_sync(0xffffffffu, s1, o);
      s2 += __shfl_xor_sync(0xffffffffu, s2, o);
    }
    if (lane == 0) {
      const double n = (double)P * cpg, mu = s1 / n;
      double var = s2 / n - mu * mu;
      if (var < 0.0) var = 0.0;
      mean_rstd[((long)b * G + g) * 2] = (float)mu;
      mean_rstd[((long)b * G + g) * 2 + 1] = (float)(1.0 / sqrt(var + (double)eps));
    }
  }
}

__global__ void __launch_bounds__(256) gn_apply_kernel(const float* __restrict__ x, const float* __restrict__ mean_rstd,
                                                       const float* __restrict__ gamma, const float* __restrict__ beta,
                                                       float* __restrict__ y, long total4, int P, int C, int G, int relu) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total4) return;
  const int nvec = C >> 2;
  const int cv = (int)(i % nvec);
  const long row = i / nvec;
  const int b = (int)(row / P);
  const int g = (cv * 4) / (C / G);
  const float mu = mean_rstd[((long)b * G + g) * 2], rs = mean_rstd[((long)b * G + g) * 2 + 1];
  const float4 v = reinterpret_cast<const float4*>(x)[i];
  const float4 ga = reinterpret_cast<const float4*>(gamma)[cv], be = reinterpret_cast<const float4*>(beta)[cv];
  float4 o = make_float4((v.x - mu) * rs * ga.x + be.x, (v.y - mu) * rs * ga.y + be.y, (v.z - mu) * rs * ga.z + be.z,
                         (v.w - mu) * rs * ga.w + be.w);
  if (relu) { o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f); }
  reinterpret_cast<float4*>(y)[i] = o;
}

// backward, stage 2: per (image, channel) sums over the chunks -> chan[b][C][2]; per (image, group): s1 = sum_c gamma_c * sum dy,
// s2 = sum_c gamma_c * sum dy*xhat -> gsum[b][G][2]
__global__ void gn_bwd_finish_kernel(const float* __restrict__ partial, const float* __restrict__ gamma, float* __restrict__ chan,
                                     float* __restrict__ gsum, int C, int G, int chunks) {
  extern __shared__ double sh[];          // 2 * C
  const int b = blockIdx.x;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    double s1 = 0.0, s2 = 0.0;
    for (int ch = 0; ch < chunks; ++ch) {
      const float* o = partial + (((long)b * chunks + ch) * C + c) * 2;
      s1 += (double)o[0]; s2 += (double)o[1];
    }
    chan[((long)b * C + c) * 2] = (float)s1; chan[((long)b * C + c) * 2 + 1] = (float)s2;
    sh[2 * c] = s1 * (double)gamma[c]; sh[2 * c + 1] = s2 * (double)gamma[c];
  }
  __syncthreads();
  const int cpg = C / G;
  for (int g = threadIdx.x; g < G; g += blockDim.x) {
    double s1 = 0.0, s2 = 0.0;
    for (int c = g * cpg; c < (g + 1) * cpg; ++c) { s1 += sh[2 * c]; s2 += sh[2 * c + 1]; }
    gsum[((long)b * G + g) * 2] = (float)s1; gsum[((long)b * G + g) * 2 + 1] = (float)s2;
  }
}

// dgamma[c] = sum_b chan[b][c][1], dbeta[c] = sum_b chan[b][c][0]
__global__ void gn_bwd_params_kernel(const float* __restrict__ chan, float* __restrict__ dgamma, float* __restrict__ dbeta, int B,
                                     int C) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  float s1 = 0.f, s2 = 0.f;
  for (int b = 0; b < B; ++b) { s1 += chan[((long)b * C + c) * 2]; s2 += chan[((long)b * C + c) * 2 + 1]; }
  dbeta[c] = s1; dgamma[c] = s2;
}

// dx = rstd * (dy*gamma - s1/n - xhat * s2/n)
__global__ void __launch_bounds__(256) gn_bwd_apply_kernel(const float* __restrict__ x, const float* __restrict__ dy,
                                                           const float* __restrict__ mean_rstd, const float* __restrict__ gsum,
                                                           const float* __restrict__ gamma, float* __restrict__ dx, long total4,
                                                           int P, int C, int G) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total4) return;
  const int nvec = C >> 2;
  const int cv = (int)(i % nvec);
  const long row = i / nvec;
  const int b = (int)(row / P);
  const int g = (cv * 4) / (C / G);
  const float mu = mean_rstd[((long)b * G + g) * 2], rs = mean_rstd[((long)b * G + g) * 2 + 1];
  const float invn = 1.0f / ((float)P * (float)(C / G));
  const float m1 = gsum[((long)b * G + g) * 2] * invn, m2 = gsum[((long)b * G + g) * 2 + 1] * invn;
  const float4 v = reinterpret_cast<const float4*>(x)[i], d = reinterpret_cast<const float4*>(dy)[i];
  const float4 ga = reinterpret_cast<const float4*>(gamma)[cv];
  float4 o;
  o.x = rs * (d.x * ga.x - m1 - (v.x - mu) * rs * m2);
  o.y = rs * (d.y * ga.y - m1 - (v.y - mu) * rs * m2);
  o.z = rs * (d.z * ga.z - m1 - (v.z - mu) * rs * m2);
  o.w = rs * (d.w * ga.w - m1 - (v.w - mu) * rs * m2);
  reinterpret_cast<float4*>(dx)[i] = o;
}

// ------------------------------------------------------------------------------------- FPN top-down step
// out[b,y,x,:] = lat[b,y,x,:] + bilinear(prev[b,:,:,:])(y,x);  lat/out (B, H*W, C), prev (B, h*w, C) with batch stride pbs
__global__ void __launch_bounds__(256) upsample_add_kernel(const float* __restrict__ lat, const float* __restrict__ prev, long pbs,
                                                           float* __restrict__ out, long total4, int H, int W, int h, int w, int C) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total4) return;
  const int nvec = C >> 2;
  const int cv = (int)(i % nvec);
  long row = i / nvec;
  const int x = (int)(row % W); row /= W;
  const int y = (int)(row % H);
  const int b = (int)(row / H);
  const BilinearAxis ay = bilinear_src((float)h / (float)H, y, h), ax = bilinear_src((float)w / (float)W, x, w);
  const float* pb = prev + (long)b * pbs + cv * 4;
  const float4 v00 = *reinterpret_cast<const float4*>(pb + ((long)ay.i0 * w + ax.i0) * C);
  const float4 v01 = *reinterpret_cast<const float4*>(pb + ((long)ay.i0 * w + ax.i1) * C);
  const float4 v10 = *reinterpret_cast<const float4*>(pb + ((long)ay.i1 * w + ax.i0) * C);
  const float4 v11 = *reinterpret_cast<const float4*>(pb + ((long)ay.i1 * w + ax.i1) * C);
  const float4 l = reinterpret_cast<const float4*>(lat)[i];
  float4 o;
  o.x = l.x + (ay.l0 * (ax.l0 * v00.x + ax.l1 * v01.x) + ay.l1 * (ax.l0 * v10.x + ax.l1 * v11.x));
  o.y = l.y + (ay.l0 * (ax.l0 * v00.y + ax.l1 * v01.y) + ay.l1 * (ax.l0 * v10.y + ax.l1 * v11.y));
  o.z = l.z + (ay.l0 * (ax.l0 * v00.z + ax.l1 * v01.z) + ay.l1 * (ax.l0 * v10.z + ax.l1 * v11.z));
  o.w = l.w + (ay.l0 * (ax.l0 * v00.w + ax.l1 * v01.w) + ay.l1 * (ax.l0 * v10.w + ax.l1 * v11.w));
  reinterpret_cast<float4*>(out)[i] = o;
}

// adjoint of the upsample: dprev (B, h*w, C) (zeroed by the caller) += scatter of dout (B, H*W, C)
__global__ void __launch_bounds__(256) upsample_add_bwd_kernel(const float* __restrict__ dout, float* __restrict__ dprev, long total4,
                                                               int H, int W, int h, int w, int C) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total4) return;
  const int nvec = C >> 2;
  const int cv = (int)(i % nvec);
  long row = i / nvec;
  const int x = (int)(row % W); row /= W;
  const int y = (int)(row % H);
  const int b = (int)(row / H);
  const BilinearAxis ay = bilinear_src((float)h / (float)H, y, h), ax = bilinear_src((float)w / (float)W, x, w);
  const float4 d = reinterpret_cast<const float4*>(dout)[i];
  float* pb = dprev + (long)b * h * w * C + cv * 4;
  auto add = [&](int yy, int xx, float wgt) {
    atomicAdd(reinterpret_cast<float4*>(pb + ((long)yy * w + xx) * C), make_float4(wgt * d.x, wgt * d.y, wgt * d.z, wgt * d.w));
  };
  add(ay.i0, ax.i0, ay.l0 * ax.l0); add(ay.i0, ax.i1, ay.l0 * ax.l1); add(ay.i1, ax.i0, ay.l1 * ax.l0); add(ay.i1, ax.i1, ay.l1 * ax.l1);
}

// ------------------------------------------------------------------------------------- layout changes
// in (B, P, C) rows with batch stride ibs (a level's slice of the token buffer) -> out (B, C, P), fp32 or bf16
template <typename OutT>
__global__ void __launch_bounds__(256) tokens_to_nchw_kernel(const float* __restrict__ in, long ibs, OutT* __restrict__ out, int P, int C) {
  __shared__ float tile[32][33];
  const int b = blockIdx.z, p0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int r = ty; r < 32; r += 8) {
    const int pp = p0 + r, c = c0 + tx;
    tile[r][tx] = (pp < P && c < C) ? in[(long)b * ibs + (long)pp * C + c] : 0.f;
  }
  __syncthreads();
  for (int r = ty; r < 32; r += 8) {
    const int c = c0 + r, pp = p0 + tx;
    if (c < C && pp < P) out[((long)b * C + c) * P + pp] = (OutT)tile[tx][r];
  }
}

// in (B, C, P) -> out (B, P, C) rows with batch stride obs; accumulate: out += in^T (a gradient joining the token buffer)
__global__ void __launch_bounds__(256) nchw_to_tokens_kernel(const float* __restrict__ in, float* __restrict__ out, long obs, int P, int C,
                                                             int accumulate) {
  __shared__ float tile[32][33];
  const int b = blockIdx.z, p0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int r = ty; r < 32; r += 8) {
    const int c = c0 + r, pp = p0 + tx;
    tile[r][tx] = (pp < P && c < C) ? in[((long)b * C + c) * P + pp] : 0.f;
  }
  __syncthreads();
  for (int r = ty; r < 32; r += 8) {
    const int pp = p0 + r, c = c0 + tx;
    if (pp < P && c < C) {
      float* o = out + (long)b * obs + (long)pp * C + c;
      *o = tile[tx][r] + (accumulate ? *o : 0.f);
    }
  }
}

}  // namespace

cudaError_t launch_ms_deform_attn(const float* value, long value_stride, const float* off, long off_stride, const float* logits,
                                  long logit_stride, float* out, int B, int S, int heads, int levels, int points, const int* hs,
                                  const int* ws, cudaStream_t s) {
  MsdaP p = {};
  p.vs = (int)value_stride; p.os = (int)off_stride; p.ls = (int)logit_stride;
  p.B = B; p.S = S; p.heads = heads; p.levels = levels; p.points = points;
  int st = 0, ps = 0;
  for (int l = 0; l < levels; ++l) {
    p.h[l] = hs[l]; p.w[l] = ws[l]; p.start[l] = st; st += hs[l] * ws[l];
    p.pw[l] = (ws[l] + 7) / 8; p.pstart[l] = ps; ps += p.pw[l] * ((hs[l] + 7) / 8);
  }
  p.pstart[levels] = ps;
  const long tq = (long)B * S;
  if (tq <= 0) return cudaSuccess;
  if ((long)S * value_stride > 0x7fffffffL) return cudaErrorInvalidValue;
  if (ps > 65535 || B > 65535) return cudaErrorInvalidValue;
  ms_deform_attn_fwd_kernel<<<dim3(heads, ps, B), 512, 0, s>>>(p, value, off, logits, out);
  count_launch();
  return cudaGetLastError();
}

cudaError_t launch_ms_deform_attn_bwd(const float* value, const float* off, const float* logits, const float* dout, float* dvalue,
                                      float* doff, float* dlogits, int B, int S, int heads, int levels, int points, const int* hs,
                                      const int* ws, cudaStream_t s) {
  MsdaP p = {};
  p.B = B; p.S = S; p.heads = heads; p.levels = levels; p.points = points;
  int st = 0, ps = 0;
  for (int l = 0; l < levels; ++l) {
    p.h[l] = hs[l]; p.w[l] = ws[l]; p.start[l] = st; st += hs[l] * ws[l];
    p.pw[l] = (ws[l] + 7) / 8; p.pstart[l] = ps; ps += p.pw[l] * ((hs[l] + 7) / 8);
  }
  p.pstart[levels] = ps;
  const long tq = (long)B * S;
  if (tq <= 0) return cudaSuccess;
  cudaError_t e = cudaMemsetAsync(dvalue, 0, (size_t)tq * heads * 32 * sizeof(float), s);
  if (e != cudaSuccess) return e;
  if (ps > 65535 || B > 65535) return cudaErrorInvalidValue;
  ms_deform_attn_kernel<true><<<dim3(heads, ps, B), 512, 0, s>>>(p, value, off, logits, nullptr, dout, dvalue, doff, dlogits);
  count_launch();
  return cudaGetLastError();
}

size_t group_norm_scratch_floats(int B, int P, int C, int G) {
  const int chunks = (P + GN_ROWS - 1) / GN_ROWS;
  return (size_t)B * chunks * C * 2 + (size_t)B * C * 2 + (size_t)B * G * 2;
}

cudaError_t launch_group_norm(const float* x, const float* gamma, const float* beta, float* y, float* mean_rstd, float* scratch, int B,
                              int P, int C, int G, float eps, bool relu, cudaStream_t s) {
  if (B <= 0 || P <= 0) return cudaSuccess;
  const int chunks = (P + GN_ROWS - 1) / GN_ROWS;
  gn_partial_kernel<<<dim3(chunks, B), 256, 0, s>>>(x, nullptr, 0, nullptr, G, scratch, P, C, chunks);
  gn_finish_kernel<<<B, 32 * (G < 32 ? G : 32), 0, s>>>(scratch, mean_rstd, P, C, G, chunks, eps);
  const long total4 = (long)B * P * (C / 4);
  gn_apply_kernel<<<(unsigned)((total4 + 255) / 256), 256, 0, s>>>(x, mean_rstd, gamma, beta, y, total4, P, C, G, relu ? 1 : 0);
  count_launch(3);
  return cudaGetLastError();
}

// dy must already carry the ReLU mask when the forward applied one
cudaError_t launch_group_norm_bwd(const float* x, const float* dy, const float* mean_rstd, const float* gamma, float* dx, float* dgamma,
                                  float* dbeta, float* scratch, int B, int P, int C, int G, cudaStream_t s) {
  if (B <= 0 || P <= 0) return cudaSuccess;
  const int chunks = (P + GN_ROWS - 1) / GN_ROWS;
  float* partial = scratch;
  float* chan = partial + (size_t)B * chunks * C * 2;
  float* gsum = chan + (size_t)B * C * 2;
  gn_partial_kernel<<<dim3(chunks, B), 256, 0, s>>>(dy, x, 1, mean_rstd, G, partial, P, C, chunks);
  gn_bwd_finish_kernel<<<B, 256, 2 * C * sizeof(double), s>>>(partial, gamma, chan, gsum, C, G, chunks);
  gn_bwd_params_kernel<<<(C + 255) / 256, 256, 0, s>>>(chan, dgamma, dbeta, B, C);
  const long total4 = (long)B * P * (C / 4);
  gn_bwd_apply_kernel<<<(unsigned)((total4 + 255) / 256), 256, 0, s>>>(x, dy, mean_rstd, gsum, gamma, dx, total4, P, C, G);
  count_launch(4);
  return cudaGetLastError();
}

cudaError_t launch_upsample_add(const float* lat, const float* prev, long prev_bstride, float* out, int B, int H, int W, int h, int w,
                                int C, cudaStream_t s) {
  const long total4 = (long)B * H * W * (C / 4);
  if (total4 <= 0) return cudaSuccess;
  upsample_add_kernel<<<(unsigned)((total4 + 255) / 256), 256, 0, s>>>(lat, prev, prev_bstride, out, total4, H, W, h, w, C);
  count_launch();
  return cudaGetLastError();
}

cudaError_t launch_upsample_add_bwd(const float* dout, float* dprev, int B, int H, int W, int h, int w, int C, cudaStream_t s) {
  const long total4 = (long)B * H * W * (C / 4);
  if (total4 <= 0) return cudaSuccess;
  cudaError_t e = cudaMemsetAsync(dprev, 0, (size_t)B * h * w * C * sizeof(float), s);
  if (e != cudaSuccess) return e;
  upsample_add_bwd_kernel<<<(unsigned)((total4 + 255) / 256), 256, 0, s>>>(dout, dprev, total4, H, W, h, w, C);
  count_launch();
  return cudaGetLastError();
}

cudaError_t launch_tokens_to_nchw(const float* in, long in_bstride, void* out, bool out_bf16, int B, int P, int C, cudaStream_t s) {
  if (B <= 0 || P <= 0) return cudaSuccess;
  dim3 grid((P + 31) / 32, (C + 31) / 32, B);
  if (out_bf16) tokens_to_nchw_kernel<__nv_bfloat16><<<grid, 256, 0, s>>>(in, in_bstride, (__nv_bfloat16*)out, P, C);
  else tokens_to_nchw_kernel<float><<<grid, 256, 0, s>>>(in, in_bstride, (float*)out, P, C);
  count_launch();
  return cudaGetLastError();
}

cudaError_t launch_nchw_to_tokens(const float* in, float* out, long out_bstride, int B, int P, int C, bool accumulate, cudaStream_t s) {
  if (B <= 0 || P <= 0) return cudaSuccess;
  dim3 grid((P + 31) / 32, (C + 31) / 32, B);
  nchw_to_tokens_kernel<<<grid, 256, 0, s>>>(in, out, out_bstride, P, C, accumulate ? 1 : 0);
  count_launch();
  return cudaGetLastError();
}

}  // namespace cgg

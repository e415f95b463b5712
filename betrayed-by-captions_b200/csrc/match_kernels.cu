// The step after the path at training time (SURVEY.md section 8 row f2): point sampling of mask logits / ground-truth
// masks, the Hungarian cost matrix, the point-sampled dice + BCE losses and the class-weighted cross entropy of
// `loss_single` (open_set/models/mask2former_head.py:464-629; targets :320-390; assigner
// open_set/assigners/mask_hungarian_assigner.py:98-125).  All fp32; HBM / latency bound gathers and reductions.
#include "common.cuh"
#include "kernels.h"

#include <math.h>

namespace cgg {
namespace {

// block-wide sum of up to 3 values (blockDim = 256); result valid in every thread
__device__ __forceinline__ void block_sum3(float& a, float& b, float& c, float (*sh)[3]) {
  a = warp_sum(a); b = warp_sum(b); c = warp_sum(c);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) { sh[warp][0] = a; sh[warp][1] = b; sh[warp][2] = c; }
  __syncthreads();
  a = b = c = 0.f;
  for (int i = 0; i < (int)(blockDim.x >> 5); ++i) { a += sh[i][0]; b += sh[i][1]; c += sh[i][2]; }
}

// ---- mmcv point_sample = F.grid_sample(input, 2 p - 1, bilinear, zeros padding, align_corners=False); index math and
// tap order of ATen's grid_sampler_2d kernel.  One thread per (plane, point).
struct Taps { int x0, y0; float nw, ne, sw, se; };
__device__ __forceinline__ Taps taps_of(float px, float py, int H, int W) {
  const float gx = 2.0f * px - 1.0f, gy = 2.0f * py - 1.0f;
  const float ix = ((gx + 1.f) * (float)W - 1.f) / 2.f, iy = ((gy + 1.f) * (float)H - 1.f) / 2.f;
  const float fx = floorf(ix), fy = floorf(iy);
  Taps t;
  t.x0 = (int)fx; t.y0 = (int)fy;
  const float ex = fx + 1.f, ey = fy + 1.f;
  t.nw = (ex - ix) * (ey - iy);
  t.ne = (ix - fx) * (ey - iy);
  t.sw = (ex - ix) * (iy - fy);
  t.se = (ix - fx) * (iy - fy);
  return t;
}
__global__ void __launch_bounds__(256) point_sample_kernel(const float* __restrict__ in, const float* __restrict__ coords,
                                                           float* __restrict__ out, int N, int H, int W, int P,
                                                           int coords_shared) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long)N * P) return;
  const int p = (int)(i % P);
  const long n = i / P;
  const float* c = coords + ((coords_shared ? 0 : n) * P + p) * 2;
  const Taps t = taps_of(c[0], c[1], H, W);
  const float* plane = in + n * H * W;
  const bool x0 = t.x0 >= 0 && t.x0 < W, x1 = t.x0 + 1 >= 0 && t.x0 + 1 < W;
  const bool y0 = t.y0 >= 0 && t.y0 < H, y1 = t.y0 + 1 >= 0 && t.y0 + 1 < H;
  float acc = 0.f;
  if (y0 && x0) acc += plane[(long)t.y0 * W + t.x0] * t.nw;
  if (y0 && x1) acc += plane[(long)t.y0 * W + t.x0 + 1] * t.ne;
  if (y1 && x0) acc += plane[(long)(t.y0 + 1) * W + t.x0] * t.sw;
  if (y1 && x1) acc += plane[(long)(t.y0 + 1) * W + t.x0 + 1] * t.se;
  out[i] = acc;
}
__global__ void __launch_bounds__(256) point_sample_bwd_kernel(const float* __restrict__ dout, const float* __restrict__ coords,
                                                               float* __restrict__ din, int N, int H, int W, int P,
                                                               int coords_shared) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long)N * P) return;
  const int p = (int)(i % P);
  const long n = i / P;
  const float* c = coords + ((coords_shared ? 0 : n) * P + p) * 2;
  const Taps t = taps_of(c[0], c[1], H, W);
  float* plane = din + n * H * W;
  const float g = dout[i];
  const bool x0 = t.x0 >= 0 && t.x0 < W, x1 = t.x0 + 1 >= 0 && t.x0 + 1 < W;
  const bool y0 = t.y0 >= 0 && t.y0 < H, y1 = t.y0 + 1 >= 0 && t.y0 + 1 < H;
  if (y0 && x0) atomicAdd(plane + (long)t.y0 * W + t.x0, g * t.nw);
  if (y0 && x1) atomicAdd(plane + (long)t.y0 * W + t.x0 + 1, g * t.ne);
  if (y1 && x0) atomicAdd(plane + (long)(t.y0 + 1) * W + t.x0, g * t.sw);
  if (y1 && x1) atomicAdd(plane + (long)(t.y0 + 1) * W + t.x0 + 1, g * t.se);
}

__device__ __forceinline__ float softplus_f(float x) { return fmaxf(x, 0.f) + log1pf(expf(-fabsf(x))); }

// ---- cost matrix, stage 1: per query row  sp = sum softplus(x), sg = sum sigmoid(x), log-sum-exp of the class rows;
// per ground-truth row  gs = sum g.   One CTA per row (rows 0..Q-1 queries, Q..Q+G-1 ground truths).
__global__ void __launch_bounds__(256) match_rowstats_kernel(const float* __restrict__ x, const float* __restrict__ g,
                                                             const float* __restrict__ cls, const float* __restrict__ emb,
                                                             int Q, int G, int C1, int P, float* __restrict__ stats) {
  __shared__ float sh[8][3];
  const int r = blockIdx.x, t = threadIdx.x;
  if (r < Q) {
    float sp = 0.f, sg = 0.f, z = 0.f;
    for (int p = t; p < P; p += 256) { const float v = x[(long)r * P + p]; sp += softplus_f(v); sg += sigmoid_f32(v); }
    block_sum3(sp, sg, z, sh);
    if (t == 0) { stats[r * 4 + 0] = sp; stats[r * 4 + 1] = sg; }
    if (t < 64) {                                            // warp 0: lse of cls, warp 1: lse of emb
      const float* row = (t < 32) ? cls : emb;
      const int lane = t & 31;
      if (row) {
        row += (long)r * C1;
        float m = -INFINITY;
        for (int c = lane; c < C1; c += 32) m = fmaxf(m, row[c]);
        m = warp_max(m);
        float s = 0.f;
        for (int c = lane; c < C1; c += 32) s += expf(row[c] - m);
        s = warp_sum(s);
        if (lane == 0) stats[r * 4 + (t < 32 ? 2 : 3)] = m + logf(s);
      }
    }
  } else {
    const int gi = r - Q;
    float gs = 0.f, z0 = 0.f, z1 = 0.f;
    for (int p = t; p < P; p += 256) gs += g[(long)gi * P + p];
    block_sum3(gs, z0, z1, sh);
    if (t == 0) stats[Q * 4 + gi] = gs;
  }
}
// stage 2: one warp per (query, ground truth):  x . g  and  sigmoid(x) . g, then the weighted sum of the four terms.
//   class terms  -softmax(row)[label]              (ClassificationCost)
//   mask term    (sum softplus(x) - x . g) / P     (CrossEntropyLossCost: BCE(x,1).g + BCE(x,0).(1-g) = softplus(x) - x g)
//   dice term    1 - (2 s.g + eps) / (sum s + sum g + eps)
__global__ void __launch_bounds__(256) match_pairs_kernel(const float* __restrict__ x, const float* __restrict__ g,
                                                          const float* __restrict__ cls, const float* __restrict__ emb,
                                                          const int64_t* __restrict__ labels, const float* __restrict__ stats,
                                                          int Q, int G, int C1, int P, float w_cls, float w_emb, float w_mask,
                                                          float w_dice, float eps, float* __restrict__ cost) {
  const long pair = (long)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (pair >= (long)Q * G) return;
  const int q = (int)(pair / G), gi = (int)(pair % G);
  const float* xr = x + (long)q * P;
  const float* gr = g + (long)gi * P;
  float xg = 0.f, sgd = 0.f;
  for (int p = lane; p < P; p += 32) {
    const float v = xr[p], t = gr[p];
    xg = fmaf(v, t, xg);
    sgd = fmaf(sigmoid_f32(v), t, sgd);
  }
  xg = warp_sum(xg);
  sgd = warp_sum(sgd);
  if (lane == 0) {
    const int64_t lab = labels[gi];
    float c = 0.f;
    if (w_cls != 0.f && cls) c += -expf(cls[(long)q * C1 + lab] - stats[q * 4 + 2]) * w_cls;
    if (w_emb != 0.f && emb) c += -expf(emb[(long)q * C1 + lab] - stats[q * 4 + 3]) * w_emb;
    if (w_mask != 0.f) c += (stats[q * 4 + 0] - xg) / (float)P * w_mask;
    if (w_dice != 0.f) c += (1.f - (2.f * sgd + eps) / (stats[q * 4 + 1] + stats[Q * 4 + gi] + eps)) * w_dice;
    cost[pair] = c;
  }
}

// ---- point-sampled dice + BCE: one CTA per matched mask row.
// out_rows[n] = (a, b, c) = (sum s t, sum s, sum t); dice_rows[n] = 1 - (2a + eps)/(b + c + eps); bce_rows[n] = sum BCE(x, t)
__global__ void __launch_bounds__(256) point_losses_kernel(const float* __restrict__ x, const float* __restrict__ t, int P,
                                                           float eps, float* __restrict__ abc, float* __restrict__ dice_rows,
                                                           float* __restrict__ bce_rows) {
  __shared__ float sh[8][3];
  const long n = blockIdx.x;
  float a = 0.f, b = 0.f, c = 0.f, e = 0.f;
  for (int p = threadIdx.x; p < P; p += 256) {
    const float v = x[n * P + p], tt = t[n * P + p];
    const float s = sigmoid_f32(v);
    a = fmaf(s, tt, a); b += s; c += tt;
    e += fmaxf(v, 0.f) - v * tt + log1pf(expf(-fabsf(v)));
  }
  block_sum3(a, b, c, sh);
  float z0 = 0.f, z1 = 0.f;
  block_sum3(e, z0, z1, sh);
  if (threadIdx.x == 0) {
    abc[n * 3 + 0] = a; abc[n * 3 + 1] = b; abc[n * 3 + 2] = c;
    dice_rows[n] = 1.f - (2.f * a + eps) / (b + c + eps);
    bce_rows[n] = e;
  }
}
// dx = g_dice[n] * d(1 - d_row)/dx + g_bce[n] * (s - t)   (per-row upstream gradients, device resident)
__global__ void __launch_bounds__(256) point_losses_bwd_kernel(const float* __restrict__ x, const float* __restrict__ t,
                                                               const float* __restrict__ abc, int P, float eps,
                                                               const float* __restrict__ g_dice_rows,
                                                               const float* __restrict__ g_bce_rows, float* __restrict__ dx) {
  const long n = blockIdx.y;
  const int p = blockIdx.x * 256 + threadIdx.x;
  if (p >= P) return;
  const float g_dice = g_dice_rows[n], g_bce = g_bce_rows[n];
  const float a = abc[n * 3], b = abc[n * 3 + 1], c = abc[n * 3 + 2];
  const float den = b + c + eps, num = 2.f * a + eps;
  const float v = x[n * P + p], tt = t[n * P + p];
  const float s = sigmoid_f32(v);
  const float dd_ds = (2.f * tt * den - num) / (den * den);      // d d_row / d s_p
  dx[n * P + p] = g_dice * (-dd_ds) * s * (1.f - s) + g_bce * (s - tt);
}

// ---- class-weighted cross entropy (F.cross_entropy(weight=class_weight, reduction='none') summed): one warp per row.
// row_loss[r] = w[label] (lse - x[label]); row_w[r] = w[label]; lse[r] kept for the backward.
__global__ void __launch_bounds__(256) weighted_ce_kernel(const float* __restrict__ logits, const int64_t* __restrict__ labels,
                                                          const float* __restrict__ cw, int R, int C1,
                                                          float* __restrict__ row_loss, float* __restrict__ row_w,
                                                          float* __restrict__ lse) {
  const int r = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (r >= R) return;
  const float* row = logits + (long)r * C1;
  float m = -INFINITY;
  for (int c = lane; c < C1; c += 32) m = fmaxf(m, row[c]);
  m = warp_max(m);
  float s = 0.f;
  for (int c = lane; c < C1; c += 32) s += expf(row[c] - m);
  s = warp_sum(s);
  if (lane == 0) {
    const int64_t lab = labels[r];
    const float l = m + logf(s), w = cw[lab];
    lse[r] = l;
    row_w[r] = w;
    row_loss[r] = w * (l - row[lab]);
  }
}
__global__ void __launch_bounds__(256) weighted_ce_bwd_kernel(const float* __restrict__ logits, const int64_t* __restrict__ labels,
                                                              const float* __restrict__ cw, const float* __restrict__ lse, int R,
                                                              int C1, const float* __restrict__ grow, float* __restrict__ dlogits) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long)R * C1) return;
  const int c = (int)(i % C1);
  const long r = i / C1;
  const int64_t lab = labels[r];
  dlogits[i] = grow[r] * cw[lab] * (expf(logits[i] - lse[r]) - (c == lab ? 1.f : 0.f));
}

}  // namespace

cudaError_t launch_point_sample(const float* in, const float* coords, float* out, int N, int H, int W, int P,
                                bool coords_shared, cudaStream_t s) {
  const long total = (long)N * P;
  if (total <= 0) return cudaSuccess;
  point_sample_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(in, coords, out, N, H, W, P, coords_shared ? 1 : 0);
  count_launch();
  return cudaGetLastError();
}
cudaError_t launch_point_sample_bwd(const float* dout, const float* coords, float* din, int N, int H, int W, int P,
                                    bool coords_shared, cudaStream_t s) {
  const long total = (long)N * P;
  if (N <= 0) return cudaSuccess;
  cudaError_t e = cudaMemsetAsync(din, 0, (size_t)N * H * W * sizeof(float), s);
  if (e != cudaSuccess || total <= 0) return e;
  point_sample_bwd_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(dout, coords, din, N, H, W, P, coords_shared ? 1 : 0);
  count_launch();
  return cudaGetLastError();
}
cudaError_t launch_matching_cost(const float* x, const float* g, const float* cls, const float* emb, const int64_t* labels,
                                 int Q, int G, int C1, int P, float w_cls, float w_emb, float w_mask, float w_dice, float eps,
                                 float* stats, float* cost, cudaStream_t s) {
  if (Q <= 0 || G <= 0) return cudaSuccess;
  match_rowstats_kernel<<<Q + G, 256, 0, s>>>(x, g, cls, emb, Q, G, C1, P, stats);
  const long pairs = (long)Q * G;
  match_pairs_kernel<<<(unsigned)((pairs + 7) / 8), 256, 0, s>>>(x, g, cls, emb, labels, stats, Q, G, C1, P, w_cls, w_emb,
                                                                 w_mask, w_dice, eps, cost);
  count_launch(2);
  return cudaGetLastError();
}
cudaError_t launch_point_losses(const float* x, const float* t, int N, int P, float eps, float* abc, float* dice_rows,
                                float* bce_rows, cudaStream_t s) {
  if (N <= 0) return cudaSuccess;
  point_losses_kernel<<<N, 256, 0, s>>>(x, t, P, eps, abc, dice_rows, bce_rows);
  count_launch();
  return cudaGetLastError();
}
cudaError_t launch_point_losses_bwd(const float* x, const float* t, const float* abc, int N, int P, float eps,
                                    const float* g_dice, const float* g_bce, float* dx, cudaStream_t s) {
  if (N <= 0 || P <= 0) return cudaSuccess;
  point_losses_bwd_kernel<<<dim3((P + 255) / 256, N), 256, 0, s>>>(x, t, abc, P, eps, g_dice, g_bce, dx);
  count_launch();
  return cudaGetLastError();
}
cudaError_t launch_weighted_ce(const float* logits, const int64_t* labels, const float* cw, int R, int C1, float* row_loss,
                               float* row_w, float* lse, cudaStream_t s) {
  if (R <= 0) return cudaSuccess;
  weighted_ce_kernel<<<(R + 7) / 8, 256, 0, s>>>(logits, labels, cw, R, C1, row_loss, row_w, lse);
  count_launch();
  return cudaGetLastError();
}
cudaError_t launch_weighted_ce_bwd(const float* logits, const int64_t* labels, const float* cw, const float* lse, int R, int C1,
                                   const float* grow, float* dlogits, cudaStream_t s) {
  const long total = (long)R * C1;
  if (total <= 0) return cudaSuccess;
  weighted_ce_bwd_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(logits, labels, cw, lse, R, C1, grow, dlogits);
  count_launch();
  return cudaGetLastError();
}

}  // namespace cgg

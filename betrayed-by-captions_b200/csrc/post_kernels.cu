// The step after the path at test time (SURVEY.md section 8f rank 1): final mask upsample + fusion-head scoring.
//   reference: simple_test upsamples the last head call's mask logits to the padded input size with
//   F.interpolate(bilinear, align_corners=False) (open_set/models/mask2former_head.py:957-964) -- 6.7 GB of fp32 per
//   16-image batch at 1024^2 -- and MaskFormerFusionHeadOpen then crops to img_shape, optionally resamples to ori_shape
//   (maskformer_fusion_head.py:412-425) and, per kept (query, class) pair, thresholds `> 0`, averages sigmoid over the
//   positive pixels and takes the bounding box (instance_postprocess_emb, :318-366; mmdet mask2bbox).
// instance_mask_stats_kernel does all of it in ONE pass that reads only the (B, Q, H/4, W/4) logits: the full-resolution
// logits are never written.  Both resampling stages follow ATen's upsample_bilinear2d index math and operation order
// (src = scale (dst + 0.5) - 0.5 clamped at 0; v = h0 (w0 a + w1 b) + h1 (w0 c + w1 d)), evaluated in fp32.
#include "common.cuh"
#include "kernels.h"
#include <cuda_bf16.h>
#include <limits.h>
#include <math.h>

namespace cgg {

namespace {

template <typename T> __device__ __forceinline__ float ldf(const T* p);
template <> __device__ __forceinline__ float ldf<float>(const float* p) { return __ldg(p); }
template <> __device__ __forceinline__ float ldf<__nv_bfloat16>(const __nv_bfloat16* p) { return __bfloat162float(*p); }

// value of the first-stage upsample (logits (h4, w4) -> (up_h, up_w)) at (y, x) given precomputed axes
template <typename T>
__device__ __forceinline__ float up1(const T* __restrict__ src, int w4, const BilinearAxis& ay, const BilinearAxis& ax) {
  const float a = ldf(src + (long)ay.i0 * w4 + ax.i0), b = ldf(src + (long)ay.i0 * w4 + ax.i1);
  const float c = ldf(src + (long)ay.i1 * w4 + ax.i0), d = ldf(src + (long)ay.i1 * w4 + ax.i1);
  return ay.l0 * (ax.l0 * a + ax.l1 * b) + ay.l1 * (ax.l0 * c + ax.l1 * d);
}

// value of the two-stage resample (logits -> (up_h, up_w) -> crop -> (out_h, out_w)) at an output pixel whose second-stage
// axes are (by, bx) and whose first-stage axes at the two source rows / columns are (ay0, ay1) / (ax0, ax1)
template <typename T>
__device__ __forceinline__ float up2(const T* __restrict__ src, int w4, const BilinearAxis& by, const BilinearAxis& ay0,
                                     const BilinearAxis& ay1, const BilinearAxis& bx, const BilinearAxis& ax0,
                                     const BilinearAxis& ax1) {
  const float a = up1(src, w4, ay0, ax0), bb = up1(src, w4, ay0, ax1);
  const float c = up1(src, w4, ay1, ax0), d = up1(src, w4, ay1, ax1);
  return by.l0 * (bx.l0 * a + bx.l1 * bb) + by.l1 * (bx.l0 * c + bx.l1 * d);
}

// materialised first stage: out (B*Q, up_h, up_w) fp32 = F.interpolate(logits, (up_h, up_w))   (head.py:957-964)
template <typename T>
__global__ void __launch_bounds__(256) upsample_kernel(const T* __restrict__ logits, float* __restrict__ out, int h4, int w4,
                                                       int up_h, int up_w) {
  const int x = blockIdx.x * 64 + (threadIdx.x & 63), y0 = (blockIdx.y * 4 + (threadIdx.x >> 6)) * 8;
  const long plane = blockIdx.z;
  if (x >= up_w) return;
  const float sy = (float)h4 / (float)up_h, sx = (float)w4 / (float)up_w;
  const BilinearAxis ax = bilinear_src(sx, x, w4);
  const T* src = logits + plane * (long)h4 * w4;
  for (int y = y0; y < y0 + 8 && y < up_h; ++y) {
    const BilinearAxis ay = bilinear_src(sy, y, h4);
    out[(plane * up_h + y) * (long)up_w + x] = up1(src, w4, ay, ax);
  }
}

// geom[b] = {crop_h, crop_w, out_h, out_w}: crop of the upsampled map (img_shape), final size (ori_shape when rescaling,
// else the crop).  One warp = one 32-pixel column strip over ROWS_PER_WARP output rows of one (image, query) plane.
constexpr int ROWS_PER_BLOCK = 64;
template <typename T>
__global__ void __launch_bounds__(256) instance_mask_stats_kernel(const T* __restrict__ logits, const int* __restrict__ geom,
                                                                  int Q, int h4, int w4, int up_h, int up_w,
                                                                  uint32_t* __restrict__ bits, long bits_plane, int bits_w32,
                                                                  int* __restrict__ count, float* __restrict__ sig_sum,
                                                                  int* __restrict__ bbox) {
  const int plane = blockIdx.z, b = plane / Q;
  const int crop_h = geom[4 * b], crop_w = geom[4 * b + 1], out_h = geom[4 * b + 2], out_w = geom[4 * b + 3];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int strip = blockIdx.x * 8 + warp, x = strip * 32 + lane;
  const int y_begin = blockIdx.y * ROWS_PER_BLOCK;
  if (strip * 32 >= out_w || y_begin >= out_h) return;
  const bool rescale = out_h != crop_h || out_w != crop_w;
  const float s1y = (float)h4 / (float)up_h, s1x = (float)w4 / (float)up_w;
  const float s2y = (float)crop_h / (float)out_h, s2x = (float)crop_w / (float)out_w;
  const bool x_ok = x < out_w;
  const int xc = x_ok ? x : out_w - 1;
  // x axes: second stage (out -> crop) and, for its two source columns, first stage (up -> logits)
  BilinearAxis bx = {xc, xc, 1.f, 0.f};
  if (rescale) bx = bilinear_src(s2x, xc, crop_w);
  const BilinearAxis ax0 = bilinear_src(s1x, bx.i0, w4), ax1 = bilinear_src(s1x, bx.i1, w4);
  const T* src = logits + (long)plane * h4 * w4;
  int cnt = 0, xmin = INT_MAX, xmax = -1, ymin = INT_MAX, ymax = -1;
  float ssum = 0.f;
  for (int y = y_begin; y < y_begin + ROWS_PER_BLOCK && y < out_h; ++y) {
    float v;
    if (rescale) {
      const BilinearAxis by = bilinear_src(s2y, y, crop_h);
      const BilinearAxis ay0 = bilinear_src(s1y, by.i0, h4), ay1 = bilinear_src(s1y, by.i1, h4);
      v = up2(src, w4, by, ay0, ay1, bx, ax0, ax1);
    } else {
      v = up1(src, w4, bilinear_src(s1y, y, h4), ax0);
    }
    const bool pos = x_ok && v > 0.f;
    const uint32_t word = __ballot_sync(0xffffffffu, pos);
    if (bits && lane == 0) bits[(long)plane * bits_plane + (long)y * bits_w32 + strip] = word;
    if (pos) {
      ++cnt;
      ssum += sigmoid_f32(v);
      xmin = min(xmin, x); xmax = max(xmax, x);
      ymin = min(ymin, y); ymax = max(ymax, y);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    ssum += __shfl_xor_sync(0xffffffffu, ssum, o);
    xmin = min(xmin, __shfl_xor_sync(0xffffffffu, xmin, o));
    xmax = max(xmax, __shfl_xor_sync(0xffffffffu, xmax, o));
    ymin = min(ymin, __shfl_xor_sync(0xffffffffu, ymin, o));
    ymax = max(ymax, __shfl_xor_sync(0xffffffffu, ymax, o));
  }
  if (lane == 0 && cnt > 0) {
    atomicAdd(count + plane, cnt);
    atomicAdd(sig_sum + plane, ssum);
    atomicMin(bbox + 4 * plane, xmin);
    atomicMin(bbox + 4 * plane + 1, ymin);
    atomicMax(bbox + 4 * plane + 2, xmax + 1);
    atomicMax(bbox + 4 * plane + 3, ymax + 1);
  }
}

__global__ void stats_init_kernel(int* count, float* sig_sum, int* bbox, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  count[i] = 0;
  sig_sum[i] = 0.f;
  bbox[4 * i] = INT_MAX; bbox[4 * i + 1] = INT_MAX; bbox[4 * i + 2] = 0; bbox[4 * i + 3] = 0;
}
// empty masks: mmdet mask2bbox leaves the box at zeros
__global__ void stats_finish_kernel(const int* count, int* bbox, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  if (count[i] == 0) { bbox[4 * i] = 0; bbox[4 * i + 1] = 0; }
}

// in-place softmax over rows of length n (get_cls_emb_scores, maskformer_fusion_head.py:297-315), one warp per row
__global__ void __launch_bounds__(256) softmax_rows_kernel(float* __restrict__ x, int rows, int n) {
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= rows) return;
  float* r = x + (long)row * n;
  float m = -INFINITY;
  for (int i = lane; i < n; i += 32) m = fmaxf(m, r[i]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  float s = 0.f;
  for (int i = lane; i < n; i += 32) s += expf(r[i] - m);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  for (int i = lane; i < n; i += 32) r[i] = expf(r[i] - m) / s;
}

// ---- panoptic fusion: mmdet 2.28.2 MaskFormerFusionHead.panoptic_postprocess on the class-embedding probabilities.
// Four launches, no host round trip: keep list -> fused pixel pass (winner + areas) -> per-image decision -> paint.
// Scratch (per image, Q entries each): kept query id, kept score, kept label, mask_area, original_area, segment value per
// kept index; then the kept count per image.
struct PanScratch {
  int *kept_q, *kept_label, *area_m, *area_o, *seg, *kept_count;
  float* kept_score;
};

__host__ __device__ inline PanScratch pan_scratch(void* base, int B, int Q) {
  int* p = static_cast<int*>(base);
  const long n = (long)B * Q;
  PanScratch s;
  s.kept_q = p; s.kept_label = p + n; s.area_m = p + 2 * n; s.area_o = p + 3 * n; s.seg = p + 4 * n;
  s.kept_score = reinterpret_cast<float*>(p + 5 * n);
  s.kept_count = p + 6 * n;
  return s;
}

constexpr int PAN_INSTANCE_OFFSET = 1000;
constexpr int PAN_FLAG = 1 << 30;      // pixel-pass code: winner's kept index | PAN_FLAG when the winner's sigmoid >= 0.5

// One CTA per image: scores, labels = probs.max(-1) (first index on ties); keep = label != C & score > fp32(thr); the kept
// query ids compacted in query order.  Also zeroes the area accumulators of the pixel pass.
__global__ void __launch_bounds__(256) pan_keep_kernel(const float* __restrict__ probs, int Q, int n_cls_p1, float thr,
                                                       PanScratch s) {
  extern __shared__ unsigned char pan_keep_smem[];
  float* s_score = reinterpret_cast<float*>(pan_keep_smem);
  int* s_label = reinterpret_cast<int*>(s_score + Q);
  const int b = blockIdx.x, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = threadIdx.x; i < Q; i += blockDim.x) { s.area_m[b * Q + i] = 0; s.area_o[b * Q + i] = 0; }
  for (int q = warp; q < Q; q += blockDim.x >> 5) {
    const float* r = probs + ((long)b * Q + q) * n_cls_p1;
    float best = -INFINITY;
    int arg = INT_MAX;
    for (int i = lane; i < n_cls_p1; i += 32) {
      const float v = r[i];
      if (v > best) { best = v; arg = i; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, best, o);
      const int oi = __shfl_xor_sync(0xffffffffu, arg, o);
      if (ov > best || (ov == best && oi < arg)) { best = ov; arg = oi; }
    }
    if (lane == 0) { s_score[q] = best; s_label[q] = arg; }
  }
  __syncthreads();
  if (warp != 0) return;
  int base = 0;
  for (int c = 0; c < Q; c += 32) {
    const int q = c + lane;
    const bool keep = q < Q && s_label[q] != n_cls_p1 - 1 && s_score[q] > thr;
    const unsigned m = __ballot_sync(0xffffffffu, keep);
    if (keep) {
      const int k = base + __popc(m & ((1u << lane) - 1u));
      s.kept_q[b * Q + k] = q;
      s.kept_score[b * Q + k] = s_score[q];
      s.kept_label[b * Q + k] = s_label[q];
    }
    base += __popc(m);
  }
  if (lane == 0) s.kept_count[b] = base;
}

// Fused pixel pass.  CTA = 32 x 32 output pixels of one image, thread = one column x 4 rows (8 apart).  The resample axes of
// a pixel are derived once; per kept query k the pixel's two-stage logit v, sigmoid(v) (torch's fp32 expression), the
// product score_k * sigmoid and the first-index argmax are evaluated.  Writes the code of the winner (kept index |
// PAN_FLAG if its sigmoid >= 0.5; -1 when nothing is kept) into pan, and accumulates mask_area[k] (winner histogram) and
// original_area[k] (#sigmoid_k >= 0.5) per CTA in shared memory, then one global atomic per (CTA, query) with a count.
constexpr int PAN_TILE = 32, PAN_ROWS = 4;
template <typename T>
__global__ void __launch_bounds__(256) pan_pixel_kernel(const T* __restrict__ logits, const int* __restrict__ geom, int Q,
                                                        int h4, int w4, int up_h, int up_w, int* __restrict__ pan,
                                                        int max_out_h, int max_out_w, PanScratch s) {
  extern __shared__ int pan_pix_smem[];
  const int b = blockIdx.z;
  const int crop_h = geom[4 * b], crop_w = geom[4 * b + 1], out_h = geom[4 * b + 2], out_w = geom[4 * b + 3];
  const int x0 = blockIdx.x * PAN_TILE, y0 = blockIdx.y * PAN_TILE;
  if (x0 >= out_w || y0 >= out_h) return;
  const int K = s.kept_count[b];
  int* s_m = pan_pix_smem;
  int* s_o = s_m + Q;
  int* s_q = s_o + Q;
  float* s_sc = reinterpret_cast<float*>(s_q + Q);
  for (int i = threadIdx.x; i < K; i += blockDim.x) {
    s_m[i] = 0; s_o[i] = 0;
    s_q[i] = s.kept_q[b * Q + i];
    s_sc[i] = s.kept_score[b * Q + i];
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const bool rescale = out_h != crop_h || out_w != crop_w;
  const float s1y = (float)h4 / (float)up_h, s1x = (float)w4 / (float)up_w;
  const float s2y = (float)crop_h / (float)out_h, s2x = (float)crop_w / (float)out_w;
  const int x = x0 + lane;
  const bool x_ok = x < out_w;
  const int xc = x_ok ? x : out_w - 1;
  BilinearAxis bx = {xc, xc, 1.f, 0.f};
  if (rescale) bx = bilinear_src(s2x, xc, crop_w);
  const BilinearAxis ax0 = bilinear_src(s1x, bx.i0, w4), ax1 = bilinear_src(s1x, bx.i1, w4);
  BilinearAxis by[PAN_ROWS], ay0[PAN_ROWS], ay1[PAN_ROWS];
  bool ok[PAN_ROWS];
  float best[PAN_ROWS];
  int code[PAN_ROWS];
#pragma unroll
  for (int r = 0; r < PAN_ROWS; ++r) {
    const int y = y0 + ty + 8 * r;
    ok[r] = x_ok && y < out_h;
    const int yc = y < out_h ? y : out_h - 1;
    by[r] = BilinearAxis{yc, yc, 1.f, 0.f};
    if (rescale) by[r] = bilinear_src(s2y, yc, crop_h);
    ay0[r] = bilinear_src(s1y, by[r].i0, h4);
    ay1[r] = bilinear_src(s1y, by[r].i1, h4);
    best[r] = -1.f;
    code[r] = -1;
  }
  for (int k = 0; k < K; ++k) {
    const T* src = logits + ((long)b * Q + s_q[k]) * h4 * w4;
    const float sc = s_sc[k];
    unsigned pos = 0;
#pragma unroll
    for (int r = 0; r < PAN_ROWS; ++r) {
      const float v = rescale ? up2(src, w4, by[r], ay0[r], ay1[r], bx, ax0, ax1) : up1(src, w4, ay0[r], ax0);
      const float sg = sigmoid_f32(v);
      const float p = sc * sg;
      const bool half = sg >= 0.5f;
      if (p > best[r]) { best[r] = p; code[r] = k | (half ? PAN_FLAG : 0); }
      pos += (ok[r] && half) ? 1u : 0u;
    }
    pos = __reduce_add_sync(0xffffffffu, pos);
    if (lane == 0 && pos) atomicAdd(s_o + k, (int)pos);
  }
#pragma unroll
  for (int r = 0; r < PAN_ROWS; ++r) {
    const int key = (ok[r] && code[r] >= 0) ? (code[r] & (PAN_FLAG - 1)) : -1;
    const unsigned grp = __match_any_sync(0xffffffffu, key);
    if (key >= 0 && lane == __ffs(grp) - 1) atomicAdd(s_m + key, __popc(grp));
    if (ok[r]) pan[((long)b * max_out_h + y0 + ty + 8 * r) * max_out_w + x] = code[r];
  }
  __syncthreads();
  for (int i = threadIdx.x; i < K; i += blockDim.x) {
    if (s_m[i]) atomicAdd(s.area_m + b * Q + i, s_m[i]);
    if (s_o[i]) atomicAdd(s.area_o + b * Q + i, s_o[i]);
  }
}

// One warp per image: the validity test of each kept query in kept order (Python's float division of two ints, i.e.
// double) and its segment value; thing instance ids are 1 + the number of valid thing queries before it.  Optionally
// writes the per-query statistics (indexed by query id; 0 / 0 / -1 for queries that were not kept).
__global__ void __launch_bounds__(32) pan_decide_kernel(int Q, int num_things, double iou_thr, PanScratch s,
                                                        int* __restrict__ mask_area, int* __restrict__ original_area,
                                                        int* __restrict__ seg_value) {
  const int b = blockIdx.x, lane = threadIdx.x;
  const int K = s.kept_count[b];
  for (int q = lane; q < Q; q += 32) {
    if (mask_area) mask_area[b * Q + q] = 0;
    if (original_area) original_area[b * Q + q] = 0;
    if (seg_value) seg_value[b * Q + q] = -1;
  }
  __syncwarp();
  int inst = 0;
  for (int c = 0; c < K; c += 32) {
    const int k = c + lane, i = b * Q + k;
    bool valid = false, thing = false;
    int ma = 0, oa = 0, label = 0;
    if (k < K) {
      ma = s.area_m[i]; oa = s.area_o[i]; label = s.kept_label[i];
      valid = ma > 0 && oa > 0 && !((double)ma / (double)oa < iou_thr);
      thing = label < num_things;
    }
    const unsigned m = __ballot_sync(0xffffffffu, valid && thing);
    if (k < K) {
      const int id = inst + __popc(m & ((1u << lane) - 1u)) + 1;
      const int v = valid ? (thing ? label + id * PAN_INSTANCE_OFFSET : label) : -1;
      s.seg[i] = v;
      const int q = b * Q + s.kept_q[i];
      if (mask_area) mask_area[q] = ma;
      if (original_area) original_area[q] = oa;
      if (seg_value) seg_value[q] = v;
    }
    inst += __popc(m);
  }
}

// pixel code -> segment value; C (void) where nothing was kept, the winner's segment was dropped, or (filter_low_score)
// the winner's sigmoid < 0.5
__global__ void __launch_bounds__(256) pan_paint_kernel(const int* __restrict__ geom, int Q, int void_label, int filter,
                                                        int* __restrict__ pan, int max_out_h, int max_out_w, PanScratch s) {
  const int b = blockIdx.z, y = blockIdx.y, x = blockIdx.x * blockDim.x + threadIdx.x;
  if (y >= geom[4 * b + 2] || x >= geom[4 * b + 3]) return;
  int* p = pan + ((long)b * max_out_h + y) * max_out_w + x;
  const int code = *p;
  int v = void_label;
  if (code >= 0 && (!filter || (code & PAN_FLAG))) {
    const int seg = s.seg[b * Q + (code & (PAN_FLAG - 1))];
    if (seg >= 0) v = seg;
  }
  *p = v;
}

}  // namespace

cudaError_t launch_upsample_masks(const void* logits, bool bf16, float* out, int planes, int h4, int w4, int up_h, int up_w,
                                  cudaStream_t s) {
  if (planes <= 0) return cudaSuccess;
  dim3 grid((up_w + 63) / 64, (up_h + 31) / 32, planes);
  if (bf16) upsample_kernel<__nv_bfloat16><<<grid, 256, 0, s>>>(static_cast<const __nv_bfloat16*>(logits), out, h4, w4, up_h, up_w);
  else upsample_kernel<float><<<grid, 256, 0, s>>>(static_cast<const float*>(logits), out, h4, w4, up_h, up_w);
  count_launch();
  return cudaGetLastError();
}

cudaError_t launch_instance_mask_stats(const void* logits, bool bf16, const int* geom, int B, int Q, int h4, int w4, int up_h,
                                       int up_w, int max_out_h, int max_out_w, uint32_t* bits, int* count, float* sig_sum,
                                       int* bbox, cudaStream_t s) {
  const int n = B * Q;
  if (n <= 0) return cudaSuccess;
  stats_init_kernel<<<(n + 255) / 256, 256, 0, s>>>(count, sig_sum, bbox, n);
  const int w32 = (max_out_w + 31) / 32;
  dim3 grid((w32 + 7) / 8, (max_out_h + ROWS_PER_BLOCK - 1) / ROWS_PER_BLOCK, n);
  const long plane = (long)max_out_h * w32;
  if (bf16)
    instance_mask_stats_kernel<__nv_bfloat16><<<grid, 256, 0, s>>>(static_cast<const __nv_bfloat16*>(logits), geom, Q, h4, w4,
                                                                   up_h, up_w, bits, plane, w32, count, sig_sum, bbox);
  else
    instance_mask_stats_kernel<float><<<grid, 256, 0, s>>>(static_cast<const float*>(logits), geom, Q, h4, w4, up_h, up_w, bits,
                                                           plane, w32, count, sig_sum, bbox);
  stats_finish_kernel<<<(n + 255) / 256, 256, 0, s>>>(count, bbox, n);
  count_launch(3);
  return cudaGetLastError();
}

cudaError_t launch_softmax_rows(float* x, int rows, int n, cudaStream_t s) {
  if (rows <= 0) return cudaSuccess;
  softmax_rows_kernel<<<(rows + 7) / 8, 256, 0, s>>>(x, rows, n);
  count_launch();
  return cudaGetLastError();
}

size_t panoptic_scratch_bytes(int B, int Q) { return ((size_t)6 * B * Q + B) * sizeof(int); }

cudaError_t launch_panoptic_fuse(const void* logits, bool bf16, const float* probs, const int* geom, int B, int Q, int n_cls_p1,
                                 int num_things, int h4, int w4, int up_h, int up_w, int max_out_h, int max_out_w,
                                 double object_mask_thr, double iou_thr, bool filter_low_score, int* pan, int* mask_area,
                                 int* original_area, int* seg_value, void* scratch, cudaStream_t st) {
  const PanScratch s = pan_scratch(scratch, B, Q);
  // `scores > object_mask_thr` compares an fp32 tensor with a Python float: the threshold is rounded to fp32
  pan_keep_kernel<<<B, 256, (size_t)Q * 8, st>>>(probs, Q, n_cls_p1, (float)object_mask_thr, s);
  dim3 grid((max_out_w + PAN_TILE - 1) / PAN_TILE, (max_out_h + PAN_TILE - 1) / PAN_TILE, B);
  const size_t smem = (size_t)Q * 16;
  if (bf16)
    pan_pixel_kernel<__nv_bfloat16><<<grid, 256, smem, st>>>(static_cast<const __nv_bfloat16*>(logits), geom, Q, h4, w4, up_h,
                                                             up_w, pan, max_out_h, max_out_w, s);
  else
    pan_pixel_kernel<float><<<grid, 256, smem, st>>>(static_cast<const float*>(logits), geom, Q, h4, w4, up_h, up_w, pan,
                                                     max_out_h, max_out_w, s);
  pan_decide_kernel<<<B, 32, 0, st>>>(Q, num_things, iou_thr, s, mask_area, original_area, seg_value);
  pan_paint_kernel<<<dim3((max_out_w + 255) / 256, max_out_h, B), 256, 0, st>>>(geom, Q, n_cls_p1 - 1, filter_low_score ? 1 : 0,
                                                                               pan, max_out_h, max_out_w, s);
  count_launch(4);
  return cudaGetLastError();
}

}  // namespace cgg

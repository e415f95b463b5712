// Test-time caption generation (beam search of open_set/utils/eval/inference.py:84-157) for a batch of images, with the
// decoder's self-attention state cached per beam and the candidate selection on the device.  The contractions (every
// linear layer, the cross-attention over the query embeddings, the 30 522-way generator) are cgg_gemm_f32 products issued
// by the caller; the four kernels here are what is left of a step:
//   cached_self_attn_kernel  append the new token's k / v to its beam's cache at position t, attend its q over t+1 keys
//   cache_reorder_kernel     each beam's K/V history gathered from its parent beam (double-buffered caches)
//   beam_scores_kernel       mean of the blocks' logits, log_softmax, the length-normalised beam score, per-row top-W
//   beam_select_kernel       flattened top-W of an image's rows and the reference's candidate bookkeeping
// Scores follow torch's fp32 arithmetic on the CPU: `(logp + w) / length**alpha` and `weights * length**alpha` are fp32
// operations with the power computed in double and rounded to fp32 (the caller passes the rounded powers).
#include "../../include/cgg_b200.h"
#include "common.cuh"
#include "kernels.h"
#include <math.h>

namespace cgg {

namespace {

constexpr int SCORE_THREADS = 512;

// (value, index) order of torch.topk: larger value first, the lower index first on equal values
__device__ __forceinline__ bool ranks_before(float v, int i, float u, int j) { return v > u || (v == u && i < j); }

// warp-wide best (value, index) under ranks_before; lanes with !valid do not take part.  Returns the winner in every lane.
__device__ __forceinline__ void warp_best(float& v, int& i, bool& valid) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float u = __shfl_xor_sync(0xffffffffu, v, o);
    const int j = __shfl_xor_sync(0xffffffffu, i, o);
    const bool ok = __shfl_xor_sync(0xffffffffu, valid, o);
    if (ok && (!valid || ranks_before(u, j, v, i))) { v = u; i = j; valid = true; }
  }
}

// grid (rows, heads).  qkv row r: heads x [q | k | v] of head_dim each (the reference's fused qkv_layer split per head);
// caches (rows, cache_len, heads * head_dim).  smem: head_dim + cache_len floats.
__global__ void __launch_bounds__(128) cached_self_attn_kernel(const float* __restrict__ qkv, float* kc, float* vc,
                                                               float* __restrict__ out, int t, int cache_len, int heads,
                                                               int hd, float scale) {
  extern __shared__ float sm[];
  float* q = sm;
  float* p = sm + hd;
  const int r = blockIdx.x, h = blockIdx.y, C = heads * hd;
  const float* src = qkv + (long)r * 3 * C + (long)h * 3 * hd;
  float* kr = kc + (long)r * cache_len * C + (long)h * hd;
  float* vr = vc + (long)r * cache_len * C + (long)h * hd;
  for (int i = threadIdx.x; i < hd; i += blockDim.x) {
    q[i] = src[i];
    kr[(long)t * C + i] = src[hd + i];
    vr[(long)t * C + i] = src[2 * hd + i];
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  for (int j = warp; j <= t; j += nw) {          // the causal mask: keys 0..t are exactly what the cache holds
    const float* kj = kr + (long)j * C;
    float s = 0.f;
    for (int i = lane; i < hd; i += 32) s = fmaf(q[i], kj[i], s);
    s = warp_sum(s);
    if (lane == 0) p[j] = s * scale;
  }
  __syncthreads();
  float m = -INFINITY, sum = 0.f;
  for (int j = 0; j <= t; ++j) m = fmaxf(m, p[j]);
  for (int j = 0; j <= t; ++j) sum += expf(p[j] - m);
  __syncthreads();
  for (int j = threadIdx.x; j <= t; j += blockDim.x) p[j] = expf(p[j] - m) / sum;
  __syncthreads();
  for (int c = threadIdx.x; c < hd; c += blockDim.x) {
    float acc = 0.f;
    for (int j = 0; j <= t; ++j) acc = fmaf(p[j], vr[(long)j * C + c], acc);
    out[(long)r * C + (long)h * hd + c] = acc;
  }
}

// grid (positions, batch * beam_width, 2 * blocks): dst[slab][row][pos] = src[slab][image row of parent[row]][pos]
__global__ void __launch_bounds__(256) cache_reorder_kernel(const float4* __restrict__ src, float4* __restrict__ dst,
                                                            const int* __restrict__ parent, int W, int cache_len, int dim4,
                                                            long rows) {
  const int pos = blockIdx.x, row = blockIdx.y;
  const long slab = blockIdx.z;
  const int from = row - row % W + parent[row];
  const float4* s = src + ((slab * rows + from) * cache_len + pos) * dim4;
  float4* d = dst + ((slab * rows + row) * cache_len + pos) * dim4;
  for (int i = threadIdx.x; i < dim4; i += blockDim.x) d[i] = s[i];
}

// block-wide best (value, index) under ranks_before.  red: 2 * 32 words of shared memory.
__device__ __forceinline__ void block_best(float& v, int& i, bool& valid, float* red_v, int* red_i) {
  warp_best(v, i, valid);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  __syncthreads();
  if (lane == 0) { red_v[warp] = v; red_i[warp] = valid ? i : -1; }
  __syncthreads();
  if (warp == 0) {
    valid = lane < nw && red_i[lane] >= 0;
    v = valid ? red_v[lane] : 0.f;
    i = valid ? red_i[lane] : 0;
    warp_best(v, i, valid);
    if (lane == 0) { red_v[0] = v; red_i[0] = valid ? i : -1; }
  }
  __syncthreads();
  v = red_v[0];
  i = red_i[0];
  valid = i >= 0;
}

__device__ __forceinline__ float block_reduce(float v, float* red, bool is_max) {
  v = is_max ? warp_max(v) : warp_sum(v);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  __syncthreads();
  if (lane == 0) red[warp] = v;
  __syncthreads();
  if (warp == 0) {
    v = lane < nw ? red[lane] : (is_max ? -INFINITY : 0.f);
    v = is_max ? warp_max(v) : warp_sum(v);
    if (lane == 0) red[0] = v;
  }
  __syncthreads();
  v = red[0];
  return v;
}

// One block per (image, beam) row of an image that is still searching and a beam that is active (the first step: beam 0
// only).  logits (blocks, rows, V); row r of block 0 is overwritten with the row's beam scores.
__global__ void __launch_bounds__(SCORE_THREADS) beam_scores_kernel(float* __restrict__ logits, int blocks, int rows, int V,
                                                                    int W, int first, cgg_beam_state st, float pow_len,
                                                                    float* __restrict__ cand_val, int* __restrict__ cand_col) {
  __shared__ float red_v[32];
  __shared__ int red_i[32];
  const int r = blockIdx.x, b = r / W, j = r % W;
  if (st.done[b] || j >= (first ? 1 : st.n_active[b])) return;
  float* x = logits + (long)r * V;
  const long bstride = (long)rows * V;
  float m = -INFINITY;
  for (int c = threadIdx.x; c < V; c += blockDim.x) {     // torch.mean over the stacked block logits
    float s = x[c];
    for (int k = 1; k < blocks; ++k) s += x[k * bstride + c];
    s = s / (float)blocks;
    x[c] = s;
    m = fmaxf(m, s);
  }
  m = block_reduce(m, red_v, true);
  float sum = 0.f;
  for (int c = threadIdx.x; c < V; c += blockDim.x) sum += expf(x[c] - m);
  const float lse = logf(block_reduce(sum, red_v, false));
  const float w = first ? 0.f : st.weights[r];
  for (int c = threadIdx.x; c < V; c += blockDim.x) {
    const float logp = (x[c] - m) - lse;
    x[c] = first ? logp : (logp + w) / pow_len;
  }
  // top-W in torch.topk order.  Each thread keeps the best of its own columns that ranks after the last pick; a pick is
  // the block's best of those, and only the thread that owned it has to look again.
  float v = 0.f;
  int i = 0;
  bool valid = false;
  for (int c = threadIdx.x; c < V; c += blockDim.x)
    if (!valid || ranks_before(x[c], c, v, i)) { v = x[c]; i = c; valid = true; }
  for (int k = 0; k < W; ++k) {
    float bv = v;
    int bi = i;
    bool bvalid = valid;
    block_best(bv, bi, bvalid, red_v, red_i);
    if (threadIdx.x == 0) { cand_val[(long)r * W + k] = bv; cand_col[(long)r * W + k] = bi; }
    if (valid && i == bi) {
      valid = false;
      for (int c = threadIdx.x; c < V; c += blockDim.x) {
        const float u = x[c];
        if (ranks_before(bv, bi, u, c) && (!valid || ranks_before(u, c, v, i))) { v = u; i = c; valid = true; }
      }
    }
  }
}

// beam_select_kernel's static shared memory: the picks of the pass and the continuing beams
struct SelectShared {
  float pick_w[32], cont_w[32];
  int pick_row[32], pick_col[32], cont_row[32], cont_col[32], n_cont;
};
static_assert(sizeof(SelectShared) <= BEAM_SELECT_STATIC_SMEM, "the token staging is sized against this bound");

// One warp per image.  smem: W * token_cap ints (the active beams' tokens before this step).
__global__ void __launch_bounds__(32) beam_select_kernel(const float* __restrict__ cand_val, const int* __restrict__ cand_col,
                                                         int W, int first, int length, int max_len, float pow_len,
                                                         float pow_len1, int eos, cgg_beam_state st) {
  extern __shared__ int old_tokens[];
  __shared__ SelectShared sh;
  const int b = blockIdx.x, lane = threadIdx.x, T = st.token_cap;
  if (st.done[b]) return;                                   // a finished image keeps its state
  const int na = first ? 1 : st.n_active[b];
  int* tokens = st.tokens + (long)b * W * T;
  for (int i = lane; i < na * T; i += 32) old_tokens[i] = tokens[i];
  // flattened top-W over the active rows: a merge of the rows' sorted candidate lists.  The flat index row * V + col
  // orders equal values by row, then by column, and each row's list is already in column order on ties.
  const float* cv = cand_val + (long)b * W * W;
  const int* cc = cand_col + (long)b * W * W;
  int head = 0;
  for (int k = 0; k < W; ++k) {
    bool valid = lane < na && head < W;
    float v = valid ? cv[lane * W + head] : 0.f;
    int i = lane;
    warp_best(v, i, valid);
    const int col = __shfl_sync(0xffffffffu, (lane < na && head < W) ? cc[lane * W + head] : 0, i);
    if (lane == i) ++head;
    if (lane == 0) {
      sh.pick_w[k] = first ? v : v * pow_len;                  // weights = topk * length**alpha (the BOS step: log p)
      sh.pick_row[k] = i;
      sh.pick_col[k] = col;
    }
  }
  __syncwarp();
  float* wts = st.weights + (long)b * W;
  int* parent = st.parent + (long)b * W;
  int64_t* next = st.next_ids + (long)b * W;
  if (first) {                       // every candidate of the BOS step becomes a beam [BOS, c] with weight log p
    if (lane < W) {
      wts[lane] = sh.pick_w[lane];
      parent[lane] = 0;
      next[lane] = sh.pick_col[lane];
      tokens[lane * T] = old_tokens[0];
      tokens[lane * T + 1] = sh.pick_col[lane];
    }
    if (lane == 0) { st.n_active[b] = W; st.max_idx[b] = 0; }
    return;
  }
  // the reference's walk over the picks in rank order (inference.py:117-146), serial in lane 0
  if (lane == 0) {
    float max_score = -100.f;                 // reset on every pass, as the reference does
    int max_idx = 0, n_fin = st.n_fin[b], n = 0;
    bool stop = false;
    for (int k = 0; k < W && !stop; ++k) {
      const int row = sh.pick_row[k], col = sh.pick_col[k];
      if (col == eos) {
        const float score = sh.pick_w[k] / pow_len1;           // weights[idx] / (length + 1)**alpha
        const long rec = (long)b * W + n_fin;
        int* ft = st.fin_tokens + rec * T;
        for (int i = 0; i < length; ++i) ft[i] = old_tokens[row * T + i];
        ft[length] = eos;
        st.fin_len[rec] = length + 1;
        st.fin_score[rec] = score;
        if (score > max_score) { max_score = score; max_idx = n_fin; }
        stop = ++n_fin == W;
      } else if (length + 1 < max_len - 1) {
        sh.cont_row[n] = row;
        sh.cont_col[n] = col;
        sh.cont_w[n] = sh.pick_w[row];                            // the reference's weights[row]: the parent-indexed pick
        ++n;
      }
    }
    st.n_fin[b] = n_fin;
    st.max_idx[b] = max_idx;
    if (stop || n == 0) {
      st.done[b] = 1;
      atomicAdd(st.n_done, 1);
      n = 0;
    }
    sh.n_cont = n;
  }
  __syncwarp();
  const int n = sh.n_cont;
  if (n == 0) return;
  for (int j = 0; j < n; ++j)
    for (int i = lane; i < length; i += 32) tokens[j * T + i] = old_tokens[sh.cont_row[j] * T + i];
  if (lane < W) {
    const bool on = lane < n;
    if (on) tokens[lane * T + length] = sh.cont_col[lane];
    wts[lane] = on ? sh.cont_w[lane] : 0.f;
    parent[lane] = on ? sh.cont_row[lane] : lane;              // rows past n_active are computed but never read
    next[lane] = on ? sh.cont_col[lane] : 0;
  }
  if (lane == 0) st.n_active[b] = n;
}

}  // namespace

cudaError_t launch_caption_self_attn(const float* qkv, float* k_cache, float* v_cache, float* out, int rows, int heads, int hd,
                                     int t, int cache_len, float scale, cudaStream_t s) {
  cached_self_attn_kernel<<<dim3(rows, heads), 128, (size_t)(hd + cache_len) * sizeof(float), s>>>(
      qkv, k_cache, v_cache, out, t, cache_len, heads, hd, scale);
  count_launch();
  return cudaGetLastError();
}

cudaError_t launch_caption_cache_reorder(const float* src, float* dst, const int* parent, int blocks, int rows, int W,
                                         int cache_len, int positions, int dim, cudaStream_t s) {
  cache_reorder_kernel<<<dim3(positions, rows, 2 * blocks), 256, 0, s>>>(reinterpret_cast<const float4*>(src),
                                                                          reinterpret_cast<float4*>(dst), parent, W,
                                                                          cache_len, dim / 4, rows);
  count_launch();
  return cudaGetLastError();
}

cudaError_t launch_beam_scores(float* logits, int blocks, int rows, int V, int W, bool first, const cgg_beam_state& st,
                               float pow_len, float* cand_val, int* cand_col, cudaStream_t s) {
  beam_scores_kernel<<<rows, SCORE_THREADS, 0, s>>>(logits, blocks, rows, V, W, first ? 1 : 0, st, pow_len, cand_val,
                                                    cand_col);
  count_launch();
  return cudaGetLastError();
}

cudaError_t launch_beam_select(const float* cand_val, const int* cand_col, int B, int W, bool first, int length, int max_len,
                               float pow_len, float pow_len1, int eos, const cgg_beam_state& st, cudaStream_t s) {
  beam_select_kernel<<<B, 32, (size_t)W * st.token_cap * sizeof(int), s>>>(cand_val, cand_col, W, first ? 1 : 0, length,
                                                                           max_len, pow_len, pow_len1, eos, st);
  count_launch();
  return cudaGetLastError();
}

}  // namespace cgg

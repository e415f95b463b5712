// Backward-side kernels of the training step (BASELINE.json configs[3]: forward + backward of the decoder head with
// the caption-grounding loss; reference: open_set/models/mask2former_head.py:851-921 forward_train -> loss, autograd
// through the path of :763-849).  fp32 SIMT.  The dense contractions of the backward (dX = dY W, dW = dY^T X, the
// two gradients of the mask einsum, the K/V in-projection) go through the generic strided GEMM of kernels_f32.cu;
// this file holds what is not a GEMM: LayerNorm backward, the masked-attention backward, ReLU masking, and the
// forward attention variant that also returns the row log-sum-exp.
#include "common.cuh"
#include "kernels.h"
#include <math.h>

namespace cgg {

namespace {

// ----------------------------------------------------------------------------------------------- LayerNorm
// y = (x - mu) * rstd * w + b  (torch.nn.LayerNorm, biased variance).  One warp per row:
//   xhat = (x - mu) rstd ; g = dy w ; dx = rstd (g - mean(g) - xhat mean(g xhat))
// dw / db partial sums: one row of (2, n) per CTA in `partial` (deterministic second pass below).
__global__ void __launch_bounds__(256) layernorm_bwd_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                                            const float* __restrict__ dy, float* __restrict__ dx,
                                                            float* __restrict__ partial, int rows, int n, float eps) {
  extern __shared__ float sm[];          // [8 warps][2][n]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int row = blockIdx.x * 8 + warp;
  float* my = sm + (size_t)warp * 2 * n;
  for (int i = lane; i < 2 * n; i += 32) my[i] = 0.f;
  if (row < rows) {
    const float* xr = x + (long)row * n;
    const float* gr = dy + (long)row * n;
    float s = 0.f;
    for (int i = lane; i < n; i += 32) s += xr[i];
    const float mu = warp_sum(s) / (float)n;
    float v = 0.f;
    for (int i = lane; i < n; i += 32) { const float d = xr[i] - mu; v = fmaf(d, d, v); }
    const float rstd = 1.0f / sqrtf(warp_sum(v) / (float)n + eps);
    float sg = 0.f, sgx = 0.f;
    for (int i = lane; i < n; i += 32) {
      const float xh = (xr[i] - mu) * rstd, g = gr[i] * w[i];
      sg += g;
      sgx = fmaf(g, xh, sgx);
      my[i] = gr[i] * xh;        // dw contribution
      my[n + i] = gr[i];         // db contribution
    }
    sg = warp_sum(sg) / (float)n;
    sgx = warp_sum(sgx) / (float)n;
    for (int i = lane; i < n; i += 32) {
      const float xh = (xr[i] - mu) * rstd, g = gr[i] * w[i];
      dx[(long)row * n + i] = rstd * (g - sg - xh * sgx);
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 2 * n; i += 256) {
    float a = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) a += sm[(size_t)k * 2 * n + i];
    partial[(long)blockIdx.x * 2 * n + i] = a;
  }
}

// dw[i] = sum_blocks partial[blk][i], db[i] = sum_blocks partial[blk][n + i].  32 columns x 32 row lanes per CTA: lane r of a
// column sums blocks r, r + 32, ... and the 32 lane sums are folded in a fixed order (deterministic).  (One thread per column
// walking all blocks took 0.22 ms at the pixel decoder's 43 k rows.)
__global__ void __launch_bounds__(1024) layernorm_bwd_reduce_kernel(const float* __restrict__ partial, int nblocks, int n,
                                                                    float* __restrict__ dw, float* __restrict__ db) {
  __shared__ float red[32][33];
  const int c = threadIdx.x & 31, r = threadIdx.x >> 5;
  const int i = blockIdx.x * 32 + c;
  float a = 0.f;
  if (i < 2 * n)
    for (int k = r; k < nblocks; k += 32) a += partial[(long)k * 2 * n + i];
  red[r][c] = a;
  __syncthreads();
  if (r == 0 && i < 2 * n) {
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < 32; ++k) t += red[k][c];
    if (i < n) dw[i] = t; else db[i - n] = t;
  }
}

// --------------------------------------------------------------------------------------------------- ReLU
// dx = dy where y > 0 (y = the ReLU output), times alpha
__global__ void relu_bwd_kernel(const float* __restrict__ y, const float* __restrict__ dy, float* __restrict__ dx, long n,
                                float alpha) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dx[i] = y[i] > 0.f ? dy[i] * alpha : 0.f;
}
__global__ void relu_bwd4_kernel(const float4* __restrict__ y, const float4* __restrict__ dy, float4* __restrict__ dx, long n4,
                                 float alpha) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n4) return;
  const float4 a = y[i], g = dy[i];
  dx[i] = make_float4(a.x > 0.f ? g.x * alpha : 0.f, a.y > 0.f ? g.y * alpha : 0.f, a.z > 0.f ? g.z * alpha : 0.f,
                      a.w > 0.f ? g.w * alpha : 0.f);
}

// out[i] += in[i]  (gradient accumulation of a tensor consumed twice inside one fused stage)
__global__ void axpy_kernel(const float* __restrict__ in, float* __restrict__ out, long n, float alpha) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = fmaf(alpha, in[i], out[i]);
}

// out[b,m,:] = x[b,m,:] + add[m,:]   (x may be null = zeros: the query_feat broadcast of head.py:808-809)
__global__ void add_rows_kernel(const float* __restrict__ x, const float* __restrict__ add, float* __restrict__ out,
                                long per, long total) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < total) out[i] = (x ? x[i] : 0.f) + add[i % per];
}
// out[i] = sum_b g[b*per + i]   (gradient of a row table broadcast over the batch), fixed order
__global__ void sum_batch_kernel(const float* __restrict__ g, float* __restrict__ out, long per, int batch) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= per) return;
  float a = 0.f;
  for (int b = 0; b < batch; ++b) a += g[(long)b * per + i];
  out[i] = a;
}
__global__ void sum_batch4_kernel(const float4* __restrict__ g, float4* __restrict__ out, long per4, int batch) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= per4) return;
  float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int b = 0; b < batch; ++b) {
    const float4 v = g[(long)b * per4 + i];
    a.x += v.x; a.y += v.y; a.z += v.z; a.w += v.w;
  }
  out[i] = a;
}
// out[b] = x[b] + add, float4 form: blockIdx.y = batch entry (no modulo per element)
__global__ void add_rows4_kernel(const float4* __restrict__ x, const float4* __restrict__ add, float4* __restrict__ out, long per4) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= per4) return;
  const long o = (long)blockIdx.y * per4 + i;
  const float4 a = add[i];
  float4 v = x ? x[o] : make_float4(0.f, 0.f, 0.f, 0.f);
  out[o] = make_float4(v.x + a.x, v.y + a.y, v.z + a.z, v.w + a.w);
}

// key_in[b,key,c] = mem[b,c,key] + level[c] + pos[key,c] ; val_in[b,key,c] = mem[b,c,key] + level[c]
// (head.py:792-804).  32 x 32 shared-memory transpose tiles; pos_level = pos + level (K, C) from cgg_prepare.
__global__ void __launch_bounds__(256) mem_prep_kernel(const float* __restrict__ mem, const float* __restrict__ level,
                                                       const float* __restrict__ pos_level, float* __restrict__ key_in,
                                                       float* __restrict__ val_in, int C, int K) {
  __shared__ float tile[32][33];
  const int b = blockIdx.z, k0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int r = ty; r < 32; r += 8) {
    const int c = c0 + r, k = k0 + tx;
    tile[r][tx] = (c < C && k < K) ? mem[((long)b * C + c) * K + k] : 0.f;
  }
  __syncthreads();
  for (int r = ty; r < 32; r += 8) {
    const int k = k0 + r, c = c0 + tx;
    if (k < K && c < C) {
      const float m = tile[tx][r];
      const long o = ((long)b * K + k) * C + c;
      key_in[o] = m + pos_level[(long)k * C + c];
      val_in[o] = m + level[c];
    }
  }
}
// dmem[b,c,key] = dkey_in[b,key,c] + dval_in[b,key,c]
__global__ void __launch_bounds__(256) mem_prep_bwd_kernel(const float* __restrict__ dkey, const float* __restrict__ dval,
                                                           float* __restrict__ dmem, int C, int K) {
  __shared__ float tile[32][33];
  const int b = blockIdx.z, k0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int r = ty; r < 32; r += 8) {
    const int k = k0 + r, c = c0 + tx;
    float v = 0.f;
    if (k < K && c < C) {
      const long o = ((long)b * K + k) * C + c;
      v = dkey[o] + dval[o];
    }
    tile[r][tx] = v;
  }
  __syncthreads();
  for (int r = ty; r < 32; r += 8) {
    const int c = c0 + r, k = k0 + tx;
    if (c < C && k < K) dmem[((long)b * C + c) * K + k] = tile[tx][r];
  }
}

// out[n] += sum_rows g[row, n]  (bias gradients; out zeroed by the launcher; row chunks of 256 per CTA)
__global__ void __launch_bounds__(256) colsum_kernel(const float* __restrict__ g, float* __restrict__ out, long rows, int n,
                                                     float alpha) {
  const int col = blockIdx.x * 32 + (threadIdx.x & 31), ty = threadIdx.x >> 5;
  const long r0 = (long)blockIdx.y * 256;
  __shared__ float red[8][33];
  float a = 0.f;
  if (col < n) {
    const long rend = (r0 + 256 < rows) ? r0 + 256 : rows;
    long r = r0 + ty;
    for (; r + 56 < rend; r += 64) {                     // 8 independent loads in flight per thread
      float v[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) v[u] = g[(r + 8 * u) * n + col];
#pragma unroll
      for (int u = 0; u < 8; ++u) a += v[u];
    }
    for (; r < rend; r += 8) a += g[r * n + col];
  }
  red[ty][threadIdx.x & 31] = a;
  __syncthreads();
  if (ty == 0 && col < n) {
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) t += red[k][threadIdx.x];
    atomicAdd(out + col, t * alpha);
  }
}

// ------------------------------------------------------------------------------- attention: row statistics
// lse[b,h,q] = log sum_k exp(s_qk) over the unmasked keys (fallback rows: all keys), D[b,h,q] = do . o.
// One warp per (b, h, q) row; K/V may be fp32 only here (the training path of the parity mode).
constexpr int HD = 32;
__global__ void __launch_bounds__(256) attn_rowstats_kernel(const float* __restrict__ q, const float* __restrict__ k,
                                                            long kv_stride, long kv_bstride,
                                                            const uint32_t* __restrict__ bitmap,
                                                            const uint8_t* __restrict__ all_masked,
                                                            const float* __restrict__ o, const float* __restrict__ dout,
                                                            float* __restrict__ lse, float* __restrict__ dsum, int B, int Q,
                                                            int K, int heads) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long r = (long)blockIdx.x * 8 + warp;            // (b, h, q)
  if (r >= (long)B * heads * Q) return;
  const int qi = (int)(r % Q), h = (int)((r / Q) % heads), b = (int)(r / ((long)Q * heads));
  const int C = heads * HD, W32 = (K + 31) / 32;
  const float* qr = q + ((long)b * Q + qi) * C + h * HD;
  float qv[HD];
#pragma unroll
  for (int d = 0; d < HD; ++d) qv[d] = qr[d];
  const bool use_mask = bitmap != nullptr && !(all_masked && all_masked[(long)b * Q + qi]);
  const uint32_t* brow = bitmap ? bitmap + ((long)b * Q + qi) * W32 : nullptr;
  float m = -INFINITY, l = 0.f;
  for (int k0 = 0; k0 < K; k0 += 32) {
    const int kk = k0 + lane;
    float s = -INFINITY;
    if (kk < K) {
      const uint32_t word = use_mask ? brow[k0 >> 5] : 0u;
      if (!((word >> lane) & 1u)) {
        const float* kr = k + (long)b * kv_bstride + (long)kk * kv_stride + h * HD;
        float acc = 0.f;
#pragma unroll
        for (int d = 0; d < HD; ++d) acc = fmaf(qv[d], kr[d], acc);
        s = acc;
      }
    }
    float mt = s;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) mt = fmaxf(mt, __shfl_xor_sync(0xffffffffu, mt, off));
    const float mn = fmaxf(m, mt);
    if (mn != -INFINITY) {
      const float e = (s == -INFINITY) ? 0.f : expf(s - mn);
      l = l * ((m == -INFINITY) ? 0.f : expf(m - mn)) + warp_sum(e);
      m = mn;
    }
  }
  float dd = 0.f;
  {
    const float* orow = o + ((long)b * Q + qi) * C + h * HD;
    const float* drow = dout + ((long)b * Q + qi) * C + h * HD;
    dd = warp_sum(orow[lane] * drow[lane]);
  }
  if (lane == 0) {
    lse[r] = (l > 0.f) ? m + logf(l) : -INFINITY;
    dsum[r] = dd;
  }
}

// ------------------------------------------------------ attention as tensor-core products: the two row-wise stages
// Training step with tf32 contractions: S = q k^T, O = P v, dP = dO v^T, dQ = dS k, dK = dS^T q, dV = P^T dO are calls
// of the tcgen05 GEMM over (image, head) batches; what is left is row-wise work on the (B, heads, Q, K) score tensor.
//
// P = softmax over the unmasked keys of a row, in place (bit = 1 in the bitmap excludes the key, unless the row's
// all_masked flag is set: mask2former_head.py:825-826).  One CTA per row; the row (<= 144 KB) is re-read from L1/L2.
template <bool CACHED>
__global__ void __launch_bounds__(256) attn_softmax_rows_kernel(float* __restrict__ S, const uint32_t* __restrict__ bitmap,
                                                                const uint8_t* __restrict__ all_masked, int heads, int Q,
                                                                int K) {
  extern __shared__ float srow[];                       // CACHED: the row (K floats), read from HBM once
  __shared__ float red[8];
  __shared__ float bcast;
  const long r = blockIdx.x;                            // (b, h, q)
  const int qi = (int)(r % Q);
  const long b = r / ((long)Q * heads);
  float* row = S + r * K;
  const int W32 = (K + 31) / 32;
  const bool use_mask = bitmap != nullptr && !(all_masked && all_masked[b * Q + qi]);
  const uint32_t* brow = use_mask ? bitmap + (b * Q + qi) * W32 : nullptr;
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  auto masked = [&](int k) { return brow && ((brow[k >> 5] >> (k & 31)) & 1u); };
  float m = -INFINITY;
  for (int k = t; k < K; k += 256) {
    const float v = masked(k) ? -INFINITY : row[k];
    if (CACHED) srow[k] = v;
    m = fmaxf(m, v);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if (lane == 0) red[warp] = m;
  __syncthreads();
  if (t == 0) {
    float mm = red[0];
    for (int i = 1; i < 8; ++i) mm = fmaxf(mm, red[i]);
    bcast = mm;
  }
  __syncthreads();
  m = bcast;
  float l = 0.f;
  if (m != -INFINITY)
    for (int k = t; k < K; k += 256) {
      const float v = CACHED ? srow[k] : (masked(k) ? -INFINITY : row[k]);
      const float e = expf(v - m);                      // exp(-inf) = 0 for the masked keys
      if (CACHED) srow[k] = e;
      l += e;
    }
  l = warp_sum(l);
  __syncthreads();
  if (lane == 0) red[warp] = l;
  __syncthreads();
  if (t == 0) {
    float ll = 0.f;
    for (int i = 0; i < 8; ++i) ll += red[i];
    bcast = ll;
  }
  __syncthreads();
  l = bcast;
  const float inv = l > 0.f ? 1.f / l : 0.f;
  for (int k = t; k < K; k += 256) {
    float e;
    if (CACHED) e = (m != -INFINITY) ? srow[k] : 0.f;
    else e = (m != -INFINITY && !masked(k)) ? expf(row[k] - m) : 0.f;
    row[k] = e * inv;
  }
}

// dS = P o (dP - D), D[b,h,q] = dO[b,q,h,:] . O[b,q,h,:]; written over dP.
__global__ void __launch_bounds__(256) attn_dscore_kernel(const float* __restrict__ P, float* __restrict__ dP,
                                                          const float* __restrict__ O, const float* __restrict__ dO,
                                                          int heads, int hd, int Q, int K) {
  __shared__ float Dsh;
  const long r = blockIdx.x;
  const int qi = (int)(r % Q), h = (int)((r / Q) % heads);
  const long b = r / ((long)Q * heads);
  if (threadIdx.x < 32) {
    const long off = (b * Q + qi) * (long)(heads * hd) + (long)h * hd;
    float d = 0.f;
    for (int i = threadIdx.x; i < hd; i += 32) d = fmaf(O[off + i], dO[off + i], d);
    d = warp_sum(d);
    if (threadIdx.x == 0) Dsh = d;
  }
  __syncthreads();
  const float D = Dsh;
  const float* prow = P + r * K;
  float* drow = dP + r * K;
  for (int k = threadIdx.x; k < K; k += 256) drow[k] = prow[k] * (drow[k] - D);
}

// ----------------------------------------------------------------------------- attention backward (fp32 SIMT)
// One CTA per (key tile of 64 keys, head, image): it owns dK, dV of its keys (no atomics) and adds its share of dQ
// with atomicAdd.  p = exp(s - lse); dP = dO . v; dS = p (dP - D); dQ += dS k; dK += dS^T q; dV += p^T dO.
// q is the SCALED query (the 1/sqrt(d) factor belongs to the producing linear layer).
constexpr int BK_T = 64, BQ_T = 32;
__global__ void __launch_bounds__(256) attn_bwd_kernel(const float* __restrict__ q, const float* __restrict__ k,
                                                       const float* __restrict__ v, long kv_stride, long kv_bstride,
                                                       const uint32_t* __restrict__ bitmap,
                                                       const uint8_t* __restrict__ all_masked,
                                                       const float* __restrict__ dout, const float* __restrict__ lse,
                                                       const float* __restrict__ dsum, float* __restrict__ dq,
                                                       float* __restrict__ dk, float* __restrict__ dv, long dkv_stride,
                                                       long dkv_bstride, int Q, int K, int heads) {
  __shared__ float Ks[BK_T][HD + 1], Vs[BK_T][HD + 1];
  __shared__ float Qs[BQ_T][HD + 1], dOs[BQ_T][HD + 1];
  __shared__ float Ps[BQ_T][BK_T + 1], dSs[BQ_T][BK_T + 1];
  __shared__ float Ls[BQ_T], Ds[BQ_T];
  const int k0 = blockIdx.x * BK_T, h = blockIdx.y, b = blockIdx.z;
  const int t = threadIdx.x;
  const int C = heads * HD, W32 = (K + 31) / 32;
  for (int i = t; i < BK_T * HD; i += 256) {
    const int kk = i / HD, d = i % HD, gk = k0 + kk;
    float kv = 0.f, vv = 0.f;
    if (gk < K) {
      const long off = (long)b * kv_bstride + (long)gk * kv_stride + h * HD + d;
      kv = k[off];
      vv = v[off];
    }
    Ks[kk][d] = kv;
    Vs[kk][d] = vv;
  }
  // each thread accumulates dK, dV for (key = t / 4, dims 8 * (t % 4) .. + 7)
  const int my_k = t >> 2, my_d0 = (t & 3) * 8;
  float dk_acc[8], dv_acc[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) dk_acc[i] = dv_acc[i] = 0.f;
  for (int q0 = 0; q0 < Q; q0 += BQ_T) {
    __syncthreads();
    for (int i = t; i < BQ_T * HD; i += 256) {
      const int qq = i / HD, d = i % HD, gq = q0 + qq;
      float qv = 0.f, dv_ = 0.f;
      if (gq < Q) {
        const long off = ((long)b * Q + gq) * C + h * HD + d;
        qv = q[off];
        dv_ = dout[off];
      }
      Qs[qq][d] = qv;
      dOs[qq][d] = dv_;
    }
    if (t < BQ_T) {
      const int gq = q0 + t;
      Ls[t] = gq < Q ? lse[((long)b * heads + h) * Q + gq] : -INFINITY;
      Ds[t] = gq < Q ? dsum[((long)b * heads + h) * Q + gq] : 0.f;
    }
    __syncthreads();
    // P and dS for the (BQ_T x BK_T) block: 2048 entries, 8 per thread
    for (int e = t; e < BQ_T * BK_T; e += 256) {
      const int qq = e / BK_T, kk = e % BK_T, gq = q0 + qq, gk = k0 + kk;
      float p = 0.f, ds = 0.f;
      if (gq < Q && gk < K && Ls[qq] != -INFINITY) {
        bool masked = false;
        if (bitmap && !(all_masked && all_masked[(long)b * Q + gq]))
          masked = (bitmap[((long)b * Q + gq) * W32 + (gk >> 5)] >> (gk & 31)) & 1u;
        if (!masked) {
          float s = 0.f, dp = 0.f;
#pragma unroll
          for (int d = 0; d < HD; ++d) {
            s = fmaf(Qs[qq][d], Ks[kk][d], s);
            dp = fmaf(dOs[qq][d], Vs[kk][d], dp);
          }
          p = expf(s - Ls[qq]);
          ds = p * (dp - Ds[qq]);
        }
      }
      Ps[qq][kk] = p;
      dSs[qq][kk] = ds;
    }
    __syncthreads();
    // dK, dV: sum over the block's queries
#pragma unroll 4
    for (int qq = 0; qq < BQ_T; ++qq) {
      const float p = Ps[qq][my_k], ds = dSs[qq][my_k];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        dk_acc[i] = fmaf(ds, Qs[qq][my_d0 + i], dk_acc[i]);
        dv_acc[i] = fmaf(p, dOs[qq][my_d0 + i], dv_acc[i]);
      }
    }
    // dQ: thread -> (query = t / 8, dims 4 * (t % 8) .. + 3), sum over the tile's keys, then atomicAdd
    {
      const int qq = t >> 3, d0 = (t & 7) * 4, gq = q0 + qq;
      float a[4] = {0.f, 0.f, 0.f, 0.f};
      for (int kk = 0; kk < BK_T; ++kk) {
        const float ds = dSs[qq][kk];
#pragma unroll
        for (int i = 0; i < 4; ++i) a[i] = fmaf(ds, Ks[kk][d0 + i], a[i]);
      }
      if (gq < Q) {
        float* dst = dq + ((long)b * Q + gq) * C + h * HD + d0;
#pragma unroll
        for (int i = 0; i < 4; ++i) atomicAdd(dst + i, a[i]);
      }
    }
  }
  const int gk = k0 + my_k;
  if (gk < K) {
    const long off = (long)b * dkv_bstride + (long)gk * dkv_stride + h * HD + my_d0;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      dk[off + i] = dk_acc[i];
      dv[off + i] = dv_acc[i];
    }
  }
}

}  // namespace

cudaError_t launch_attn_softmax_rows(float* S, const uint32_t* bitmap, const uint8_t* all_masked, int B, int heads, int Q,
                                     int K, cudaStream_t s) {
  const long rows = (long)B * heads * Q;
  if (rows <= 0 || K <= 0) return cudaSuccess;
  const size_t smem = (size_t)K * sizeof(float);
  if (smem <= 96 * 1024) {                              // row cached in shared memory: one HBM read, one write
    static bool attr = false;
    if (!attr) {
      cudaError_t e = cudaFuncSetAttribute(attn_softmax_rows_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024);
      if (e != cudaSuccess) return e;
      attr = true;
    }
    attn_softmax_rows_kernel<true><<<(unsigned)rows, 256, smem, s>>>(S, bitmap, all_masked, heads, Q, K);
  } else {
    attn_softmax_rows_kernel<false><<<(unsigned)rows, 256, 0, s>>>(S, bitmap, all_masked, heads, Q, K);
  }
  count_launch();
  return cudaGetLastError();
}

cudaError_t launch_attn_dscore(const float* P, float* dP, const float* O, const float* dO, int B, int heads, int head_dim,
                               int Q, int K, cudaStream_t s) {
  const long rows = (long)B * heads * Q;
  if (rows <= 0 || K <= 0) return cudaSuccess;
  attn_dscore_kernel<<<(unsigned)rows, 256, 0, s>>>(P, dP, O, dO, heads, head_dim, Q, K);
  count_launch();
  return cudaGetLastError();
}

cudaError_t launch_layernorm_bwd(const float* x, const float* w, const float* dy, float* dx, float* dw, float* db,
                                 float* partial, int rows, int n, float eps, cudaStream_t s) {
  if (rows <= 0) return cudaSuccess;
  const int nblocks = (rows + 7) / 8;
  const size_t smem = (size_t)8 * 2 * n * sizeof(float);
  cudaError_t e = cudaFuncSetAttribute(layernorm_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  layernorm_bwd_kernel<<<nblocks, 256, smem, s>>>(x, w, dy, dx, partial, rows, n, eps);
  layernorm_bwd_reduce_kernel<<<(2 * n + 31) / 32, 1024, 0, s>>>(partial, nblocks, n, dw, db);
  count_launch(2);
  return cudaGetLastError();
}

cudaError_t launch_relu_bwd(const float* y, const float* dy, float* dx, long n, float alpha, cudaStream_t s) {
  if (n <= 0) return cudaSuccess;
  auto al16 = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15) == 0; };
  if (n % 4 == 0 && al16(y) && al16(dy) && al16(dx))
    relu_bwd4_kernel<<<(unsigned)((n / 4 + 255) / 256), 256, 0, s>>>((const float4*)y, (const float4*)dy, (float4*)dx, n / 4, alpha);
  else
    relu_bwd_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(y, dy, dx, n, alpha);
  count_launch();
  return cudaGetLastError();
}

cudaError_t launch_axpy(const float* in, float* out, long n, float alpha, cudaStream_t s) {
  if (n <= 0) return cudaSuccess;
  axpy_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(in, out, n, alpha);
  count_launch();
  return cudaGetLastError();
}

cudaError_t launch_add_rows(const float* x, const float* add, float* out, int batch, long per, cudaStream_t s) {
  const long total = per * batch;
  if (total <= 0) return cudaSuccess;
  auto al16 = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15) == 0; };
  if (per % 4 == 0 && batch <= 65535 && al16(x) && al16(add) && al16(out))
    add_rows4_kernel<<<dim3((unsigned)((per / 4 + 255) / 256), batch), 256, 0, s>>>((const float4*)x, (const float4*)add, (float4*)out, per / 4);
  else
    add_rows_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(x, add, out, per, total);
  count_launch();
  return cudaGetLastError();
}

cudaError_t launch_sum_batch(const float* g, float* out, int batch, long per, cudaStream_t s) {
  if (per <= 0) return cudaSuccess;
  auto al16 = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15) == 0; };
  if (per % 4 == 0 && al16(g) && al16(out))
    sum_batch4_kernel<<<(unsigned)((per / 4 + 255) / 256), 256, 0, s>>>((const float4*)g, (float4*)out, per / 4, batch);
  else
    sum_batch_kernel<<<(unsigned)((per + 255) / 256), 256, 0, s>>>(g, out, per, batch);
  count_launch();
  return cudaGetLastError();
}

cudaError_t launch_mem_prep(const float* mem, const float* level, const float* pos_level, float* key_in, float* val_in,
                            int B, int C, int K, cudaStream_t s) {
  if (B <= 0) return cudaSuccess;
  mem_prep_kernel<<<dim3((K + 31) / 32, (C + 31) / 32, B), 256, 0, s>>>(mem, level, pos_level, key_in, val_in, C, K);
  count_launch();
  return cudaGetLastError();
}

cudaError_t launch_mem_prep_bwd(const float* dkey, const float* dval, float* dmem, int B, int C, int K, cudaStream_t s) {
  if (B <= 0) return cudaSuccess;
  mem_prep_bwd_kernel<<<dim3((K + 31) / 32, (C + 31) / 32, B), 256, 0, s>>>(dkey, dval, dmem, C, K);
  count_launch();
  return cudaGetLastError();
}

cudaError_t launch_colsum(const float* g, float* out, long rows, int n, float alpha, cudaStream_t s, bool accumulate) {
  if (n <= 0) return cudaSuccess;
  cudaError_t e = accumulate ? cudaSuccess : cudaMemsetAsync(out, 0, (size_t)n * sizeof(float), s);
  if (e != cudaSuccess || rows <= 0) return e;
  colsum_kernel<<<dim3((n + 31) / 32, (unsigned)((rows + 255) / 256)), 256, 0, s>>>(g, out, rows, n, alpha);
  count_launch();
  return cudaGetLastError();
}

cudaError_t launch_attention_bwd(const float* q, const float* k, const float* v, long kv_stride, long kv_bstride,
                                 const uint32_t* bitmap, const uint8_t* all_masked, const float* o, const float* dout,
                                 float* lse, float* dsum, float* dq, float* dk, float* dv, long dkv_stride,
                                 long dkv_bstride, int B, int Q, int K, int heads, cudaStream_t s) {
  if (B <= 0 || Q <= 0 || K <= 0) return cudaSuccess;
  const long rows = (long)B * heads * Q;
  attn_rowstats_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, s>>>(q, k, kv_stride, kv_bstride, bitmap, all_masked, o, dout,
                                                                  lse, dsum, B, Q, K, heads);
  cudaError_t e = cudaMemsetAsync(dq, 0, (size_t)B * Q * heads * HD * sizeof(float), s);
  if (e != cudaSuccess) return e;
  dim3 grid((K + BK_T - 1) / BK_T, heads, B);
  attn_bwd_kernel<<<grid, 256, 0, s>>>(q, k, v, kv_stride, kv_bstride, bitmap, all_masked, dout, lse, dsum, dq, dk, dv,
                                       dkv_stride, dkv_bstride, Q, K, heads);
  count_launch(2);
  return cudaGetLastError();
}

}  // namespace cgg

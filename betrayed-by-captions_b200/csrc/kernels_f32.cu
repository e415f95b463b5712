// fp32 SIMT kernels of the decoder-head path: the parity mode (CGG_FP32) runs entirely on
// these, and the throughput mode (CGG_BF16) keeps using them for the latency-bound small-M
// work.  No fast-math: the sigmoid threshold and the softmax follow IEEE expf / division so the
// attention-mask bits match the PyTorch CUDA reference (SURVEY.md section 7, hard part 2).
#include "common.cuh"
#include "kernels.h"
#include <cuda_fp16.h>
#include <math.h>
#include <atomic>

namespace cgg {

static std::atomic<unsigned long long> g_launches{0};
void count_launch(int n) { g_launches.fetch_add((unsigned long long)n, std::memory_order_relaxed); }
unsigned long long launch_count() { return g_launches.load(std::memory_order_relaxed); }

// ------------------------------------------------------------------------------- GEMM
template <bool A_MMAJOR, bool C_MMAJOR>
__global__ void __launch_bounds__(256) gemm_f32_kernel(GemmF32 p) {
  constexpr int BM = 64, BN = 64, BK = 16;
  __shared__ __align__(16) float As[BK][BM + 4];
  __shared__ __align__(16) float Bs[BK][BN + 4];
  const int b = blockIdx.z;
  const int m0 = blockIdx.x * BM, n0 = blockIdx.y * BN;
  const int t = threadIdx.x, tx = t & 15, ty = t >> 4;
  const int mb = C_MMAJOR ? tx : ty, nb = C_MMAJOR ? ty : tx;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  const long bo = b / p.batch_inner, bi = b % p.batch_inner;
  const float* __restrict__ A = p.A + bo * p.sAb + bi * p.sAb2;
  const float* __restrict__ W = p.W + bo * p.sWb + bi * p.sWb2;
  for (int k0 = 0; k0 < p.K; k0 += BK) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int idx = t + i * 256;
      int m, k;
      if (A_MMAJOR) { m = idx & 63; k = idx >> 6; } else { k = idx & 15; m = idx >> 4; }
      const int gm = m0 + m, gk = k0 + k;
      float v = 0.f;
      if (gm < p.M && gk < p.K) {
        if (p.conv_cin > 0) {          // implicit 3x3 convolution: k = (tap, channel), taps outside the image are zero
          const int tap = gk / p.conv_cin, cc = gk - tap * p.conv_cin;
          const int yy = (int)bi + tap / 3 - 1, xx = gm + tap % 3 - 1;
          if (yy >= 0 && yy < p.batch_inner && xx >= 0 && xx < p.M)
            v = p.A[bo * p.sAb + (long)yy * p.sAb2 + (long)xx * p.sAm + (long)cc * p.sAk];
        } else {
          v = A[(long)gm * p.sAm + (long)gk * p.sAk];
          if (p.A2) v += p.A2[(long)(gm % p.a2_mod) * p.sA2m + (long)gk * p.sA2k];
        }
      }
      As[k][m] = v;
      const int kb = idx & 15, n = idx >> 4;
      const int gn = n0 + n, gkb = k0 + kb;
      Bs[kb][n] = (gn < p.N && gkb < p.K) ? W[(long)gn * p.sWn + (long)gkb * p.sWk] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < BK; ++k) {
      const float4 a4 = *reinterpret_cast<const float4*>(&As[k][mb * 4]);
      const float4 b4 = *reinterpret_cast<const float4*>(&Bs[k][nb * 4]);
      const float a[4] = {a4.x, a4.y, a4.z, a4.w};
      const float bb[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], bb[j], acc[i][j]);
    }
    __syncthreads();
  }
  float* __restrict__ C = p.C + bo * p.sCb + bi * p.sCb2;
  const float* __restrict__ R = p.R ? p.R + (long)b * p.sRb : nullptr;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int gm = m0 + mb * 4 + i;
    if (gm >= p.M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int gn = n0 + nb * 4 + j;
      if (gn >= p.N) continue;
      float v = acc[i][j];
      if (p.bias) v += p.bias[gn];
      v *= p.alpha;
      if (R && gn < p.r_ncols) v += R[(long)(gm % p.r_mod) * p.sRm + (long)gn * p.sRn];
      if (gn >= p.relu_from) v = fmaxf(v, 0.f);
      if (p.accumulate) v += C[(long)gm * p.sCm + (long)gn * p.sCn];
      C[(long)gm * p.sCm + (long)gn * p.sCn] = v;
    }
  }
}

cudaError_t launch_gemm_f32(const GemmF32& p, cudaStream_t s) {
  if (p.M <= 0 || p.N <= 0 || p.batch <= 0) return cudaSuccess;
  dim3 grid((p.M + 63) / 64, (p.N + 63) / 64, p.batch), block(256);
  if (p.a_mmajor && p.c_mmajor) gemm_f32_kernel<true, true><<<grid, block, 0, s>>>(p);
  else if (p.a_mmajor) gemm_f32_kernel<true, false><<<grid, block, 0, s>>>(p);
  else if (p.c_mmajor) gemm_f32_kernel<false, true><<<grid, block, 0, s>>>(p);
  else gemm_f32_kernel<false, false><<<grid, block, 0, s>>>(p);
  count_launch();
  return cudaGetLastError();
}

// -------------------------------------------------------------------------- LayerNorm
__global__ void __launch_bounds__(256) layernorm_kernel(const float* __restrict__ x,
                                                        const int64_t* __restrict__ gather,
                                                        const float* __restrict__ w,
                                                        const float* __restrict__ b,
                                                        float* __restrict__ y, int rows, int n,
                                                        float eps, bool apply_norm) {
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float* xr = x + (gather ? gather[row] : (int64_t)row) * n;
  float* yr = y + (long)row * n;
  if (!apply_norm) {
    for (int i = lane; i < n; i += 32) yr[i] = xr[i];
    return;
  }
  float s = 0.f;
  for (int i = lane; i < n; i += 32) s += xr[i];
  const float mu = warp_sum(s) / (float)n;
  float v = 0.f;
  for (int i = lane; i < n; i += 32) { const float d = xr[i] - mu; v = fmaf(d, d, v); }
  const float rstd = 1.0f / sqrtf(warp_sum(v) / (float)n + eps);
  for (int i = lane; i < n; i += 32) yr[i] = (xr[i] - mu) * rstd * w[i] + b[i];
}

cudaError_t launch_layernorm(const float* x, const int64_t* gather, const float* w, const float* b,
                             float* y, int rows, int n, float eps, bool apply_norm, cudaStream_t s) {
  if (rows <= 0) return cudaSuccess;
  layernorm_kernel<<<(rows + 7) / 8, 256, 0, s>>>(x, gather, w, b, y, rows, n, eps, apply_norm);
  count_launch();
  return cudaGetLastError();
}

__global__ void broadcast_rows_kernel(const float* __restrict__ src, float* __restrict__ dst,
                                      long per, long total) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < total) dst[i] = src[i % per];
}
cudaError_t launch_broadcast_rows(const float* src, float* dst, int batch, int rows, int n, cudaStream_t s) {
  const long per = (long)rows * n, total = per * batch;
  broadcast_rows_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(src, dst, per, total);
  count_launch();
  return cudaGetLastError();
}

// -------------------------------------------------------------------- positional table
__global__ void pos_level_kernel(const float* __restrict__ level_embed, float* __restrict__ out,
                                 int h, int w, int C) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  const long total = (long)h * w * C;
  if (i >= total) return;
  const int c = (int)(i % C);
  const int key = (int)(i / C);
  const int row = key / w, col = key % w;
  const int F = C / 2;
  const bool is_y = c < F;
  const int cc = is_y ? c : c - F;
  const float scale = 6.283185307179586f;  // float32(2*pi)
  const float num = is_y ? (float)(row + 1) : (float)(col + 1);
  const float den = (is_y ? (float)h : (float)w) + 1e-6f;
  const float e = num / den * scale;
  const float dim_t = (float)pow(10000.0, (double)(2 * (cc / 2)) / (double)F);
  const float a = e / dim_t;
  const float v = (cc & 1) ? (float)cos((double)a) : (float)sin((double)a);
  out[i] = v + (level_embed ? level_embed[c] : 0.f);
}
cudaError_t launch_pos_level(const float* level_embed, float* out, int h, int w, int C, cudaStream_t s) {
  const long total = (long)h * w * C;
  pos_level_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(level_embed, out, h, w, C);
  count_launch();
  return cudaGetLastError();
}

// ---------------------------------------------------------------- K3: attention-mask bits
// F.interpolate(bilinear, align_corners=False) -> sigmoid() < 0.5 -> bit-pack, with the index math and threshold of
// common.cuh; all_masked_kernel (gemm_tc.cu) then flags the rows that are masked at every key.
// one warp per (row, 32-key word): 400 rows alone would leave most of the machine idle
__global__ void __launch_bounds__(256) mask_bits_kernel(const float* __restrict__ mask_pred, long words, int W32,
                                                        int H4, int W4, int th, int tw,
                                                        uint32_t* __restrict__ bitmap) {
  const long wid = (long)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (wid >= words) return;
  const long row = wid / W32;
  const int wi = (int)(wid % W32);
  const float* mp = mask_pred + row * H4 * W4;
  const int K = th * tw;
  const float sh = (float)H4 / (float)th, sw = (float)W4 / (float)tw;
  const int key = wi * 32 + lane;
  bool m = false;
  if (key < K) {
    const int r = key / tw, c = key % tw;
    const BilinearAxis y = bilinear_src(sh, r, H4), x = bilinear_src(sw, c, W4);
    const float a = mp[(long)y.i0 * W4 + x.i0], bq = mp[(long)y.i0 * W4 + x.i1];
    const float cq = mp[(long)y.i1 * W4 + x.i0], dq = mp[(long)y.i1 * W4 + x.i1];
    const float d = y.l0 * (x.l0 * a + x.l1 * bq) + y.l1 * (x.l0 * cq + x.l1 * dq);
    m = masked_from_logit(d);
  }
  const uint32_t word = __ballot_sync(0xffffffffu, m);
  if (lane == 0) bitmap[wid] = word;
}
cudaError_t launch_mask_bits(const float* mask_pred, int rows, int H4, int W4, int th, int tw,
                             uint32_t* bitmap, uint8_t* all_masked, cudaStream_t s) {
  if (rows <= 0) return cudaSuccess;
  const int K = th * tw, W32 = (K + 31) / 32;
  const long words = (long)rows * W32;
  mask_bits_kernel<<<(unsigned)((words + 7) / 8), 256, 0, s>>>(mask_pred, words, W32, H4, W4, th, tw, bitmap);
  all_masked_kernel<<<(rows + 7) / 8, 256, 0, s>>>(bitmap, rows, W32, K, all_masked);
  count_launch(2);
  return cudaGetLastError();
}

// --------------------------------------------------------------- attention core (fp32)
constexpr int AQT = 16, AKT = 128, AHD = 32;

__global__ void __launch_bounds__(128) attention_f32_kernel(
    const float* __restrict__ q, const float* __restrict__ k, const float* __restrict__ v,
    long kv_stride, long kv_bstride, const uint32_t* __restrict__ bitmap,
    const uint8_t* __restrict__ all_masked, float* __restrict__ out, int Q, int K, int heads) {
  __shared__ float qs[AQT][AHD];
  __shared__ float Ks[AKT][AHD + 1];
  __shared__ __align__(16) float Vs[AKT][AHD];
  __shared__ float Ps[AQT][AKT];
  __shared__ float red[4][AQT];
  __shared__ float m_run[AQT], scale_s[AQT];
  __shared__ uint32_t Ms[AQT][AKT / 32];
  const int q0 = blockIdx.x * AQT, h = blockIdx.y, b = blockIdx.z;
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const int C = heads * AHD;
  for (int i = t; i < AQT * AHD; i += 128) {
    const int qq = i / AHD, d = i % AHD;
    qs[qq][d] = (q0 + qq < Q) ? q[((long)b * Q + q0 + qq) * C + h * AHD + d] : 0.f;
  }
  if (t < AQT) m_run[t] = -INFINITY;
  const int pq = t >> 3, pd = (t & 7) * 4;
  float o[4] = {0.f, 0.f, 0.f, 0.f};
  float l = 0.f;
  const int W32 = (K + 31) / 32;
  const bool use_mask = bitmap != nullptr;
  for (int kt0 = 0; kt0 < K; kt0 += AKT) {
    __syncthreads();
    if (use_mask) {
      bool all_ones = true;
      if (t < AQT * 4) {
        const int qq = t >> 2, wi = t & 3, gq = q0 + qq, widx = kt0 / 32 + wi;
        uint32_t wv = 0xffffffffu;
        if (gq < Q && widx < W32) {
          wv = bitmap[((long)b * Q + gq) * W32 + widx];
          if (all_masked && all_masked[(long)b * Q + gq]) wv = 0u;   // fallback: attend everywhere
          if (widx == W32 - 1 && (K & 31)) wv |= ~((1u << (K & 31)) - 1u);  // tail = not a key
        }
        Ms[qq][wi] = wv;
        all_ones = (wv == 0xffffffffu);
      }
      if (__syncthreads_and(all_ones)) continue;   // whole key tile masked for every query here
    }
    for (int i = t; i < AKT * AHD; i += 128) {
      const int kk = i / AHD, d = i % AHD, gk = kt0 + kk;
      float kv = 0.f, vv = 0.f;
      if (gk < K) {
        const long off = (long)b * kv_bstride + (long)gk * kv_stride + h * AHD + d;
        kv = k[off];
        vv = v[off];
      }
      Ks[kk][d] = kv;
      Vs[kk][d] = vv;
    }
    __syncthreads();
    float kr[AHD];
#pragma unroll
    for (int d = 0; d < AHD; ++d) kr[d] = Ks[t][d];
    const bool kvalid = (kt0 + t) < K;
    float sc[AQT];
#pragma unroll
    for (int qq = 0; qq < AQT; ++qq) {
      float acc = 0.f;
#pragma unroll
      for (int d = 0; d < AHD; ++d) acc = fmaf(qs[qq][d], kr[d], acc);
      bool masked = !kvalid;
      if (use_mask) masked = masked || ((Ms[qq][t >> 5] >> (t & 31)) & 1u);
      sc[qq] = masked ? -INFINITY : acc;
      const float mx = warp_max(sc[qq]);
      if (lane == 0) red[warp][qq] = mx;
    }
    __syncthreads();
    if (t < AQT) {
      const float mold = m_run[t];
      const float mt = fmaxf(fmaxf(red[0][t], red[1][t]), fmaxf(red[2][t], red[3][t]));
      const float mnew = fmaxf(mold, mt);
      scale_s[t] = (mnew == -INFINITY) ? 1.f : expf(mold - mnew);
      m_run[t] = mnew;
    }
    __syncthreads();
#pragma unroll
    for (int qq = 0; qq < AQT; ++qq)
      Ps[qq][t] = (sc[qq] == -INFINITY) ? 0.f : expf(sc[qq] - m_run[qq]);
    __syncthreads();
    const float s0 = scale_s[pq];
    o[0] *= s0; o[1] *= s0; o[2] *= s0; o[3] *= s0;
    l *= s0;
#pragma unroll 8
    for (int kk = 0; kk < AKT; ++kk) {
      const float pv = Ps[pq][kk];
      const float4 vv = *reinterpret_cast<const float4*>(&Vs[kk][pd]);
      o[0] = fmaf(pv, vv.x, o[0]);
      o[1] = fmaf(pv, vv.y, o[1]);
      o[2] = fmaf(pv, vv.z, o[2]);
      o[3] = fmaf(pv, vv.w, o[3]);
      l += pv;
    }
  }
  if (q0 + pq < Q) {
    const float inv = (l > 0.f) ? 1.0f / l : 0.f;
    const long off = ((long)b * Q + q0 + pq) * C + h * AHD + pd;
    out[off] = o[0] * inv; out[off + 1] = o[1] * inv; out[off + 2] = o[2] * inv; out[off + 3] = o[3] * inv;
  }
}

cudaError_t launch_attention_f32(const float* q, const float* k, const float* v, long kv_stride, long kv_bstride,
                                 const uint32_t* bitmap, const uint8_t* all_masked, float* out, int B, int Q, int K,
                                 int heads, cudaStream_t s) {
  if (B <= 0 || Q <= 0) return cudaSuccess;
  dim3 grid((Q + AQT - 1) / AQT, heads, B);
  attention_f32_kernel<<<grid, 128, 0, s>>>(q, k, v, kv_stride, kv_bstride, bitmap, all_masked, out, Q, K, heads);
  count_launch();
  return cudaGetLastError();
}

// -------------------------------------------------------------------------- K7 grounding
// One CTA per (caption i, image j): S[t,q] = cap_i[t].pred_j[q]/T in shared memory, then the
// l2v softmax over queries (token-masked) and the v2l softmax over ALL max_tokens.
__global__ void __launch_bounds__(256) grounding_pairs_kernel(
    const float* __restrict__ pred, const float* __restrict__ cap, const int64_t* __restrict__ cap_mask,
    int Bg, int Q, int T, int D, float inv_temp, float* __restrict__ g_l2v, float* __restrict__ g_v2l,
    const float* __restrict__ S_pre) {
  extern __shared__ float sm[];
  float* S = sm;                 // T*Q
  float* part_t = S + T * Q;     // T
  float* part_q = part_t + T;    // Q
  const int i = blockIdx.y, j = blockIdx.x, t = threadIdx.x;
  const float* ci = cap + (long)i * T * D;
  const float* pj = pred + (long)j * Q * D;
  // S_pre: the similarities of ALL pairs, (Bg*T, Bg*Q) row-major, already divided by the temperature -- one tcgen05
  // GEMM (cgg_grounding_loss, tensor-core mode) instead of T*Q dot products per CTA
  if (S_pre) {
    for (int idx = t; idx < T * Q; idx += 256) {
      const int tt = idx / Q, qq = idx % Q;
      S[idx] = S_pre[((long)i * T + tt) * ((long)Bg * Q) + (long)j * Q + qq];
    }
  } else
  for (int idx = t; idx < T * Q; idx += 256) {
    const int tt = idx / Q, qq = idx % Q;
    const float4* a = reinterpret_cast<const float4*>(ci + (long)tt * D);
    const float4* bq = reinterpret_cast<const float4*>(pj + (long)qq * D);
    float acc = 0.f;
    for (int d = 0; d < D / 4; ++d) {
      const float4 x = a[d], y = bq[d];
      acc = fmaf(x.x, y.x, acc); acc = fmaf(x.y, y.y, acc);
      acc = fmaf(x.z, y.z, acc); acc = fmaf(x.w, y.w, acc);
    }
    S[idx] = acc * inv_temp;
  }
  __syncthreads();
  const int lane = t & 31, warp = t >> 5;
  for (int tt = warp; tt < T; tt += 8) {       // l2v: softmax over queries for token tt
    float mx = -INFINITY;
    for (int qq = lane; qq < Q; qq += 32) mx = fmaxf(mx, S[tt * Q + qq]);
    mx = warp_max(mx);
    float se = 0.f, sd = 0.f;
    for (int qq = lane; qq < Q; qq += 32) {
      const float sv = S[tt * Q + qq], e = expf(sv - mx);
      se += e;
      sd = fmaf(e, -sv, sd);
    }
    se = warp_sum(se);
    sd = warp_sum(sd);
    if (lane == 0) part_t[tt] = (cap_mask[(long)i * T + tt] != 0) ? sd / se : 0.f;
  }
  for (int qq = t; qq < Q; qq += 256) {        // v2l: softmax over tokens for query qq
    float mx = -INFINITY;
    for (int tt = 0; tt < T; ++tt) mx = fmaxf(mx, S[tt * Q + qq]);
    float se = 0.f, sd = 0.f;
    for (int tt = 0; tt < T; ++tt) {
      const float sv = S[tt * Q + qq], e = expf(sv - mx);
      se += e;
      sd = fmaf(e, -sv, sd);
    }
    part_q[qq] = sd / se;
  }
  __syncthreads();
  if (t == 0) {
    float a = 0.f;
    long ntok = 0;
    for (int tt = 0; tt < T; ++tt) { a += part_t[tt]; ntok += (cap_mask[(long)i * T + tt] != 0); }
    g_l2v[i * Bg + j] = a / (float)(ntok > 0 ? ntok : 1);
  } else if (t == 32) {
    float a = 0.f;
    for (int qq = 0; qq < Q; ++qq) a += part_q[qq];
    g_v2l[i * Bg + j] = a / (float)Q;
  }
}

cudaError_t launch_grounding_pairs(const float* pred, const float* cap, const int64_t* cap_mask,
                                   int Bg, int Q, int T, int D, float temperature,
                                   float* g_l2v, float* g_v2l, cudaStream_t s, const float* S_pre) {
  const size_t smem = (size_t)(T * Q + T + Q) * sizeof(float);
  cudaError_t e = cudaFuncSetAttribute(grounding_pairs_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  grounding_pairs_kernel<<<dim3(Bg, Bg), 256, smem, s>>>(pred, cap, cap_mask, Bg, Q, T, D,
                                                         1.0f / temperature, g_l2v, g_v2l, S_pre);
  count_launch();
  return cudaGetLastError();
}

// cost (Bg,Bg): rows = captions, cols = images.  Empty captions -> max()+100, then the four
// log-softmax diagonals (grounding_loss.py:52-75).
__global__ void __launch_bounds__(256) grounding_finish_kernel(
    const float* __restrict__ g_l2v, const float* __restrict__ g_v2l, const int64_t* __restrict__ cap_mask,
    int Bg, int T, float loss_weight, float* __restrict__ loss, float* __restrict__ dg_l2v, float* __restrict__ dg_v2l) {
  extern __shared__ float sm[];
  float* cost = sm;                 // Bg*Bg
  float* diag = cost + Bg * Bg;     // Bg (per-row loss terms)
  __shared__ float total;
  __shared__ float gmax;
  const int t = threadIdx.x;
  if (t == 0) total = 0.f;
  for (int which = 0; which < 2; ++which) {
    const float* g = which == 0 ? g_l2v : g_v2l;
    __syncthreads();
    if (t == 0) {
      float m = -INFINITY;
      for (int x = 0; x < Bg * Bg; ++x) m = fmaxf(m, g[x]);
      gmax = m;
    }
    __syncthreads();
    for (int x = t; x < Bg * Bg; x += 256) {
      const int i = x / Bg;
      long ntok = 0;
      for (int tt = 0; tt < T; ++tt) ntok += (cap_mask[(long)i * T + tt] != 0);
      cost[x] = -((ntok > 0) ? g[x] : gmax + 100.0f);   // logits = -cost
    }
    __syncthreads();
    for (int d = t; d < Bg; d += 256) {
      // log_softmax over dim 0 (captions) at column d, and over dim 1 (images) at row d
      float m0 = -INFINITY, m1 = -INFINITY;
      for (int x = 0; x < Bg; ++x) { m0 = fmaxf(m0, cost[x * Bg + d]); m1 = fmaxf(m1, cost[d * Bg + x]); }
      float s0 = 0.f, s1 = 0.f;
      for (int x = 0; x < Bg; ++x) { s0 += expf(cost[x * Bg + d] - m0); s1 += expf(cost[d * Bg + x] - m1); }
      const float c = cost[d * Bg + d];
      diag[d] = -((c - m0) - logf(s0)) - ((c - m1) - logf(s1));
    }
    __syncthreads();
    if (t == 0) {
      float a = 0.f;
      for (int d = 0; d < Bg; ++d) a += diag[d];
      total += a / (float)Bg;
    }
    float* dg = which == 0 ? dg_l2v : dg_v2l;
    if (dg) {
      // d loss / d cost[i,j] = w/(4 Bg) * (2 delta_ij - softmax_dim0(-cost)[i,j] - softmax_dim1(-cost)[i,j]); rows of
      // empty captions were replaced by a detached constant (grounding_loss.py:52-61) -> zero gradient
      __syncthreads();
      for (int x = t; x < Bg * Bg; x += 256) {
        const int i = x / Bg, j = x % Bg;
        long ntok = 0;
        for (int tt = 0; tt < T; ++tt) ntok += (cap_mask[(long)i * T + tt] != 0);
        float m0 = -INFINITY, m1 = -INFINITY;
        for (int y = 0; y < Bg; ++y) { m0 = fmaxf(m0, cost[y * Bg + j]); m1 = fmaxf(m1, cost[i * Bg + y]); }
        float s0 = 0.f, s1 = 0.f;
        for (int y = 0; y < Bg; ++y) { s0 += expf(cost[y * Bg + j] - m0); s1 += expf(cost[i * Bg + y] - m1); }
        const float p0 = expf(cost[x] - m0) / s0, p1 = expf(cost[x] - m1) / s1;
        dg[x] = ntok > 0 ? loss_weight / (4.0f * (float)Bg) * ((i == j ? 2.0f : 0.0f) - p0 - p1) : 0.f;
      }
    }
  }
  __syncthreads();
  if (t == 0) loss[0] = loss_weight * total / 4.0f;
}

cudaError_t launch_grounding_finish(const float* g_l2v, const float* g_v2l, const int64_t* cap_mask,
                                    int Bg, int T, float loss_weight, float* loss, cudaStream_t s, float* dg_l2v,
                                    float* dg_v2l) {
  const size_t smem = (size_t)(Bg * Bg + Bg) * sizeof(float);
  cudaError_t e = cudaFuncSetAttribute(grounding_finish_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  grounding_finish_kernel<<<1, 256, smem, s>>>(g_l2v, g_v2l, cap_mask, Bg, T, loss_weight, loss, dg_l2v, dg_v2l);
  count_launch();
  return cudaGetLastError();
}

// Backward of the pair distances w.r.t. the similarities: one CTA per (caption i, image j) recomputes
// S in shared memory and writes dS[j][i][t][q] * (1/temperature) (image-major so that the following
// batched GEMM  dpred_j = dS_j^T . cap  is deterministic).
//   l2v: f_t = -sum_q a_tq S_tq, a = softmax_q  ->  d f_t / d S_tq = -a_tq (1 + S_tq + f_t)
//   v2l: g_q = -sum_t b_tq S_tq, b = softmax_t  ->  d g_q / d S_tq = -b_tq (1 + S_tq + g_q)
__global__ void __launch_bounds__(256) grounding_bwd_pairs_kernel(
    const float* __restrict__ pred, const float* __restrict__ cap, const int64_t* __restrict__ cap_mask,
    int Bg, int Q, int T, int D, float inv_temp, const float* __restrict__ dg_l2v, const float* __restrict__ dg_v2l,
    float grad_scale, float* __restrict__ dS, const float* __restrict__ S_pre, __nv_bfloat16* __restrict__ dS_hl, int Kp) {
  extern __shared__ float sm[];
  float* S = sm;                   // T*Q
  float* st_max = S + T * Q;       // per token: max, 1/sum, f_t
  float* st_inv = st_max + T;
  float* st_f = st_inv + T;
  float* sq_max = st_f + T;        // per query: max, 1/sum, g_q
  float* sq_inv = sq_max + Q;
  float* sq_g = sq_inv + Q;
  const int i = blockIdx.y, j = blockIdx.x, t = threadIdx.x;
  const float* ci = cap + (long)i * T * D;
  const float* pj = pred + (long)j * Q * D;
  if (S_pre) {
    for (int idx = t; idx < T * Q; idx += 256) {
      const int tt = idx / Q, qq = idx % Q;
      S[idx] = S_pre[((long)i * T + tt) * ((long)Bg * Q) + (long)j * Q + qq];
    }
  } else
  for (int idx = t; idx < T * Q; idx += 256) {
    const int tt = idx / Q, qq = idx % Q;
    const float4* a = reinterpret_cast<const float4*>(ci + (long)tt * D);
    const float4* bq = reinterpret_cast<const float4*>(pj + (long)qq * D);
    float acc = 0.f;
    for (int d = 0; d < D / 4; ++d) {
      const float4 x = a[d], y = bq[d];
      acc = fmaf(x.x, y.x, acc); acc = fmaf(x.y, y.y, acc);
      acc = fmaf(x.z, y.z, acc); acc = fmaf(x.w, y.w, acc);
    }
    S[idx] = acc * inv_temp;
  }
  __syncthreads();
  const int lane = t & 31, warp = t >> 5;
  for (int tt = warp; tt < T; tt += 8) {
    float mx = -INFINITY;
    for (int qq = lane; qq < Q; qq += 32) mx = fmaxf(mx, S[tt * Q + qq]);
    mx = warp_max(mx);
    float se = 0.f, sd = 0.f;
    for (int qq = lane; qq < Q; qq += 32) {
      const float sv = S[tt * Q + qq], e = expf(sv - mx);
      se += e;
      sd = fmaf(e, -sv, sd);
    }
    se = warp_sum(se);
    sd = warp_sum(sd);
    if (lane == 0) { st_max[tt] = mx; st_inv[tt] = 1.0f / se; st_f[tt] = sd / se; }
  }
  for (int qq = t; qq < Q; qq += 256) {
    float mx = -INFINITY;
    for (int tt = 0; tt < T; ++tt) mx = fmaxf(mx, S[tt * Q + qq]);
    float se = 0.f, sd = 0.f;
    for (int tt = 0; tt < T; ++tt) {
      const float sv = S[tt * Q + qq], e = expf(sv - mx);
      se += e;
      sd = fmaf(e, -sv, sd);
    }
    sq_max[qq] = mx; sq_inv[qq] = 1.0f / se; sq_g[qq] = sd / se;
  }
  __syncthreads();
  long ntok = 0;
  for (int tt = 0; tt < T; ++tt) ntok += (cap_mask[(long)i * T + tt] != 0);
  const float gl = dg_l2v[i * Bg + j] * grad_scale / (float)(ntok > 0 ? ntok : 1);
  const float gv = dg_v2l[i * Bg + j] * grad_scale / (float)Q;
  float* out = dS + (((long)j * Bg + i) * T) * Q;
  for (int idx = t; idx < T * Q; idx += 256) {
    const int tt = idx / Q, qq = idx % Q;
    const float sv = S[idx];
    const float a = expf(sv - st_max[tt]) * st_inv[tt];
    const float b = expf(sv - sq_max[qq]) * sq_inv[qq];
    const float m = (cap_mask[(long)i * T + tt] != 0) ? 1.f : 0.f;
    const float d = (gl * m * (-a) * (1.0f + sv + st_f[tt]) + gv * (-b) * (1.0f + sv + sq_g[qq])) * inv_temp;
    if (dS_hl) {
      // tensor-core mode: row (j, q) of the K-major operand of dpred = dS . cap, column (i, t), as a bf16 hi/lo pair
      const __nv_bfloat16 hi = __float2bfloat16_rn(d);
      __nv_bfloat16* row = dS_hl + ((long)j * Q + qq) * 2 * Kp + (long)i * T + tt;
      row[0] = hi;
      row[Kp] = __float2bfloat16_rn(d - __bfloat162float(hi));
    } else {
      out[idx] = d;
    }
  }
}

// cap (R rows, D) fp32 -> capT (D rows, 2*Kp) bf16 [hi | lo], column = source row (zero padded to Kp)
__global__ void transpose_split_kernel(const float* __restrict__ in, __nv_bfloat16* __restrict__ out, int R, int D, int Kp) {
  const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long)D * Kp) return;
  const int r = (int)(idx % Kp), d = (int)(idx / Kp);
  const float x = r < R ? in[(long)r * D + d] : 0.f;
  const __nv_bfloat16 hi = __float2bfloat16_rn(x);
  out[(long)d * 2 * Kp + r] = hi;
  out[(long)d * 2 * Kp + Kp + r] = __float2bfloat16_rn(x - __bfloat162float(hi));
}
cudaError_t launch_transpose_split(const float* in, __nv_bfloat16* out, int R, int D, int Kp, cudaStream_t s) {
  const long n = (long)D * Kp;
  transpose_split_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(in, out, R, D, Kp);
  count_launch();
  return cudaGetLastError();
}

cudaError_t launch_grounding_bwd_pairs(const float* pred, const float* cap, const int64_t* cap_mask, int Bg, int Q, int T,
                                       int D, float temperature, const float* dg_l2v, const float* dg_v2l,
                                       float grad_scale, float* dS, cudaStream_t s, const float* S_pre, __nv_bfloat16* dS_hl, int Kp) {
  const size_t smem = (size_t)(T * Q + 3 * T + 3 * Q) * sizeof(float);
  cudaError_t e = cudaFuncSetAttribute(grounding_bwd_pairs_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  grounding_bwd_pairs_kernel<<<dim3(Bg, Bg), 256, smem, s>>>(pred, cap, cap_mask, Bg, Q, T, D, 1.0f / temperature, dg_l2v,
                                                             dg_v2l, grad_scale, dS, S_pre, dS_hl, Kp);
  count_launch();
  return cudaGetLastError();
}

// x[row, :] /= ||x[row, :]||_2 in place (pred_emb_norm, head.py:743-744); one warp per row
__global__ void __launch_bounds__(256) l2norm_rows_kernel(float* __restrict__ x, int rows, int D) {
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= rows) return;
  float* r = x + (long)row * D;
  float ss = 0.f;
  for (int i = lane; i < D; i += 32) ss = fmaf(r[i], r[i], ss);
  ss = warp_sum(ss);
  const float n = sqrtf(ss);
  for (int i = lane; i < D; i += 32) r[i] = r[i] / n;
}

cudaError_t launch_l2norm_rows(float* x, int rows, int D, cudaStream_t s) {
  l2norm_rows_kernel<<<(rows + 7) / 8, 256, 0, s>>>(x, rows, D);
  count_launch();
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------- cast
__global__ void cast_bf16_kernel(const float* __restrict__ in, __nv_bfloat16* __restrict__ out, size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = __float2bfloat16_rn(in[i]);
}
cudaError_t launch_cast_bf16(const float* in, __nv_bfloat16* out, size_t n, cudaStream_t s) {
  if (n == 0) return cudaSuccess;
  cast_bf16_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(in, out, n);
  count_launch();
  return cudaGetLastError();
}

__global__ void cast_f16_kernel(const float* __restrict__ in, __half* __restrict__ out, size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = __float2half_rn(in[i]);
}
cudaError_t launch_cast_f16(const float* in, void* out, size_t n, cudaStream_t s) {
  if (n == 0) return cudaSuccess;
  cast_f16_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(in, static_cast<__half*>(out), n);
  count_launch();
  return cudaGetLastError();
}

__global__ void cast_bf16_split_kernel(const float* __restrict__ in, __nv_bfloat16* __restrict__ out, long n, int cols) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const long r = i / cols;
  const int c = (int)(i % cols);
  const float x = in[i];
  const __nv_bfloat16 hi = __float2bfloat16_rn(x);
  out[r * 2 * cols + c] = hi;
  out[r * 2 * cols + cols + c] = __float2bfloat16_rn(x - __bfloat162float(hi));
}
cudaError_t launch_cast_bf16_split(const float* in, __nv_bfloat16* out, int rows, int cols, cudaStream_t s) {
  const long n = (long)rows * cols;
  if (n == 0) return cudaSuccess;
  cast_bf16_split_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(in, out, n, cols);
  count_launch();
  return cudaGetLastError();
}

}  // namespace cgg

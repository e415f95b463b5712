// Throughput-mode (CGG_BF16) orchestration of the query-side ("small-M") work: every linear layer
// of the decoder layer and of the query heads runs on the tcgen05 GEMM (gemm_tc.cu) with bf16
// K-major activations through TMA; bias / scale / ReLU / residual + LayerNorm live in the GEMM
// epilogues.  The decoder state x stays fp32 between layers (residual stream); only GEMM operands
// are rounded to bf16.
#include "common.cuh"
#include "gemm_tc.h"
#include "kernels.h"
#include "tc_ptx.cuh"
#include "tc_state.h"
#include <cuda_fp16.h>

#include <math.h>
#include <stdlib.h>

namespace cgg {

namespace {

// hi/lo bf16 pair of a float pair, packed
__device__ __forceinline__ void split_pack(float a, float b, uint32_t& hi, uint32_t& lo) {
  const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  const float2 back = __bfloat1622float2(h);
  const __nv_bfloat162 l = __floats2bfloat162_rn(a - back.x, b - back.y);
  hi = *reinterpret_cast<const uint32_t*>(&h);
  lo = *reinterpret_cast<const uint32_t*>(&l);
}

// dst = half(x + qe[row % Q]): the IEEE-half operand of the layer's q / k projections
__global__ void add_qe_cast_kernel(const float* __restrict__ x, const float* __restrict__ qe,
                                   __nv_bfloat16* __restrict__ dst, long total, int per /* Q*C */) {
  ptx::grid_dep_launch();
  ptx::grid_dep_wait();
  const long i = ((long)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (i >= total) return;
  const float4 a = *reinterpret_cast<const float4*>(x + i);
  const float4 b = *reinterpret_cast<const float4*>(qe + (i % per));
  const __half2 lo = __floats2half2_rn(a.x + b.x, a.y + b.y), hi = __floats2half2_rn(a.z + b.z, a.w + b.w);
  uint2 pk;
  pk.x = *reinterpret_cast<const uint32_t*>(&lo);
  pk.y = *reinterpret_cast<const uint32_t*>(&hi);
  *reinterpret_cast<uint2*>(dst + i) = pk;
}

// Row LayerNorm over 256 channels, one warp per row, every access coalesced.  Optional outputs: fp32 y; IEEE-half rows
// of y (out_bf16) and of y + qe[row % Q] (out_bf16_q) -- the operands of the layer's linear layers, which run on
// kind::f16 MMAs with HALF operands (11 significand bits: the residual stream is LayerNorm-scaled, so the range is no
// issue, and a CPU study shows bf16 operands here cost the attention masks ~0.1 % of their bits after 9 layers, half
// operands 0.01 %; DESIGN.md section 3) -- and a bf16 hi/lo pair row [hi(256) | lo(256)] of y or of its chained second
// LayerNorm (out_hl), the split-precision operand of the query heads.
__global__ void __launch_bounds__(256) ln_rows_kernel(const float* __restrict__ x, int nparts, long part_stride,
                                                      const float* __restrict__ w,
                                                      const float* __restrict__ b, int rows, float* __restrict__ out_f32,
                                                      __nv_bfloat16* __restrict__ out_bf16,
                                                      __nv_bfloat16* __restrict__ out_bf16_q,
                                                      const float* __restrict__ qe, int Q,
                                                      __nv_bfloat16* __restrict__ out_hl,
                                                      const float* __restrict__ w2, const float* __restrict__ b2) {
  ptx::grid_dep_launch();
  ptx::grid_dep_wait();
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= rows) return;
  const int n0 = lane * 8;
  const float4* xr = reinterpret_cast<const float4*>(x + (long)row * 256 + n0);
  const float4 a = xr[0], c = xr[1];
  float v[8] = {a.x, a.y, a.z, a.w, c.x, c.y, c.z, c.w};
  for (int pt = 1; pt < nparts; ++pt) {      // K-split partial sums of the producing GEMM, fixed order
    const float4* xp = reinterpret_cast<const float4*>(x + pt * part_stride + (long)row * 256 + n0);
    const float4 e = xp[0], f = xp[1];
    v[0] += e.x; v[1] += e.y; v[2] += e.z; v[3] += e.w; v[4] += f.x; v[5] += f.y; v[6] += f.z; v[7] += f.w;
  }
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) s += v[i];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  const float mu = s * (1.0f / 256.0f);
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) { const float d = v[i] - mu; q = fmaf(d, d, q); }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
  const float rstd = 1.0f / sqrtf(q * (1.0f / 256.0f) + 1e-5f);
  float y[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) y[i] = (v[i] - mu) * rstd * __ldg(w + n0 + i) + __ldg(b + n0 + i);
  if (out_f32) {
    float4* d = reinterpret_cast<float4*>(out_f32 + (long)row * 256 + n0);
    d[0] = make_float4(y[0], y[1], y[2], y[3]);
    d[1] = make_float4(y[4], y[5], y[6], y[7]);
  }
  auto store_hl = [&](__nv_bfloat16* dst, const float* v8) {
    uint4 ph, pl;
    split_pack(v8[0], v8[1], ph.x, pl.x);
    split_pack(v8[2], v8[3], ph.y, pl.y);
    split_pack(v8[4], v8[5], ph.z, pl.z);
    split_pack(v8[6], v8[7], ph.w, pl.w);
    *reinterpret_cast<uint4*>(dst + (long)row * 512 + n0) = ph;
    *reinterpret_cast<uint4*>(dst + (long)row * 512 + 256 + n0) = pl;
  };
  auto store_h = [&](__nv_bfloat16* dst, const float* v8) {
    uint4 pk;
    uint32_t* w = reinterpret_cast<uint32_t*>(&pk);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const __half2 h2 = __floats2half2_rn(v8[2 * i], v8[2 * i + 1]);
      w[i] = *reinterpret_cast<const uint32_t*>(&h2);
    }
    *reinterpret_cast<uint4*>(dst + (long)row * 256 + n0) = pk;
  };
  if (out_bf16) store_h(out_bf16, y);
  if (out_bf16_q) {
    const float* e = qe + (long)(row % Q) * 256 + n0;
    float yq[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) yq[i] = y[i] + e[i];
    store_h(out_bf16_q, yq);
  }
  if (out_hl && w2) {
    // chained second LayerNorm (post_norm of the head call that follows): z = LN(y; w2, b2)
    float s2 = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) s2 += y[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s2 += __shfl_xor_sync(0xffffffffu, s2, o);
    const float mu2 = s2 * (1.0f / 256.0f);
    float q2 = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) { const float d = y[i] - mu2; q2 = fmaf(d, d, q2); }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) q2 += __shfl_xor_sync(0xffffffffu, q2, o);
    const float rstd2 = 1.0f / sqrtf(q2 * (1.0f / 256.0f) + 1e-5f);
#pragma unroll
    for (int i = 0; i < 8; ++i) y[i] = (y[i] - mu2) * rstd2 * __ldg(w2 + n0 + i) + __ldg(b2 + n0 + i);
  }
  if (out_hl) store_hl(out_hl, y);
}

cudaError_t launch_ln_rows(const float* x, const float* w, const float* b, int rows, float* out_f32,
                           __nv_bfloat16* out_bf16, __nv_bfloat16* out_bf16_q, const float* qe, int Q,
                           __nv_bfloat16* out_hl, cudaStream_t s, const float* w2 = nullptr, const float* b2 = nullptr,
                           int nparts = 1, long part_stride = 0) {
  cudaError_t e = launch_pdl(ln_rows_kernel, dim3((rows + 7) / 8), dim3(256), 0, s, x, nparts, part_stride, w, b, rows, out_f32, out_bf16, out_bf16_q,
                             qe, Q > 0 ? Q : 1, out_hl, w2, b2);
  count_launch();
  return e != cudaSuccess ? e : cudaGetLastError();
}

template <typename T>
T* at(void* ws, size_t off) { return reinterpret_cast<T*>(static_cast<char*>(ws) + off); }

TcSeg seg(int col0, int ncols, void* ptr, long ld, bool bf16, bool relu, float alpha = 1.f, const float* rowbias = nullptr,
          int rb_mod = 1, long rb_ld = 0, bool split = false, const float* res = nullptr, long res_ld = 0) {
  TcSeg s;
  s.res = res; s.res_ld = res_ld; s.remap_q = 0; s.remap_rows = 0; s.remap_row0 = 0;
  s.col0 = col0; s.ncols = ncols; s.ptr = ptr; s.ld = ld; s.is_bf16 = bf16 ? 1 : 0; s.relu = relu ? 1 : 0;
  s.split = split ? 1 : 0;
  s.alpha = alpha; s.rowbias = rowbias; s.rb_mod = rb_mod; s.rb_ld = rb_ld;
  return s;
}

// CGG_DEBUG_SYNC=1: synchronise after every stage so a faulting kernel is named in the error.
inline bool debug_sync_on() {
  static const bool on = getenv("CGG_DEBUG_SYNC") != nullptr;
  return on;
}
#define TST(call)                                                                                      \
  do {                                                                                                 \
    int st__ = (call);                                                                                 \
    if (st__ != CGG_OK) return st__;                                                                   \
    if (debug_sync_on()) {                                                                             \
      cudaError_t e2__ = cudaStreamSynchronize(s);                                                     \
      if (e2__ != cudaSuccess)                                                                         \
        return tc_fail(t, CGG_ERR_CUDA, std::string("after ") + #call + ": " + cudaGetErrorString(e2__)); \
    }                                                                                                  \
  } while (0)

}  // namespace

// bf16 copies of every small-M weight, in the row order the fused GEMMs want.
int tc_pack_weights(TcState* t, const cgg_weights* w, cudaStream_t s) {
  const cgg_config& c = t->cfg;
  const int C = c.embed_dim, F = c.ffn_dim, Q = c.num_queries, L = c.num_layers;
  const int nh = round_up(c.d_lang + C + c.num_classes_p1, 256);
  if (c.d_lang % 16 != 0) return tc_fail(t, CGG_ERR_UNSUPPORTED, "d_lang must be a multiple of 16");
  if (!t->packed_alloc || t->nh_padded != nh) {
    t->free_packed();
    for (int i = 0; i < L; ++i) {
      TcState::LayerW& l = t->pl[i];
      // the layer chain's weights are kept in IEEE half (DESIGN.md section 3)
      TCU(cudaMalloc(&l.wq_c, (size_t)C * C * 2));
      TCU(cudaMalloc(&l.wo_c, (size_t)C * C * 2));
      TCU(cudaMalloc(&l.wqkv_s, (size_t)3 * C * C * 2));
      TCU(cudaMalloc(&l.wo_s, (size_t)C * C * 2));
      TCU(cudaMalloc(&l.w1, (size_t)F * C * 2));
      TCU(cudaMalloc(&l.w2, (size_t)C * F * 2));
      TCU(cudaMalloc(&l.rowbias_v, (size_t)Q * C * 4));
    }
    TCU(cudaMalloc(&t->wh, (size_t)nh * 2 * C * 2));       // hi/lo rows: the head chain runs at split precision
    TCU(cudaMalloc(&t->wme1, (size_t)C * 2 * C * 2));
    TCU(cudaMalloc(&t->wme2, (size_t)C * 2 * C * 2));
    TCU(cudaMalloc(&t->bias_h, (size_t)nh * 4));
    t->nh_padded = nh;
    t->packed_alloc = true;
  }
  for (int i = 0; i < L; ++i) {
    const cgg_layer_weights& lw = w->layers[i];
    TcState::LayerW& l = t->pl[i];
    TCU(launch_cast_f16(lw.cross_in_w, l.wq_c, (size_t)C * C, s));                  // Wq of the cross-attention
    TCU(launch_cast_f16(lw.cross_out_w, l.wo_c, (size_t)C * C, s));
    TCU(launch_cast_f16(lw.self_in_w, l.wqkv_s, (size_t)3 * C * C, s));             // [Wq; Wk; Wv] as stored
    TCU(launch_cast_f16(lw.self_out_w, l.wo_s, (size_t)C * C, s));
    TCU(launch_cast_f16(lw.ffn_w1, l.w1, (size_t)F * C, s));
    TCU(launch_cast_f16(lw.ffn_w2, l.w2, (size_t)C * F, s));
    // v = x Wv^T + bv = (x + qe) Wv^T + bv - qe Wv^T : the last term is a per-query constant
    GemmF32 g;
    g.A = w->query_embed; g.sAm = C; g.sAk = 1;
    g.W = lw.self_in_w + (size_t)2 * C * C; g.sWn = C; g.sWk = 1;
    g.C = l.rowbias_v; g.sCm = C; g.sCn = 1;
    g.M = Q; g.N = C; g.K = C; g.alpha = -1.f;
    TCU(launch_gemm_f32(g, s));
  }
  TCU(cudaMemsetAsync(t->wh, 0, (size_t)nh * 2 * C * 2, s));
  TCU(cudaMemsetAsync(t->bias_h, 0, (size_t)nh * 4, s));
  if (c.d_lang > 0) TCU(launch_cast_bf16_split(w->v2l_w, t->wh, c.d_lang, C, s));
  TCU(launch_cast_bf16_split(w->me_w[0], t->wh + (size_t)c.d_lang * 2 * C, C, C, s));
  TCU(launch_cast_bf16_split(w->cls_w, t->wh + (size_t)(c.d_lang + C) * 2 * C, c.num_classes_p1, C, s));
  if (c.d_lang > 0) TCU(cudaMemcpyAsync(t->bias_h, w->v2l_b, (size_t)c.d_lang * 4, cudaMemcpyDeviceToDevice, s));
  TCU(cudaMemcpyAsync(t->bias_h + c.d_lang, w->me_b[0], (size_t)C * 4, cudaMemcpyDeviceToDevice, s));
  TCU(cudaMemcpyAsync(t->bias_h + c.d_lang + C, w->cls_b, (size_t)c.num_classes_p1 * 4, cudaMemcpyDeviceToDevice, s));
  TCU(launch_cast_bf16_split(w->me_w[1], t->wme1, C, C, s));
  TCU(launch_cast_bf16_split(w->me_w[2], t->wme2, C, C, s));
  return CGG_OK;
}

// K1: post_norm -> [v2l_transform | mask_embed.0 + ReLU | cls_embed] in one GEMM -> mask_embed.2 -> .4
int tc_query_heads(TcState* t, const cgg_weights* w, int batch, const float* x, float* cls, float* emb, float* me,
                   void* ws, cudaStream_t s, int call_slot, bool z_ready) {
  const cgg_config& c = t->cfg;
  const int C = c.embed_dim, M = batch * c.num_queries;
  TcWs o;
  o.carve(t, batch);
  __nv_bfloat16* zb = at<__nv_bfloat16>(ws, o.zb);
  __nv_bfloat16* h1b = at<__nv_bfloat16>(ws, o.h1b);
  __nv_bfloat16* h2b = at<__nv_bfloat16>(ws, o.h2b);
  if (!z_ready) TCU(launch_ln_rows(x, w->post_norm_w, w->post_norm_b, M, nullptr, nullptr, nullptr, nullptr, 0, zb, s));
  // split precision (hi/lo bf16 pairs, 3 MMAs per product): the mask embedding feeds the
  // sigmoid<0.5 threshold, where plain bf16 operands flip ~0.15% of the attention-mask bits
  TcSeg sh[3] = {seg(0, c.d_lang, emb, c.d_lang, false, false),
                 seg(c.d_lang, C, h1b, 2 * C, true, true, 1.f, nullptr, 1, 0, /*split=*/true),
                 seg(c.d_lang + C, c.num_classes_p1, cls, c.num_classes_p1, false, false)};
  TST(tc_linear(t, zb, M, C, t->wh, t->nh_padded, t->bias_h, sh, 3, s, true));
  TcSeg s2[1] = {seg(0, C, h2b, 2 * C, true, true, 1.f, nullptr, 1, 0, true)};
  TST(tc_linear(t, h1b, M, C, t->wme1, C, w->me_b[1], s2, 1, s, true));
  TcSeg s3[1] = {seg(0, C, me, C, false, false)};
  if (!me) {
    // straight into the all-call B operand of the mask einsum / attention-mask GEMMs: hi | lo rows of 2C
    s3[0] = seg(0, C, at<__nv_bfloat16>(ws, o.me_all), 2 * C, true, false, 1.f, nullptr, 1, 0, /*split=*/true);
    s3[0].remap_q = c.num_queries; s3[0].remap_rows = t->rows_per_batch; s3[0].remap_row0 = call_slot * t->q_pad;
  }
  TST(tc_linear(t, h2b, M, C, t->wme2, C, w->me_b[2], s3, 1, s, true));
  return CGG_OK;
}

// K5 + K6: one DetrTransformerDecoderLayer (head.py:829-840), bf16 operands on tensor cores.
int tc_decoder_layer(TcState* t, const cgg_weights* w, int batch, int layer, const float* x_in, const void* k,
                     const void* v, long kv_stride, long kv_bstride, int num_keys, const uint32_t* bitmap,
                     const uint8_t* all_masked, float* x_out, void* ws, cudaStream_t s, bool chained_in, bool chained_out,
                     bool q_ready) {
  const cgg_config& c = t->cfg;
  const int C = c.embed_dim, Q = c.num_queries, M = batch * Q, F = c.ffn_dim;
  const cgg_layer_weights& lw = w->layers[layer];
  const TcState::LayerW& pw = t->pl[layer];
  const float qscale = 1.0f / sqrtf((float)(C / c.num_heads));
  TcWs o;
  o.carve(t, batch);
  __nv_bfloat16* xqb = at<__nv_bfloat16>(ws, o.xqb);
  __nv_bfloat16* xb = at<__nv_bfloat16>(ws, o.xb);
  __nv_bfloat16* ob = at<__nv_bfloat16>(ws, o.ob);
  __nv_bfloat16* fb = at<__nv_bfloat16>(ws, o.fb);
  float* qf = at<float>(ws, o.qf);
  float* qs = at<float>(ws, o.qs);
  float* kvs = at<float>(ws, o.kvs);
  float* x1 = at<float>(ws, o.x1);
  float* x2 = at<float>(ws, o.x2);
  float* t1 = at<float>(ws, o.t1);
  // ---- cross-attention: q = ((x + query_embed) Wq^T + bq) / sqrt(d)
  const long total = (long)M * C;
  if (!chained_in) {
    TCU(launch_pdl(add_qe_cast_kernel, dim3((unsigned)((total / 4 + 255) / 256)), dim3(256), 0, s, x_in, w->query_embed, xqb,
                   total, Q * C));
    count_launch();
    TCU(cudaGetLastError());
  }
  if (!q_ready) {      // (q_ready: tc_layer_qproj already ran, on a branch parallel to the head call)
    TcSeg sq[1] = {seg(0, C, qf, C, false, false, qscale)};
    TST(tc_linear(t, xqb, M, C, pw.wq_c, C, lw.cross_in_b, sq, 1, s, false, 1, 0, /*f16=*/true));
  }
  {
    const int level = layer % CGG_NUM_LEVELS, slot = layer / CGG_NUM_LEVELS;
    long rcols = 0;
    const void* rtab = tc_key_bias_table(t, level, &rcols);
    TST(tc_attention(t, batch, num_keys, qf, k, v, kv_stride, kv_bstride, bitmap, all_masked, nullptr, ob, s, rtab, rcols,
                     slot * C, /*out_mode: IEEE half*/ 2));
  }
  // x1 = LN(x + o Wo^T + bo);  also bf16(x1 + query_embed) for the self-attention projections
  TcSeg so[1] = {seg(0, C, t1, C, false, false, 1.f, nullptr, 1, 0, false, x_in, C)};
  TST(tc_linear(t, ob, M, C, pw.wo_c, C, lw.cross_out_b, so, 1, s, false, 1, 0, true));
  TCU(launch_ln_rows(t1, lw.norm_w[0], lw.norm_b[0], M, x1, nullptr, xqb, w->query_embed, Q, nullptr, s));
  // ---- self-attention: q, k from x1 + query_embed, v from x1 (per-query constant folded into rowbias_v)
  __nv_bfloat16* kvb = reinterpret_cast<__nv_bfloat16*>(kvs);          // (M, 2C) bf16: [k | v]
  TcSeg sk[3] = {seg(0, C, qs, C, false, false, qscale), seg(C, C, kvb, 2 * C, true, false),
                 seg(2 * C, C, kvb + C, 2 * C, true, false, 1.f, pw.rowbias_v, Q, C)};
  TST(tc_linear(t, xqb, M, C, pw.wqkv_s, 3 * C, lw.self_in_b, sk, 3, s, false, 1, 0, true));
  // the 100 x 100 self-attention runs on the same tcgen05 attention kernel (one key tile, no mask)
  TST(tc_attention(t, batch, Q, qs, kvb, kvb + C, 2 * C, (long)Q * 2 * C, nullptr, nullptr, nullptr, ob, s, nullptr, 0, 0,
                   /*out_mode: IEEE half*/ 2));
  TcSeg so2[1] = {seg(0, C, t1, C, false, false, 1.f, nullptr, 1, 0, false, x1, C)};
  TST(tc_linear(t, ob, M, C, pw.wo_s, C, lw.self_out_b, so2, 1, s, false, 1, 0, true));
  TCU(launch_ln_rows(t1, lw.norm_w[1], lw.norm_b[1], M, x2, xb, nullptr, nullptr, 0, nullptr, s));
  // ---- FFN
  TcSeg sf[1] = {seg(0, F, fb, F, true, true)};
  sf[0].is_bf16 = 3;                                   // IEEE half: the operand of FFN2
  TST(tc_linear(t, xb, M, C, pw.w1, F, lw.ffn_b1, sf, 1, s, false, 1, 0, true));
  TcSeg sf2[1] = {seg(0, C, t1, C, false, false, 1.f, nullptr, 1, 0, false, x2, C)};
  // K = 2048 over 4 K-parts (4x the CTAs, each a quarter of the chunk chain); the LayerNorm adds the parts
  const int kparts = (F / 64) % 4 == 0 ? 4 : 1;
  const long pstride = (long)M * C;
  TST(tc_linear(t, fb, M, F, pw.w2, C, lw.ffn_b2, sf2, 1, s, false, kparts, pstride, true));
  if (chained_out)   // also bf16(x_out + query_embed) for the next layer and post_norm(x_out) for the next head call
    TCU(launch_ln_rows(t1, lw.norm_w[2], lw.norm_b[2], M, x_out, nullptr, xqb, w->query_embed, Q, at<__nv_bfloat16>(ws, o.zb), s,
                       w->post_norm_w, w->post_norm_b, kparts, pstride));
  else
    TCU(launch_ln_rows(t1, lw.norm_w[2], lw.norm_b[2], M, x_out, nullptr, nullptr, nullptr, 0, nullptr, s, nullptr, nullptr,
                       kparts, pstride));
  return CGG_OK;
}

// The cross-attention query projection of `layer` from the bf16 (x + query_embed) copy the previous layer left in
// the workspace.  It depends on the decoder state only, not on the head call, so the whole-path entry point runs
// it on a helper stream underneath the head call's six kernels.
int tc_layer_qproj(TcState* t, const cgg_weights* w, int batch, int layer, void* ws, cudaStream_t s) {
  const cgg_config& c = t->cfg;
  const int C = c.embed_dim, M = batch * c.num_queries;
  const float qscale = 1.0f / sqrtf((float)(C / c.num_heads));
  TcWs o;
  o.carve(t, batch);
  TcSeg sq[1] = {seg(0, C, at<float>(ws, o.qf), C, false, false, qscale)};
  TST(tc_linear(t, at<__nv_bfloat16>(ws, o.xqb), M, C, t->pl[layer].wq_c, C, w->layers[layer].cross_in_b, sq, 1, s, false, 1, 0,
                true));
  return CGG_OK;
}

}  // namespace cgg

// Throughput-mode (CGG_BF16) side: bf16 operands on tcgen05 tensor cores, TMA-fed, fp32
// accumulation in TMEM.  Internal interface used by api.cu.
#pragma once
#include "../../include/cgg_b200.h"
#include <cuda_runtime.h>
#include <cuda_bf16.h>

namespace cgg {

struct TcState;

// One column segment of a row-major GEMM output: columns [col0, col0+ncols) of
//   y = (acc + bias[n] + rowbias[(m % rb_mod), n-col0]) * alpha + res[m, n-col0], optional ReLU, fp32 or bf16.
// col0 must be a multiple of 32 (a warp of the epilogue holds 32 consecutive features).
struct TcSeg {
  int col0, ncols;
  void* ptr; long ld;
  int is_bf16, relu;   // is_bf16: 0 = fp32 output, 1 = bf16, 3 = IEEE half
  int split;      // bf16 only: write x as a hi/lo pair, hi at column n, lo at column ncols+n of the row
  float alpha;
  const float* rowbias; int rb_mod; long rb_ld;
  const float* res; long res_ld;   // fp32 residual added after the scale: res[token*res_ld + (n - col0)]
  // optional output-row remap (split outputs): row = (token / remap_q) * remap_rows + remap_row0 + token % remap_q
  int remap_q, remap_rows, remap_row0;
};

TcState* tc_create(const cgg_config& cfg);
void tc_destroy(TcState* t);
const char* tc_last_error(const TcState* t);
size_t tc_workspace_bytes(const TcState* t, int batch);  // t may be null (fp32 mode) -> 0
size_t tc_workspace_offset(const TcState* t, int batch, const char* what);  // (size_t)-1 if unknown

// bf16 copies of the K/V projection weights and key-bias tables for the given sizes.
int tc_prepare(TcState* t, const cgg_weights* w, int H4, int W4, const int* lh, const int* lw, const int* nl,
               float* const* wkv_f32, float* const* rk_f32, float* const* bkv_f32, cudaStream_t s);

// K4: kv[b, key, :] = mem[b, :, key]^T Wkv^T + bias tables, bf16 out (B, K_l, nl*2C)
// cta_cap > 0: run on at most that many CTAs, for launches that overlap a latency-bound chain
int tc_kv_project(TcState* t, int level, int batch, const void* mem_bf16, void* kv_bf16, void* ws, cudaStream_t s,
                  int cta_cap = 0);

// Once per forward: the centre-2x2 averages of mask_features at the three level resolutions
// (bf16, (B,C,K_l) each) that the attention-mask GEMMs contract against.
int tc_downsample(TcState* t, int batch, const void* mask_features_bf16, void* ws, cudaStream_t s);

// Stores head call `call_idx`'s mask embeddings (fp32 (B,Q,C)) as bf16 rows of the all-layer
// B operand in the workspace.
int tc_store_mask_embed(TcState* t, int batch, int call_idx, const float* me_f32, void* ws, cudaStream_t s);

// K3 on tensor cores: attention-mask bitmap of head call `call_idx` for `level`:
//   bits = sigmoid( me . Fds_level ) < 0.5, ballot-packed in the epilogue; then all_masked.
int tc_mask_bits(TcState* t, int batch, int call_idx, int level, uint32_t* bitmap, uint8_t* all_masked, void* ws,
                 cudaStream_t s);

// K2: mask[b,q,p] = sum_c me[b,q,c] F[b,c,p], bf16 out.  first_call..first_call+num_calls-1 head
// calls in ONE pass over mask_features (A tile resident in shared memory across all of them).
// mask points at call `first_call`'s slice; consecutive calls are call_stride elements apart.
int tc_mask_einsum(TcState* t, int batch, int first_call, int num_calls, const void* mask_features_bf16,
                   void* mask_bf16, long call_stride, void* ws, cudaStream_t s);

// Small-M linear layers on tensor cores (rows = flattened (image, query)); bf16 K-major operands.
// split_k: A and W rows are [hi(256) | lo(256)] bf16 pairs and the contraction is evaluated as
// hi.hi + lo.hi + hi.lo (fp32 accumulate), i.e. with ~16 mantissa bits per operand (K must be 256).
int tc_linear(TcState* t, const __nv_bfloat16* A, int M, int K, const __nv_bfloat16* W, int n_padded, const float* bias,
              const TcSeg* segs, int nsegs, cudaStream_t s, bool split_k = false, int kparts = 1, long kpart_stride = 0,
              bool f16 = false);   // f16: both operands are IEEE half (11 significand bits) instead of bf16
// kparts > 1: the K range is split over gridDim.z CTAs; part z writes fp32 partial sums at ptr + z*kpart_stride
// (bias / residual added by part 0); the consumer (LayerNorm) adds the parts.
// The bf16-mode decoder layer (K5 + K6) and the query heads (K1) built from the pieces above.
// chained_in: the workspace already holds bf16(x_in + query_embed) (written by the previous layer's last
// LayerNorm); chained_out: the last LayerNorm also emits bf16(x_out + query_embed) and post_norm(x_out) as
// hi/lo pairs for the next head call / layer, which then skip their own preparation kernels.
int tc_decoder_layer(TcState* t, const cgg_weights* w, int batch, int layer, const float* x_in, const void* k,
                     const void* v, long kv_stride, long kv_bstride, int num_keys, const uint32_t* bitmap,
                     const uint8_t* all_masked, float* x_out, void* ws, cudaStream_t s, bool chained_in = false,
                     bool chained_out = false, bool q_ready = false);
int tc_layer_qproj(TcState* t, const cgg_weights* w, int batch, int layer, void* ws, cudaStream_t s);
// me_f32 == nullptr: the mask embeddings go straight into the all-call hi/lo operand (slot call_slot)
// from the last GEMM's epilogue; z_ready: post_norm(x) is already in the workspace.
int tc_query_heads(TcState* t, const cgg_weights* w, int batch, const float* x, float* cls, float* emb, float* me_f32,
                   void* ws, cudaStream_t s, int call_slot = 0, bool z_ready = false);

// K5 on tensor cores: masked multi-head cross-attention, flash-style over 128-key tiles.
// q (B,Q,heads*32) fp32 pre-scaled; k, v bf16 rows (b*kv_bstride + key*kv_stride); out fp32 and/or bf16
// (either may be null).
int tc_attention(TcState* t, int batch, int num_keys, const float* q, const void* k, const void* v, long kv_stride,
                 long kv_bstride, const uint32_t* bitmap, const uint8_t* all_masked, float* out,
                 __nv_bfloat16* out_bf16, cudaStream_t s, const void* r_table = nullptr, long r_cols = 0, int r_col0 = 0,
                 int out_mode = 0);   // out_bf16 format: 0 = bf16 rows, 1 = [hi(C) | lo(C)] bf16 pairs, 2 = IEEE half rows
// r_table: optional bf16 (num_keys, r_cols) key-bias table stored as [hi | lo] column halves;
// S += Q . (R_hi + R_lo)[:, r_col0 + head*32 ...]^T
const void* tc_key_bias_table(const TcState* t, int level, long* cols);
// K5 with the arguments of decoder layer `layer`'s cross-attention (its level's key-bias table at its slot's columns),
// or without a table for layer < 0; out fp32 and / or out_half IEEE half rows (either may be null).
int tc_layer_attention(TcState* t, int layer, int batch, int num_keys, const float* q, const void* k, const void* v,
                       long kv_stride, long kv_bstride, const uint32_t* bitmap, const uint8_t* all_masked, float* out,
                       void* out_half, cudaStream_t s);

}  // namespace cgg

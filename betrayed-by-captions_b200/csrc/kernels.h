// Internal launch interface between the C-ABI layer (api.cu) and the kernels.
// Not part of the public ABI.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>

struct cgg_beam_state;   // include/cgg_b200.h
struct cgg_gt_image;     // include/cgg_b200.h

namespace cgg {

// launch counter (cgg_launch_count)
void count_launch(int n = 1);
unsigned long long launch_count();

// ---------------------------------------------------------------------------------------
// Generic strided fp32 SIMT GEMM (parity mode + every latency-bound small-M op):
//   C[b,m,n] = epi( sum_k (A[b,m,k] + A2[m % a2_mod, k]) * W[b,n,k] )
//   epi(v)   = relu_{n >= relu_from}( (v + bias[n]) * alpha + R[b, m % r_mod, n] (n < r_ncols) )
// Element (m,k) of A lives at A + b*sAb + m*sAm + k*sAk, etc.  A_MMAJOR / C_MMAJOR only
// select which index is walked by consecutive lanes (coalescing), never the result.
struct GemmF32 {
  const float* A = nullptr; long sAb = 0, sAm = 0, sAk = 0;
  const float* A2 = nullptr; long sA2m = 0, sA2k = 0; int a2_mod = 1;
  const float* W = nullptr; long sWb = 0, sWn = 0, sWk = 0;
  const float* bias = nullptr;
  const float* R = nullptr; long sRb = 0, sRm = 0, sRn = 0; int r_mod = 1; int r_ncols = 1 << 30;
  float* C = nullptr; long sCb = 0, sCm = 0, sCn = 0;
  int M = 0, N = 0, K = 0, batch = 1;
  // two-level batch: z in [0, batch) -> (z / batch_inner) * sXb + (z % batch_inner) * sXb2 for A, W and C (R: z * sRb)
  int batch_inner = 1; long sAb2 = 0, sWb2 = 0, sCb2 = 0;
  bool accumulate = false;   // C = epi(...) + C  (gradient accumulation in place)
  int slot = 0;              // workspace slot of the split-K partial sums (one per concurrently used stream)
  // conv_cin > 0: 3x3 convolution (stride 1, zero padding 1) as an implicit GEMM over token-major images.  The batch is
  // (image, row y) = (z / batch_inner, z % batch_inner) with batch_inner = H, m = column x (M = W), k = tap * conv_cin + c
  // (K = 9 * conv_cin, tap = 3 * (dy + 1) + (dx + 1)):  A[z, m, k] = X[image, y + dy, x + dx, c], zero outside the image.
  int conv_cin = 0;
  int relu_from = 1 << 30;   // relu applied to columns n >= relu_from
  float alpha = 1.f;
  bool a_mmajor = false, c_mmajor = false;
};
cudaError_t launch_gemm_f32(const GemmF32& p, cudaStream_t s);

// Row LayerNorm: y[r,:] = (x[r,:]-mu)/sqrt(var+eps)*w + b ; rows of length n (n % 32 == 0 not
// required).  gather != nullptr: row r of x is x[gather[r], :] (BERT table lookup).
cudaError_t launch_layernorm(const float* x, const int64_t* gather, const float* w, const float* b,
                             float* y, int rows, int n, float eps, bool apply_norm, cudaStream_t s);

// x[b,q,:] = src[q,:]  (query_feat broadcast over the batch, head.py:808-809)
cudaError_t launch_broadcast_rows(const float* src, float* dst, int batch, int rows, int n, cudaStream_t s);

// mmdet SinePositionalEncoding(num_feats=C/2, normalize=True) + level embedding:
//   out[key, c] = pos(key, c) + level_embed[c]     (K, C) fp32
cudaError_t launch_pos_level(const float* level_embed, float* out, int h, int w, int C, cudaStream_t s);

// K3: mask logits (B*Q rows of H4*W4 fp32) -> bitmap words + all_masked flags for target (th,tw)
cudaError_t launch_mask_bits(const float* mask_pred, int rows, int H4, int W4, int th, int tw,
                             uint32_t* bitmap, uint8_t* all_masked, cudaStream_t s);
// all_masked[row] = every one of the row's K keys is masked (the reference's all-masked-row fallback,
// mask2former_head.py:825-826).  One warp per row, 256 threads per block; defined in gemm_tc.cu, where the bf16 route
// launches it with programmatic dependent launch.
__global__ void all_masked_kernel(const uint32_t* __restrict__ bitmap, int rows, int W32, int K,
                                  uint8_t* __restrict__ all_masked);

// K5/K6 attention core, fp32 SIMT flash-style.  q, out (B,Q,heads*32), q pre-scaled; k,v rows of heads*32 at
// (b*kv_bstride + key*kv_stride); bitmap (B,Q,ceil(K/32)) or nullptr.
cudaError_t launch_attention_f32(const float* q, const float* k, const float* v, long kv_stride, long kv_bstride,
                                 const uint32_t* bitmap, const uint8_t* all_masked, float* out, int B, int Q, int K,
                                 int heads, cudaStream_t s);

// K7 grounding: per (caption i, image j) pair distances, then the contrastive reduction.
cudaError_t launch_grounding_pairs(const float* pred, const float* cap, const int64_t* cap_mask,
                                   int Bg, int Q, int T, int D, float temperature,
                                   float* g_l2v, float* g_v2l, cudaStream_t s, const float* S_pre = nullptr);
// in-place L2 normalisation of rows (pred_emb_norm, head.py:743-744)
cudaError_t launch_l2norm_rows(float* x, int rows, int D, cudaStream_t s);
cudaError_t launch_grounding_finish(const float* g_l2v, const float* g_v2l, const int64_t* cap_mask,
                                    int Bg, int T, float loss_weight, float* loss, cudaStream_t s,
                                    float* dg_l2v = nullptr, float* dg_v2l = nullptr);
// backward: dS[j][i][t][q] = d loss / d (cap_i[t].pred_j[q]) (already divided by the temperature)
cudaError_t launch_grounding_bwd_pairs(const float* pred, const float* cap, const int64_t* cap_mask, int Bg, int Q, int T,
                                       int D, float temperature, const float* dg_l2v, const float* dg_v2l,
                                       float grad_scale, float* dS, cudaStream_t s, const float* S_pre = nullptr,
                                       __nv_bfloat16* dS_hl = nullptr, int Kp = 0);
// (R, D) fp32 -> (D, 2*Kp) bf16 [hi | lo] transposed, zero padded columns
cudaError_t launch_transpose_split(const float* in, __nv_bfloat16* out, int R, int D, int Kp, cudaStream_t s);

// ---- training step (train_kernels.cu)
cudaError_t launch_layernorm_bwd(const float* x, const float* w, const float* dy, float* dx, float* dw, float* db,
                                 float* partial, int rows, int n, float eps, cudaStream_t s);
cudaError_t launch_relu_bwd(const float* y, const float* dy, float* dx, long n, float alpha, cudaStream_t s);
cudaError_t launch_axpy(const float* in, float* out, long n, float alpha, cudaStream_t s);
cudaError_t launch_add_rows(const float* x, const float* add, float* out, int batch, long per, cudaStream_t s);
cudaError_t launch_sum_batch(const float* g, float* out, int batch, long per, cudaStream_t s);
cudaError_t launch_mem_prep(const float* mem, const float* level, const float* pos_level, float* key_in, float* val_in,
                            int B, int C, int K, cudaStream_t s);
cudaError_t launch_mem_prep_bwd(const float* dkey, const float* dval, float* dmem, int B, int C, int K, cudaStream_t s);
cudaError_t launch_colsum(const float* g, float* out, long rows, int n, float alpha, cudaStream_t s, bool accumulate = false);
// lse, dsum: (B, heads, Q) scratch each
cudaError_t launch_attention_bwd(const float* q, const float* k, const float* v, long kv_stride, long kv_bstride,
                                 const uint32_t* bitmap, const uint8_t* all_masked, const float* o, const float* dout,
                                 float* lse, float* dsum, float* dq, float* dk, float* dv, long dkv_stride,
                                 long dkv_bstride, int B, int Q, int K, int heads, cudaStream_t s);

// attention as tensor-core products (tf32 training mode): row softmax with the bitmap / dS = P o (dP - D), in place
cudaError_t launch_attn_softmax_rows(float* S, const uint32_t* bitmap, const uint8_t* all_masked, int B, int heads, int Q,
                                     int K, cudaStream_t s);
cudaError_t launch_attn_dscore(const float* P, float* dP, const float* O, const float* dO, int B, int heads, int head_dim,
                               int Q, int K, cudaStream_t s);

// ---- the matching-based losses after the path at training time (match_kernels.cu; SURVEY.md 8 row f2)
// mmcv point_sample: in (N, H, W), coords (N or 1, P, 2) as (x, y) in [0, 1] -> out (N, P); backward scatters into din
cudaError_t launch_point_sample(const float* in, const float* coords, float* out, int N, int H, int W, int P,
                                bool coords_shared, cudaStream_t s);
cudaError_t launch_point_sample_bwd(const float* dout, const float* coords, float* din, int N, int H, int W, int P,
                                    bool coords_shared, cudaStream_t s);
// Hungarian cost matrix (Q, G) from sampled mask logits x (Q, P), sampled ground truth g (G, P), class rows (Q, C1);
// stats: 4*Q + G floats of scratch
cudaError_t launch_matching_cost(const float* x, const float* g, const float* cls, const float* emb, const int64_t* labels,
                                 int Q, int G, int C1, int P, float w_cls, float w_emb, float w_mask, float w_dice, float eps,
                                 float* stats, float* cost, cudaStream_t s);
cudaError_t launch_point_losses(const float* x, const float* t, int N, int P, float eps, float* abc, float* dice_rows,
                                float* bce_rows, cudaStream_t s);
cudaError_t launch_point_losses_bwd(const float* x, const float* t, const float* abc, int N, int P, float eps,
                                    const float* g_dice, const float* g_bce, float* dx, cudaStream_t s);
// panoptic targets: ascending stuff labels (B, num_classes - num_things) and counts (B,) of the semantic maps (B, pixels);
// bitmap: B * ceil(num_stuff / 32) words of scratch.  Ground-truth point samples of (image, target) rows -> out (R, P)
cudaError_t launch_panoptic_stuff_labels(const void* sem, bool sem_i64, int B, long pixels, int num_things, int num_classes,
                                         uint32_t* bitmap, int64_t* labels, int* counts, cudaStream_t s);
cudaError_t launch_gt_point_sample(const cgg_gt_image* images, const int* rows, const float* coords, float* out, int R, int P,
                                   bool coords_per_image, cudaStream_t s);
cudaError_t launch_weighted_ce(const float* logits, const int64_t* labels, const float* cw, int R, int C1, float* row_loss,
                               float* row_w, float* lse, cudaStream_t s);
cudaError_t launch_weighted_ce_bwd(const float* logits, const int64_t* labels, const float* cw, const float* lse, int R, int C1,
                                   const float* grow, float* dlogits, cudaStream_t s);

// ---- the pixel decoder before the path (pixdec_kernels.cu; SURVEY.md 8 row f3), token-major fp32 activations
cudaError_t launch_ms_deform_attn(const float* value, long value_stride, const float* off, long off_stride, const float* logits,
                                  long logit_stride, float* out, int B, int S, int heads, int levels, int points, const int* hs,
                                  const int* ws, cudaStream_t s);
cudaError_t launch_ms_deform_attn_bwd(const float* value, const float* off, const float* logits, const float* dout, float* dvalue,
                                      float* doff, float* dlogits, int B, int S, int heads, int levels, int points, const int* hs,
                                      const int* ws, cudaStream_t s);
size_t group_norm_scratch_floats(int B, int P, int C, int G);
cudaError_t launch_group_norm(const float* x, const float* gamma, const float* beta, float* y, float* mean_rstd, float* scratch, int B,
                              int P, int C, int G, float eps, bool relu, cudaStream_t s);
cudaError_t launch_group_norm_bwd(const float* x, const float* dy, const float* mean_rstd, const float* gamma, float* dx, float* dgamma,
                                  float* dbeta, float* scratch, int B, int P, int C, int G, cudaStream_t s);
cudaError_t launch_upsample_add(const float* lat, const float* prev, long prev_bstride, float* out, int B, int H, int W, int h, int w,
                                int C, cudaStream_t s);
cudaError_t launch_upsample_add_bwd(const float* dout, float* dprev, int B, int H, int W, int h, int w, int C, cudaStream_t s);
cudaError_t launch_tokens_to_nchw(const float* in, long in_bstride, void* out, bool out_bf16, int B, int P, int C, cudaStream_t s);
cudaError_t launch_nchw_to_tokens(const float* in, float* out, long out_bstride, int B, int P, int C, bool accumulate, cudaStream_t s);

// ---- test-time step after the path (post_kernels.cu)
cudaError_t launch_upsample_masks(const void* logits, bool bf16, float* out, int planes, int h4, int w4, int up_h, int up_w,
                                  cudaStream_t s);
cudaError_t launch_instance_mask_stats(const void* logits, bool bf16, const int* geom, int B, int Q, int h4, int w4, int up_h,
                                       int up_w, int max_out_h, int max_out_w, uint32_t* bits, int* count, float* sig_sum,
                                       int* bbox, cudaStream_t s);
cudaError_t launch_softmax_rows(float* x, int rows, int n, cudaStream_t s);
size_t panoptic_scratch_bytes(int B, int Q);
cudaError_t launch_panoptic_fuse(const void* logits, bool bf16, const float* probs, const int* geom, int B, int Q, int n_cls_p1,
                                 int num_things, int h4, int w4, int up_h, int up_w, int max_out_h, int max_out_w,
                                 double object_mask_thr, double iou_thr, bool filter_low_score, int* pan, int* mask_area,
                                 int* original_area, int* seg_value, void* scratch, cudaStream_t s);

// ---- test-time caption beam search (caption_kernels.cu)
// cached self-attention step: qkv (rows, heads x [q | k | v]), caches (rows, cache_len, heads * hd), new key at position t
cudaError_t launch_caption_self_attn(const float* qkv, float* k_cache, float* v_cache, float* out, int rows, int heads, int hd,
                                     int t, int cache_len, float scale, cudaStream_t s);
// caches (blocks, 2, rows, cache_len, dim): positions [0, positions) of each row copied from its parent beam's row
cudaError_t launch_caption_cache_reorder(const float* src, float* dst, const int* parent, int blocks, int rows, int W,
                                         int cache_len, int positions, int dim, cudaStream_t s);
cudaError_t launch_beam_scores(float* logits, int blocks, int rows, int V, int W, bool first, const cgg_beam_state& st,
                               float pow_len, float* cand_val, int* cand_col, cudaStream_t s);
// beam_select_kernel stages beam_width * token_cap ints in dynamic shared memory; with its static shared memory (at most
// BEAM_SELECT_STATIC_SMEM bytes) that stays within the default 48 KiB a launch may use without an opt-in
constexpr int BEAM_SELECT_STATIC_SMEM = 1024;
constexpr int BEAM_SELECT_MAX_TOKENS = (48 * 1024 - BEAM_SELECT_STATIC_SMEM) / 4;
cudaError_t launch_beam_select(const float* cand_val, const int* cand_col, int B, int W, bool first, int length, int max_len,
                               float pow_len, float pow_len1, int eos, const cgg_beam_state& st, cudaStream_t s);

// fp32 (rows, cols) -> bf16 (rows, 2*cols) hi/lo pairs: [hi | lo] per row
cudaError_t launch_cast_bf16_split(const float* in, __nv_bfloat16* out, int rows, int cols, cudaStream_t s);
// fp32 -> IEEE half cast (n elements)
cudaError_t launch_cast_f16(const float* in, void* out, size_t n, cudaStream_t s);
// fp32 -> bf16 cast (n elements)
cudaError_t launch_cast_bf16(const float* in, __nv_bfloat16* out, size_t n, cudaStream_t s);

}  // namespace cgg

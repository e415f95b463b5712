/*
 * cgg_b200.h -- C ABI of the B200-native decoder-head hot path of CGG
 * ("Betrayed by Captions", jianzongwu/betrayed-by-captions).
 *
 * Every entry point replaces a piece of the reference's PyTorch path; the reference
 * location is cited beside each declaration (paths relative to the reference root,
 * "head.py" = open_set/models/mask2former_head.py).  The reference has no FFI of its own
 * (it is pure Python on torch/mmcv), so this header IS the boundary a maintainer binds:
 * INTEGRATION.md shows the ctypes stub and the mmdet HEADS registration that sit on it.
 *
 * Conventions (all entry points)
 *   - plain C: raw DEVICE pointers, sizes, enums, a cudaStream_t passed as void*.
 *   - the caller allocates and owns every input, output and workspace buffer; the
 *     library only owns what cgg_create() allocates inside the handle (cached positional
 *     tables, per-level K/V bias tables, bf16 weight copies, TMA descriptors) and frees it
 *     in cgg_destroy().
 *   - all work is enqueued on the given stream; no hidden synchronisation, no global
 *     mutable state; one handle per (device, stream); graph-capturable after cgg_prepare().
 *   - return value: 0 = CGG_OK, negative = cgg_status; no C++ exception crosses the ABI.
 *     cgg_last_error(handle) gives a human-readable message for the last failure.
 *   - there is NO CPU fallback: without a CUDA device every compute entry point returns
 *     CGG_ERR_CUDA.
 *
 * Tensor layouts (row-major, innermost last)
 *   x / decoder state        (B, Q, C)            fp32      [reference keeps (Q,B,C)]
 *   mask_features            (B, C, H4, W4)       fp32 (CGG_FP32) or bf16 (CGG_BF16), NCHW as
 *                                                 the pixel decoder emits it (head.py:787)
 *   memories[l]              (B, C, h_l, w_l)     same dtype rule, l = 0..2 = 1/32,1/16,1/8
 *   cls                      (L+1, B, Q, ncls1)   fp32
 *   emb                      (L+1, B, Q, d_l)     fp32
 *   mask                     (L+1, B, Q, H4, W4)  fp32 (CGG_FP32) or bf16 (CGG_BF16)
 *   attention-mask bitmap    (B, Q, ceil(K_l/32)) u32, bit (k%32) of word (k/32) = 1  <=>
 *                                                 reference attn_mask[b*heads+h, q, k] == True
 *                                                 ("do not attend"), identical for all heads
 *                                                 (head.py:756-758); tail bits are 0
 *   all_masked               (B, Q)               u8, 1 <=> every key of the row is masked
 *                                                 (the fallback of head.py:825-826 applies)
 */
#ifndef CGG_B200_H
#define CGG_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CGG_MAX_LAYERS 16
#define CGG_NUM_LEVELS 3

typedef enum {
  CGG_OK = 0,
  CGG_ERR_BAD_SHAPE = -1,
  CGG_ERR_UNSUPPORTED = -2,
  CGG_ERR_CUDA = -3,
  CGG_ERR_NOT_PREPARED = -4,
  CGG_ERR_WORKSPACE = -5,
  CGG_ERR_NULL = -6
} cgg_status;

typedef enum {
  CGG_FP32 = 0, /* parity mode: fp32 operands, fp32 FFMA accumulation, fp32 masks out       */
  CGG_BF16 = 1  /* throughput mode: bf16 operands on tcgen05, fp32 accumulate, bf16 masks out */
} cgg_precision;

/* Hyper-parameters of the head (configs/instance/coco_b48n17.py:28-100). */
typedef struct {
  int num_queries;   /* Q      (100..300)                                   :36  */
  int embed_dim;     /* C      must be 256                                  :82  */
  int num_heads;     /* must be 8 (head_dim 32)                             :83  */
  int ffn_dim;       /* 2048                                                :90  */
  int num_layers;    /* 9                                                   :77  */
  int num_classes_p1;/* ncls+1: 49 (instance) / 118 (OSPS)                       */
  int d_lang;        /* 768 (BERT width of v2l_transform, head.py:219); 0 = no
                        v2l_transform: use_class_emb=False, emb output = cls (:739-744) */
  int precision;     /* cgg_precision                                            */
  int pred_emb_norm; /* head.py:743-744 (only with d_lang > 0)                   */
} cgg_config;

/* Per-layer weights: state_dict keys transformer_decoder.layers.<i>.* (SURVEY.md 8b). */
typedef struct {
  const float *cross_in_w, *cross_in_b;   /* attentions.0.attn.in_proj_{weight (3C,C),bias (3C)} */
  const float *cross_out_w, *cross_out_b; /* attentions.0.attn.out_proj.{weight (C,C),bias}     */
  const float *self_in_w, *self_in_b;     /* attentions.1.attn.in_proj_*                        */
  const float *self_out_w, *self_out_b;   /* attentions.1.attn.out_proj.*                       */
  const float *ffn_w1, *ffn_b1;           /* ffns.0.layers.0.0.{weight (F,C),bias}              */
  const float *ffn_w2, *ffn_b2;           /* ffns.0.layers.1.{weight (C,F),bias}                */
  const float *norm_w[3], *norm_b[3];     /* norms.{0,1,2}.{weight,bias}                        */
} cgg_layer_weights;

/* All fp32 DEVICE pointers in the reference's own layouts; never retained past a call
 * except by cgg_prepare(), which derives handle-owned tables from them. */
typedef struct {
  const float *query_embed;  /* query_embed.weight (Q,C)   head.py:133 */
  const float *query_feat;   /* query_feat.weight  (Q,C)   head.py:134 */
  const float *level_embed;  /* level_embed.weight (3,C)   head.py:136 */
  const float *cls_w, *cls_b;        /* cls_embed (ncls1,C)        head.py:139 */
  const float *me_w[3], *me_b[3];    /* mask_embed.{0,2,4} (C,C)   head.py:140-143 */
  const float *v2l_w, *v2l_b;        /* v2l_transform (d_l,C)      head.py:219 */
  const float *post_norm_w, *post_norm_b; /* transformer_decoder.post_norm */
  cgg_layer_weights layers[CGG_MAX_LAYERS];
} cgg_weights;

typedef struct cgg_handle cgg_handle;

/* ---- lifetime ------------------------------------------------------------------- */
int cgg_create(cgg_handle **out, const cgg_config *cfg);
void cgg_destroy(cgg_handle *h);
const char *cgg_last_error(const cgg_handle *h);
/* "major.minor" of this ABI and the SM arch the kernels were compiled for (sm_100a). */
const char *cgg_version(void);
/* Number of kernels this library has launched in this process (monotonic; bench.py reports the
 * difference over its timed region as "gpu_launches"). */
uint64_t cgg_launch_count(void);

/* Derives, for the given weights and feature sizes, the handle-owned tables: sine
 * positional encodings (mmdet SinePositionalEncoding, head.py:798-804), per-layer
 * key-bias tables  PosK_i = (pos_l + level_embed[l]) Wk_i^T + bk_i,  value biases
 * Wv_i level_embed[l] + bv_i  (head.py:792-796 folded through the cross-attention
 * in-projection) and, in CGG_BF16 mode, bf16 copies of the GEMM weights.  Must be called
 * again when weights or sizes change. */
int cgg_prepare(cgg_handle *h, const cgg_weights *w, int H4, int W4,
                const int level_h[CGG_NUM_LEVELS], const int level_w[CGG_NUM_LEVELS],
                void *stream);

/* Bytes of caller-provided workspace cgg_decoder_forward needs for this batch size. */
size_t cgg_workspace_bytes(const cgg_handle *h, int batch);
/* Introspection for the stage-level parity tests: byte offset inside the workspace of a named
 * intermediate ("kv0","kv1","kv2": projected keys/values of level l, (B,K_l,nl*2C), columns
 * [k_0..k_{nl-1} | v_0..v_{nl-1}]; "me_all": bf16 mask embeddings of all head calls; "fds0".."fds2":
 * mask_features resampled to level l (bf16 mode)).  Returns (size_t)-1 for an unknown name. */
size_t cgg_workspace_offset(const cgg_handle *h, int batch, const char *what);

/* ---- whole path: Mask2FormerHeadOpen.forward after the pixel decoder (head.py:787-849)
 * mask_features, memories: dtype per precision (see layouts).  Outputs as listed above.
 * Optional (may be NULL) introspection outputs used by the parity tests:
 *   x_states (L+1,B,Q,C) fp32  : decoder state fed to each head call
 *   bitmaps[j], j=0..L-1       : bitmap produced by head call j (for level j%3), BEFORE
 *                                the fallback; all_masked (L,B,Q) u8.                    */
int cgg_decoder_forward(cgg_handle *h, const cgg_weights *w, int batch,
                        const void *mask_features, const void *const memories[CGG_NUM_LEVELS],
                        float *cls, float *emb, void *mask,
                        float *x_states, uint32_t *const *bitmaps, uint8_t *all_masked,
                        void *workspace, size_t workspace_bytes, void *stream);

/* ---- stages (each is what cgg_decoder_forward enqueues; exported for stage-level and
 *      teacher-forced parity tests and for microbenchmarks) ---------------------------- */

/* K4: cross-attention key/value in-projection of every layer from the three memories
 * (torch.nn.MultiheadAttention in-proj reached from head.py:829-840) into the workspace. */
int cgg_kv_project(cgg_handle *h, const cgg_weights *w, int batch,
                   const void *const memories[CGG_NUM_LEVELS], void *workspace,
                   size_t workspace_bytes, void *stream);

/* K1+K2+K3: forward_head (head.py:711-761) for head call `call_idx` (0..L): post_norm,
 * cls_embed, v2l_transform, mask_embed MLP, mask einsum, and -- when bitmap != NULL -- the
 * bilinear downsample to level `target_level`, sigmoid<0.5 threshold, bit-pack and
 * all-masked flags.  x (B,Q,C).  cls/emb/mask point at this call's slice. */
int cgg_head_call(cgg_handle *h, const cgg_weights *w, int batch, const float *x,
                  const void *mask_features, int target_level, float *cls, float *emb,
                  void *mask, float *mask_embed_out, uint32_t *bitmap, uint8_t *all_masked,
                  void *workspace, size_t workspace_bytes, void *stream);

/* K2 alone (CGG_BF16 mode): the mask einsum of head calls first_call .. first_call+num_calls-1 in ONE
 * pass over mask_features, from the mask embeddings that cgg_head_call / cgg_decoder_forward left in
 * the workspace (head.py:748, x num_calls).  mask points at call `first_call`'s (B,Q,H4,W4) bf16
 * slice; consecutive calls must be contiguous.  Used by the roofline measurement in bench.py. */
int cgg_mask_einsum(cgg_handle *h, int batch, int first_call, int num_calls, const void *mask_features,
                    void *mask, void *workspace, size_t workspace_bytes, void *stream);

/* K3 alone on given fp32 logits (stage-level bit-exactness test): mask_pred (B,Q,H4,W4)
 * -> bitmap, all_masked for a target (h,w).  head.py:749-759. */
int cgg_attn_mask_from_logits(cgg_handle *h, int batch, const float *mask_pred, int H4, int W4,
                              int th, int tw, uint32_t *bitmap, uint8_t *all_masked, void *stream);

/* K5+K6: one DetrTransformerDecoderLayer (cross-attn, norm, self-attn, norm, FFN, norm;
 * head.py:829-840) with the K/V that cgg_kv_project left in the workspace.  The fallback
 * (head.py:825-826) is applied from all_masked.  x_in, x_out (B,Q,C) fp32. */
int cgg_decoder_layer(cgg_handle *h, const cgg_weights *w, int batch, int layer,
                      const float *x_in, const uint32_t *bitmap, const uint8_t *all_masked,
                      float *x_out, void *workspace, size_t workspace_bytes, void *stream);

/* K5 alone: masked multi-head cross-attention core softmax(q k^T + mask) v.
 * q (B,Q,C) fp32 already scaled by 1/sqrt(d); k, v (B,K,C) fp32 (CGG_FP32) or bf16 with row
 * stride kv_stride elements; bitmap/all_masked may be NULL (= no mask). out (B,Q,C) fp32. */
int cgg_masked_attention(cgg_handle *h, int batch, int num_keys, const float *q, const void *k,
                         const void *v, long kv_stride, long kv_batch_stride,
                         const uint32_t *bitmap, const uint8_t *all_masked,
                         float *out, void *stream);

/* ---- grounding side -------------------------------------------------------------- */

/* extract_word_embeddings (head.py:686-698) + BertEmbeddings (utils/bert_embeddings.py:4-13):
 * out[n,:] = LayerNorm_eps(table[ids[n],:]) (no LN when text_emb_norm == 0). ids int64. */
int cgg_noun_embeddings(cgg_handle *h, const float *table, const float *ln_w, const float *ln_b,
                        const int64_t *ids, int n_ids, int d_lang, float eps, int text_emb_norm,
                        float *out, void *stream);

/* _get_cls_emb_logits (head.py:631-648) and test-time `att` (head.py:973-978):
 * out (M,N) = a (M,D) . b (N,D)^T * scale. */
int cgg_similarity(cgg_handle *h, const float *a, const float *b, int M, int N, int D,
                   float scale, float *out, void *stream);

/* K7 forward: grounding_loss (losses/grounding_loss.py:9-77) for Bg images x Bg captions as one
 * similarity contraction + fused dual softmax / masked reductions + the 4 contrastive CE terms.
 * pred (Bg,Q,D) fp32, cap (Bg,T,D) fp32, cap_mask (Bg,T) int64 -> loss (1) fp32 = weight*loss.
 * scratch: >= cgg_grounding_scratch_bytes(Bg) bytes. */
size_t cgg_grounding_scratch_bytes(int Bg, int Q, int T);
int cgg_grounding_loss(cgg_handle *h, const float *pred, const float *cap, const int64_t *cap_mask,
                       int Bg, int Q, int T, int D, float temperature, float loss_weight,
                       float *loss, void *scratch, size_t scratch_bytes, void *stream);

/* Inference shortcut (opt-in, changes the output contract; SURVEY.md section 8f): only the LAST head call's mask
 * logits are consumed at test time (mask2former_head.py:943-945).  With the option on, cgg_decoder_forward writes
 * that one map only -- `mask` then points to a (B,Q,H4,W4) buffer -- and the mask einsum of the nine intermediate
 * head calls is skipped (their attention-mask bits never needed full-resolution logits).  CGG_BF16 only. */
int cgg_set_final_mask_only(cgg_handle *h, int on);

/* K7 backward: d loss / d pred (Bg,Q,D) fp32 of the same loss, times grad_out (the upstream scalar gradient).
 * Captions are frozen BERT embeddings in the reference (head.py:251-254), so no caption gradient is produced.
 * scratch: >= cgg_grounding_bwd_scratch_bytes(Bg,Q,T) bytes. */
size_t cgg_grounding_bwd_scratch_bytes(int Bg, int Q, int T);
int cgg_grounding_loss_backward(cgg_handle *h, const float *pred, const float *cap, const int64_t *cap_mask,
                                int Bg, int Q, int T, int D, float temperature, float loss_weight, float grad_out,
                                float *dpred, void *scratch, size_t scratch_bytes, void *stream);

/* ---- training step (BASELINE.json configs[3]): stage kernels with their backward -----------------------------
 * The reference trains through autograd over the path (forward_train head.py:851-921 -> loss :393-462 -> backward);
 * the replacement exposes each stage's forward and backward so that a tape (betrayed-by-captions_b200/train.py builds
 * one with torch.autograd.Function) reaches every head parameter, the mask features and the memories.  All fp32. */

/* Generic strided GEMM: C[b,m,n] = relu?((sum_k A[b,m,k] W[b,n,k] + bias[n]) * alpha + R[b, m % r_mod, n]); strides in
 * elements.  Every linear layer's forward, dX = dY W and dW = dY^T X, the mask einsum (head.py:748) and both of its
 * gradients are calls of this entry point.  a_mmajor / c_mmajor only say which index consecutive lanes walk. */
typedef struct {
  const float *A; long sAb, sAm, sAk;
  const float *A2; long sA2m, sA2k; int a2_mod;      /* optional addend A2[m % a2_mod, k] of A (may be NULL) */
  const float *W; long sWb, sWn, sWk;
  const float *bias;
  const float *R; long sRb, sRm, sRn; int r_mod; int r_ncols;
  float *C; long sCb, sCm, sCn;
  int M, N, K, batch;
  int relu;
  float alpha;
  int a_mmajor, c_mmajor;
  int tf32;      /* 0: fp32 FMA (parity mode, exact); 1: tcgen05 kind::tf32 MMAs fed by TMA from the same fp32 tensors
                  * (10-bit operand mantissas, fp32 accumulate, split-K summed in a fixed order).  Products whose strides
                  * TMA cannot describe (a row pitch that is not a multiple of 16 bytes) run on the FMA kernel. */
  int batch_inner;            /* two-level batch (0 or 1 = off): item z of A / W / C sits at (z / batch_inner) * sXb +
                               * (z % batch_inner) * sXb2 -- (image, head) batches of the attention products */
  long sAb2, sWb2, sCb2;
  int accumulate;             /* 1: C = (the above) + C, in place (a gradient that several products contribute to) */
  int slot;                   /* 0 / 1: which split-K workspace to use -- calls issued concurrently on two streams (the
                               * weight-gradient products of the training step run on a side stream) pass different slots */
  int conv_cin;               /* > 0: 3x3 convolution (stride 1, zero padding 1: the pixel decoder's output_convs) as an
                               * implicit GEMM over a token-major image batch X (images, H, W, conv_cin): batch = images * H
                               * with batch_inner = H (sAb / sAb2 = image / row strides of X), M = W, sAm = pixel stride,
                               * K = 9 * conv_cin, W[n, tap * conv_cin + c] with tap = 3 * ky + kx.  The tf32 form fetches
                               * each tap with TMA, whose out-of-bounds zero fill is the padding. */
} cgg_gemm_desc;
int cgg_gemm_f32(cgg_handle *h, const cgg_gemm_desc *d, void *stream);

/* torch.nn.LayerNorm forward / backward over rows of length n (post_norm, norms.{0,1,2}). */
int cgg_layernorm(cgg_handle *h, const float *x, const float *w, const float *b, float *y, int rows, int n, float eps,
                  void *stream);
size_t cgg_layernorm_bwd_scratch_bytes(int rows, int n);
int cgg_layernorm_backward(cgg_handle *h, const float *x, const float *w, const float *dy, float *dx, float *dw,
                           float *db, void *scratch, size_t scratch_bytes, int rows, int n, float eps, void *stream);
/* dx = dy * alpha where the ReLU output y > 0 */
int cgg_relu_backward(cgg_handle *h, const float *y, const float *dy, float *dx, long n, float alpha, void *stream);
/* out += alpha * in */
int cgg_axpy(cgg_handle *h, const float *in, float *out, long n, float alpha, void *stream);
/* out[b,i] = (x ? x[b,i] : 0) + add[i], i < per   (x + query_embed; the query_feat broadcast, head.py:808-811) */
int cgg_add_rows(cgg_handle *h, const float *x, const float *add, float *out, int batch, long per, void *stream);
/* out[i] = sum_b g[b,i]   (its backward) */
int cgg_sum_batch(cgg_handle *h, const float *g, float *out, int batch, long per, void *stream);
/* out[n] (+)= alpha * sum_rows g[row,n]   (bias gradients; accumulate = 1 adds to out in place) */
int cgg_colsum(cgg_handle *h, const float *g, float *out, long rows, int n, float alpha, int accumulate, void *stream);
/* head.py:792-804: key_in[b,key,:] = mem[b,:,key] + level + pos[key,:], val_in = mem[b,:,key] + level, and the backward
 * dmem[b,c,key] = dkey_in[b,key,c] + dval_in[b,key,c].  pos_level (K,C) = pos + level. */
int cgg_mem_prep(cgg_handle *h, const float *mem, const float *level, const float *pos_level, float *key_in,
                 float *val_in, int batch, int C, int K, void *stream);
int cgg_mem_prep_backward(cgg_handle *h, const float *dkey_in, const float *dval_in, float *dmem, int batch, int C,
                          int K, void *stream);
/* mmdet SinePositionalEncoding(normalize=True) of an (hh, ww) map -> (hh*ww, C) fp32 (head.py:798-804) */
int cgg_sine_pos(cgg_handle *h, float *out, int hh, int ww, int C, void *stream);
/* softmax(q k^T + mask) v for num_q queries (cross-attention: Q queries; self-attention: num_q = num_keys), fp32, and
 * its backward (dq, dk, dv; softmax recomputed from the saved q, k; bitmap as in the forward).
 * scratch: 2 * batch * heads * num_q floats. */
int cgg_attention_f32(cgg_handle *h, int batch, int num_q, int num_keys, const float *q, const float *k, const float *v,
                      long kv_stride, long kv_batch_stride, const uint32_t *bitmap, const uint8_t *all_masked,
                      float *out, void *stream);
int cgg_attention_backward(cgg_handle *h, int batch, int num_q, int num_keys, const float *q, const float *k,
                           const float *v, long kv_stride, long kv_batch_stride, const uint32_t *bitmap,
                           const uint8_t *all_masked, const float *out, const float *dout, float *dq, float *dk,
                           float *dv, long dkv_stride, long dkv_batch_stride, float *scratch, void *stream);
/* The same attention as tensor-core products (training step with tf32 contractions): S = q k^T, O = P v and the four
 * gradient products are cgg_gemm_f32 calls over (image, head) batches (batch_inner = heads); these two entry points are
 * the row-wise stages in between, in place on the (batch, heads, num_q, num_keys) fp32 score tensor:
 *   cgg_attn_softmax_rows: scores -> softmax over the keys the bitmap leaves (all keys for all_masked rows; a row with
 *                          no key left becomes zeros);
 *   cgg_attn_dscore:       dprobs -> probs * (dprobs - D),  D[b,h,q] = dout[b,q,h,:] . out[b,q,h,:].
 * heads / head_dim: 0 = the handle's (8 x 32); the caption transformer (row f4) passes its own (8 x 96). */
int cgg_attn_softmax_rows(cgg_handle *h, float *scores, const uint32_t *bitmap, const uint8_t *all_masked, int batch,
                          int heads, int num_q, int num_keys, void *stream);
int cgg_attn_dscore(cgg_handle *h, const float *probs, float *dprobs, const float *out, const float *dout, int batch,
                    int heads, int head_dim, int num_q, int num_keys, void *stream);

/* ---- the matching-based losses after the path at training time (SURVEY.md section 8 row f2) -------------------
 * loss_single (open_set/models/mask2former_head.py:464-629) and its target assignment (:320-390; assigner
 * open_set/assigners/mask_hungarian_assigner.py:98-125).  The reference reaches into mmcv / mmdet for these steps
 * (mmcv.ops.point_sample, mmdet match costs, DiceLoss, CrossEntropyLoss); each entry names what it replaces.  fp32. */

/* mmcv.ops.point_sample (F.grid_sample on 2p-1, bilinear, zeros padding, align_corners=False) of `planes` maps (hh, ww)
 * at num_points points (x, y) in [0,1]^2; coords (planes, P, 2), or (1, P, 2) when coords_shared (the matching step
 * samples every query and every ground-truth mask of an image at the same points, head.py:352-363).  -> out (planes, P).
 * The backward scatters dout into din (planes, hh, ww) (zeroed here). */
int cgg_point_sample(cgg_handle *h, const float *in, const float *coords, float *out, int planes, int hh, int ww,
                     int num_points, int coords_shared, void *stream);
int cgg_point_sample_backward(cgg_handle *h, const float *dout, const float *coords, float *din, int planes, int hh, int ww,
                              int num_points, int coords_shared, void *stream);
/* cost (num_q, num_gt) = w_cls * ClassificationCost(cls_scores) + w_cls_emb * ClassificationCost(cls_emb_logits)
 *                      + w_mask * CrossEntropyLossCost(use_sigmoid) + w_dice * DiceCost(pred_act, eps)   (assigner :98-125)
 * on the sampled mask logits (num_q, P) and sampled ground-truth masks (num_gt, P).  A class term with weight 0 may pass
 * NULL.  scratch: 4 * num_q + num_gt floats.  The Hungarian solve itself stays on the host, as in the reference (:127-134). */
int cgg_matching_cost(cgg_handle *h, const float *mask_points, const float *gt_points, const float *cls_scores,
                      const float *cls_emb_logits, const int64_t *gt_labels, int num_q, int num_gt, int classes_p1,
                      int num_points, float w_cls, float w_cls_emb, float w_mask, float w_dice, float dice_eps,
                      float *scratch, float *cost, void *stream);
/* Per matched mask row: dice_rows = 1 - (2 s.t + eps) / (sum s + sum t + eps), s = sigmoid(pred)  (DiceLoss naive_dice,
 * head.py:614-616) and bce_rows = sum_p BCE-with-logits(pred, t)  (loss_mask, :618-627); abc (rows, 3) is kept for the
 * backward, which takes per-row upstream gradients (device resident). */
int cgg_point_losses(cgg_handle *h, const float *pred_points, const float *target_points, int rows, int num_points,
                     float dice_eps, float *abc, float *dice_rows, float *bce_rows, void *stream);
int cgg_point_losses_backward(cgg_handle *h, const float *pred_points, const float *target_points, const float *abc,
                              int rows, int num_points, float dice_eps, const float *g_dice_rows, const float *g_bce_rows,
                              float *dpred, void *stream);
/* F.cross_entropy(logits, labels, weight=class_weight, reduction='none') (loss_cls / loss_cls_emb, head.py:520-538):
 * row_loss = w[label] (lse - x[label]), row_weight = w[label] (the avg_factor is their sum), lse kept for the backward
 * dlogits[r, c] = g_rows[r] w[label_r] (softmax_c - [c == label_r]). */
int cgg_weighted_ce(cgg_handle *h, const float *logits, const int64_t *labels, const float *class_weight, int rows,
                    int classes_p1, float *row_loss, float *row_weight, float *lse, void *stream);
int cgg_weighted_ce_backward(cgg_handle *h, const float *logits, const int64_t *labels, const float *class_weight,
                             const float *lse, int rows, int classes_p1, const float *g_rows, float *dlogits, void *stream);

/* ---- the step after the path at test time (SURVEY.md 8f rank 1) ---------------------------------------------------
 * logits: the LAST head call's mask logits (B, Q, h4, w4), fp32 (is_bf16 = 0) or bf16 (is_bf16 = 1).
 * cgg_upsample_masks: F.interpolate(logits, (up_h, up_w), bilinear, align_corners=False) materialised in fp32, the
 *   tensor simple_test returns (head.py:957-964).
 * cgg_instance_mask_stats: the same upsample FUSED with what MaskFormerFusionHeadOpen does next -- crop to img_shape,
 *   optional second bilinear resample to ori_shape (maskformer_fusion_head.py:412-425), `> 0`, sum of sigmoid over the
 *   positive pixels, pixel count and bounding box (instance_postprocess_emb :352-362, mmdet mask2bbox) -- without ever
 *   writing full-resolution logits.  geom (DEVICE, B x 4 int32) = {crop_h, crop_w, out_h, out_w} per image (out = crop
 *   when not rescaling).  Outputs: bits (B, Q, max_out_h, ceil(max_out_w/32)) u32 packed binary masks (may be NULL),
 *   count (B,Q) int32, sig_sum (B,Q) fp32, bbox (B,Q,4) int32 = x0, y0, x1+1, y1+1 (zeros for an empty mask).
 * cgg_softmax_rows: in-place row softmax (get_cls_emb_scores, maskformer_fusion_head.py:312-313).
 * cgg_panoptic_fuse: the fusion head's panoptic output (mmdet 2.28.2 MaskFormerFusionHead.panoptic_postprocess with the
 *   class-embedding probabilities) from the same logits and the same resample / crop / rescale as cgg_instance_mask_stats,
 *   with no host round trip.  probs (B, Q, classes_p1) fp32 on the device (column classes_p1 - 1 = void); geom as above.
 *   scores, labels = probs.max(-1); keep = label != void & score > (float)object_mask_thr; per pixel the kept query with
 *   the largest score * sigmoid(logit) wins (first in query order on ties); a kept query whose winning area over its
 *   #(sigmoid >= 0.5) is >= iou_thr (double) becomes a segment: label + 1000 * instance_id for things (label <
 *   num_things, ids 1, 2, ... in query order over the valid things), label for stuff (one value per class).  pan
 *   (B, max_out_h, max_out_w) int32 is written inside each image's out_h x out_w only: the segment value, or classes_p1 - 1
 *   where no segment covers the pixel (with filter_low_score, also where the winner's sigmoid is < 0.5).  mask_area,
 *   original_area, seg_value (B, Q) int32 per query id (may be NULL): winning pixels, pixels with sigmoid >= 0.5, segment
 *   value; 0, 0, -1 for queries not kept, seg_value -1 for a dropped query.  scratch: device memory of at least
 *   cgg_panoptic_scratch_bytes(batch, num_q) bytes, else CGG_ERR_WORKSPACE.  num_q <= 4096. */
int cgg_upsample_masks(cgg_handle *h, const void *logits, int is_bf16, float *out, int planes, int h4, int w4, int up_h,
                       int up_w, void *stream);
int cgg_instance_mask_stats(cgg_handle *h, const void *logits, int is_bf16, const int *geom, int batch, int num_q, int h4,
                            int w4, int up_h, int up_w, int max_out_h, int max_out_w, uint32_t *bits, int *count,
                            float *sig_sum, int *bbox, void *stream);
int cgg_softmax_rows(cgg_handle *h, float *x, int rows, int n, void *stream);
size_t cgg_panoptic_scratch_bytes(int batch, int num_q);
int cgg_panoptic_fuse(cgg_handle *h, const void *logits, int is_bf16, const float *probs, const int *geom, int batch,
                      int num_q, int classes_p1, int num_things, int h4, int w4, int up_h, int up_w, int max_out_h,
                      int max_out_w, double object_mask_thr, double iou_thr, int filter_low_score, int *pan,
                      int *mask_area, int *original_area, int *seg_value, void *scratch, size_t scratch_bytes,
                      void *stream);

/* ---- test-time caption generation: the beam search of open_set/utils/eval/inference.py:84-157 ---------------------
 * For `batch` images at once, W = beam_width beams each (1..32), rows = batch * W in (image, beam) order.  The caller runs
 * the decoder blocks with cgg_gemm_f32 / cgg_layernorm and these four stages; nothing here synchronises with the host.
 * Search state, device arrays (T = token_cap, the longest sequence the search can produce):
 *   tokens (batch, W, T) int32   the active beams' token ids, BOS first
 *   weights (batch, W) fp32      the beams' weights;  n_active (batch) int32;  parent (batch, W) int32: beam of the previous
 *                                step each beam continues;  next_ids (batch, W) int64: the token each beam feeds next
 *   fin_tokens (batch, W, T) int32, fin_len (batch, W) int32, fin_score (batch, W) fp32, n_fin (batch) int32: finished
 *                                sequences in the order the reference appends them
 *   max_idx (batch) int32: the reference's max_idx of the image's last pass (its result is fin[max_idx], if n_fin > 0)
 *   done (batch) int32: the image's search has ended (later calls leave its state unchanged);  n_done (1) int32: count of
 *                                done images (each image adds 1 once)
 * A new search starts from tokens[:, :, 0] = BOS, n_fin = done = n_done = 0. */
typedef struct cgg_beam_state {
  int *tokens;
  int token_cap;
  float *weights;
  int *n_active, *parent;
  int64_t *next_ids;
  int *fin_tokens, *fin_len;
  float *fin_score;
  int *n_fin, *max_idx, *done, *n_done;
} cgg_beam_state;

/* cgg_caption_self_attn_step: masked self-attention of one new position t with cached keys: per row and head, k and v of
 *   qkv (rows, heads x [q | k | v] of head_dim each, the caption transformer's fused qkv_layer output) are stored at
 *   position t of k_cache / v_cache (rows, cache_len, heads * head_dim), then softmax(scale q k^T) v over positions 0..t
 *   -> out (rows, heads * head_dim).  t < cache_len; head_dim + cache_len <= 12288.
 * cgg_caption_cache_reorder: src / dst caches (blocks, 2 [k, v], rows, cache_len, dim): dst[., ., image * W + w, p] =
 *   src[., ., image * W + parent[image * W + w], p] for p < positions (dim % 4 == 0).
 * cgg_caption_beam_scores: logits (blocks, rows, vocab), the generator applied to every block's output.  For each row of
 *   an image that is not done and a beam < n_active (first != 0: beam 0 only): logp = log_softmax(mean over blocks), the
 *   score logp (first) or (logp + weights[row]) / pow_len, and the row's top W scores in torch.topk order (descending,
 *   ties to the lower column) -> cand_val / cand_col (rows, W).  Overwrites block 0 of logits.  vocab >= W.
 * cgg_caption_beam_select: per image, the flattened top W of its active rows' candidates (flat index row * vocab + col,
 *   torch.topk order) and the reference's bookkeeping.  first != 0 (the BOS step, length 1): the W picks become the
 *   beams [BOS, c] with weight log p.  Otherwise, with the picks' weights = score * pow_len and in rank order: EOS
 *   appends (sequence + EOS, weights[k] / pow_len1) to the finished list, the walk stops at W finished; another token
 *   continues if length + 1 < max_len - 1 with weight weights[parent row]; the image is done on the stop or when no
 *   beam continues.  pow_len = fp32(length ** alpha), pow_len1 = fp32((length + 1) ** alpha), alpha in double as the
 *   reference computes them.  max_len <= num_positions (the position table's rows), length + 1 <= token_cap,
 *   W * token_cap <= 12032.  Bad sizes: CGG_ERR_BAD_SHAPE. */
int cgg_caption_self_attn_step(cgg_handle *h, const float *qkv, float *k_cache, float *v_cache, float *out, int rows,
                               int heads, int head_dim, int t, int cache_len, float scale, void *stream);
int cgg_caption_cache_reorder(cgg_handle *h, const float *src, float *dst, const int *parent, int blocks, int batch,
                              int beam_width, int cache_len, int positions, int dim, void *stream);
int cgg_caption_beam_scores(cgg_handle *h, float *logits, int blocks, int batch, int beam_width, int vocab, int first,
                            const cgg_beam_state *state, float pow_len, float *cand_val, int *cand_col, void *stream);
int cgg_caption_beam_select(cgg_handle *h, const float *cand_val, const int *cand_col, int batch, int beam_width,
                            int first, int length, int max_len, int num_positions, float pow_len, float pow_len1,
                            int eos, const cgg_beam_state *state, void *stream);

/* ---- the step before the path: mmdet MSDeformAttnPixelDecoder (SURVEY.md 8f rank 3) ------------------------------
 * `mask_features, multi_scale_memorys = self.pixel_decoder(feats)` (mask2former_head.py:787; configured at
 * configs/instance/coco_b48n17.py:38-70).  mmdet 2.28.2 / mmcv-full 1.7.1 are un-vendored dependencies of the reference;
 * each entry point names the third-party function it stands for.  Activations are TOKEN-MAJOR fp32: (images, pixels,
 * channels), the levels of the encoder concatenated along the pixel axis, lowest resolution first.  The contractions (1x1
 * convs, the 3x3 conv via cgg_gemm_desc.conv_cin, all linear layers) are cgg_gemm_f32 calls; LayerNorm is cgg_layernorm.
 *
 * cgg_ms_deform_attn: mmcv MultiScaleDeformableAttention core (ops/multi_scale_deform_attn.py, CUDA op
 *   ms_deform_attn_forward): value (B, S, heads*32) = value_proj(x); offsets (B, S, heads*levels*points*2) = the
 *   sampling_offsets projection of (x + pos), (x, y) in pixels of the sampled level; weight_logits (B, S, heads*levels*
 *   points) = the attention_weights projection BEFORE its softmax (done here, over levels*points).  Reference point of
 *   token s = its own pixel centre ((x+.5)/w, (y+.5)/h) in every level (all-valid padding mask, as the reference runs it);
 *   bilinear taps, zero outside, align_corners=False.  out (B, S, heads*32).  level_h / level_w: HOST arrays.
 *   The three inputs of the forward carry their own token stride (elements between consecutive tokens), so that they can
 *   be column blocks of ONE fused projection [offsets | logits | value] of the token buffer.
 *   The backward returns dvalue (zeroed here, then scattered with atomics), doffsets and dweight_logits (through the
 *   softmax). */
int cgg_ms_deform_attn(cgg_handle *h, const float *value, long value_stride, const float *offsets, long offset_stride,
                       const float *weight_logits, long logit_stride, float *out, int batch, int tokens, int heads,
                       int levels, int points, const int *level_h, const int *level_w, void *stream);
int cgg_ms_deform_attn_backward(cgg_handle *h, const float *value, const float *offsets, const float *weight_logits,
                                const float *dout, float *dvalue, float *doffsets, float *dweight_logits, int batch,
                                int tokens, int heads, int levels, int points, const int *level_h, const int *level_w,
                                void *stream);
/* GroupNorm of mmcv's ConvModule (norm_cfg GN, num_groups 32; eps 1e-5) + optional ReLU over token-major x (B, pixels,
 * channels): statistics per (image, group of channels/groups consecutive channels).  mean_rstd (B, groups, 2) is kept
 * for the backward; dy of the backward must already carry the ReLU mask (cgg_relu_backward).  Deterministic. */
size_t cgg_group_norm_scratch_bytes(int batch, int pixels, int channels, int groups);
int cgg_group_norm_tokens(cgg_handle *h, const float *x, const float *gamma, const float *beta, float *y, float *mean_rstd,
                          void *scratch, size_t scratch_bytes, int batch, int pixels, int channels, int groups, float eps,
                          int relu, void *stream);
int cgg_group_norm_tokens_backward(cgg_handle *h, const float *x, const float *dy, const float *mean_rstd,
                                   const float *gamma, float *dx, float *dgamma, float *dbeta, void *scratch,
                                   size_t scratch_bytes, int batch, int pixels, int channels, int groups, void *stream);
/* FPN top-down step of MSDeformAttnPixelDecoder.forward: out = lateral + F.interpolate(coarse, size=(H, W), bilinear,
 * align_corners=False); lateral / out (B, H*W, C), coarse (B, ch*cw, C) with its own batch stride (a level's slice of the
 * encoder's token buffer).  Backward: dlateral = dout; dcoarse (B, ch*cw, C) contiguous, zeroed here, then scattered. */
int cgg_upsample_add_tokens(cgg_handle *h, const float *lateral, const float *coarse, long coarse_batch_stride, float *out,
                            int batch, int H, int W, int ch, int cw, int channels, void *stream);
int cgg_upsample_add_tokens_backward(cgg_handle *h, const float *dout, float *dcoarse, int batch, int H, int W, int ch,
                                     int cw, int channels, void *stream);
/* Layout change at the boundary: tokens (B, pixels, C) with a batch stride -> NCHW (B, C, pixels) fp32 or bf16 (what
 * cgg_decoder_forward consumes), and back (optionally accumulating: a gradient joining the token buffer). */
int cgg_tokens_to_nchw(cgg_handle *h, const float *tokens, long token_batch_stride, void *out, int out_bf16, int batch,
                       int pixels, int channels, void *stream);
int cgg_nchw_to_tokens(cgg_handle *h, const float *in, float *tokens, long token_batch_stride, int batch, int pixels,
                       int channels, int accumulate, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* CGG_B200_H */

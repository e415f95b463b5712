// C-ABI layer + host-side orchestration of the decoder-head path (include/cgg_b200.h).
// Everything here only enqueues kernels on the caller's stream.
#include "../../include/cgg_b200.h"
#include "common.cuh"
#include "kernels.h"
#include "gemm_tc.h"
#include "gemm_tf32.h"
#include "tc_state.h"

#include <math.h>
#include <stdio.h>
#include <string.h>
#include <stdlib.h>
#include <string>
#include <vector>

using namespace cgg;

struct cgg_handle {
  cgg_config cfg;
  std::string err;
  bool prepared = false;
  int H4 = 0, W4 = 0, lh[CGG_NUM_LEVELS] = {0, 0, 0}, lw[CGG_NUM_LEVELS] = {0, 0, 0};
  int nl[CGG_NUM_LEVELS] = {0, 0, 0};  // decoder layers that read level l
  // handle-owned device tables (fp32)
  float* pos_level[CGG_NUM_LEVELS] = {nullptr, nullptr, nullptr};  // (K_l, C)   pos + level_embed
  float* wkv[CGG_NUM_LEVELS] = {nullptr, nullptr, nullptr};        // (nl*2C, C) [Wk.. | Wv..]
  float* rk[CGG_NUM_LEVELS] = {nullptr, nullptr, nullptr};         // (K_l, nl*C) key bias table
  float* bkv[CGG_NUM_LEVELS] = {nullptr, nullptr, nullptr};        // (nl*2C)    0 | value bias
  TcState* tc = nullptr;                                           // bf16 / tcgen05 side
  // Helper streams of cgg_decoder_forward (bf16 mode): throughput kernels that are off the critical
  // chain (K/V projection of the later levels, the mask einsum of finished head calls) are forked
  // from the caller's stream with events and joined back before the call's work ends on it.
  cudaStream_t side[2] = {nullptr, nullptr};
  cudaEvent_t ev_fork = nullptr, ev_join[2] = {nullptr, nullptr}, ev_kv[CGG_NUM_LEVELS] = {nullptr, nullptr, nullptr};
  cudaEvent_t ev_me[CGG_MAX_LAYERS + 1] = {};   // fork of layer j's q projection
  bool overlap_kv = false;   // K/V levels 1,2 and the layers' q projections on helper streams (set when the streams exist)
  bool final_mask_only = false;   // cgg_set_final_mask_only
  // K7 on tensor cores: the similarity contraction of the grounding loss (and its backward contraction) as split-precision
  // tcgen05 GEMMs.  Operand buffers live in the handle (grown on demand); tc_aux serves handles created in CGG_FP32 mode.
  TcState* tc_aux = nullptr;
  Tf32Ctx* tf32 = nullptr;   // training-step contractions on tcgen05 (gemm_tf32.cu), created on first use
  struct K7Buf {
    __nv_bfloat16 *pred_hl = nullptr, *cap_hl = nullptr, *dst_hl = nullptr, *capT_hl = nullptr;
    float* S = nullptr;
    size_t n_pred = 0, n_cap = 0, n_dst = 0, n_capT = 0, n_S = 0;
    void release() {
      cudaFree(pred_hl); cudaFree(cap_hl); cudaFree(dst_hl); cudaFree(capT_hl); cudaFree(S);
      pred_hl = cap_hl = dst_hl = capT_hl = nullptr; S = nullptr; n_pred = n_cap = n_dst = n_capT = n_S = 0;
    }
  } k7;
  void free_tables() {
    for (int l = 0; l < CGG_NUM_LEVELS; ++l) {
      cudaFree(pos_level[l]); cudaFree(wkv[l]); cudaFree(rk[l]); cudaFree(bkv[l]);
      pos_level[l] = wkv[l] = rk[l] = bkv[l] = nullptr;
    }
  }
};

namespace {

int fail(cgg_handle* h, int code, const std::string& msg) {
  if (h) h->err = msg;
  return code;
}
#define CU(call)                                                                              \
  do {                                                                                        \
    cudaError_t e__ = (call);                                                                 \
    if (e__ != cudaSuccess)                                                                   \
      return fail(h, CGG_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__));      \
  } while (0)
#define ST(call)                       \
  do {                                 \
    int s__ = (call);                  \
    if (s__ != CGG_OK) return s__;     \
  } while (0)
// a tc_* stage on TcState `t`: a failure hands its message to the handle
#define TC(t, call)                                                                          \
  do {                                                                                       \
    int s__ = (call);                                                                        \
    if (s__ != CGG_OK) return fail(h, s__, std::string(#call) + ": " + tc_last_error(t));   \
  } while (0)

// Workspace carving shared by cgg_workspace_bytes and the entry points.
struct Workspace {
  size_t total = 0;
  size_t kv[CGG_NUM_LEVELS];
  size_t z, h1, h2, me, qb, kb, vb, o, t, x1, x2, f, xs, bitmap, allm, tcws;
  void carve(const cgg_handle* h, int B) {
    const cgg_config& c = h->cfg;
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off += align256(bytes); return o; };
    const size_t kv_elt = (c.precision == CGG_BF16) ? 2 : 4;
    for (int l = 0; l < CGG_NUM_LEVELS; ++l)
      kv[l] = take((size_t)B * h->lh[l] * h->lw[l] * h->nl[l] * 2 * c.embed_dim * kv_elt);
    const size_t bqc = (size_t)B * c.num_queries * c.embed_dim * sizeof(float);
    z = take(bqc); h1 = take(bqc); h2 = take(bqc); me = take(bqc); qb = take(bqc); kb = take(bqc);
    vb = take(bqc); o = take(bqc); t = take(bqc); x1 = take(bqc); x2 = take(bqc);
    f = take((size_t)B * c.num_queries * c.ffn_dim * sizeof(float));
    xs = take(bqc * (c.num_layers + 1));
    int maxk = 0;
    for (int l = 0; l < CGG_NUM_LEVELS; ++l) maxk = max(maxk, h->lh[l] * h->lw[l]);
    bitmap = take((size_t)B * c.num_queries * ((maxk + 31) / 32) * sizeof(uint32_t));
    allm = take((size_t)B * c.num_queries);
    tcws = take(tc_workspace_bytes(h->tc, B));
    total = off;
  }
};

template <typename T>
T* at(void* ws, size_t off) { return reinterpret_cast<T*>(static_cast<char*>(ws) + off); }

int check_ws(cgg_handle* h, int B, void* ws, size_t bytes, Workspace& w) {
  if (!h->prepared) return fail(h, CGG_ERR_NOT_PREPARED, "cgg_prepare() has not been called");
  if (B <= 0) return fail(h, CGG_ERR_BAD_SHAPE, "batch must be positive");
  w.carve(h, B);
  if (!ws || bytes < w.total) return fail(h, CGG_ERR_WORKSPACE, "workspace too small");
  return CGG_OK;
}

// y = (x [+ qe]) W^T + b, rows = B*Q
int linear_rows(cgg_handle* h, cudaStream_t s, const float* x, const float* a2, int a2_mod, const float* W,
                const float* bias, float* y, int rows, int N, int K, float alpha = 1.f,
                const float* R = nullptr, bool relu = false) {
  GemmF32 p;
  p.A = x; p.sAm = K; p.sAk = 1;
  if (a2) { p.A2 = a2; p.sA2m = K; p.sA2k = 1; p.a2_mod = a2_mod; }
  p.W = W; p.sWn = K; p.sWk = 1;
  p.bias = bias; p.alpha = alpha;
  if (R) { p.R = R; p.sRm = N; p.sRn = 1; p.r_mod = rows; }
  p.C = y; p.sCm = N; p.sCn = 1;
  p.M = rows; p.N = N; p.K = K; p.batch = 1;
  if (relu) p.relu_from = 0;
  CU(launch_gemm_f32(p, s));
  return CGG_OK;
}

}  // namespace

// ============================================================================ lifetime
extern "C" const char* cgg_version(void) { return "1.0 sm_100a"; }

extern "C" uint64_t cgg_launch_count(void) { return (uint64_t)cgg::launch_count(); }

extern "C" const char* cgg_last_error(const cgg_handle* h) { return h ? h->err.c_str() : "null handle"; }

extern "C" int cgg_create(cgg_handle** out, const cgg_config* cfg) {
  if (!out || !cfg) return CGG_ERR_NULL;
  *out = nullptr;
  if (cfg->embed_dim != 256 || cfg->num_heads != 8) return CGG_ERR_UNSUPPORTED;
  if (cfg->num_layers < 1 || cfg->num_layers > CGG_MAX_LAYERS) return CGG_ERR_BAD_SHAPE;
  // d_lang == 0: no v2l_transform (use_class_emb=False, head.py:739-744): the embedding output is not produced
  if (cfg->num_queries < 1 || cfg->num_queries > 1024 || cfg->ffn_dim < 1 || cfg->num_classes_p1 < 1 ||
      cfg->d_lang < 0 || (cfg->d_lang == 0 && cfg->pred_emb_norm))
    return CGG_ERR_BAD_SHAPE;
  if (cfg->precision != CGG_FP32 && cfg->precision != CGG_BF16) return CGG_ERR_UNSUPPORTED;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return CGG_ERR_CUDA;  // no CPU fallback
  cgg_handle* h = new (std::nothrow) cgg_handle();
  if (!h) return CGG_ERR_CUDA;
  h->cfg = *cfg;
  if (cfg->precision == CGG_BF16) {
    h->tc = tc_create(*cfg);
    if (!h->tc) { delete h; return CGG_ERR_CUDA; }
    // helper streams: the K/V projection of levels 1 and 2 (5/6 of that work, first needed by layers 1 and 2) and each
    // layer's query projection run underneath the latency-bound head-call / layer chain (measured on B200 at B=16,
    // 1024^2: 3.536 ms/step without, 3.468 with; putting the mask einsums there as well was slower and is gone)
    {
      int lo = 0, hi = 0;
      cudaDeviceGetStreamPriorityRange(&lo, &hi);
      bool ok = true;
      for (int i = 0; i < 2; ++i) ok = ok && cudaStreamCreateWithPriority(&h->side[i], cudaStreamNonBlocking, lo) == cudaSuccess;
      ok = ok && cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming) == cudaSuccess;
      for (int i = 0; i < 2; ++i) ok = ok && cudaEventCreateWithFlags(&h->ev_join[i], cudaEventDisableTiming) == cudaSuccess;
      for (int i = 0; i < CGG_NUM_LEVELS; ++i) ok = ok && cudaEventCreateWithFlags(&h->ev_kv[i], cudaEventDisableTiming) == cudaSuccess;
      for (int i = 0; i <= CGG_MAX_LAYERS; ++i) ok = ok && cudaEventCreateWithFlags(&h->ev_me[i], cudaEventDisableTiming) == cudaSuccess;
      h->overlap_kv = ok;
    }
  }
  *out = h;
  return CGG_OK;
}

extern "C" void cgg_destroy(cgg_handle* h) {
  if (!h) return;
  h->free_tables();
  if (h->tc) tc_destroy(h->tc);
  if (h->tc_aux) tc_destroy(h->tc_aux);
  if (h->tf32) tf32_destroy(h->tf32);
  h->k7.release();
  for (int i = 0; i < 2; ++i) if (h->side[i]) cudaStreamDestroy(h->side[i]);
  if (h->ev_fork) cudaEventDestroy(h->ev_fork);
  for (int i = 0; i < 2; ++i) if (h->ev_join[i]) cudaEventDestroy(h->ev_join[i]);
  for (int i = 0; i < CGG_NUM_LEVELS; ++i) if (h->ev_kv[i]) cudaEventDestroy(h->ev_kv[i]);
  for (int i = 0; i <= CGG_MAX_LAYERS; ++i) if (h->ev_me[i]) cudaEventDestroy(h->ev_me[i]);
  delete h;
}

extern "C" int cgg_prepare(cgg_handle* h, const cgg_weights* w, int H4, int W4, const int level_h[CGG_NUM_LEVELS],
                           const int level_w[CGG_NUM_LEVELS], void* stream) {
  if (!h || !w || !level_h || !level_w) return CGG_ERR_NULL;
  cudaStream_t s = (cudaStream_t)stream;
  const cgg_config& c = h->cfg;
  const int C = c.embed_dim;
  if (H4 <= 0 || W4 <= 0) return fail(h, CGG_ERR_BAD_SHAPE, "bad mask feature size");
  bool same = h->prepared && h->H4 == H4 && h->W4 == W4;
  for (int l = 0; l < CGG_NUM_LEVELS; ++l) {
    if (level_h[l] <= 0 || level_w[l] <= 0) return fail(h, CGG_ERR_BAD_SHAPE, "bad level size");
    same = same && h->lh[l] == level_h[l] && h->lw[l] == level_w[l];
  }
  if (!same) {
    // (re)allocation is the only place that may synchronise; steady-state re-prepare
    // (new weights, same sizes) reuses the tables and stays asynchronous.
    CU(cudaStreamSynchronize(s));
    h->prepared = false;     // stays false until every table below exists (a failed re-prepare must not leave a usable handle)
    h->free_tables();
    h->H4 = H4; h->W4 = W4;
    for (int l = 0; l < CGG_NUM_LEVELS; ++l) {
      h->lh[l] = level_h[l]; h->lw[l] = level_w[l];
      h->nl[l] = 0;
    }
    for (int i = 0; i < c.num_layers; ++i) h->nl[i % CGG_NUM_LEVELS]++;
    for (int l = 0; l < CGG_NUM_LEVELS; ++l) {
      const size_t K = (size_t)level_h[l] * level_w[l];
      const int n = h->nl[l] > 0 ? h->nl[l] : 1;
      CU(cudaMalloc(&h->pos_level[l], K * C * sizeof(float)));
      CU(cudaMalloc(&h->wkv[l], (size_t)n * 2 * C * C * sizeof(float)));
      CU(cudaMalloc(&h->rk[l], K * n * C * sizeof(float)));
      CU(cudaMalloc(&h->bkv[l], (size_t)n * 2 * C * sizeof(float)));
    }
  }
  for (int l = 0; l < CGG_NUM_LEVELS; ++l) {
    const int K = level_h[l] * level_w[l], n = h->nl[l];
    CU(launch_pos_level(w->level_embed + (size_t)l * C, h->pos_level[l], level_h[l], level_w[l], C, s));
    CU(cudaMemsetAsync(h->bkv[l], 0, (size_t)(n > 0 ? n : 1) * 2 * C * sizeof(float), s));
    for (int sl = 0; sl < n; ++sl) {
      const cgg_layer_weights& lw = w->layers[sl * CGG_NUM_LEVELS + l];
      if (!lw.cross_in_w || !lw.cross_in_b) return fail(h, CGG_ERR_NULL, "missing cross-attention weights");
      const float* Wk = lw.cross_in_w + (size_t)C * C;
      const float* Wv = lw.cross_in_w + (size_t)2 * C * C;
      CU(cudaMemcpyAsync(h->wkv[l] + (size_t)sl * C * C, Wk, (size_t)C * C * sizeof(float), cudaMemcpyDeviceToDevice, s));
      CU(cudaMemcpyAsync(h->wkv[l] + (size_t)(n + sl) * C * C, Wv, (size_t)C * C * sizeof(float), cudaMemcpyDeviceToDevice, s));
      // key bias table: (pos + level_embed) Wk^T + bk   -> rk[l][:, sl*C:(sl+1)*C]
      GemmF32 p;
      p.A = h->pos_level[l]; p.sAm = C; p.sAk = 1;
      p.W = Wk; p.sWn = C; p.sWk = 1;
      p.bias = lw.cross_in_b + C;
      p.C = h->rk[l] + (size_t)sl * C; p.sCm = (long)n * C; p.sCn = 1;
      p.M = K; p.N = C; p.K = C;
      CU(launch_gemm_f32(p, s));
      // value bias: level_embed Wv^T + bv -> bkv[l][(n+sl)*C ...]
      GemmF32 v;
      v.A = w->level_embed + (size_t)l * C; v.sAm = C; v.sAk = 1;
      v.W = Wv; v.sWn = C; v.sWk = 1;
      v.bias = lw.cross_in_b + 2 * C;
      v.C = h->bkv[l] + (size_t)(n + sl) * C; v.sCm = C; v.sCn = 1;
      v.M = 1; v.N = C; v.K = C;
      CU(launch_gemm_f32(v, s));
    }
  }
  if (h->tc) TC(h->tc, tc_prepare(h->tc, w, H4, W4, h->lh, h->lw, h->nl, h->wkv, h->rk, h->bkv, s));
  h->prepared = true;
  return CGG_OK;
}

extern "C" size_t cgg_workspace_bytes(const cgg_handle* h, int batch) {
  if (!h || !h->prepared || batch <= 0) return 0;
  Workspace w;
  w.carve(h, batch);
  return w.total;
}

extern "C" size_t cgg_workspace_offset(const cgg_handle* h, int batch, const char* what) {
  if (!h || !h->prepared || batch <= 0 || !what) return (size_t)-1;
  Workspace w;
  w.carve(h, batch);
  const std::string n(what);
  if (n == "kv0") return w.kv[0];
  if (n == "kv1") return w.kv[1];
  if (n == "kv2") return w.kv[2];
  const size_t o = tc_workspace_offset(h->tc, batch, what);
  return o == (size_t)-1 ? o : w.tcws + o;
}

// ============================================================================== stages
static int kv_project_levels(cgg_handle* h, const cgg_weights* w, int batch, const void* const memories[CGG_NUM_LEVELS],
                             void* workspace, size_t workspace_bytes, cudaStream_t s, int l_begin, int l_end,
                             int cta_cap = 0) {
  if (!h || !w || !memories) return CGG_ERR_NULL;
  Workspace ws;
  ST(check_ws(h, batch, workspace, workspace_bytes, ws));
  const int C = h->cfg.embed_dim;
  for (int l = l_begin; l < l_end; ++l) {
    if (h->nl[l] == 0) continue;
    if (!memories[l]) return fail(h, CGG_ERR_NULL, "null memory level");
    const int K = h->lh[l] * h->lw[l], N = h->nl[l] * 2 * C;
    if (h->cfg.precision == CGG_BF16) {
      TC(h->tc, tc_kv_project(h->tc, l, batch, memories[l], at<void>(workspace, ws.kv[l]), at<void>(workspace, ws.tcws), s,
                              cta_cap));
      continue;
    }
    GemmF32 p;
    p.A = static_cast<const float*>(memories[l]); p.sAb = (long)C * K; p.sAm = 1; p.sAk = K; p.a_mmajor = true;
    p.W = h->wkv[l]; p.sWn = C; p.sWk = 1;
    p.bias = h->bkv[l];
    p.R = h->rk[l]; p.sRm = (long)h->nl[l] * C; p.sRn = 1; p.r_mod = K; p.r_ncols = h->nl[l] * C;
    p.C = at<float>(workspace, ws.kv[l]); p.sCb = (long)K * N; p.sCm = N; p.sCn = 1;
    p.M = K; p.N = N; p.K = C; p.batch = batch;
    CU(launch_gemm_f32(p, s));
  }
  return CGG_OK;
}

extern "C" int cgg_kv_project(cgg_handle* h, const cgg_weights* w, int batch, const void* const memories[CGG_NUM_LEVELS],
                              void* workspace, size_t workspace_bytes, void* stream) {
  return kv_project_levels(h, w, batch, memories, workspace, workspace_bytes, (cudaStream_t)stream, 0, CGG_NUM_LEVELS);
}

extern "C" int cgg_attn_mask_from_logits(cgg_handle* h, int batch, const float* mask_pred, int H4, int W4, int th,
                                         int tw, uint32_t* bitmap, uint8_t* all_masked, void* stream) {
  if (!h || !mask_pred || !bitmap || !all_masked) return CGG_ERR_NULL;
  if (batch <= 0 || H4 <= 0 || W4 <= 0 || th <= 0 || tw <= 0) return fail(h, CGG_ERR_BAD_SHAPE, "bad shape");
  CU(launch_mask_bits(mask_pred, batch * h->cfg.num_queries, H4, W4, th, tw, bitmap, all_masked, (cudaStream_t)stream));
  return CGG_OK;
}

// forward_head (head.py:711-761).  call_slot: row block of the all-call mask-embedding operand
// (bf16 mode); defer_einsum: leave K2 to the batched pass at the end of cgg_decoder_forward;
// fds_ready: the per-level downsampled features are already in the workspace.
static int head_call_impl(cgg_handle* h, const cgg_weights* w, int batch, const float* x, const void* mask_features,
                          int target_level, float* cls, float* emb, void* mask, float* mask_embed_out,
                          uint32_t* bitmap, uint8_t* all_masked, void* workspace, size_t workspace_bytes,
                          cudaStream_t s, int call_slot, bool defer_einsum, bool fds_ready, bool z_ready = false) {
  if (!h || !w || !x || !mask_features || !cls || (!emb && h->cfg.d_lang > 0)) return CGG_ERR_NULL;
  if (!mask && !defer_einsum) return CGG_ERR_NULL;
  Workspace ws;
  ST(check_ws(h, batch, workspace, workspace_bytes, ws));
  if (bitmap && (target_level < 0 || target_level >= CGG_NUM_LEVELS)) return fail(h, CGG_ERR_BAD_SHAPE, "bad level");
  if (bitmap && !all_masked) return CGG_ERR_NULL;
  const cgg_config& c = h->cfg;
  const int C = c.embed_dim, Q = c.num_queries, rows = batch * Q, HW = h->H4 * h->W4;
  float* z = at<float>(workspace, ws.z);
  float* h1 = at<float>(workspace, ws.h1);
  float* h2 = at<float>(workspace, ws.h2);
  float* me = mask_embed_out ? mask_embed_out : at<float>(workspace, ws.me);
  // K1: post_norm + the three heads (head.py:734-746)
  if (c.precision == CGG_BF16) {
    TC(h->tc, tc_query_heads(h->tc, w, batch, x, cls, emb, me, at<void>(workspace, ws.tcws), s, call_slot, z_ready));
  } else {
  CU(launch_layernorm(x, nullptr, w->post_norm_w, w->post_norm_b, z, rows, C, 1e-5f, true, s));
  ST(linear_rows(h, s, z, nullptr, 1, w->cls_w, w->cls_b, cls, rows, c.num_classes_p1, C));
  if (c.d_lang > 0) ST(linear_rows(h, s, z, nullptr, 1, w->v2l_w, w->v2l_b, emb, rows, c.d_lang, C));
  ST(linear_rows(h, s, z, nullptr, 1, w->me_w[0], w->me_b[0], h1, rows, C, C, 1.f, nullptr, true));
  ST(linear_rows(h, s, h1, nullptr, 1, w->me_w[1], w->me_b[1], h2, rows, C, C, 1.f, nullptr, true));
  ST(linear_rows(h, s, h2, nullptr, 1, w->me_w[2], w->me_b[2], me, rows, C, C));
  }
  // head.py:743-744; on in the class-agnostic pre-training configs, which run with use_class_emb=False (d_lang == 0 here)
  if (c.pred_emb_norm && c.d_lang > 0) CU(launch_l2norm_rows(emb, rows, c.d_lang, s));
  if (c.precision == CGG_BF16) {
    void* tws = at<void>(workspace, ws.tcws);
    TC(h->tc, tc_store_mask_embed(h->tc, batch, call_slot, me, tws, s));
    if (bitmap) {
      // K3 on tensor cores: me x (mask_features resampled to the level) -> threshold -> ballot
      if (!fds_ready) TC(h->tc, tc_downsample(h->tc, batch, mask_features, tws, s));
      TC(h->tc, tc_mask_bits(h->tc, batch, call_slot, target_level, bitmap, all_masked, tws, s));
    }
    if (!defer_einsum) TC(h->tc, tc_mask_einsum(h->tc, batch, call_slot, 1, mask_features, mask, 0, tws, s));
    return CGG_OK;
  }
  // K2: mask_pred[b,q,p] = sum_c me[b,q,c] F[b,c,p]   (head.py:748)
  GemmF32 p;
  p.A = static_cast<const float*>(mask_features); p.sAb = (long)C * HW; p.sAm = 1; p.sAk = HW; p.a_mmajor = true;
  p.W = me; p.sWb = (long)Q * C; p.sWn = C; p.sWk = 1;
  p.C = static_cast<float*>(mask); p.sCb = (long)Q * HW; p.sCm = 1; p.sCn = HW; p.c_mmajor = true;
  p.M = HW; p.N = Q; p.K = C; p.batch = batch;
  CU(launch_gemm_f32(p, s));
  // K3: downsample + threshold + bit-pack (head.py:749-759)
  if (bitmap)
    CU(launch_mask_bits(static_cast<const float*>(mask), rows, h->H4, h->W4, h->lh[target_level], h->lw[target_level],
                        bitmap, all_masked, s));
  return CGG_OK;
}

extern "C" int cgg_head_call(cgg_handle* h, const cgg_weights* w, int batch, const float* x, const void* mask_features,
                             int target_level, float* cls, float* emb, void* mask, float* mask_embed_out,
                             uint32_t* bitmap, uint8_t* all_masked, void* workspace, size_t workspace_bytes,
                             void* stream) {
  if (!mask) return CGG_ERR_NULL;
  return head_call_impl(h, w, batch, x, mask_features, target_level, cls, emb, mask, mask_embed_out, bitmap, all_masked,
                        workspace, workspace_bytes, (cudaStream_t)stream, 0, false, false);
}

extern "C" int cgg_mask_einsum(cgg_handle* h, int batch, int first_call, int num_calls, const void* mask_features,
                               void* mask, void* workspace, size_t workspace_bytes, void* stream) {
  if (!h || !mask_features || !mask) return CGG_ERR_NULL;
  if (h->cfg.precision != CGG_BF16) return fail(h, CGG_ERR_UNSUPPORTED, "cgg_mask_einsum is a CGG_BF16 stage");
  Workspace ws;
  ST(check_ws(h, batch, workspace, workspace_bytes, ws));
  if (first_call < 0 || num_calls < 1 || first_call + num_calls > h->cfg.num_layers + 1)
    return fail(h, CGG_ERR_BAD_SHAPE, "bad head-call range");
  const long call_stride = (long)batch * h->cfg.num_queries * h->H4 * h->W4;
  TC(h->tc, tc_mask_einsum(h->tc, batch, first_call, num_calls, mask_features, mask, call_stride,
                           at<void>(workspace, ws.tcws), (cudaStream_t)stream));
  return CGG_OK;
}

extern "C" int cgg_masked_attention(cgg_handle* h, int batch, int num_keys, const float* q, const void* k,
                                    const void* v, long kv_stride, long kv_batch_stride, const uint32_t* bitmap,
                                    const uint8_t* all_masked, int layer, float* out, void* out_half, void* stream) {
  if (!h || !q || !k || !v || (!out && !out_half)) return CGG_ERR_NULL;
  if (batch <= 0 || num_keys <= 0) return fail(h, CGG_ERR_BAD_SHAPE, "bad shape");
  if (layer < -1 || layer >= h->cfg.num_layers) return fail(h, CGG_ERR_BAD_SHAPE, "bad layer index");
  if (h->cfg.precision != CGG_BF16 && (layer >= 0 || out_half))
    return fail(h, CGG_ERR_UNSUPPORTED, "key-bias table and half output are CGG_BF16 options (fp32 keys carry their bias)");
  if (layer >= 0) {
    const int l = layer % CGG_NUM_LEVELS;
    if (!h->prepared) return fail(h, CGG_ERR_BAD_SHAPE, "a layer's key-bias table needs cgg_prepare()");
    if (num_keys != h->lh[l] * h->lw[l]) return fail(h, CGG_ERR_BAD_SHAPE, "num_keys is not the layer level's key count");
  }
  cudaStream_t s = (cudaStream_t)stream;
  if (h->cfg.precision == CGG_BF16) {
    TC(h->tc, tc_layer_attention(h->tc, layer, batch, num_keys, q, k, v, kv_stride, kv_batch_stride, bitmap, all_masked,
                                 out, out_half, s));
    return CGG_OK;
  }
  CU(launch_attention_f32(q, (const float*)k, (const float*)v, kv_stride, kv_batch_stride, bitmap, all_masked, out, batch,
                          h->cfg.num_queries, num_keys, h->cfg.num_heads, s));
  return CGG_OK;
}

static int decoder_layer_impl(cgg_handle* h, const cgg_weights* w, int batch, int layer, const float* x_in,
                              const uint32_t* bitmap, const uint8_t* all_masked, float* x_out, void* workspace,
                              size_t workspace_bytes, void* stream, bool chained_in, bool chained_out,
                              bool q_ready = false);

extern "C" int cgg_decoder_layer(cgg_handle* h, const cgg_weights* w, int batch, int layer, const float* x_in,
                                 const uint32_t* bitmap, const uint8_t* all_masked, float* x_out, void* workspace,
                                 size_t workspace_bytes, void* stream) {
  return decoder_layer_impl(h, w, batch, layer, x_in, bitmap, all_masked, x_out, workspace, workspace_bytes, stream, false,
                            false);
}

static int decoder_layer_impl(cgg_handle* h, const cgg_weights* w, int batch, int layer, const float* x_in,
                              const uint32_t* bitmap, const uint8_t* all_masked, float* x_out, void* workspace,
                              size_t workspace_bytes, void* stream, bool chained_in, bool chained_out, bool q_ready) {
  if (!h || !w || !x_in || !x_out) return CGG_ERR_NULL;
  cudaStream_t s = (cudaStream_t)stream;
  Workspace ws;
  ST(check_ws(h, batch, workspace, workspace_bytes, ws));
  const cgg_config& c = h->cfg;
  if (layer < 0 || layer >= c.num_layers) return fail(h, CGG_ERR_BAD_SHAPE, "bad layer index");
  const int C = c.embed_dim, Q = c.num_queries, rows = batch * Q, F = c.ffn_dim;
  const int l = layer % CGG_NUM_LEVELS, sl = layer / CGG_NUM_LEVELS, n = h->nl[l];
  const int K = h->lh[l] * h->lw[l];
  if (c.precision == CGG_BF16) {
    const long kvs = (long)n * 2 * C, kvb = (long)K * kvs;
    const __nv_bfloat16* kv = at<__nv_bfloat16>(workspace, ws.kv[l]);
    TC(h->tc, tc_decoder_layer(h->tc, w, batch, layer, x_in, kv + (size_t)sl * C, kv + (size_t)(n + sl) * C, kvs, kvb, K,
                               bitmap, all_masked, x_out, at<void>(workspace, ws.tcws), s, chained_in, chained_out, q_ready));
    return CGG_OK;
  }
  const cgg_layer_weights& lw = w->layers[layer];
  const float qscale = 1.0f / sqrtf((float)(C / c.num_heads));
  float* qb = at<float>(workspace, ws.qb);
  float* kb = at<float>(workspace, ws.kb);
  float* vb = at<float>(workspace, ws.vb);
  float* o = at<float>(workspace, ws.o);
  float* t = at<float>(workspace, ws.t);
  float* x1 = at<float>(workspace, ws.x1);
  float* x2 = at<float>(workspace, ws.x2);
  float* f = at<float>(workspace, ws.f);
  // ---- masked cross-attention (K5): q = ((x + query_embed) Wq^T + bq) / sqrt(d)
  ST(linear_rows(h, s, x_in, w->query_embed, Q, lw.cross_in_w, lw.cross_in_b, qb, rows, C, C, qscale));
  const long kv_stride = (long)n * 2 * C, kv_bstride = (long)K * kv_stride;
  const float* kv = at<float>(workspace, ws.kv[l]);
  ST(cgg_masked_attention(h, batch, K, qb, kv + (size_t)sl * C, kv + (size_t)(n + sl) * C, kv_stride, kv_bstride,
                          bitmap, all_masked, -1, o, nullptr, stream));
  ST(linear_rows(h, s, o, nullptr, 1, lw.cross_out_w, lw.cross_out_b, t, rows, C, C, 1.f, x_in));
  CU(launch_layernorm(t, nullptr, lw.norm_w[0], lw.norm_b[0], x1, rows, C, 1e-5f, true, s));
  // ---- self-attention (K6): q = k-input = x1 + query_embed, v-input = x1
  ST(linear_rows(h, s, x1, w->query_embed, Q, lw.self_in_w, lw.self_in_b, qb, rows, C, C, qscale));
  ST(linear_rows(h, s, x1, w->query_embed, Q, lw.self_in_w + (size_t)C * C, lw.self_in_b + C, kb, rows, C, C));
  ST(linear_rows(h, s, x1, nullptr, 1, lw.self_in_w + (size_t)2 * C * C, lw.self_in_b + 2 * C, vb, rows, C, C));
  CU(launch_attention_f32(qb, kb, vb, C, (long)Q * C, nullptr, nullptr, o, batch, Q, Q, c.num_heads, s));
  ST(linear_rows(h, s, o, nullptr, 1, lw.self_out_w, lw.self_out_b, t, rows, C, C, 1.f, x1));
  CU(launch_layernorm(t, nullptr, lw.norm_w[1], lw.norm_b[1], x2, rows, C, 1e-5f, true, s));
  // ---- FFN
  ST(linear_rows(h, s, x2, nullptr, 1, lw.ffn_w1, lw.ffn_b1, f, rows, F, C, 1.f, nullptr, true));
  ST(linear_rows(h, s, f, nullptr, 1, lw.ffn_w2, lw.ffn_b2, t, rows, C, F, 1.f, x2));
  CU(launch_layernorm(t, nullptr, lw.norm_w[2], lw.norm_b[2], x_out, rows, C, 1e-5f, true, s));
  return CGG_OK;
}

extern "C" int cgg_set_final_mask_only(cgg_handle* h, int on) {
  if (!h) return CGG_ERR_NULL;
  if (on && h->cfg.precision != CGG_BF16) return fail(h, CGG_ERR_UNSUPPORTED, "final-mask-only is a CGG_BF16 option");
  h->final_mask_only = on != 0;
  return CGG_OK;
}

// ========================================================================== whole path
extern "C" int cgg_decoder_forward(cgg_handle* h, const cgg_weights* w, int batch, const void* mask_features,
                                   const void* const memories[CGG_NUM_LEVELS], float* cls, float* emb, void* mask,
                                   float* x_states, uint32_t* const* bitmaps, uint8_t* all_masked, void* workspace,
                                   size_t workspace_bytes, void* stream) {
  if (!h || !w || !mask_features || !memories || !cls || (!emb && h->cfg.d_lang > 0) || !mask) return CGG_ERR_NULL;
  cudaStream_t s = (cudaStream_t)stream;
  Workspace ws;
  ST(check_ws(h, batch, workspace, workspace_bytes, ws));
  const cgg_config& c = h->cfg;
  const int C = c.embed_dim, Q = c.num_queries, L = c.num_layers;
  const size_t bqc = (size_t)batch * Q * C;
  const size_t HW = (size_t)h->H4 * h->W4;
  const size_t mask_elt = (c.precision == CGG_BF16) ? 2 : 4;
  float* xs = x_states ? x_states : at<float>(workspace, ws.xs);
  const bool tcm = c.precision == CGG_BF16;
  const bool ovl_kv = tcm && h->overlap_kv && L >= CGG_NUM_LEVELS;
  void* tws = at<void>(workspace, ws.tcws);
  if (ovl_kv) {
    // Level 0 K/V on the caller's stream (layer 0 needs it first).  Levels 1 and 2 -- 5/6 of the projection
    // work, first needed by layers 1 and 2 -- run on a helper stream on a capped number of persistent CTAs,
    // underneath head call 0 / layer 0 / head call 1 / layer 1, which are latency-bound and leave most SMs idle.
    CU(cudaEventRecord(h->ev_fork, s));
    CU(cudaStreamWaitEvent(h->side[0], h->ev_fork, 0));
    ST(kv_project_levels(h, w, batch, memories, workspace, workspace_bytes, s, 0, 1));
    for (int l = 1; l < CGG_NUM_LEVELS; ++l) {
      ST(kv_project_levels(h, w, batch, memories, workspace, workspace_bytes, h->side[0], l, l + 1));
      CU(cudaEventRecord(h->ev_kv[l], h->side[0]));
    }
  } else {
    ST(cgg_kv_project(h, w, batch, memories, workspace, workspace_bytes, stream));
  }
  if (tcm) TC(h->tc, tc_downsample(h->tc, batch, mask_features, tws, s));
  CU(launch_broadcast_rows(w->query_feat, xs, batch, Q, C, s));          // head.py:808-809
  for (int j = 0; j <= L; ++j) {
    const bool need_mask = j < L;                                           // the last mask is never used
    // layer j's query projection needs the decoder state only: it runs on a helper stream underneath head call j
    const bool q_par = ovl_kv && j > 0 && j < L;
    if (q_par) {
      CU(cudaEventRecord(h->ev_me[j], s));
      CU(cudaStreamWaitEvent(h->side[1], h->ev_me[j], 0));
      TC(h->tc, tc_layer_qproj(h->tc, w, batch, j, tws, h->side[1]));
      CU(cudaEventRecord(h->ev_join[1], h->side[1]));
    }
    uint32_t* bm = need_mask ? ((bitmaps && bitmaps[j]) ? bitmaps[j] : at<uint32_t>(workspace, ws.bitmap)) : nullptr;
    uint8_t* am = need_mask ? (all_masked ? all_masked + (size_t)j * batch * Q : at<uint8_t>(workspace, ws.allm))
                            : nullptr;
    ST(head_call_impl(h, w, batch, xs + j * bqc, mask_features, j % CGG_NUM_LEVELS,
                      cls + (size_t)j * batch * Q * c.num_classes_p1, emb ? emb + (size_t)j * batch * Q * c.d_lang : nullptr,
                      static_cast<char*>(mask) + (size_t)j * batch * Q * HW * mask_elt, nullptr, bm, am, workspace,
                      workspace_bytes, s, j, /*defer_einsum=*/tcm, /*fds_ready=*/true, /*z_ready=*/tcm && j > 0));
    if (j < L) {
      const int lvl = j % CGG_NUM_LEVELS;
      if (ovl_kv && j == lvl && lvl > 0) CU(cudaStreamWaitEvent(s, h->ev_kv[lvl], 0));   // first use of this level's K/V
      if (q_par) CU(cudaStreamWaitEvent(s, h->ev_join[1], 0));
      ST(decoder_layer_impl(h, w, batch, j, xs + j * bqc, bm, am, xs + (j + 1) * bqc, workspace, workspace_bytes, stream,
                            /*chained_in=*/tcm && j > 0, /*chained_out=*/tcm, /*q_ready=*/q_par));
    }
  }
  if (tcm && h->final_mask_only) {
    // inference shortcut: the last head call's logits only, into a (B,Q,H4,W4) buffer
    TC(h->tc, tc_mask_einsum(h->tc, batch, L, 1, mask_features, mask, (long)batch * Q * HW, tws, s));
  } else if (tcm) {
    // K2 of all L+1 head calls in one pass over mask_features
    TC(h->tc, tc_mask_einsum(h->tc, batch, 0, L + 1, mask_features, mask, (long)batch * Q * HW, tws, s));
  }
  return CGG_OK;
}

// ====================================================================== grounding side
extern "C" int cgg_noun_embeddings(cgg_handle* h, const float* table, const float* ln_w, const float* ln_b,
                                   const int64_t* ids, int n_ids, int d_lang, float eps, int text_emb_norm, float* out,
                                   void* stream) {
  if (!h || !table || !ids || !out) return CGG_ERR_NULL;
  if (text_emb_norm && (!ln_w || !ln_b)) return CGG_ERR_NULL;
  if (n_ids < 0 || d_lang <= 0) return fail(h, CGG_ERR_BAD_SHAPE, "bad shape");
  CU(launch_layernorm(table, ids, ln_w, ln_b, out, n_ids, d_lang, eps, text_emb_norm != 0, (cudaStream_t)stream));
  return CGG_OK;
}

extern "C" int cgg_similarity(cgg_handle* h, const float* a, const float* b, int M, int N, int D, float scale,
                              float* out, void* stream) {
  if (!h || !a || !b || !out) return CGG_ERR_NULL;
  if (M <= 0 || N <= 0 || D <= 0) return fail(h, CGG_ERR_BAD_SHAPE, "bad shape");
  GemmF32 p;
  p.A = a; p.sAm = D; p.sAk = 1;
  p.W = b; p.sWn = D; p.sWk = 1;
  p.C = out; p.sCm = N; p.sCn = 1;
  p.M = M; p.N = N; p.K = D; p.alpha = scale;
  CU(launch_gemm_f32(p, (cudaStream_t)stream));
  return CGG_OK;
}

namespace {

template <typename T>
int grow(cgg_handle* h, T** p, size_t* have, size_t want_elems, cudaStream_t s, bool zero) {
  if (*have >= want_elems) return CGG_OK;
  CU(cudaStreamSynchronize(s));
  cudaFree(*p);
  *p = nullptr; *have = 0;
  CU(cudaMalloc(p, want_elems * sizeof(T)));
  if (zero) CU(cudaMemsetAsync(*p, 0, want_elems * sizeof(T), s));
  *have = want_elems;
  return CGG_OK;
}

// S[(i,t), (j,q)] = cap_i[t] . pred_j[q] / T for ALL caption x image pairs: ONE tcgen05 GEMM (M = Bg*T tokens,
// N = Bg*Q, K = D) at split (hi/lo bf16, 3-term) precision -- the raw similarities reach |120| (BERT rows of norm ~24),
// so plain bf16 operands would move the softmax arguments by ~0.05.
int k7_similarity(cgg_handle* h, const float* pred, const float* cap, int Bg, int Q, int T, int D, float temperature,
                  cudaStream_t s) {
  TcState* t = h->tc ? h->tc : h->tc_aux;
  if (!t) {
    h->tc_aux = tc_create(h->cfg);
    if (!h->tc_aux) return fail(h, CGG_ERR_CUDA, "tc_create (grounding) failed");
    t = h->tc_aux;
  }
  const int rows_p = Bg * Q, rows_c = Bg * T, np = round_up(rows_p, 128);
  ST(grow(h, &h->k7.pred_hl, &h->k7.n_pred, (size_t)np * 2 * D, s, true));      // pad rows stay zero
  ST(grow(h, &h->k7.cap_hl, &h->k7.n_cap, (size_t)rows_c * 2 * D, s, false));
  ST(grow(h, &h->k7.S, &h->k7.n_S, (size_t)rows_c * rows_p, s, false));
  CU(launch_cast_bf16_split(pred, h->k7.pred_hl, rows_p, D, s));
  CU(launch_cast_bf16_split(cap, h->k7.cap_hl, rows_c, D, s));
  TcSeg sg = {};
  sg.col0 = 0; sg.ncols = rows_p; sg.ptr = h->k7.S; sg.ld = rows_p; sg.alpha = 1.0f / temperature; sg.rb_mod = 1;
  TC(t, tc_linear(t, h->k7.cap_hl, rows_c, D, h->k7.pred_hl, np, nullptr, &sg, 1, s, /*split_k=*/true));
  return CGG_OK;
}

}  // namespace

extern "C" size_t cgg_grounding_scratch_bytes(int Bg, int Q, int T) {
  (void)Q; (void)T;
  return Bg > 0 ? (size_t)2 * Bg * Bg * sizeof(float) : 0;
}

extern "C" int cgg_grounding_loss(cgg_handle* h, const float* pred, const float* cap, const int64_t* cap_mask, int Bg,
                                  int Q, int T, int D, float temperature, float loss_weight, float* loss,
                                  void* scratch, size_t scratch_bytes, void* stream) {
  if (!h || !pred || !cap || !cap_mask || !loss || !scratch) return CGG_ERR_NULL;
  if (Bg <= 0 || Bg > 128 || Q <= 0 || T <= 0 || D <= 0 || (D % 4) != 0) return fail(h, CGG_ERR_BAD_SHAPE, "bad shape");
  if ((size_t)(T * Q + T + Q) * sizeof(float) > 200 * 1024) return fail(h, CGG_ERR_BAD_SHAPE, "T*Q too large");
  if (scratch_bytes < cgg_grounding_scratch_bytes(Bg, Q, T)) return fail(h, CGG_ERR_WORKSPACE, "scratch too small");
  cudaStream_t s = (cudaStream_t)stream;
  float* g1 = static_cast<float*>(scratch);
  float* g2 = g1 + (size_t)Bg * Bg;
  const float* S_pre = nullptr;
  if (D % 64 == 0) {
    ST(k7_similarity(h, pred, cap, Bg, Q, T, D, temperature, s));
    S_pre = h->k7.S;
  }
  CU(launch_grounding_pairs(pred, cap, cap_mask, Bg, Q, T, D, temperature, g1, g2, s, S_pre));
  CU(launch_grounding_finish(g1, g2, cap_mask, Bg, T, loss_weight, loss, s));
  return CGG_OK;
}

extern "C" size_t cgg_grounding_bwd_scratch_bytes(int Bg, int Q, int T) {
  if (Bg <= 0 || Q <= 0 || T <= 0) return 0;
  return ((size_t)4 * Bg * Bg + (size_t)Bg * Bg * T * Q + 1) * sizeof(float);
}

extern "C" int cgg_grounding_loss_backward(cgg_handle* h, const float* pred, const float* cap, const int64_t* cap_mask,
                                           int Bg, int Q, int T, int D, float temperature, float loss_weight,
                                           float grad_out, float* dpred, void* scratch, size_t scratch_bytes,
                                           void* stream) {
  if (!h || !pred || !cap || !cap_mask || !dpred || !scratch) return CGG_ERR_NULL;
  if (Bg <= 0 || Bg > 128 || Q <= 0 || T <= 0 || D <= 0 || (D % 4) != 0) return fail(h, CGG_ERR_BAD_SHAPE, "bad shape");
  if ((size_t)(T * Q + 3 * T + 3 * Q) * sizeof(float) > 200 * 1024) return fail(h, CGG_ERR_BAD_SHAPE, "T*Q too large");
  if (scratch_bytes < cgg_grounding_bwd_scratch_bytes(Bg, Q, T)) return fail(h, CGG_ERR_WORKSPACE, "scratch too small");
  cudaStream_t s = (cudaStream_t)stream;
  float* g1 = static_cast<float*>(scratch);
  float* g2 = g1 + (size_t)Bg * Bg;
  float* d1 = g2 + (size_t)Bg * Bg;
  float* d2 = d1 + (size_t)Bg * Bg;
  float* loss = d2 + (size_t)Bg * Bg;
  float* dS = loss + 1;
  if (D % 64 == 0) {
    // tensor-core mode: S once (tcgen05), pair kernels on S, then dpred[(j,q), :] = sum_(i,t) dS[(j,q), (i,t)] cap[(i,t), :]
    // as a second split-precision tcgen05 GEMM (M = Bg*Q tokens, N = D, K = Bg*T padded to 64)
    ST(k7_similarity(h, pred, cap, Bg, Q, T, D, temperature, s));
    const int rows_p = Bg * Q, rows_c = Bg * T, Kp = round_up(rows_c, 64), nd = round_up(D, 128);
    ST(grow(h, &h->k7.dst_hl, &h->k7.n_dst, (size_t)rows_p * 2 * Kp, s, true));    // pad columns stay zero
    ST(grow(h, &h->k7.capT_hl, &h->k7.n_capT, (size_t)nd * 2 * Kp, s, true));
    CU(launch_grounding_pairs(pred, cap, cap_mask, Bg, Q, T, D, temperature, g1, g2, s, h->k7.S));
    CU(launch_grounding_finish(g1, g2, cap_mask, Bg, T, loss_weight, loss, s, d1, d2));
    CU(launch_grounding_bwd_pairs(pred, cap, cap_mask, Bg, Q, T, D, temperature, d1, d2, grad_out, nullptr, s, h->k7.S,
                                  h->k7.dst_hl, Kp));
    CU(launch_transpose_split(cap, h->k7.capT_hl, rows_c, D, Kp, s));
    TcState* t = h->tc ? h->tc : h->tc_aux;
    TcSeg sg = {};
    sg.col0 = 0; sg.ncols = D; sg.ptr = dpred; sg.ld = D; sg.alpha = 1.0f; sg.rb_mod = 1;
    TC(t, tc_linear(t, h->k7.dst_hl, rows_p, Kp, h->k7.capT_hl, nd, nullptr, &sg, 1, s, /*split_k=*/true));
    return CGG_OK;
  }
  // recompute the pair distances, then d loss / d cost, d loss / d S, and dpred_j = sum_{i,t} dS[j][i][t][:]^T cap[i][t][:]
  CU(launch_grounding_pairs(pred, cap, cap_mask, Bg, Q, T, D, temperature, g1, g2, s));
  CU(launch_grounding_finish(g1, g2, cap_mask, Bg, T, loss_weight, loss, s, d1, d2));
  CU(launch_grounding_bwd_pairs(pred, cap, cap_mask, Bg, Q, T, D, temperature, d1, d2, grad_out, dS, s));
  GemmF32 p;
  p.A = dS; p.sAb = (long)Bg * T * Q; p.sAm = 1; p.sAk = Q; p.a_mmajor = true;     // A[q, (i,t)]
  p.W = cap; p.sWn = 1; p.sWk = D;                                                  // W[d, (i,t)]
  p.C = dpred; p.sCb = (long)Q * D; p.sCm = D; p.sCn = 1;
  p.M = Q; p.N = D; p.K = Bg * T; p.batch = Bg;
  CU(launch_gemm_f32(p, s));
  return CGG_OK;
}

// ====================================================================== training-step stages
extern "C" int cgg_gemm_f32(cgg_handle* h, const cgg_gemm_desc* d, void* stream) {
  if (!h || !d || !d->A || !d->W || !d->C) return CGG_ERR_NULL;
  if (d->M < 0 || d->N < 0 || d->K < 0 || d->batch < 1) return fail(h, CGG_ERR_BAD_SHAPE, "bad gemm shape");
  if ((long)d->batch > 65535 || ((long)d->N + 63) / 64 > 65535) return fail(h, CGG_ERR_BAD_SHAPE, "gemm grid too large");
  GemmF32 p;
  p.A = d->A; p.sAb = d->sAb; p.sAm = d->sAm; p.sAk = d->sAk;
  if (d->A2) { p.A2 = d->A2; p.sA2m = d->sA2m; p.sA2k = d->sA2k; p.a2_mod = d->a2_mod > 0 ? d->a2_mod : 1; }
  p.W = d->W; p.sWb = d->sWb; p.sWn = d->sWn; p.sWk = d->sWk;
  p.bias = d->bias;
  if (d->R) { p.R = d->R; p.sRb = d->sRb; p.sRm = d->sRm; p.sRn = d->sRn; p.r_mod = d->r_mod > 0 ? d->r_mod : 1; p.r_ncols = d->r_ncols; }
  p.C = d->C; p.sCb = d->sCb; p.sCm = d->sCm; p.sCn = d->sCn;
  p.M = d->M; p.N = d->N; p.K = d->K; p.batch = d->batch;
  if (d->relu) p.relu_from = 0;
  p.alpha = d->alpha;
  p.a_mmajor = d->a_mmajor != 0; p.c_mmajor = d->c_mmajor != 0;
  if (d->batch_inner > 1) {
    if (d->batch % d->batch_inner) return fail(h, CGG_ERR_BAD_SHAPE, "batch must be a multiple of batch_inner");
    p.batch_inner = d->batch_inner; p.sAb2 = d->sAb2; p.sWb2 = d->sWb2; p.sCb2 = d->sCb2;
  }
  p.accumulate = d->accumulate != 0;
  p.slot = d->slot;
  if (d->conv_cin > 0) {
    if (d->K != 9 * d->conv_cin || d->A2 || d->batch_inner < 1) return fail(h, CGG_ERR_BAD_SHAPE, "conv_cin: K must be 9 * conv_cin, batch_inner = image height");
    p.conv_cin = d->conv_cin;
    p.batch_inner = d->batch_inner; p.sAb2 = d->sAb2; p.sWb2 = d->sWb2; p.sCb2 = d->sCb2;
  }
  if (d->tf32) {
    if (!h->tf32 && !(h->tf32 = tf32_create())) return fail(h, CGG_ERR_CUDA, "tf32_create failed");
    const int r = launch_gemm_tf32(h->tf32, p, (cudaStream_t)stream);
    if (r == 0) return CGG_OK;
    if (r < 0) return fail(h, CGG_ERR_CUDA, tf32_last_error(h->tf32));
  }
  CU(launch_gemm_f32(p, (cudaStream_t)stream));
  return CGG_OK;
}

extern "C" int cgg_layernorm(cgg_handle* h, const float* x, const float* w, const float* b, float* y, int rows, int n,
                             float eps, void* stream) {
  if (!h || !x || !w || !b || !y) return CGG_ERR_NULL;
  if (rows < 0 || n <= 0) return fail(h, CGG_ERR_BAD_SHAPE, "bad shape");
  CU(launch_layernorm(x, nullptr, w, b, y, rows, n, eps, true, (cudaStream_t)stream));
  return CGG_OK;
}

extern "C" size_t cgg_layernorm_bwd_scratch_bytes(int rows, int n) {
  return rows > 0 && n > 0 ? (size_t)((rows + 7) / 8) * 2 * n * sizeof(float) : 0;
}

extern "C" int cgg_layernorm_backward(cgg_handle* h, const float* x, const float* w, const float* dy, float* dx, float* dw,
                                      float* db, void* scratch, size_t scratch_bytes, int rows, int n, float eps,
                                      void* stream) {
  if (!h || !x || !w || !dy || !dx || !dw || !db || !scratch) return CGG_ERR_NULL;
  if (rows <= 0 || n <= 0 || (size_t)8 * 2 * n * sizeof(float) > 200 * 1024) return fail(h, CGG_ERR_BAD_SHAPE, "bad shape");
  if (scratch_bytes < cgg_layernorm_bwd_scratch_bytes(rows, n)) return fail(h, CGG_ERR_WORKSPACE, "scratch too small");
  CU(launch_layernorm_bwd(x, w, dy, dx, dw, db, static_cast<float*>(scratch), rows, n, eps, (cudaStream_t)stream));
  return CGG_OK;
}

extern "C" int cgg_relu_backward(cgg_handle* h, const float* y, const float* dy, float* dx, long n, float alpha, void* stream) {
  if (!h || !y || !dy || !dx) return CGG_ERR_NULL;
  CU(launch_relu_bwd(y, dy, dx, n, alpha, (cudaStream_t)stream));
  return CGG_OK;
}

extern "C" int cgg_axpy(cgg_handle* h, const float* in, float* out, long n, float alpha, void* stream) {
  if (!h || !in || !out) return CGG_ERR_NULL;
  CU(launch_axpy(in, out, n, alpha, (cudaStream_t)stream));
  return CGG_OK;
}

extern "C" int cgg_add_rows(cgg_handle* h, const float* x, const float* add, float* out, int batch, long per, void* stream) {
  if (!h || !add || !out) return CGG_ERR_NULL;
  if (batch < 1 || per < 1) return fail(h, CGG_ERR_BAD_SHAPE, "bad shape");
  CU(launch_add_rows(x, add, out, batch, per, (cudaStream_t)stream));
  return CGG_OK;
}

extern "C" int cgg_sum_batch(cgg_handle* h, const float* g, float* out, int batch, long per, void* stream) {
  if (!h || !g || !out) return CGG_ERR_NULL;
  if (batch < 1 || per < 1) return fail(h, CGG_ERR_BAD_SHAPE, "bad shape");
  CU(launch_sum_batch(g, out, batch, per, (cudaStream_t)stream));
  return CGG_OK;
}

extern "C" int cgg_colsum(cgg_handle* h, const float* g, float* out, long rows, int n, float alpha, int accumulate,
                          void* stream) {
  if (!h || !g || !out) return CGG_ERR_NULL;
  if (rows < 0 || n < 1 || (rows + 255) / 256 > 65535) return fail(h, CGG_ERR_BAD_SHAPE, "bad shape");
  CU(launch_colsum(g, out, rows, n, alpha, (cudaStream_t)stream, accumulate != 0));
  return CGG_OK;
}

extern "C" int cgg_mem_prep(cgg_handle* h, const float* mem, const float* level, const float* pos_level, float* key_in,
                            float* val_in, int batch, int C, int K, void* stream) {
  if (!h || !mem || !level || !pos_level || !key_in || !val_in) return CGG_ERR_NULL;
  if (batch < 1 || batch > 65535 || C < 1 || K < 1) return fail(h, CGG_ERR_BAD_SHAPE, "bad shape");
  CU(launch_mem_prep(mem, level, pos_level, key_in, val_in, batch, C, K, (cudaStream_t)stream));
  return CGG_OK;
}

extern "C" int cgg_mem_prep_backward(cgg_handle* h, const float* dkey_in, const float* dval_in, float* dmem, int batch,
                                     int C, int K, void* stream) {
  if (!h || !dkey_in || !dval_in || !dmem) return CGG_ERR_NULL;
  if (batch < 1 || batch > 65535 || C < 1 || K < 1) return fail(h, CGG_ERR_BAD_SHAPE, "bad shape");
  CU(launch_mem_prep_bwd(dkey_in, dval_in, dmem, batch, C, K, (cudaStream_t)stream));
  return CGG_OK;
}

extern "C" int cgg_sine_pos(cgg_handle* h, float* out, int hh, int ww, int C, void* stream) {
  if (!h || !out) return CGG_ERR_NULL;
  if (hh < 1 || ww < 1 || C < 2 || (C & 1)) return fail(h, CGG_ERR_BAD_SHAPE, "bad shape");
  CU(launch_pos_level(nullptr, out, hh, ww, C, (cudaStream_t)stream));
  return CGG_OK;
}

extern "C" int cgg_attention_f32(cgg_handle* h, int batch, int num_q, int num_keys, int heads, const float* q,
                                 const float* k, const float* v, long kv_stride, long kv_batch_stride,
                                 const uint32_t* bitmap, const uint8_t* all_masked, float* out, void* stream) {
  if (!h || !q || !k || !v || !out) return CGG_ERR_NULL;
  if (batch < 1 || num_q < 1 || num_keys < 1) return fail(h, CGG_ERR_BAD_SHAPE, "bad shape");
  if (heads < 1 || kv_stride < 32L * heads) return fail(h, CGG_ERR_BAD_SHAPE, "heads < 1 or kv_stride < heads * 32");
  CU(launch_attention_f32(q, k, v, kv_stride, kv_batch_stride, bitmap, all_masked, out, batch, num_q, num_keys, heads,
                          (cudaStream_t)stream));
  return CGG_OK;
}

extern "C" int cgg_attention_backward(cgg_handle* h, int batch, int num_q, int num_keys, int heads, const float* q,
                                      const float* k, const float* v, long kv_stride, long kv_batch_stride,
                                      const uint32_t* bitmap, const uint8_t* all_masked, const float* out,
                                      const float* dout, float* dq, float* dk, float* dv, long dkv_stride,
                                      long dkv_batch_stride, float* scratch, void* stream) {
  if (!h || !q || !k || !v || !out || !dout || !dq || !dk || !dv || !scratch) return CGG_ERR_NULL;
  if (batch < 1 || batch > 65535 || num_q < 1 || num_keys < 1) return fail(h, CGG_ERR_BAD_SHAPE, "bad shape");
  if (heads < 1 || kv_stride < 32L * heads) return fail(h, CGG_ERR_BAD_SHAPE, "heads < 1 or kv_stride < heads * 32");
  const size_t n = (size_t)batch * heads * num_q;
  CU(launch_attention_bwd(q, k, v, kv_stride, kv_batch_stride, bitmap, all_masked, out, dout, scratch, scratch + n, dq, dk,
                          dv, dkv_stride, dkv_batch_stride, batch, num_q, num_keys, heads, (cudaStream_t)stream));
  return CGG_OK;
}

extern "C" int cgg_attn_softmax_rows(cgg_handle* h, float* scores, const uint32_t* bitmap, const uint8_t* all_masked,
                                     int batch, int heads, int num_q, int num_keys, void* stream) {
  if (!h || !scores) return CGG_ERR_NULL;
  if (batch < 1 || heads < 1 || num_q < 1 || num_keys < 1) return fail(h, CGG_ERR_BAD_SHAPE, "bad shape");
  CU(launch_attn_softmax_rows(scores, bitmap, all_masked, batch, heads, num_q, num_keys, (cudaStream_t)stream));
  return CGG_OK;
}

extern "C" int cgg_attn_dscore(cgg_handle* h, const float* probs, float* dprobs, const float* out, const float* dout,
                               int batch, int heads, int head_dim, int num_q, int num_keys, void* stream) {
  if (!h || !probs || !dprobs || !out || !dout) return CGG_ERR_NULL;
  if (batch < 1 || heads < 1 || head_dim < 1 || num_q < 1 || num_keys < 1) return fail(h, CGG_ERR_BAD_SHAPE, "bad shape");
  CU(launch_attn_dscore(probs, dprobs, out, dout, batch, heads, head_dim, num_q, num_keys, (cudaStream_t)stream));
  return CGG_OK;
}

// ====================================================================== the step after the path (training time, f2)
extern "C" int cgg_point_sample(cgg_handle* h, const float* in, const float* coords, float* out, int planes, int hh, int ww,
                                int num_points, int coords_shared, void* stream) {
  if (!h || !in || !coords || !out) return CGG_ERR_NULL;
  if (planes < 0 || hh < 1 || ww < 1 || num_points < 0) return fail(h, CGG_ERR_BAD_SHAPE, "bad shape");
  CU(launch_point_sample(in, coords, out, planes, hh, ww, num_points, coords_shared != 0, (cudaStream_t)stream));
  return CGG_OK;
}

extern "C" int cgg_point_sample_backward(cgg_handle* h, const float* dout, const float* coords, float* din, int planes, int hh,
                                         int ww, int num_points, int coords_shared, void* stream) {
  if (!h || !dout || !coords || !din) return CGG_ERR_NULL;
  if (planes < 0 || hh < 1 || ww < 1 || num_points < 0) return fail(h, CGG_ERR_BAD_SHAPE, "bad shape");
  CU(launch_point_sample_bwd(dout, coords, din, planes, hh, ww, num_points, coords_shared != 0, (cudaStream_t)stream));
  return CGG_OK;
}

extern "C" int cgg_panoptic_stuff_labels(cgg_handle* h, const void* sem, int sem_is_i64, int batch, int hs, int ws,
                                         int num_things, int num_classes, uint32_t* bitmap, int64_t* stuff_labels, int* counts,
                                         void* stream) {
  if (!h || !sem || !bitmap || !stuff_labels || !counts) return CGG_ERR_NULL;
  if (batch < 1 || hs < 1 || ws < 1 || num_things < 0 || num_classes <= num_things || num_classes - num_things > 8192)
    return fail(h, CGG_ERR_BAD_SHAPE, "bad shape");
  CU(launch_panoptic_stuff_labels(sem, sem_is_i64 != 0, batch, (long)hs * ws, num_things, num_classes, bitmap, stuff_labels,
                                  counts, (cudaStream_t)stream));
  return CGG_OK;
}

extern "C" int cgg_gt_point_sample(cgg_handle* h, const cgg_gt_image* images, const int* rows, const float* coords, float* out,
                                   int num_rows, int num_points, int coords_per_image, void* stream) {
  if (!h || !images || !rows || !coords || !out) return CGG_ERR_NULL;
  if (num_rows < 0 || num_points < 0) return fail(h, CGG_ERR_BAD_SHAPE, "bad shape");
  CU(launch_gt_point_sample(images, rows, coords, out, num_rows, num_points, coords_per_image != 0, (cudaStream_t)stream));
  return CGG_OK;
}

extern "C" int cgg_matching_cost(cgg_handle* h, const float* mask_points, const float* gt_points, const float* cls_scores,
                                 const float* cls_emb_logits, const int64_t* gt_labels, int num_q, int num_gt, int classes_p1,
                                 int num_points, float w_cls, float w_cls_emb, float w_mask, float w_dice, float dice_eps,
                                 float* scratch, float* cost, void* stream) {
  if (!h || !mask_points || !gt_points || !gt_labels || !scratch || !cost) return CGG_ERR_NULL;
  if (num_q < 0 || num_gt < 0 || num_points < 1 || classes_p1 < 1) return fail(h, CGG_ERR_BAD_SHAPE, "bad shape");
  if ((w_cls != 0.f && !cls_scores) || (w_cls_emb != 0.f && !cls_emb_logits)) return CGG_ERR_NULL;
  CU(launch_matching_cost(mask_points, gt_points, cls_scores, cls_emb_logits, gt_labels, num_q, num_gt, classes_p1, num_points,
                          w_cls, w_cls_emb, w_mask, w_dice, dice_eps, scratch, cost, (cudaStream_t)stream));
  return CGG_OK;
}

extern "C" int cgg_point_losses(cgg_handle* h, const float* pred_points, const float* target_points, int rows, int num_points,
                                float dice_eps, float* abc, float* dice_rows, float* bce_rows, void* stream) {
  if (!h || !pred_points || !target_points || !abc || !dice_rows || !bce_rows) return CGG_ERR_NULL;
  if (rows < 0 || rows > 65535 || num_points < 1) return fail(h, CGG_ERR_BAD_SHAPE, "bad shape");
  CU(launch_point_losses(pred_points, target_points, rows, num_points, dice_eps, abc, dice_rows, bce_rows, (cudaStream_t)stream));
  return CGG_OK;
}

extern "C" int cgg_point_losses_backward(cgg_handle* h, const float* pred_points, const float* target_points, const float* abc,
                                         int rows, int num_points, float dice_eps, const float* g_dice_rows,
                                         const float* g_bce_rows, float* dpred, void* stream) {
  if (!h || !pred_points || !target_points || !abc || !g_dice_rows || !g_bce_rows || !dpred) return CGG_ERR_NULL;
  if (rows < 0 || rows > 65535 || num_points < 1) return fail(h, CGG_ERR_BAD_SHAPE, "bad shape");
  CU(launch_point_losses_bwd(pred_points, target_points, abc, rows, num_points, dice_eps, g_dice_rows, g_bce_rows, dpred,
                             (cudaStream_t)stream));
  return CGG_OK;
}

extern "C" int cgg_weighted_ce(cgg_handle* h, const float* logits, const int64_t* labels, const float* class_weight, int rows,
                               int classes_p1, float* row_loss, float* row_weight, float* lse, void* stream) {
  if (!h || !logits || !labels || !class_weight || !row_loss || !row_weight || !lse) return CGG_ERR_NULL;
  if (rows < 0 || classes_p1 < 1) return fail(h, CGG_ERR_BAD_SHAPE, "bad shape");
  CU(launch_weighted_ce(logits, labels, class_weight, rows, classes_p1, row_loss, row_weight, lse, (cudaStream_t)stream));
  return CGG_OK;
}

extern "C" int cgg_weighted_ce_backward(cgg_handle* h, const float* logits, const int64_t* labels, const float* class_weight,
                                        const float* lse, int rows, int classes_p1, const float* g_rows, float* dlogits,
                                        void* stream) {
  if (!h || !logits || !labels || !class_weight || !lse || !g_rows || !dlogits) return CGG_ERR_NULL;
  if (rows < 0 || classes_p1 < 1) return fail(h, CGG_ERR_BAD_SHAPE, "bad shape");
  CU(launch_weighted_ce_bwd(logits, labels, class_weight, lse, rows, classes_p1, g_rows, dlogits, (cudaStream_t)stream));
  return CGG_OK;
}

// ====================================================================== the step after the path (test time)
extern "C" int cgg_upsample_masks(cgg_handle* h, const void* logits, int is_bf16, float* out, int planes, int h4, int w4,
                                  int up_h, int up_w, void* stream) {
  if (!h || !logits || !out) return CGG_ERR_NULL;
  if (planes < 1 || planes > 65535 || h4 < 1 || w4 < 1 || up_h < 1 || up_w < 1) return fail(h, CGG_ERR_BAD_SHAPE, "bad shape");
  CU(launch_upsample_masks(logits, is_bf16 != 0, out, planes, h4, w4, up_h, up_w, (cudaStream_t)stream));
  return CGG_OK;
}

extern "C" int cgg_instance_mask_stats(cgg_handle* h, const void* logits, int is_bf16, const int* geom, int batch, int num_q,
                                       int h4, int w4, int up_h, int up_w, int max_out_h, int max_out_w, uint32_t* bits,
                                       int* count, float* sig_sum, int* bbox, void* stream) {
  if (!h || !logits || !geom || !count || !sig_sum || !bbox) return CGG_ERR_NULL;
  if (batch < 1 || num_q < 1 || (long)batch * num_q > 65535 || h4 < 1 || w4 < 1 || up_h < 1 || up_w < 1 || max_out_h < 1 ||
      max_out_w < 1)
    return fail(h, CGG_ERR_BAD_SHAPE, "bad shape");
  CU(launch_instance_mask_stats(logits, is_bf16 != 0, geom, batch, num_q, h4, w4, up_h, up_w, max_out_h, max_out_w, bits, count,
                                sig_sum, bbox, (cudaStream_t)stream));
  return CGG_OK;
}

extern "C" int cgg_softmax_rows(cgg_handle* h, float* x, int rows, int n, void* stream) {
  if (!h || !x) return CGG_ERR_NULL;
  if (rows < 0 || n < 1) return fail(h, CGG_ERR_BAD_SHAPE, "bad shape");
  CU(launch_softmax_rows(x, rows, n, (cudaStream_t)stream));
  return CGG_OK;
}

extern "C" size_t cgg_panoptic_scratch_bytes(int batch, int num_q) {
  if (batch < 1 || num_q < 1) return 0;
  return panoptic_scratch_bytes(batch, num_q);
}

extern "C" int cgg_panoptic_fuse(cgg_handle* h, const void* logits, int is_bf16, const float* probs, const int* geom, int batch,
                                 int num_q, int classes_p1, int num_things, int h4, int w4, int up_h, int up_w, int max_out_h,
                                 int max_out_w, double object_mask_thr, double iou_thr, int filter_low_score, int* pan,
                                 int* mask_area, int* original_area, int* seg_value, void* scratch, size_t scratch_bytes,
                                 void* stream) {
  if (!h || !logits || !probs || !geom || !pan || !scratch) return CGG_ERR_NULL;
  if (batch < 1 || batch > 65535 || num_q < 1 || num_q > 4096 || classes_p1 < 2 || num_things < 0 ||
      num_things > classes_p1 - 1 || h4 < 1 || w4 < 1 || up_h < 1 || up_w < 1 || max_out_h < 1 || max_out_h > 65535 ||
      max_out_w < 1)
    return fail(h, CGG_ERR_BAD_SHAPE, "bad shape");
  if (scratch_bytes < panoptic_scratch_bytes(batch, num_q)) return fail(h, CGG_ERR_WORKSPACE, "panoptic scratch too small");
  CU(launch_panoptic_fuse(logits, is_bf16 != 0, probs, geom, batch, num_q, classes_p1, num_things, h4, w4, up_h, up_w, max_out_h,
                          max_out_w, object_mask_thr, iou_thr, filter_low_score != 0, pan, mask_area, original_area, seg_value,
                          scratch, (cudaStream_t)stream));
  return CGG_OK;
}

// ====================================================================== the pixel decoder before the path (row f3)
extern "C" int cgg_ms_deform_attn(cgg_handle* h, const float* value, long value_stride, const float* offsets, long offset_stride,
                                  const float* weight_logits, long logit_stride, float* out, int batch, int tokens, int heads,
                                  int levels, int points, const int* level_h, const int* level_w, void* stream) {
  if (!h || !value || !offsets || !weight_logits || !out || !level_h || !level_w) return CGG_ERR_NULL;
  if (value_stride < heads * 32 || value_stride % 4 || offset_stride < heads * levels * points * 2 || offset_stride % 2 ||
      logit_stride < heads * levels * points || (reinterpret_cast<uintptr_t>(value) & 15) || (reinterpret_cast<uintptr_t>(offsets) & 7))
    return fail(h, CGG_ERR_BAD_SHAPE, "ms_deform_attn: token strides / alignment (value rows 16-byte, offset rows 8-byte aligned)");
  if (batch < 0 || tokens < 1 || heads < 1 || heads > 8 || levels < 1 || levels > 4 || points < 1 || levels * points > 16)
    return fail(h, CGG_ERR_BAD_SHAPE, "ms_deform_attn: heads <= 8 (x 32 channels), levels <= 4, levels * points <= 16");
  long tot = 0;
  for (int l = 0; l < levels; ++l) tot += (long)level_h[l] * level_w[l];
  if (tot != tokens) return fail(h, CGG_ERR_BAD_SHAPE, "ms_deform_attn: level sizes do not add up to the token count");
  CU(launch_ms_deform_attn(value, value_stride, offsets, offset_stride, weight_logits, logit_stride, out, batch, tokens, heads, levels, points,
                           level_h, level_w, (cudaStream_t)stream));
  return CGG_OK;
}

extern "C" int cgg_ms_deform_attn_backward(cgg_handle* h, const float* value, const float* offsets, const float* weight_logits,
                                           const float* dout, float* dvalue, float* doffsets, float* dweight_logits, int batch,
                                           int tokens, int heads, int levels, int points, const int* level_h, const int* level_w,
                                           void* stream) {
  if (!h || !value || !offsets || !weight_logits || !dout || !dvalue || !doffsets || !dweight_logits || !level_h || !level_w) return CGG_ERR_NULL;
  if (batch < 0 || tokens < 1 || heads < 1 || heads > 8 || levels < 1 || levels > 4 || points < 1 || levels * points > 16)
    return fail(h, CGG_ERR_BAD_SHAPE, "ms_deform_attn: heads <= 8 (x 32 channels), levels <= 4, levels * points <= 16");
  long tot = 0;
  for (int l = 0; l < levels; ++l) tot += (long)level_h[l] * level_w[l];
  if (tot != tokens) return fail(h, CGG_ERR_BAD_SHAPE, "ms_deform_attn: level sizes do not add up to the token count");
  CU(launch_ms_deform_attn_bwd(value, offsets, weight_logits, dout, dvalue, doffsets, dweight_logits, batch, tokens, heads, levels, points,
                               level_h, level_w, (cudaStream_t)stream));
  return CGG_OK;
}

static bool gn_shape_ok(int batch, int pixels, int channels, int groups) {
  return batch >= 0 && pixels >= 1 && channels >= 4 && groups >= 1 && channels % groups == 0 && (channels / groups) % 4 == 0 &&
         (long)batch <= 65535;
}

extern "C" size_t cgg_group_norm_scratch_bytes(int batch, int pixels, int channels, int groups) {
  return gn_shape_ok(batch, pixels, channels, groups) ? group_norm_scratch_floats(batch, pixels, channels, groups) * sizeof(float) : 0;
}

extern "C" int cgg_group_norm_tokens(cgg_handle* h, const float* x, const float* gamma, const float* beta, float* y, float* mean_rstd,
                                     void* scratch, size_t scratch_bytes, int batch, int pixels, int channels, int groups, float eps,
                                     int relu, void* stream) {
  if (!h || !x || !gamma || !beta || !y || !mean_rstd || !scratch) return CGG_ERR_NULL;
  if (!gn_shape_ok(batch, pixels, channels, groups)) return fail(h, CGG_ERR_BAD_SHAPE, "group_norm: channels / groups must be a multiple of 4");
  if (scratch_bytes < cgg_group_norm_scratch_bytes(batch, pixels, channels, groups)) return fail(h, CGG_ERR_WORKSPACE, "group_norm scratch too small");
  CU(launch_group_norm(x, gamma, beta, y, mean_rstd, (float*)scratch, batch, pixels, channels, groups, eps, relu != 0, (cudaStream_t)stream));
  return CGG_OK;
}

extern "C" int cgg_group_norm_tokens_backward(cgg_handle* h, const float* x, const float* dy, const float* mean_rstd, const float* gamma,
                                              float* dx, float* dgamma, float* dbeta, void* scratch, size_t scratch_bytes, int batch,
                                              int pixels, int channels, int groups, void* stream) {
  if (!h || !x || !dy || !mean_rstd || !gamma || !dx || !dgamma || !dbeta || !scratch) return CGG_ERR_NULL;
  if (!gn_shape_ok(batch, pixels, channels, groups)) return fail(h, CGG_ERR_BAD_SHAPE, "group_norm: channels / groups must be a multiple of 4");
  if (scratch_bytes < cgg_group_norm_scratch_bytes(batch, pixels, channels, groups)) return fail(h, CGG_ERR_WORKSPACE, "group_norm scratch too small");
  CU(launch_group_norm_bwd(x, dy, mean_rstd, gamma, dx, dgamma, dbeta, (float*)scratch, batch, pixels, channels, groups, (cudaStream_t)stream));
  return CGG_OK;
}

extern "C" int cgg_upsample_add_tokens(cgg_handle* h, const float* lateral, const float* coarse, long coarse_batch_stride, float* out,
                                       int batch, int H, int W, int ch, int cw, int channels, void* stream) {
  if (!h || !lateral || !coarse || !out) return CGG_ERR_NULL;
  if (batch < 0 || H < 1 || W < 1 || ch < 1 || cw < 1 || channels < 4 || channels % 4) return fail(h, CGG_ERR_BAD_SHAPE, "bad shape");
  CU(launch_upsample_add(lateral, coarse, coarse_batch_stride, out, batch, H, W, ch, cw, channels, (cudaStream_t)stream));
  return CGG_OK;
}

extern "C" int cgg_upsample_add_tokens_backward(cgg_handle* h, const float* dout, float* dcoarse, int batch, int H, int W, int ch, int cw,
                                                int channels, void* stream) {
  if (!h || !dout || !dcoarse) return CGG_ERR_NULL;
  if (batch < 0 || H < 1 || W < 1 || ch < 1 || cw < 1 || channels < 4 || channels % 4) return fail(h, CGG_ERR_BAD_SHAPE, "bad shape");
  CU(launch_upsample_add_bwd(dout, dcoarse, batch, H, W, ch, cw, channels, (cudaStream_t)stream));
  return CGG_OK;
}

extern "C" int cgg_tokens_to_nchw(cgg_handle* h, const float* tokens, long token_batch_stride, void* out, int out_bf16, int batch,
                                  int pixels, int channels, void* stream) {
  if (!h || !tokens || !out) return CGG_ERR_NULL;
  if (batch < 0 || batch > 65535 || pixels < 1 || channels < 1) return fail(h, CGG_ERR_BAD_SHAPE, "bad shape");
  CU(launch_tokens_to_nchw(tokens, token_batch_stride, out, out_bf16 != 0, batch, pixels, channels, (cudaStream_t)stream));
  return CGG_OK;
}

extern "C" int cgg_nchw_to_tokens(cgg_handle* h, const float* in, float* tokens, long token_batch_stride, int batch, int pixels,
                                  int channels, int accumulate, void* stream) {
  if (!h || !in || !tokens) return CGG_ERR_NULL;
  if (batch < 0 || batch > 65535 || pixels < 1 || channels < 1) return fail(h, CGG_ERR_BAD_SHAPE, "bad shape");
  CU(launch_nchw_to_tokens(in, tokens, token_batch_stride, batch, pixels, channels, accumulate != 0, (cudaStream_t)stream));
  return CGG_OK;
}

// ====================================================================== test-time caption generation (beam search)
namespace {
int check_beam_state(cgg_handle* h, const cgg_beam_state* st) {
  if (!st || !st->tokens || !st->weights || !st->n_active || !st->parent || !st->next_ids || !st->fin_tokens ||
      !st->fin_len || !st->fin_score || !st->n_fin || !st->max_idx || !st->done || !st->n_done)
    return CGG_ERR_NULL;
  if (st->token_cap < 2) return fail(h, CGG_ERR_BAD_SHAPE, "token_cap must be at least 2");
  return CGG_OK;
}
int check_beams(cgg_handle* h, int batch, int beam_width) {
  if (beam_width < 1 || beam_width > 32) return fail(h, CGG_ERR_BAD_SHAPE, "beam_width must be in 1..32");
  if (batch < 1 || (long)batch * beam_width > 65535) return fail(h, CGG_ERR_BAD_SHAPE, "bad batch");
  return CGG_OK;
}
}  // namespace

extern "C" int cgg_caption_self_attn_step(cgg_handle* h, const float* qkv, float* k_cache, float* v_cache, float* out,
                                          int rows, int heads, int head_dim, int t, int cache_len, float scale,
                                          void* stream) {
  if (!h || !qkv || !k_cache || !v_cache || !out) return CGG_ERR_NULL;
  if (rows < 1 || rows > 0x7fffffff / 2 || heads < 1 || heads > 65535 || head_dim < 1 || cache_len < 1 || t < 0 ||
      t >= cache_len || head_dim + cache_len > 12288)
    return fail(h, CGG_ERR_BAD_SHAPE, "bad shape");
  CU(launch_caption_self_attn(qkv, k_cache, v_cache, out, rows, heads, head_dim, t, cache_len, scale, (cudaStream_t)stream));
  return CGG_OK;
}

extern "C" int cgg_caption_cache_reorder(cgg_handle* h, const float* src, float* dst, const int* parent, int blocks, int batch,
                                         int beam_width, int cache_len, int positions, int dim, void* stream) {
  if (!h || !src || !dst || !parent) return CGG_ERR_NULL;
  ST(check_beams(h, batch, beam_width));
  if (blocks < 1 || 2 * blocks > 65535 || cache_len < 1 || positions < 1 || positions > cache_len || dim < 4 || dim % 4)
    return fail(h, CGG_ERR_BAD_SHAPE, "bad shape");
  CU(launch_caption_cache_reorder(src, dst, parent, blocks, batch * beam_width, beam_width, cache_len, positions, dim,
                                  (cudaStream_t)stream));
  return CGG_OK;
}

extern "C" int cgg_caption_beam_scores(cgg_handle* h, float* logits, int blocks, int batch, int beam_width, int vocab,
                                       int first, const cgg_beam_state* state, float pow_len, float* cand_val, int* cand_col,
                                       void* stream) {
  if (!h || !logits || !cand_val || !cand_col) return CGG_ERR_NULL;
  ST(check_beam_state(h, state));
  ST(check_beams(h, batch, beam_width));
  if (blocks < 1 || vocab < beam_width) return fail(h, CGG_ERR_BAD_SHAPE, "bad shape");
  CU(launch_beam_scores(logits, blocks, batch * beam_width, vocab, beam_width, first != 0, *state, pow_len, cand_val, cand_col,
                        (cudaStream_t)stream));
  return CGG_OK;
}

extern "C" int cgg_caption_beam_select(cgg_handle* h, const float* cand_val, const int* cand_col, int batch, int beam_width,
                                       int first, int length, int max_len, int num_positions, float pow_len, float pow_len1,
                                       int eos, const cgg_beam_state* state, void* stream) {
  if (!h || !cand_val || !cand_col) return CGG_ERR_NULL;
  ST(check_beam_state(h, state));
  ST(check_beams(h, batch, beam_width));
  if (max_len < 1 || num_positions < 1 || max_len > num_positions)
    return fail(h, CGG_ERR_BAD_SHAPE, "max_len must be in 1..num_positions (the position table's rows)");
  if (length < 1 || length + 1 > state->token_cap || beam_width * state->token_cap > BEAM_SELECT_MAX_TOKENS)
    return fail(h, CGG_ERR_BAD_SHAPE, "bad length / token_cap");
  CU(launch_beam_select(cand_val, cand_col, batch, beam_width, first != 0, length, max_len, pow_len, pow_len1, eos, *state,
                        (cudaStream_t)stream));
  return CGG_OK;
}

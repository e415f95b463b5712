// Internal state of the bf16 / tcgen05 side (shared by gemm_tc.cu and attention_tc.cu).
#pragma once
#include "common.cuh"
#include "gemm_tc.h"
#include <cuda.h>
#include <cuda_bf16.h>
#include <string>

namespace cgg {

struct TcState {
  cgg_config cfg;
  std::string err;
  int num_sms = 0;
  int H4 = 0, W4 = 0, lh[3] = {0, 0, 0}, lw[3] = {0, 0, 0}, nl[3] = {0, 0, 0};
  __nv_bfloat16* wkv[3] = {nullptr, nullptr, nullptr};   // (nl*2C, C) bf16
  __nv_bfloat16* rk[3] = {nullptr, nullptr, nullptr};    // (K_l, nl*C) bf16 key-bias table
  const float* bkv[3] = {nullptr, nullptr, nullptr};     // (nl*2C) fp32, owned by the handle
  // N tiling of the mask einsum / bits GEMMs (tc_create): q_pad = B-operand rows per head call;
  // ein_ntile = N tile of tc_einsum_pair_kernel, 0 when the mask einsum runs on tc_einsum_t_kernel
  int q_pad = 0, ein_ntile = 0, bits_ntile = 0, bits_nt = 0;
  int rows_per_batch = 0;
  // bf16 copies of the small-M weights (path_bf16.cu)
  struct LayerW {
    __nv_bfloat16 *wq_c = nullptr, *wo_c = nullptr, *wqkv_s = nullptr, *wo_s = nullptr, *w1 = nullptr, *w2 = nullptr;
    float* rowbias_v = nullptr;   // (Q, C) = -query_embed Wv_self^T : lets q, k, v share the A operand x + query_embed
  } pl[CGG_MAX_LAYERS];
  __nv_bfloat16 *wh = nullptr, *wme1 = nullptr, *wme2 = nullptr;   // heads [v2l | mask_embed.0 | cls | 0], mask_embed.2/.4
  float* bias_h = nullptr;
  int nh_padded = 0;
  bool packed_alloc = false;
  uint8_t* live_buf = nullptr;          // per (image, query tile, key tile) "any key unmasked" flags
  size_t live_bytes = 0;
  void free_all() {
    for (int l = 0; l < 3; ++l) { cudaFree(wkv[l]); cudaFree(rk[l]); wkv[l] = rk[l] = nullptr; }
  }
  void free_packed() {
    for (int i = 0; i < CGG_MAX_LAYERS; ++i) {
      cudaFree(pl[i].wq_c); cudaFree(pl[i].wo_c); cudaFree(pl[i].wqkv_s); cudaFree(pl[i].wo_s); cudaFree(pl[i].w1);
      cudaFree(pl[i].w2); cudaFree(pl[i].rowbias_v);
      pl[i] = LayerW();
    }
    cudaFree(wh); cudaFree(wme1); cudaFree(wme2); cudaFree(bias_h);
    wh = wme1 = wme2 = nullptr; bias_h = nullptr; packed_alloc = false;
  }
};


// carving of the caller-provided tc workspace
inline int pitch8(int k) { return (k + 7) & ~7; }

struct TcWs {
  size_t me_all, fds[3], memp[3], xqb, xb, ob, fb, zb, h1b, h2b, qf, qs, kvs, x1, x2, t1, total;
  void carve(const TcState* t, int B) {
    size_t off = 0;
    auto take = [&](size_t b) { size_t o = off; off += align256(b); return o; };
    const int C = t->cfg.embed_dim;
    const size_t M = (size_t)B * t->cfg.num_queries;
    me_all = take((size_t)B * t->rows_per_batch * 2 * C * 2 + 128 * 1024);   // [hi|lo] rows + 128 slack rows
    // resampled features, one fp16 plane per channel; the plane pitch is the key count rounded up to 8 (TMA 16-byte stride rule)
    for (int l = 0; l < 3; ++l) fds[l] = take((size_t)B * C * pitch8(t->lh[l] * t->lw[l]) * 2);
    // re-pitched copy of a memory level whose key count is not a multiple of 8 (tc_kv_project)
    for (int l = 0; l < 3; ++l) {
      const int K = t->lh[l] * t->lw[l];
      memp[l] = take((K % 8) ? (size_t)B * C * pitch8(K) * 2 : 0);
    }
    xqb = take(M * C * 2); xb = take(M * C * 2); ob = take(M * C * 2);   // IEEE-half rows
    fb = take(M * t->cfg.ffn_dim * 2);
    zb = take(M * 2 * C * 2); h1b = take(M * 2 * C * 2); h2b = take(M * 2 * C * 2);   // hi/lo rows
    qf = take(M * C * 4); qs = take(M * C * 4); kvs = take(M * 2 * C * 4);
    x1 = take(M * C * 4); x2 = take(M * C * 4); t1 = take(4 * M * C * 4);   // t1: up to 4 K-split partial sums
    total = off;
  }
};

int tc_pack_weights(TcState* t, const cgg_weights* w, cudaStream_t s);   // path_bf16.cu
cudaError_t tc_attention_setup();   // attention_tc.cu: kernel attributes, once per handle (per device)

inline int tc_fail(TcState* t, int code, const std::string& m) { t->err = m; return code; }

#define TCU(call)                                                                                  \
  do {                                                                                             \
    cudaError_t e__ = (call);                                                                      \
    if (e__ != cudaSuccess) return tc_fail(t, CGG_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__)); \
  } while (0)

}  // namespace cgg

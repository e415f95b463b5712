// tcgen05 / TMEM / TMA GEMMs of the throughput mode (CGG_BF16), sm_100a.
//
// Three dense contractions have an NCHW feature map as their big operand:
//   K2  mask einsum      D[pixel, (call,q)] = sum_c F[c,pixel]      * me[(call,q), c]
//   K3  attn-mask bits   D[key,   q]        = sum_c Fds_l[c,key]    * me[q, c]     -> sigmoid<0.5 -> ballot
//   K4  K/V projection   D[key,   n]        = sum_c mem_l[c,key]    * Wkv[n, c]    (+ bias)
// The feature map is "MN-major": pixels contiguous, channels strided -- exactly NCHW -- so it is fed to the
// tensor core as-is through TMA with a 128-byte swizzle, no transposition pass.  The other operand (mask
// embeddings / weights) is K-major [rows][256].  K2 and K4 run on CTA pairs (cta_group::2) with the feature tile
// resident in shared memory; K3 keeps the mask embeddings resident instead.  The linear layers (tc_gemm_kernel)
// stream both operands.  Ragged shapes need no code in the kernels: TMA fills the out-of-bounds part of a load
// box with zeros and clips stores at the tensor's extent.
//   warp 0 : TMA producer (one lane)        warp 1 : TMEM alloc + tcgen05.mma issue (one lane)
//   warps 2..17 : epilogue (tcgen05.ld -> registers -> global), 4 warps per TMEM lane quarter
#include "common.cuh"
#include "gemm_tc.h"
#include "kernels.h"
#include <cuda_fp16.h>
#include "tc_ptx.cuh"
#include "tc_state.h"

#include <cuda.h>
#include <cuda_bf16.h>
#include <string>

namespace cgg {

namespace {

constexpr int TC_THREADS = 64 + 16 * 32;   // TMA warp + MMA warp + 16 epilogue warps
constexpr int TC_BM = 128;      // pixels per CTA (UMMA M)
constexpr int TC_BK = 64;       // channels per smem chunk (one 128B swizzle row of bf16 K... see below)
constexpr int A_CHUNK_BYTES = 2 * 64 * 64 * 2;   // 2 pixel groups x 64 ch x 64 px x bf16 = 16 KB

// Linear layers (tc_gemm_kernel): one 128-feature x N_TILE-token tile per CTA
struct TcLinP {
  int N_TILE, KC, stages, tmem_cols;
  int f16;               // 1: operands are IEEE half instead of bf16
  // split precision: rows of both operands are [hi(split_K) | lo(split_K)] bf16 pairs and the CTA walks
  // 3 * split_cpc chunks = hi.hi, hi.lo, lo.hi terms of its K range (split_cpc chunks of 64 per term); 0 = off
  int split_cpc, split_K;
  // up to 3 FEATURE segments (32-aligned starts) of (acc + bias [+ rowbias]) * alpha [+ res] [relu]
  TcSeg seg[3]; int nseg; const float* lin_bias; int n_tokens;
  long kpart_stride;     // with gridDim.z K-parts: part z writes its partial sums at ptr + z*kpart_stride (fp32)
};

// CTA-pair kernels (K2 einsum, K2 transposed einsum, K4): persistent pairs walk work items of two 128-pixel
// tiles of one image; the feature tiles are resident in shared memory, N is walked in NT tiles.
struct TcPairP {
  int NT, N_TILE, stages;
  int b_row0;            // first B row (first_call * q_pad)
  int b_rows_per_batch;  // B row offset per image (0: weights shared by the batch)
  int acc_stride;        // TMEM columns between the two accumulator buffers
  int tmem_cols;         // power of two >= 32
  int ein_split, q_rows; // transposed einsum: 0 = two head calls per step (q_rows = q_pad rows each CTA), 1 = one call per step, CTA r takes rows [r q_rows, (r+1) q_rows)
  int m_pairs, n_batch;  // work items per image (ceil(128-pixel tiles / 2)), images
  int q_pad, n_calls;    // K2: rows per head call in the B operand, head calls of the launch
  const float* bias;     // K4: bias of all NT * N_TILE output columns
};

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}

__device__ __forceinline__ void split_bf16(float x, __nv_bfloat16& hi, __nv_bfloat16& lo) {
  hi = __float2bfloat16_rn(x);
  lo = __float2bfloat16_rn(x - __bfloat162float(hi));
}
__device__ __forceinline__ uint32_t pack2(__nv_bfloat16 a, __nv_bfloat16 b) {
  return (uint32_t)__bfloat16_as_ushort(a) | ((uint32_t)__bfloat16_as_ushort(b) << 16);
}

constexpr int EPI_WARPS = 16;                 // epilogue warps (4 per TMEM lane quarter)
constexpr int EPI_PARTS = EPI_WARPS / 4;

struct EpiCtx {
  int lane, m, batch, part, chunks, wi, col0;
  bool m_ok;
  uint32_t taddr;
};

// K2 epilogue: out[call][image][q][pixel] bf16.  TMEM lanes = pixels, columns = (call, q): the tile
// is staged in shared memory as [column][128 pixels] and leaves through one TMA store of a
// (128 px x N_TILE rows) box; a tile never spans two head calls, and rows q >= Q fall outside the tensor
// and are clipped by the TMA unit.  No per-thread global stores at all.
__device__ __forceinline__ void epi_mask_t(const TcPairP& p, const EpiCtx& c, uint8_t* sStage, const CUtensorMap* tmC,
                                           bool leader_warp, bool last, int m_tile, uint64_t* acc_empty_bar) {
  const bool leader = leader_warp && c.lane == 0;
  // 1. accumulator -> registers (up to 4 chunks of 16 columns per warp, loads in flight together).
  //    This overlaps the TMA engine still reading the previous tile out of the staging buffer.
  static_assert(EPI_PARTS == 4, "four chunk slots per warp below");
  uint32_t r0[16], r1[16], r2[16], r3[16];
  const int ch0 = c.part, ch1 = c.part + 4, ch2 = c.part + 8, ch3 = c.part + 12;
  const bool on0 = ch0 < c.chunks, on1 = ch1 < c.chunks, on2 = ch2 < c.chunks, on3 = ch3 < c.chunks;   // warp-uniform
  if (on0) ptx::tmem_ld16_issue(c.taddr + (uint32_t)(ch0 * 16), r0);
  if (on1) ptx::tmem_ld16_issue(c.taddr + (uint32_t)(ch1 * 16), r1);
  if (on2) ptx::tmem_ld16_issue(c.taddr + (uint32_t)(ch2 * 16), r2);
  if (on3) ptx::tmem_ld16_issue(c.taddr + (uint32_t)(ch3 * 16), r3);
  if (on0) ptx::tmem_ld_wait16(r0);
  if (on1) ptx::tmem_ld_wait16(r1);
  if (on2) ptx::tmem_ld_wait16(r2);
  if (on3) ptx::tmem_ld_wait16(r3);
  // 2. the accumulator buffer is free again: the MMAs of the tile after next may start
  ptx::tc_fence_before();
  __syncwarp();
  if (c.lane == 0) ptx::mbar_arrive_leader(acc_empty_bar);
  // 3. the previous tile's stores must have finished READING the staging buffer
  if (leader) ptx::tma_store_wait_read();
  asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS * 32) : "memory");
  const int row = c.m & (TC_BM - 1);
  auto stage16 = [&](const uint32_t (&r)[16], int ch) {
    __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(sStage) + (long)(ch * 16) * TC_BM + row;
#pragma unroll
    for (int i = 0; i < 16; ++i) dst[i * TC_BM] = __float2bfloat16_rn(__uint_as_float(r[i]));
  };
  if (on0) stage16(r0, ch0);
  if (on1) stage16(r1, ch1);
  if (on2) stage16(r2, ch2);
  if (on3) stage16(r3, ch3);
  ptx::fence_proxy_async_smem();
  asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS * 32) : "memory");
  if (leader) {
    const int call = c.col0 / p.q_pad, q0 = c.col0 - call * p.q_pad;   // first (call, q) row of this tile
    ptx::tma_store_3d(tmC, sStage, m_tile * TC_BM, q0, call * p.n_batch + c.batch);
    ptx::tma_store_commit();
    if (last) ptx::tma_store_wait_read();   // smem must stay valid until the last store has read it
  }
}

// K4 epilogue: out[image][key][n] bf16 = acc + bias[n].  The 128-key x N_TILE tile is staged in shared
// memory as 64-column sub-tiles in the TMA 128-byte-swizzle layout (a thread owns a key row and writes
// 16-byte chunks at chunk ^ (row & 7): conflict-free) and leaves through one TMA store per sub-tile;
// rows past the image's last key are clipped by the TMA unit.  (The positional / level part of the keys
// is not added here at all: the attention kernel adds Q R^T, see attention_tc.cu.)
__device__ __forceinline__ void epi_rowmajor(const EpiCtx& c, uint8_t* sStage, const float* sBias, const CUtensorMap* tmC,
                                             bool leader_warp, bool last, int m_tile, uint64_t* acc_empty_bar) {
  const bool leader = leader_warp && c.lane == 0;
  static_assert(EPI_PARTS == 4, "four chunk slots per warp below");
  // 1. accumulator -> registers (up to 4 chunks of 16 columns per warp, loads in flight together); this overlaps
  //    the TMA engine still reading the previous tile out of the staging buffer
  uint32_t r0[16], r1[16], r2[16], r3[16];
  const int ch0 = c.part, ch1 = c.part + 4, ch2 = c.part + 8, ch3 = c.part + 12;
  const bool on0 = ch0 < c.chunks, on1 = ch1 < c.chunks, on2 = ch2 < c.chunks, on3 = ch3 < c.chunks;   // warp-uniform
  if (on0) ptx::tmem_ld16_issue(c.taddr + (uint32_t)(ch0 * 16), r0);
  if (on1) ptx::tmem_ld16_issue(c.taddr + (uint32_t)(ch1 * 16), r1);
  if (on2) ptx::tmem_ld16_issue(c.taddr + (uint32_t)(ch2 * 16), r2);
  if (on3) ptx::tmem_ld16_issue(c.taddr + (uint32_t)(ch3 * 16), r3);
  if (on0) ptx::tmem_ld_wait16(r0);
  if (on1) ptx::tmem_ld_wait16(r1);
  if (on2) ptx::tmem_ld_wait16(r2);
  if (on3) ptx::tmem_ld_wait16(r3);
  // 2. the accumulator buffer is free again
  ptx::tc_fence_before();
  __syncwarp();
  if (c.lane == 0) ptx::mbar_arrive_leader(acc_empty_bar);
  // 3. the previous tile's stores must have finished READING the staging buffer
  if (leader) ptx::tma_store_wait_read();
  asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS * 32) : "memory");
  const int row = c.m & (TC_BM - 1);
  auto stage16 = [&](const uint32_t (&r)[16], int ch) {
    const float* bf = sBias + c.col0 + ch * 16;       // same address for the whole warp: shared-memory broadcast
    uint4 o[2];
    uint32_t* ow = reinterpret_cast<uint32_t*>(o);
#pragma unroll
    for (int i = 0; i < 8; ++i)
      ow[i] = pack_bf16x2(__uint_as_float(r[2 * i]) + bf[2 * i], __uint_as_float(r[2 * i + 1]) + bf[2 * i + 1]);
    // column chunk (16 B = 8 columns) j of sub-tile `sub`, swizzled with the row
    const int sub = ch >> 2, j = (ch & 3) * 2;
    uint8_t* base = sStage + sub * (TC_BM * 128) + row * 128;
    *reinterpret_cast<uint4*>(base + ((j ^ (row & 7)) << 4)) = o[0];
    *reinterpret_cast<uint4*>(base + (((j + 1) ^ (row & 7)) << 4)) = o[1];
  };
  if (on0) stage16(r0, ch0);
  if (on1) stage16(r1, ch1);
  if (on2) stage16(r2, ch2);
  if (on3) stage16(r3, ch3);
  ptx::fence_proxy_async_smem();
  asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS * 32) : "memory");
  if (leader) {
    const int subs = c.chunks >> 2;
    for (int sub = 0; sub < subs; ++sub)
      ptx::tma_store_3d(tmC, sStage + sub * (TC_BM * 128), c.col0 + sub * 64, m_tile * TC_BM, c.batch);
    ptx::tma_store_commit();
    if (last) ptx::tma_store_wait_read();
  }
}

// K3 epilogue: threshold (common.cuh) + ballot = 32 consecutive key bits of one query per warp instruction.
__device__ __forceinline__ void epi_bits(int Q, int W32, uint32_t* bitmap, const EpiCtx& c) {
  uint32_t* brow = bitmap + (long)c.batch * Q * W32 + c.wi;
  const bool w_ok = c.wi < W32;
  for (int ch = c.part; ch < c.chunks; ch += EPI_PARTS) {
    float v[16];
    ptx::tmem_ld16(c.taddr + (uint32_t)(ch * 16), v);
    const int q0 = c.col0 + ch * 16;
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      const uint32_t word = __ballot_sync(0xffffffffu, c.m_ok && v[i] <= MASKED_LOGIT_MAX);
      if (c.lane == 0 && w_ok && q0 + i < Q) brow[(long)(q0 + i) * W32] = word;
    }
  }
}

// Swap-AB linear layers: TMEM lanes = output FEATURES, columns = tokens; for one token a warp holds
// 32 consecutive features, so every global access is one coalesced line.  The thread's segment is
// resolved once (registers), and the inner loop is specialised on the output kind / extra operands.
struct LinCtx {
  bool on = false;
  int f = 0, mode = 0, rb_mod = 1, split_off = 0;
  long ld = 0, rb_ld = 0, res_ld = 0;
  float bias = 0.f, alpha = 1.f, floor = -INFINITY;
  void* ptr = nullptr;
  const float* rowbias = nullptr;
  const float* res = nullptr;
  __device__ __forceinline__ void init(const TcLinP& p, int m) {
#pragma unroll
    for (int sgi = 0; sgi < 3; ++sgi) {
      if (sgi < p.nseg && m >= p.seg[sgi].col0 && m < p.seg[sgi].col0 + p.seg[sgi].ncols) {
        on = true;
        f = m - p.seg[sgi].col0;
        mode = p.seg[sgi].is_bf16 == 3 ? 3 : (p.seg[sgi].is_bf16 ? (p.seg[sgi].split ? 2 : 1) : 0);   // 3 = IEEE half
        floor = p.seg[sgi].relu ? 0.f : -INFINITY;
        ptr = p.seg[sgi].ptr; ld = p.seg[sgi].ld; alpha = p.seg[sgi].alpha;
        rowbias = p.seg[sgi].rowbias; rb_mod = p.seg[sgi].rb_mod; rb_ld = p.seg[sgi].rb_ld;
        res = p.seg[sgi].res; res_ld = p.seg[sgi].res_ld; split_off = p.seg[sgi].ncols;
      }
    }
    if (on && p.lin_bias) bias = __ldg(p.lin_bias + m);
    if (blockIdx.z > 0) {   // K-split partial: bias / residual belong to part 0 only
      bias = 0.f; res = nullptr; rowbias = nullptr;
      ptr = static_cast<float*>(ptr) + (long)blockIdx.z * p.kpart_stride;
    }
  }
};

// Per-token operands of the epilogue (row bias or residual) do not depend on the accumulator: they are
// fetched while the MMAs still run (up to 2 chunks of 16 tokens per warp: N_TILE <= 128).
struct LinPre {
  float a[16], b[16];
};
__device__ __forceinline__ void lin_prefetch(const TcLinP& p, const EpiCtx& c, const LinCtx& L, LinPre& pre) {
  const int tok_base = c.batch * p.N_TILE;
#pragma unroll
  for (int i = 0; i < 16; ++i) pre.a[i] = pre.b[i] = 0.f;
  if (!L.on || (L.rowbias == nullptr && L.res == nullptr)) return;
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    const int ch = c.part + j * EPI_PARTS;
    if (ch >= c.chunks) break;
    const int tok0 = tok_base + ch * 16;
    const int nvalid = min(16, p.n_tokens - tok0);
    float* dst = j ? pre.b : pre.a;
    if (L.rowbias) {
      int tq = tok0 % L.rb_mod;
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        if (i < nvalid) dst[i] = __ldg(L.rowbias + (long)tq * L.rb_ld + L.f);
        if (++tq == L.rb_mod) tq = 0;
      }
    } else {
      const float* rp = L.res + (long)tok0 * L.res_ld + L.f;
#pragma unroll
      for (int i = 0; i < 16; ++i)
        if (i < nvalid) dst[i] = __ldg(rp + (long)i * L.res_ld);
    }
  }
}

template <int MODE, bool HAS_RB, bool HAS_RES>
__device__ __forceinline__ void epi_linear_t(const TcLinP& p, const EpiCtx& c, const LinCtx& L, const LinPre& pre) {
  const int n_tokens = p.n_tokens;
  const int tok_base = c.batch * p.N_TILE;
  int j = 0;
  for (int ch = c.part; ch < c.chunks; ch += EPI_PARTS, ++j) {
    const int tok0 = tok_base + ch * 16;
    const int nvalid = L.on ? min(16, n_tokens - tok0) : 0;      // <= 0: nothing to store
    float ex[16];                                                 // the prefetched row bias or residual
#pragma unroll
    for (int i = 0; i < 16; ++i) ex[i] = j ? pre.b[i] : pre.a[i];
    float v[16];
    ptx::tmem_ld16(c.taddr + (uint32_t)(ch * 16), v);
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      float x = v[i] + L.bias;
      if (HAS_RB) x += ex[i];
      x *= L.alpha;
      if (HAS_RES) x += ex[i];
      x = fmaxf(x, L.floor);
      if (i < nvalid) {
        const long off = (long)(tok0 + i) * L.ld + L.f;
        if (MODE == 0) {
          static_cast<float*>(L.ptr)[off] = x;
        } else if (MODE == 1) {
          static_cast<__nv_bfloat16*>(L.ptr)[off] = __float2bfloat16_rn(x);
        } else if (MODE == 3) {
          static_cast<__half*>(L.ptr)[off] = __float2half_rn(x);
        } else {
          __nv_bfloat16 hi, lo;
          split_bf16(x, hi, lo);
          static_cast<__nv_bfloat16*>(L.ptr)[off] = hi;
          static_cast<__nv_bfloat16*>(L.ptr)[off + L.split_off] = lo;
        }
      }
    }
  }
}

__device__ __forceinline__ void epi_linear_dispatch(const TcLinP& p, const EpiCtx& c, const LinCtx& L, const LinPre& pre) {
  // warp-uniform: a warp's 32 features belong to one segment (32-aligned segment starts)
  const bool rb = L.rowbias != nullptr, rs = L.res != nullptr;
  if (L.mode == 0) {
    if (rb) epi_linear_t<0, true, false>(p, c, L, pre);
    else if (rs) epi_linear_t<0, false, true>(p, c, L, pre);
    else epi_linear_t<0, false, false>(p, c, L, pre);
  } else if (L.mode == 1) {
    if (rb) epi_linear_t<1, true, false>(p, c, L, pre);
    else epi_linear_t<1, false, false>(p, c, L, pre);
  } else if (L.mode == 3) {
    epi_linear_t<3, false, false>(p, c, L, pre);
  } else {
    epi_linear_t<2, false, false>(p, c, L, pre);
  }
}

// ------------------------------------------------------------------- linear layers
// Swap-AB: A = weights [features][K] (128 features per CTA on the TMEM lanes, blockIdx.x), B = activations
// [tokens][K] (one tile of N_TILE <= 128 tokens, blockIdx.y), K range of part blockIdx.z.  Both operands are
// K-major and stream together through a ring of TMA stages; one accumulator tile per CTA.
__global__ void __launch_bounds__(TC_THREADS, 1)
tc_gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               const __grid_constant__ TcLinP p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int stage_bytes = A_CHUNK_BYTES + p.N_TILE * 128;   // ring stage = [weight chunk] [activation chunk]
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + p.stages * stage_bytes);
  uint64_t* full = bars;
  uint64_t* empty = full + p.stages;
  uint64_t* acc_full = empty + p.stages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_full + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // K coordinates of chunk kc in the weight (A) and activation (B) tensor maps
  auto kcoords = [&](int kc, int& ka, int& kb) {
    if (p.split_cpc > 0) {
      const int term = kc / p.split_cpc, j = kc - term * p.split_cpc;
      const int k0 = ((int)blockIdx.z * p.split_cpc + j) * TC_BK;
      ka = (term == 2 ? p.split_K : 0) + k0;      // weights:     hi, hi, lo
      kb = (term == 1 ? p.split_K : 0) + k0;      // activations: hi, lo, hi
    } else {
      ka = kb = ((int)blockIdx.z * p.KC + kc) * TC_BK;
    }
  };

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmA);
    ptx::prefetch_tmap(&tmB);
    for (int i = 0; i < p.stages; ++i) { ptx::mbar_init(&full[i], 1); ptx::mbar_init(&empty[i], 1); }
    ptx::mbar_init(acc_full, 1);
    ptx::fence_mbar_init();
  }
  if (warp == 1) {
    ptx::tmem_alloc(tmem_slot, (uint32_t)p.tmem_cols);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // everything above (barriers, TMEM, descriptor prefetch) overlapped the previous kernel's tail
  ptx::grid_dep_launch();
  // The A operand is a WEIGHT matrix, independent of the previous kernel: its first ring-full of chunks is
  // requested before waiting for the previous grid (the activations, operand B, follow after the wait).
  const int n_pre = p.KC < p.stages ? p.KC : p.stages;
  if (warp == 0 && lane == 0)
    for (int kc = 0; kc < n_pre; ++kc) {
      int ka, kb;
      kcoords(kc, ka, kb);
      ptx::mbar_expect_tx(&full[kc], (uint32_t)stage_bytes);
      ptx::tma_load_2d(smem + kc * stage_bytes, &tmA, &full[kc], ka, (int)blockIdx.x * TC_BM);
    }
  ptx::grid_dep_wait();

  if (warp == 0) {
    if (lane == 0) {
      // ---------------- TMA producer: a chunk is (64 k x 128 features) of A and (64 k x N_TILE tokens) of B
      for (int kc = 0; kc < p.KC; ++kc) {
        const int s = kc % p.stages;
        uint8_t* stage = smem + s * stage_bytes;
        int ka, kb;
        kcoords(kc, ka, kb);
        if (kc >= n_pre) {
          ptx::mbar_wait(&empty[s], ((uint32_t)(kc / p.stages) & 1u) ^ 1u);
          ptx::mbar_expect_tx(&full[s], (uint32_t)stage_bytes);
          ptx::tma_load_2d(stage, &tmA, &full[s], ka, (int)blockIdx.x * TC_BM);
        }
        ptx::tma_load_2d(stage + A_CHUNK_BYTES, &tmB, &full[s], kb, (int)blockIdx.y * p.N_TILE);
      }
    }
  } else if (warp == 1) {
    // ---------------- MMA issuer: the whole warp walks the loop (uniform control flow keeps the descriptors in
    // uniform registers), one elected lane issues.  Descriptors = base + constant increments of the 14-bit
    // address field (16-byte units); K-major SW128: 32 B along K per MMA, SBO 1 KB.
    const uint32_t idesc = ptx::umma_idesc_bf16(TC_BM, p.N_TILE, /*A MN-major*/ false, /*B K-major*/ false, p.f16 != 0);
    const uint64_t ad0 = ptx::umma_desc(ptx::smem_u32(smem), 16, 1024, ptx::UMMA_SW128);
    const uint64_t bd0 = ptx::umma_desc(ptx::smem_u32(smem + A_CHUNK_BYTES), 16, 1024, ptx::UMMA_SW128);
    const uint32_t stage16 = (uint32_t)stage_bytes >> 4;
    for (int kc = 0; kc < p.KC; ++kc) {
      const int s = kc % p.stages;
      ptx::mbar_wait(&full[s], (uint32_t)(kc / p.stages) & 1u);
      ptx::tc_fence_after();
      if (ptx::elect_one()) {
        const uint64_t off = (uint64_t)((uint32_t)s * stage16);
#pragma unroll
        for (int k = 0; k < TC_BK / 16; ++k)
          ptx::mma_bf16_ss(tmem_base, ad0 + off + (uint64_t)(k * 2), bd0 + off + (uint64_t)(k * 2), idesc,
                           (kc | k) != 0 ? 1u : 0u);
        ptx::mma_commit(&empty[s]);                        // frees the stage when these MMAs retire
        if (kc == p.KC - 1) ptx::mma_commit(acc_full);     // accumulator tile complete
      }
      __syncwarp();
    }
  } else {
    // ---------------- epilogue: EPI_WARPS warps, EPI_WARPS/4 per TMEM lane quarter; each warp takes
    // every (EPI_WARPS/4)-th 16-column chunk
    const int quarter = warp & 3;
    const int m = (int)blockIdx.x * TC_BM + quarter * 32 + lane;    // TMEM lane -> output feature
    EpiCtx ctx;
    ctx.lane = lane; ctx.m = m; ctx.m_ok = true; ctx.batch = blockIdx.y; ctx.part = (warp - 2) >> 2;
    ctx.chunks = p.N_TILE / 16; ctx.wi = 0; ctx.col0 = 0;
    ctx.taddr = tmem_base + ((uint32_t)(quarter * 32) << 16);
    LinCtx lin;
    LinPre pre;
    lin.init(p, m);
    lin_prefetch(p, ctx, lin, pre);
    ptx::mbar_wait(acc_full, 0);
    ptx::tc_fence_after();
    epi_linear_dispatch(p, ctx, lin, pre);
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    ptx::tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
  }
}

// ------------------------------------------------------------------- K2, CTA-pair variant
// The mask einsum with cta_group::2 MMAs (M = 256: two 128-pixel tiles, one per CTA of the pair; N =
// N_TILE).  Each CTA streams only HALF of every B chunk (N_TILE/2 mask-embedding rows), which makes room
// for TWO whole N tiles of B in shared memory (2 x 4 chunks).  That matters because the single MMA-issuing
// thread, not the tensor pipe, paces a single-CTA kernel: every tcgen05.commit costs it ~300-400
// cycles, and a 4-stage ring needs one per chunk.  Here ONE commit per N tile (acc_full) tells the
// epilogue "accumulator ready" and the producer "these four B slots are free".  An N tile never spans two
// head calls.  Persistent pairs: A tile resident and refilled chunk by chunk under the last N tile,
// double-buffered accumulators, staged TMA-store epilogue (each CTA stores its own 128 pixels).
// Work items of all three pair kernels are ceil(m_tiles / 2) tile pairs per image: with an odd tile count the
// rank-1 tile of the last pair lies wholly past the end, TMA loads it as zeros and clips its stores.
__global__ void __launch_bounds__(TC_THREADS, 1)
tc_einsum_pair_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                      const __grid_constant__ CUtensorMap tmC, const __grid_constant__ TcPairP p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  constexpr int KC = 4;
  const int half_n = p.N_TILE / 2;
  const int b_chunk_bytes = half_n * 128;
  uint8_t* sA = smem;
  uint8_t* sB = sA + KC * A_CHUNK_BYTES;                  // [2 N-tile slots][KC chunks]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sB + 2 * KC * b_chunk_bytes);
  uint64_t* a_full = bars;
  uint64_t* a_empty = bars + 4;
  uint64_t* b_full = bars + 8;                            // [2][KC]
  uint64_t* acc_full = b_full + 2 * KC;
  uint64_t* acc_empty = acc_full + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);
  uint8_t* sStage = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(tmem_slot + 4) + 1023) & ~(uintptr_t)1023);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = ptx::cluster_ctarank();          // 0 = leader
  const int pair = blockIdx.x >> 1, n_pairs = gridDim.x >> 1;
  const int mt2 = p.m_pairs;                              // pixel-tile pairs per image
  const int n_work = mt2 * p.n_batch;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmA);
    ptx::prefetch_tmap(&tmB);
    for (int i = 0; i < 4; ++i) { ptx::mbar_init(&a_full[i], 1); ptx::mbar_init(&a_empty[i], 1); }
    for (int i = 0; i < 2 * KC; ++i) ptx::mbar_init(&b_full[i], 1);
    for (int i = 0; i < 2; ++i) { ptx::mbar_init(&acc_full[i], 1); ptx::mbar_init(&acc_empty[i], 2 * EPI_WARPS); }
    ptx::fence_mbar_init();
  }
  if (warp == 1) {
    ptx::tmem_alloc_2sm(tmem_slot, (uint32_t)p.tmem_cols);
    ptx::tmem_relinquish_2sm();
  }
  __syncwarp();
  ptx::tc_fence_before();
  ptx::cluster_sync_all();        // the peer's barriers exist before anything arrives on them
  ptx::tc_fence_after();
  __syncthreads();                // (implied by the cluster barrier; spelled out for compute-sanitizer racecheck, which does not track it)
  const uint32_t tmem_base = *tmem_slot;
  ptx::grid_dep_launch();
  ptx::grid_dep_wait();

  if (warp == 0) {
    if (lane == 0) {
      // ---------------- TMA producer (both CTAs: own pixel tile, own half of B; tx bytes land on the leader)
      int g = 0, tl = 0;
      for (int w = pair; w < n_work; w += n_pairs, ++tl) {
        const int batch = w / mt2, m_tile = (w - batch * mt2) * 2 + (int)rank;
        for (int t = 0; t < p.NT; ++t, ++g) {
          const int slot = g & 1;
          // the MMAs of N tile g-2 (same slot) have completed: its accumulator commit doubles as "B slot free"
          if (g >= 2) ptx::mbar_wait(&acc_full[slot], (uint32_t)((g - 2) >> 1) & 1u);
          for (int kc = 0; kc < KC; ++kc) {
            if (t == 0) {
              if (tl > 0) ptx::mbar_wait(&a_empty[kc], (uint32_t)(tl & 1) ^ 1u);
              if (rank == 0) ptx::mbar_expect_tx(&a_full[kc], 2u * A_CHUNK_BYTES);
              for (int h = 0; h < 2; ++h)
                ptx::tma_load_3d_2sm(sA + kc * A_CHUNK_BYTES + h * (A_CHUNK_BYTES / 2), &tmA, &a_full[kc],
                                     m_tile * TC_BM + h * 64, kc * TC_BK, batch);
            }
            uint64_t* bar = &b_full[slot * KC + kc];
            if (rank == 0) ptx::mbar_expect_tx(bar, 2u * (uint32_t)b_chunk_bytes);
            ptx::tma_load_2d_2sm(sB + (slot * KC + kc) * b_chunk_bytes, &tmB, bar, kc * TC_BK,
                                 batch * p.b_rows_per_batch + p.b_row0 + t * p.N_TILE + (int)rank * half_n);
          }
        }
      }
    }
  } else if (warp == 1) {
    if (rank == 0) {
      // ---------------- MMA issuer: the leader CTA's warp walks the loop, one elected lane drives both SMs
      const uint32_t idesc = ptx::umma_idesc_bf16(2 * TC_BM, p.N_TILE, /*A MN-major*/ true, /*B K-major*/ false);
      // descriptors differ by a constant in the 14-bit address field (units of 16 bytes)
      uint64_t adesc0[KC], bdesc0[2 * KC];
#pragma unroll
      for (int kc = 0; kc < KC; ++kc)
        adesc0[kc] = ptx::umma_desc(ptx::smem_u32(sA + kc * A_CHUNK_BYTES), A_CHUNK_BYTES / 2, 1024, ptx::UMMA_SW128);
#pragma unroll
      for (int i = 0; i < 2 * KC; ++i) bdesc0[i] = ptx::umma_desc(ptx::smem_u32(sB + i * b_chunk_bytes), 16, 1024, ptx::UMMA_SW128);
      int g = 0, tl = 0;
      for (int w = pair; w < n_work; w += n_pairs, ++tl)
        for (int t = 0; t < p.NT; ++t, ++g) {
          const int buf = g & 1;
          const uint32_t use = (uint32_t)(g >> 1);
          ptx::mbar_wait(&acc_empty[buf], (use & 1u) ^ 1u);
          ptx::tc_fence_after();
          const uint32_t d_tmem = tmem_base + (uint32_t)(buf * p.acc_stride);
#pragma unroll
          for (int kc = 0; kc < KC; ++kc) {
            if (t == 0) ptx::mbar_wait(&a_full[kc], (uint32_t)(tl & 1));
            ptx::mbar_wait(&b_full[buf * KC + kc], use & 1u);
            ptx::tc_fence_after();
            if (ptx::elect_one()) {
              const uint64_t ad = adesc0[kc], bd = buf ? bdesc0[KC + kc] : bdesc0[kc];
#pragma unroll
              for (int k = 0; k < TC_BK / 16; ++k)
                ptx::mma_bf16_ss_2sm(d_tmem, ad + (uint64_t)(k * (2048 >> 4)), bd + (uint64_t)(k * (32 >> 4)), idesc,
                                     (kc | k) != 0 ? 1u : 0u);
              if (t == p.NT - 1) ptx::mma_commit_2sm(&a_empty[kc]);   // A chunk kc may be refilled for the next work item
              if (kc == KC - 1) ptx::mma_commit_2sm(&acc_full[buf]);  // accumulator ready (epilogue) + B slot free (producer), both CTAs
            }
            __syncwarp();
          }
        }
    }
  } else {
    // ---------------- epilogue (both CTAs, own 128 accumulator lanes)
    const int quarter = warp & 3;
    const int part = (warp - 2) >> 2;
    int g = 0;
    for (int w = pair; w < n_work; w += n_pairs) {
      const int batch = w / mt2, m_tile = (w - batch * mt2) * 2 + (int)rank;
      const bool last_work = w + n_pairs >= n_work;
      const int m = m_tile * TC_BM + quarter * 32 + lane;
      EpiCtx ctx;
      ctx.lane = lane; ctx.m = m; ctx.m_ok = true; ctx.batch = batch; ctx.part = part;
      ctx.chunks = p.N_TILE / 16; ctx.wi = 0;
      for (int t = 0; t < p.NT; ++t, ++g) {
        const int buf = g & 1;
        const uint32_t use = (uint32_t)(g >> 1);
        ptx::mbar_wait(&acc_full[buf], use & 1u);
        ptx::tc_fence_after();
        ctx.taddr = tmem_base + (uint32_t)(buf * p.acc_stride) + ((uint32_t)(quarter * 32) << 16);
        ctx.col0 = t * p.N_TILE;
        epi_mask_t(p, ctx, sStage, &tmC, warp == 2, last_work && t == p.NT - 1, m_tile, &acc_empty[buf]);
      }
    }
  }
  __syncwarp();                   // the single-lane roles rejoin their warps (cluster barrier is .aligned)
  ptx::tc_fence_before();
  ptx::cluster_sync_all();        // both CTAs are done with both TMEMs and with each other's barriers
  if (warp == 1) ptx::tmem_dealloc_2sm(tmem_base, (uint32_t)p.tmem_cols);
}

// ------------------------------------------------------------------- K4, CTA-pair variant
// K/V projection with cta_group::2 MMAs: M = 256 = two 128-token tiles (one per CTA, resident, refilled chunk by
// chunk under the last N tile), N = N_TILE weight rows of which each CTA streams HALF per chunk.  A single-CTA
// kernel is bound by that stream (128 KB of weights per N tile through a two-stage ring); halving it per CTA and
// doubling the ring depth moves the kernel to its HBM-write / epilogue bound.  Epilogue = epi_rowmajor.
__global__ void __launch_bounds__(TC_THREADS, 1)
tc_kv_pair_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                  const __grid_constant__ CUtensorMap tmC, const __grid_constant__ TcPairP p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  constexpr int KC = 4;
  const int half_n = p.N_TILE / 2;
  const int b_stage_bytes = half_n * 128;
  uint8_t* sA = smem;
  uint8_t* sB = sA + KC * A_CHUNK_BYTES;
  uint8_t* sStage = sB + p.stages * b_stage_bytes;                       // N_TILE x 128 tokens bf16 (1024-aligned)
  float* sBias = reinterpret_cast<float*>(sStage + (size_t)p.N_TILE * TC_BM * 2);
  uint64_t* bars = reinterpret_cast<uint64_t*>(sBias + p.NT * p.N_TILE);
  uint64_t* a_full = bars;
  uint64_t* a_empty = bars + 4;
  uint64_t* b_full = bars + 8;
  uint64_t* b_empty = b_full + p.stages;
  uint64_t* acc_full = b_empty + p.stages;
  uint64_t* acc_empty = acc_full + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = ptx::cluster_ctarank();
  const int pair = blockIdx.x >> 1, n_pairs = gridDim.x >> 1;
  const int mt2 = p.m_pairs;
  const int n_work = mt2 * p.n_batch;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmA);
    ptx::prefetch_tmap(&tmB);
    for (int i = 0; i < 4; ++i) { ptx::mbar_init(&a_full[i], 1); ptx::mbar_init(&a_empty[i], 1); }
    for (int i = 0; i < p.stages; ++i) { ptx::mbar_init(&b_full[i], 1); ptx::mbar_init(&b_empty[i], 1); }
    for (int i = 0; i < 2; ++i) { ptx::mbar_init(&acc_full[i], 1); ptx::mbar_init(&acc_empty[i], 2 * EPI_WARPS); }
    ptx::fence_mbar_init();
  }
  if (warp == 1) {
    ptx::tmem_alloc_2sm(tmem_slot, (uint32_t)p.tmem_cols);
    ptx::tmem_relinquish_2sm();
  }
  __syncwarp();
  ptx::tc_fence_before();
  ptx::cluster_sync_all();
  ptx::tc_fence_after();
  __syncthreads();                // (implied by the cluster barrier; spelled out for compute-sanitizer racecheck, which does not track it)
  const uint32_t tmem_base = *tmem_slot;
  ptx::grid_dep_launch();
  ptx::grid_dep_wait();

  if (warp == 0) {
    if (lane == 0) {
      int it = 0, tl = 0;
      for (int w = pair; w < n_work; w += n_pairs, ++tl) {
        const int batch = w / mt2, m_tile = (w - batch * mt2) * 2 + (int)rank;
        for (int t = 0; t < p.NT; ++t)
          for (int kc = 0; kc < KC; ++kc, ++it) {
            if (t == 0) {
              if (tl > 0) ptx::mbar_wait(&a_empty[kc], (uint32_t)(tl & 1) ^ 1u);
              if (rank == 0) ptx::mbar_expect_tx(&a_full[kc], 2u * A_CHUNK_BYTES);
              for (int h = 0; h < 2; ++h)
                ptx::tma_load_3d_2sm(sA + kc * A_CHUNK_BYTES + h * (A_CHUNK_BYTES / 2), &tmA, &a_full[kc],
                                     m_tile * TC_BM + h * 64, kc * TC_BK, batch);
            }
            const int s = it % p.stages;
            ptx::mbar_wait(&b_empty[s], ((uint32_t)(it / p.stages) & 1u) ^ 1u);
            if (rank == 0) ptx::mbar_expect_tx(&b_full[s], 2u * (uint32_t)b_stage_bytes);
            ptx::tma_load_2d_2sm(sB + s * b_stage_bytes, &tmB, &b_full[s], kc * TC_BK, t * p.N_TILE + (int)rank * half_n);
          }
      }
    }
  } else if (warp == 1) {
    if (rank == 0) {
      const uint32_t idesc = ptx::umma_idesc_bf16(2 * TC_BM, p.N_TILE, /*A MN-major*/ true, /*B K-major*/ false);
      const uint64_t ad0 = ptx::umma_desc(ptx::smem_u32(sA), A_CHUNK_BYTES / 2, 1024, ptx::UMMA_SW128);
      const uint64_t bd0 = ptx::umma_desc(ptx::smem_u32(sB), 16, 1024, ptx::UMMA_SW128);
      const uint32_t stage16 = (uint32_t)b_stage_bytes >> 4;
      int it = 0, g = 0, tl = 0;
      for (int w = pair; w < n_work; w += n_pairs, ++tl)
        for (int t = 0; t < p.NT; ++t, ++g) {
          const int buf = g & 1;
          ptx::mbar_wait(&acc_empty[buf], (((uint32_t)(g >> 1)) & 1u) ^ 1u);
          ptx::tc_fence_after();
          const uint32_t d_tmem = tmem_base + (uint32_t)(buf * p.acc_stride);
          for (int kc = 0; kc < KC; ++kc, ++it) {
            const int s = it % p.stages;
            if (t == 0) ptx::mbar_wait(&a_full[kc], (uint32_t)(tl & 1));
            ptx::mbar_wait(&b_full[s], (uint32_t)(it / p.stages) & 1u);
            ptx::tc_fence_after();
            if (ptx::elect_one()) {
              const uint64_t ad = ad0 + (uint64_t)(kc * (A_CHUNK_BYTES >> 4));
              const uint64_t bd = bd0 + (uint64_t)((uint32_t)s * stage16);
#pragma unroll
              for (int k = 0; k < TC_BK / 16; ++k)
                ptx::mma_bf16_ss_2sm(d_tmem, ad + (uint64_t)(k * (2048 >> 4)), bd + (uint64_t)(k * 2), idesc, (kc | k) != 0 ? 1u : 0u);
              ptx::mma_commit_2sm(&b_empty[s]);
              if (t == p.NT - 1) ptx::mma_commit_2sm(&a_empty[kc]);
              if (kc == KC - 1) ptx::mma_commit_2sm(&acc_full[buf]);
            }
            __syncwarp();
          }
        }
    }
  } else {
    const int quarter = warp & 3;
    const int part = (warp - 2) >> 2;
    for (int i = threadIdx.x - 64; i < p.NT * p.N_TILE; i += EPI_WARPS * 32) sBias[i] = __ldg(p.bias + i);
    asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS * 32) : "memory");
    int g = 0;
    for (int w = pair; w < n_work; w += n_pairs) {
      const int batch = w / mt2, m_tile = (w - batch * mt2) * 2 + (int)rank;
      const bool last_work = w + n_pairs >= n_work;
      EpiCtx ctx;
      ctx.lane = lane; ctx.m = m_tile * TC_BM + quarter * 32 + lane; ctx.m_ok = true; ctx.batch = batch;
      ctx.part = part; ctx.chunks = p.N_TILE / 16; ctx.wi = 0;
      for (int t = 0; t < p.NT; ++t, ++g) {
        const int buf = g & 1;
        ptx::mbar_wait(&acc_full[buf], ((uint32_t)(g >> 1)) & 1u);
        ptx::tc_fence_after();
        ctx.taddr = tmem_base + (uint32_t)(buf * p.acc_stride) + ((uint32_t)(quarter * 32) << 16);
        ctx.col0 = t * p.N_TILE;
        epi_rowmajor(ctx, sStage, sBias, &tmC, warp == 2, last_work && t == p.NT - 1, m_tile, &acc_empty[buf]);
      }
    }
  }
  __syncwarp();
  ptx::tc_fence_before();
  ptx::cluster_sync_all();
  if (warp == 1) ptx::tmem_dealloc_2sm(tmem_base, (uint32_t)p.tmem_cols);
}

// ------------------------------------------------------------------- K2, transposed CTA-pair variant
// D^T = E . F^T: the TMEM lanes are the QUERIES of a head call, the columns are PIXELS.  A thread of the
// epilogue then holds 16 consecutive pixels of one (call, query) row -- exactly the output's contiguous
// dimension -- and stages them with two 16-byte shared-memory stores (the pixel-on-lane form needs sixteen
// 2-byte stores for the same data); the staging tiles are 128-byte-swizzled (64 px x q_pad rows), so a warp's
// 32 rows hit 32 distinct bank groups, and leave through TMA stores.
//   cta_group::2, M = 256 = two head calls (CTA r of the pair provides the 128-row block of call 2t+r),
//   N = 256 pixels (CTA r holds the features of pixels [128 r, 128 r + 128) of the tile, resident, MN-major),
//   K = 256 channels.  Per step t each CTA streams ONE call's mask embeddings (q_pad rows per chunk; the MMA
//   reads 128 rows, the extra lanes are never stored), two steps of chunks fit the ring, and ONE commit per step
//   signals "accumulator ready" + "ring slots free".  Both accumulators (2 x 256 columns) fill the TMEM.
__global__ void __launch_bounds__(TC_THREADS, 1)
tc_einsum_t_kernel(const __grid_constant__ CUtensorMap tmF, const __grid_constant__ CUtensorMap tmE,
                   const __grid_constant__ CUtensorMap tmC, const __grid_constant__ TcPairP p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  constexpr int KC = 4;
  const int e_chunk_bytes = p.q_rows * 128;               // this CTA's query rows x 64 k
  const int sub_bytes = p.q_rows * 128;                   // staging sub-tile: query rows x 64 px
  uint8_t* sF = smem;                                     // features of this CTA's 128 pixels: 4 chunks of 16 KB
  uint8_t* sE = sF + KC * A_CHUNK_BYTES;                  // [2 step slots][KC chunks]
  uint8_t* sStage = sE + 2 * KC * e_chunk_bytes;          // 4 sub-tiles (q_pad * 128 is a multiple of 1024)
  uint64_t* bars = reinterpret_cast<uint64_t*>(sStage + 4 * sub_bytes);
  uint64_t* f_full = bars;
  uint64_t* f_empty = bars + 4;
  uint64_t* e_full = bars + 8;                            // [2][KC]
  uint64_t* acc_full = e_full + 2 * KC;
  uint64_t* acc_empty = acc_full + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = ptx::cluster_ctarank();          // 0 = leader
  const int pair = blockIdx.x >> 1, n_pairs = gridDim.x >> 1;
  const int mt2 = p.m_pairs;                              // 256-pixel tiles per image
  const int n_work = mt2 * p.n_batch;
  const int NS = p.ein_split ? p.n_calls : (p.n_calls + 1) >> 1;   // steps: two head calls each (or one, split over the pair)
  const int q0 = p.ein_split ? (int)rank * p.q_rows : 0;  // first query row of this CTA within its call

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmF);
    ptx::prefetch_tmap(&tmE);
    for (int i = 0; i < 4; ++i) { ptx::mbar_init(&f_full[i], 1); ptx::mbar_init(&f_empty[i], 1); }
    for (int i = 0; i < 2 * KC; ++i) ptx::mbar_init(&e_full[i], 1);
    for (int i = 0; i < 2; ++i) { ptx::mbar_init(&acc_full[i], 1); ptx::mbar_init(&acc_empty[i], 2 * EPI_WARPS); }
    ptx::fence_mbar_init();
  }
  if (warp == 1) {
    ptx::tmem_alloc_2sm(tmem_slot, 512u);
    ptx::tmem_relinquish_2sm();
  }
  __syncwarp();
  ptx::tc_fence_before();
  ptx::cluster_sync_all();
  ptx::tc_fence_after();
  __syncthreads();                // (implied by the cluster barrier; spelled out for compute-sanitizer racecheck, which does not track it)
  const uint32_t tmem_base = *tmem_slot;
  ptx::grid_dep_launch();
  ptx::grid_dep_wait();

  if (warp == 0) {
    if (lane == 0) {
      // ---------------- TMA producer (both CTAs: own 128 pixels, own head call; tx bytes land on the leader)
      int g = 0, tl = 0;
      for (int w = pair; w < n_work; w += n_pairs, ++tl) {
        const int batch = w / mt2, px0 = ((w - batch * mt2) * 2 + (int)rank) * TC_BM;
        for (int t = 0; t < NS; ++t, ++g) {
          const int slot = g & 1;
          if (g >= 2) ptx::mbar_wait(&acc_full[slot], (uint32_t)((g - 2) >> 1) & 1u);   // MMAs of step g-2 done
          const int call = p.ein_split ? t : 2 * t + (int)rank;
          for (int kc = 0; kc < KC; ++kc) {
            if (t == 0) {
              if (tl > 0) ptx::mbar_wait(&f_empty[kc], (uint32_t)(tl & 1) ^ 1u);
              if (rank == 0) ptx::mbar_expect_tx(&f_full[kc], 2u * A_CHUNK_BYTES);
              for (int h = 0; h < 2; ++h)
                ptx::tma_load_3d_2sm(sF + kc * A_CHUNK_BYTES + h * (A_CHUNK_BYTES / 2), &tmF, &f_full[kc], px0 + h * 64,
                                     kc * TC_BK, batch);
            }
            uint64_t* bar = &e_full[slot * KC + kc];
            if (rank == 0) ptx::mbar_expect_tx(bar, 2u * (uint32_t)e_chunk_bytes);
            ptx::tma_load_2d_2sm(sE + (slot * KC + kc) * e_chunk_bytes, &tmE, bar, kc * TC_BK,
                                 batch * p.b_rows_per_batch + p.b_row0 + call * p.q_pad + q0);
          }
        }
      }
    }
  } else if (warp == 1) {
    if (rank == 0) {
      // ---------------- MMA issuer: the leader CTA's warp walks the loop, one elected lane drives both SMs
      const uint32_t idesc = ptx::umma_idesc_bf16(2 * TC_BM, 256, /*A = E, K-major*/ false, /*B = F, MN-major*/ true);
      const uint64_t ed0 = ptx::umma_desc(ptx::smem_u32(sE), 16, 1024, ptx::UMMA_SW128);
      const uint64_t fd0 = ptx::umma_desc(ptx::smem_u32(sF), A_CHUNK_BYTES / 2, 1024, ptx::UMMA_SW128);
      const uint32_t e16 = (uint32_t)e_chunk_bytes >> 4;
      int g = 0, tl = 0;
      for (int w = pair; w < n_work; w += n_pairs, ++tl)
        for (int t = 0; t < NS; ++t, ++g) {
          const int buf = g & 1;
          const uint32_t use = (uint32_t)(g >> 1);
          ptx::mbar_wait(&acc_empty[buf], (use & 1u) ^ 1u);
          ptx::tc_fence_after();
          const uint32_t d_tmem = tmem_base + (uint32_t)(buf * 256);
#pragma unroll
          for (int kc = 0; kc < KC; ++kc) {
            if (t == 0) ptx::mbar_wait(&f_full[kc], (uint32_t)(tl & 1));
            ptx::mbar_wait(&e_full[buf * KC + kc], use & 1u);
            ptx::tc_fence_after();
            if (ptx::elect_one()) {
              const uint64_t ed = ed0 + (uint64_t)((uint32_t)(buf * KC + kc) * e16);
              const uint64_t fd = fd0 + (uint64_t)(kc * (A_CHUNK_BYTES >> 4));
#pragma unroll
              for (int k = 0; k < TC_BK / 16; ++k)
                ptx::mma_bf16_ss_2sm(d_tmem, ed + (uint64_t)(k * 2), fd + (uint64_t)(k * (2048 >> 4)), idesc, (kc | k) != 0 ? 1u : 0u);
              if (t == NS - 1) ptx::mma_commit_2sm(&f_empty[kc]);     // feature chunk kc may be refilled for the next tile
              if (kc == KC - 1) ptx::mma_commit_2sm(&acc_full[buf]);  // accumulator ready + ring slots free, both CTAs
            }
            __syncwarp();
          }
        }
    }
  } else {
    // ---------------- epilogue (both CTAs): lane = query row of this CTA's head call, 256 pixel columns
    const int quarter = warp & 3;
    const int part = (warp - 2) >> 2;                       // 16-pixel chunk `part` of every 64-pixel sub-tile
    const int row = quarter * 32 + lane;
    const bool row_ok = row < p.q_rows;
    const bool leader = warp == 2 && lane == 0;
    const uint32_t lane_off = (uint32_t)(quarter * 32) << 16;
    int g = 0;
    for (int w = pair; w < n_work; w += n_pairs) {
      const int batch = w / mt2, px_pair = (w - batch * mt2) * 2 * TC_BM;
      const bool last_work = w + n_pairs >= n_work;
      for (int t = 0; t < NS; ++t, ++g) {
        const int buf = g & 1;
        const uint32_t use = (uint32_t)(g >> 1);
        const int call = p.ein_split ? t : 2 * t + (int)rank;
        ptx::mbar_wait(&acc_full[buf], use & 1u);
        ptx::tc_fence_after();
        // 1. accumulator -> registers: sub-tile j, pixels 64 j + 16 part .. + 15
        const uint32_t ta = tmem_base + (uint32_t)(buf * 256 + part * 16) + lane_off;
        uint32_t r0[16], r1[16], r2[16], r3[16];
        ptx::tmem_ld16_issue(ta, r0);
        ptx::tmem_ld16_issue(ta + 64, r1);
        ptx::tmem_ld16_issue(ta + 128, r2);
        ptx::tmem_ld16_issue(ta + 192, r3);
        ptx::tmem_ld_wait16(r0);
        ptx::tmem_ld_wait16(r1);
        ptx::tmem_ld_wait16(r2);
        ptx::tmem_ld_wait16(r3);
        // 2. the accumulator buffer is free again
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive_leader(&acc_empty[buf]);
        // 3. the previous step's stores must have finished READING the staging tiles
        if (leader) ptx::tma_store_wait_read();
        asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS * 32) : "memory");
        auto stage16 = [&](const uint32_t (&r)[16], int j) {
          uint4 o[2];
          uint32_t* ow = reinterpret_cast<uint32_t*>(o);
#pragma unroll
          for (int i = 0; i < 8; ++i) ow[i] = pack_bf16x2(__uint_as_float(r[2 * i]), __uint_as_float(r[2 * i + 1]));
          uint8_t* base = sStage + j * sub_bytes + row * 128;
          *reinterpret_cast<uint4*>(base + (((2 * part) ^ (row & 7)) << 4)) = o[0];
          *reinterpret_cast<uint4*>(base + (((2 * part + 1) ^ (row & 7)) << 4)) = o[1];
        };
        if (row_ok) {
          stage16(r0, 0);
          stage16(r1, 1);
          stage16(r2, 2);
          stage16(r3, 3);
        }
        ptx::fence_proxy_async_smem();
        asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS * 32) : "memory");
        if (leader) {
          if (call < p.n_calls)
            for (int j = 0; j < 4; ++j)
              ptx::tma_store_3d(&tmC, sStage + j * sub_bytes, px_pair + j * 64, q0, call * p.n_batch + batch);
          ptx::tma_store_commit();
          if (last_work && t == NS - 1) ptx::tma_store_wait_read();
        }
      }
    }
  }
  __syncwarp();
  ptx::tc_fence_before();
  ptx::cluster_sync_all();
  if (warp == 1) ptx::tmem_dealloc_2sm(tmem_base, 512u);
}

// ------------------------------------------------------------------- K3, persistent variant
// Attention-mask bits with the B operand RESIDENT: the head call's mask embeddings (fp16, 4 chunks of
// N_TILE x 64) are loaded once per CTA and stay in shared memory while the CTA walks its share of the
// image's 128-key tiles; per tile only the resampled features (fp16, 4 chunks) stream in.  Above 256 queries
// the queries are split into gridDim.z slices of N_TILE: slice z holds rows z*N_TILE.. of the head call.
// Both operands are IEEE half: the resampled features are means of four bf16 values (10 significand bits,
// exact in fp16 for 3 of 4 values), and rounding the mask embeddings to 11 bits flips 0.02 % of the bits --
// plain bf16 operands flip 0.12 %, outside the 99.9 % bar (CPU study in DESIGN.md).
struct TcBitsP {
  int N_TILE, b_row, m_tiles, K_valid, Q, W32, stages, acc_stride, tmem_cols, C;
  uint32_t* bitmap;
};

__global__ void __launch_bounds__(TC_THREADS, 1)
tc_bits_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               const __grid_constant__ TcBitsP p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int bt = p.N_TILE * 128;                 // bytes of one resident B chunk
  uint8_t* sBres = smem;                         // 4 chunks: mask-embedding k-chunks 0..3 (fp16)
  uint8_t* sA = sBres + 4 * bt;                  // ring of stages, each TWO 16 KB feature chunks (one commit frees both)
  constexpr int STAGE_BYTES = 2 * A_CHUNK_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sA + p.stages * STAGE_BYTES);
  uint64_t* b_res_full = bars;
  uint64_t* a_full = bars + 1;
  uint64_t* a_empty = a_full + p.stages;
  uint64_t* acc_full = a_empty + p.stages;
  uint64_t* acc_empty = acc_full + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int batch = blockIdx.y;
  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmA);
    ptx::prefetch_tmap(&tmB);
    ptx::mbar_init(b_res_full, 1);
    for (int i = 0; i < p.stages; ++i) { ptx::mbar_init(&a_full[i], 1); ptx::mbar_init(&a_empty[i], 1); }
    for (int i = 0; i < 2; ++i) { ptx::mbar_init(&acc_full[i], 1); ptx::mbar_init(&acc_empty[i], EPI_WARPS); }
    ptx::fence_mbar_init();
  }
  if (warp == 1) {
    ptx::tmem_alloc(tmem_slot, (uint32_t)p.tmem_cols);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  __syncthreads();                // (implied by the cluster barrier; spelled out for compute-sanitizer racecheck, which does not track it)
  const uint32_t tmem_base = *tmem_slot;
  ptx::grid_dep_launch();
  ptx::grid_dep_wait();

  if (warp == 0) {
    if (lane == 0) {
      ptx::mbar_expect_tx(b_res_full, (uint32_t)(4 * bt));
      for (int j = 0; j < 4; ++j)      // the fp16 copy of the mask embeddings sits in columns [C, 2C) of the rows
        ptx::tma_load_3d(sBres + j * bt, &tmB, b_res_full, p.C + j * TC_BK, p.b_row + (int)blockIdx.z * p.N_TILE, batch);
      int it = 0;
      for (int mt = blockIdx.x; mt < p.m_tiles; mt += gridDim.x)
        for (int j2 = 0; j2 < 2; ++j2, ++it) {
          const int s = it % p.stages;
          ptx::mbar_wait(&a_empty[s], ((uint32_t)(it / p.stages) & 1u) ^ 1u);
          ptx::mbar_expect_tx(&a_full[s], STAGE_BYTES);
          for (int c = 0; c < 2; ++c) {
            const int ch = (2 * j2 + c) * TC_BK;
            for (int g = 0; g < 2; ++g)
              ptx::tma_load_3d(sA + s * STAGE_BYTES + c * A_CHUNK_BYTES + g * (A_CHUNK_BYTES / 2), &tmA, &a_full[s],
                               mt * TC_BM + g * 64, ch, batch);
          }
        }
    }
  } else if (warp == 1) {
    // MMA issuer.  The whole warp walks the loop (uniform control flow: descriptors stay in uniform registers);
    // one elected lane issues.  Descriptors = base + constant increments of the 14-bit address field.
    const uint32_t idesc = ptx::umma_idesc_bf16(TC_BM, p.N_TILE, true, false, /*f16*/ true);
    ptx::mbar_wait(b_res_full, 0);
    ptx::tc_fence_after();
    const uint64_t ad0 = ptx::umma_desc(ptx::smem_u32(sA), A_CHUNK_BYTES / 2, 1024, ptx::UMMA_SW128);
    const uint64_t bd0 = ptx::umma_desc(ptx::smem_u32(sBres), 16, 1024, ptx::UMMA_SW128);
    const uint32_t bt16 = (uint32_t)bt >> 4;
    int it = 0, t = 0;
    for (int mt = blockIdx.x; mt < p.m_tiles; mt += gridDim.x, ++t) {
      const int buf = t & 1;
      ptx::mbar_wait(&acc_empty[buf], (((uint32_t)(t >> 1)) & 1u) ^ 1u);
      ptx::tc_fence_after();
      const uint32_t d_tmem = tmem_base + (uint32_t)(buf * p.acc_stride);
      for (int j2 = 0; j2 < 2; ++j2, ++it) {
        const int s = it % p.stages;
        ptx::mbar_wait(&a_full[s], (uint32_t)(it / p.stages) & 1u);
        ptx::tc_fence_after();
        if (ptx::elect_one()) {
#pragma unroll
          for (int c = 0; c < 2; ++c) {
            const int j = 2 * j2 + c;
            const uint64_t ad = ad0 + (uint64_t)(s * (STAGE_BYTES >> 4) + c * (A_CHUNK_BYTES >> 4));
            const uint64_t bd = bd0 + (uint64_t)(j * bt16);
#pragma unroll
            for (int k = 0; k < TC_BK / 16; ++k)
              ptx::mma_bf16_ss(d_tmem, ad + (uint64_t)(k * (2048 >> 4)), bd + (uint64_t)(k * 2), idesc, (j | k) != 0 ? 1u : 0u);
          }
          ptx::mma_commit(&a_empty[s]);
          if (j2 == 1) ptx::mma_commit(&acc_full[buf]);
        }
        __syncwarp();
      }
    }
  } else {
    const int quarter = warp & 3;
    EpiCtx ctx;
    ctx.lane = lane; ctx.batch = batch; ctx.part = (warp - 2) >> 2; ctx.chunks = p.N_TILE / 16;
    ctx.col0 = (int)blockIdx.z * p.N_TILE;       // first query of this slice
    int t = 0;
    for (int mt = blockIdx.x; mt < p.m_tiles; mt += gridDim.x, ++t) {
      const int buf = t & 1;
      ptx::mbar_wait(&acc_full[buf], ((uint32_t)(t >> 1)) & 1u);
      ptx::tc_fence_after();
      ctx.m = mt * TC_BM + quarter * 32 + lane;
      ctx.m_ok = ctx.m < p.K_valid;
      ctx.wi = (mt * TC_BM + quarter * 32) >> 5;
      ctx.taddr = tmem_base + (uint32_t)(buf * p.acc_stride) + ((uint32_t)(quarter * 32) << 16);
      epi_bits(p.Q, p.W32, p.bitmap, ctx);
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&acc_empty[buf]);
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    ptx::tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
  }
}

// ---------------------------------------------------------------------------- small kernels
// One pass over mask_features (bf16 NCHW) producing the bilinear (align_corners=False) resamples to
// the three level sizes for the exact ratios 8/4/2: each is the mean of the central 2x2 of its
// block, evaluated in the reference's order 0.5*(0.5a+0.5b)+0.5*(0.5c+0.5d) in fp32.
// One thread per 8x8 block of one (image, channel) plane.
// Outputs are IEEE half (a mean of four bf16 values has 10 significand bits: fp16 holds it exactly unless the
// four exponents differ): per image the resampled map is stored as (C, pitch_l).
__global__ void __launch_bounds__(256) downsample3_kernel(const __nv_bfloat16* __restrict__ F, int planes, int C, int H4,
                                                          int W4, __half* __restrict__ d8, __half* __restrict__ d4,
                                                          __half* __restrict__ d2, int p8, int p4, int p2) {
  ptx::grid_dep_launch();
  ptx::grid_dep_wait();
  const int bw = W4 >> 3, bh = H4 >> 3;
  const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
  const long total = (long)planes * bh * bw;
  if (idx >= total) return;
  const int bx = (int)(idx % bw);
  const int by = (int)((idx / bw) % bh);
  const long plane = idx / ((long)bw * bh);
  const __nv_bfloat16* src = F + plane * (long)H4 * W4 + (long)by * 8 * W4 + bx * 8;
  float px[8][8];
#pragma unroll
  for (int r = 0; r < 8; ++r) {
    const uint4 x = *reinterpret_cast<const uint4*>(src + (long)r * W4);
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&x);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float2 f = __bfloat1622float2(h[j]);
      px[r][2 * j] = f.x;
      px[r][2 * j + 1] = f.y;
    }
  }
  auto avg = [&](int r, int c) {
    return 0.5f * (0.5f * px[r][c] + 0.5f * px[r][c + 1]) + 0.5f * (0.5f * px[r + 1][c] + 0.5f * px[r + 1][c + 1]);
  };
  auto h2 = [](float a, float b) {
    const __half2 v = __floats2half2_rn(a, b);
    return *reinterpret_cast<const uint32_t*>(&v);
  };
  // ratio 8 -> rows 3,4 cols 3,4
  d8[plane * (long)p8 + (long)by * bw + bx] = __float2half_rn(avg(3, 3));
  // ratio 4 -> centre of each 4x4: rows 1,2 / 5,6
  {
    const int w = W4 >> 2;
    const long off = (long)(by * 2) * w + bx * 2;
#pragma unroll
    for (int r = 0; r < 2; ++r)
      *reinterpret_cast<uint32_t*>(d4 + plane * (long)p4 + off + (long)r * w) = h2(avg(4 * r + 1, 1), avg(4 * r + 1, 5));
  }
  // ratio 2 -> every 2x2
  {
    const int w = W4 >> 1;
    const long off = (long)(by * 4) * w + bx * 4;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      uint2 ph;
      ph.x = h2(avg(2 * r, 0), avg(2 * r, 2));
      ph.y = h2(avg(2 * r, 4), avg(2 * r, 6));
      *reinterpret_cast<uint2*>(d2 + plane * (long)p2 + off + (long)r * w) = ph;
    }
  }
}

// (rows, K) bf16 -> (rows, pitch) bf16, zero padded
__global__ void repitch_kernel(const __nv_bfloat16* __restrict__ src, __nv_bfloat16* __restrict__ dst, long rows, int K,
                               int pitch) {
  ptx::grid_dep_launch();
  ptx::grid_dep_wait();
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * pitch) return;
  const int k = (int)(i % pitch);
  const long r = i / pitch;
  dst[i] = k < K ? src[r * K + k] : __float2bfloat16(0.f);
}

// me (B,Q,C) fp32 -> rows [b][call*q_pad + q][C] bf16 of the all-call B operand
__global__ void store_me_kernel(const float* __restrict__ me, __nv_bfloat16* __restrict__ dst, int B, int Q, int C,
                                int rows_per_batch, int row0) {
  ptx::grid_dep_launch();
  ptx::grid_dep_wait();
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  const long total = (long)B * Q * C;
  if (i >= total) return;
  const int c = (int)(i % C);
  const long bq = i / C;
  const int q = (int)(bq % Q);
  const int b = (int)(bq / Q);
  __nv_bfloat16* row = dst + ((long)b * rows_per_batch + row0 + q) * 2 * C;
  row[c] = __float2bfloat16_rn(me[i]);                                   // columns [0,C): bf16, read by the mask einsum
  reinterpret_cast<__half*>(row)[C + c] = __float2half_rn(me[i]);        // columns [C,2C): fp16, read by the attention-mask GEMM
}

}  // namespace

// all_masked[row] = (popcount of the row's bitmap == K).  The fp32 route launches it without PDL, where the two
// griddepcontrol instructions do nothing.
__global__ void __launch_bounds__(256) all_masked_kernel(const uint32_t* __restrict__ bitmap, int rows, int W32, int K,
                                                         uint8_t* __restrict__ all_masked) {
  ptx::grid_dep_launch();
  ptx::grid_dep_wait();
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= rows) return;
  int cnt = 0;
  for (int i = lane; i < W32; i += 32) cnt += __popc(bitmap[(long)row * W32 + i]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  if (lane == 0) all_masked[row] = (cnt == K) ? 1 : 0;
}

namespace {

// 3-D map over an NCHW feature tensor: dims (pixels, channels, batch), box (64 px, 64 ch, 1)
// `pitch` = elements between consecutive channel planes (>= pixels, multiple of 8); columns in [pixels, pitch)
// are never read: the map's extent is `pixels`, TMA zero-fills beyond it.
int make_map_A(TcState* t, CUtensorMap* m, const void* base, int pixels, int C, int B, int pitch = -1) {
  if (pitch < 0) pitch = pixels;
  if ((pitch * 2) % 16 != 0 || (reinterpret_cast<uintptr_t>(base) & 15))
    return tc_fail(t, CGG_ERR_UNSUPPORTED, "TMA needs 16-byte aligned channel planes (pixel pitch multiple of 8)");
  const cuuint64_t dims[3] = {(cuuint64_t)pixels, (cuuint64_t)C, (cuuint64_t)B};
  const cuuint64_t strides[2] = {(cuuint64_t)pitch * 2, (cuuint64_t)pitch * C * 2};
  const cuuint32_t box[3] = {64, 64, 1};
  if (!encode_tensor_map(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, base, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B,
                         CU_TENSOR_MAP_L2_PROMOTION_L2_128B, "A", &t->err))
    return CGG_ERR_CUDA;
  return CGG_OK;
}
// 2-D map over a K-major [rows][C] bf16 matrix: box (64 k, n_tile rows)
int make_map_B(TcState* t, CUtensorMap* m, const void* base, long rows, int C, int n_tile) {
  // C = row length in elements (pitch == length)
  const cuuint64_t dims[2] = {(cuuint64_t)C, (cuuint64_t)rows};
  const cuuint64_t strides[1] = {(cuuint64_t)C * 2};
  const cuuint32_t box[2] = {64, (cuuint32_t)n_tile};
  if (!encode_tensor_map(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, base, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B,
                         CU_TENSOR_MAP_L2_PROMOTION_L2_256B, "B", &t->err))
    return CGG_ERR_CUDA;
  return CGG_OK;
}

// TMEM columns of one N_TILE-wide fp32 accumulator: a power of two >= 32
int tmem_cols_for(int n_tile) { return n_tile <= 32 ? 32 : n_tile <= 64 ? 64 : n_tile <= 128 ? 128 : 256; }

// Launches a CTA-pair kernel over the tile pairs of `pixels` per image: ceil(pixels / 256) work items per image,
// at most one CTA per SM and, when cta_cap > 0, at most cta_cap CTAs (leaving SMs to a concurrent latency-bound chain).
template <typename Kernel>
int launch_pairs(TcState* t, Kernel kernel, size_t smem, cudaStream_t s, const CUtensorMap& mA, const CUtensorMap& mB,
                 const CUtensorMap& mC, TcPairP p, long pixels, int batch, int cta_cap = 0) {
  p.m_pairs = (int)((pixels + 2 * TC_BM - 1) / (2 * TC_BM)); p.n_batch = batch;
  const int items = p.m_pairs * batch;
  int pairs = t->num_sms / 2;
  if (cta_cap > 0 && pairs > cta_cap / 2) pairs = cta_cap / 2;
  if (pairs > items) pairs = items;
  TCU(launch_pdl_cluster(2, kernel, dim3(2 * pairs), dim3(TC_THREADS), smem, s, mA, mB, mC, p));
  count_launch();
  TCU(cudaGetLastError());
  return CGG_OK;
}

}  // namespace

// =========================================================================== host interface
TcState* tc_create(const cgg_config& cfg) {
  TcState* t = new (std::nothrow) TcState();
  if (!t) return nullptr;
  t->cfg = cfg;
  // the SM count and the kernels' shared-memory limit belong to the device: a handle lives on the one it is created on
  int dev = 0;
  const auto max_smem = [](auto kernel) {
    return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024) == cudaSuccess;
  };
  if (cudaGetDevice(&dev) != cudaSuccess ||
      cudaDeviceGetAttribute(&t->num_sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess ||
      !max_smem(tc_gemm_kernel) || !max_smem(tc_kv_pair_kernel) || !max_smem(tc_bits_kernel) ||
      !max_smem(tc_einsum_t_kernel) || !max_smem(tc_einsum_pair_kernel) ||
      tc_attention_setup() != cudaSuccess) {
    delete t;
    return nullptr;
  }
  const int Q = cfg.num_queries, calls = cfg.num_layers + 1;
  // Mask-einsum routing.  Shared memory holds tc_einsum_t_kernel's query rows up to 104 per CTA and
  // tc_einsum_pair_kernel's N tile up to 208 columns.  q_pad = B-operand rows per head call.
  //   Q <= 104   einsum_t, q_pad = max(16, round8(Q)) rows per CTA, two head calls per step
  //   105..128   pair kernel, one head call per N tile of round16(Q)
  //   129..208   einsum_t, q_pad = round16(Q), one head call per step split over the pair
  //   > 208      pair kernel, T = ceil(Q / 208) N tiles of round16(ceil(Q / T)) per head call
  if (Q <= 104) {
    t->q_pad = round_up(Q, 8) < 16 ? 16 : round_up(Q, 8);
  } else if (Q <= 128) {
    t->q_pad = t->ein_ntile = round_up(Q, 16);
  } else if (Q <= 208) {
    t->q_pad = round_up(Q, 16);
  } else {
    const int T = (Q + 207) / 208;
    t->ein_ntile = round_up((Q + T - 1) / T, 16);
    t->q_pad = T * t->ein_ntile;
  }
  // attention-mask bits: one N tile of round16(Q) queries, above 256 queries two slices of round32(Q) / 2
  if (round_up(Q, 16) <= 256) { t->bits_ntile = round_up(Q, 16); t->bits_nt = 1; }
  else { t->bits_ntile = round_up(Q, 32) / 2; t->bits_nt = 2; }
  if (t->bits_ntile > 256) { delete t; return nullptr; }
  t->rows_per_batch = calls * t->q_pad;
  t->live_bytes = 1 << 20;
  if (cudaMalloc(&t->live_buf, t->live_bytes) != cudaSuccess) { delete t; return nullptr; }
  return t;
}

void tc_destroy(TcState* t) {
  if (!t) return;
  t->free_all();
  t->free_packed();
  cudaFree(t->live_buf);
  delete t;
}

const char* tc_last_error(const TcState* t) { return t ? t->err.c_str() : ""; }

size_t tc_workspace_bytes(const TcState* t, int batch) {
  if (!t) return 0;
  TcWs w;
  w.carve(t, batch);
  return w.total;
}

size_t tc_workspace_offset(const TcState* t, int batch, const char* what) {
  if (!t || !what) return (size_t)-1;
  TcWs w;
  w.carve(t, batch);
  const std::string n(what);
  if (n == "me_all") return w.me_all;
  if (n == "fds0") return w.fds[0];
  if (n == "fds1") return w.fds[1];
  if (n == "fds2") return w.fds[2];
  return (size_t)-1;
}
const void* tc_key_bias_table(const TcState* t, int level, long* cols) {
  if (cols) *cols = 2L * t->nl[level] * t->cfg.embed_dim;   // [hi | lo]
  return t->rk[level];
}

int tc_prepare(TcState* t, const cgg_weights* w, int H4, int W4, const int* lh, const int* lw, const int* nl,
               float* const* wkv_f32, float* const* rk_f32, float* const* bkv_f32, cudaStream_t s) {
  const int C = t->cfg.embed_dim;
  const int ratio[3] = {8, 4, 2};
  for (int l = 0; l < 3; ++l)
    if (lh[l] * ratio[l] != H4 || lw[l] * ratio[l] != W4)
      return tc_fail(t, CGG_ERR_UNSUPPORTED,
                     "bf16 mode needs level sizes at exactly 1/8, 1/4, 1/2 of the mask-feature size (inputs padded to /32)");
  bool same = t->H4 == H4 && t->W4 == W4;
  for (int l = 0; l < 3; ++l) same = same && t->lh[l] == lh[l] && t->lw[l] == lw[l] && t->nl[l] == nl[l] && t->wkv[l];
  if (!same) {
    t->free_all();
    t->H4 = H4; t->W4 = W4;
    for (int l = 0; l < 3; ++l) {
      t->lh[l] = lh[l]; t->lw[l] = lw[l]; t->nl[l] = nl[l];
      const int n = nl[l] > 0 ? nl[l] : 1;
      TCU(cudaMalloc(&t->wkv[l], (size_t)n * 2 * C * C * 2));
      TCU(cudaMalloc(&t->rk[l], (size_t)lh[l] * lw[l] * n * C * 2 * 2));   // hi | lo
    }
  }
  for (int l = 0; l < 3; ++l) {
    if (nl[l] == 0) continue;
    TCU(launch_cast_bf16(wkv_f32[l], t->wkv[l], (size_t)nl[l] * 2 * C * C, s));
    TCU(launch_cast_bf16_split(rk_f32[l], t->rk[l], lh[l] * lw[l], nl[l] * C, s));
    t->bkv[l] = bkv_f32[l];
  }
  return tc_pack_weights(t, w, s);
}

int tc_kv_project(TcState* t, int level, int batch, const void* mem_bf16, void* kv_bf16, void* ws, cudaStream_t s,
                  int cta_cap) {
  const int C = t->cfg.embed_dim, K = t->lh[level] * t->lw[level], N = t->nl[level] * 2 * C;
  CUtensorMap mA, mB;
  int pitch = K;
  if (K % 8) {
    // ragged level (e.g. 33x25 keys of a 1056x800 input): copy to 16-byte aligned channel planes first
    TcWs w;
    w.carve(t, batch);
    pitch = pitch8(K);
    __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(static_cast<char*>(ws) + w.memp[level]);
    const long total = (long)batch * C * pitch;
    TCU(launch_pdl(repitch_kernel, dim3((unsigned)((total + 255) / 256)), dim3(256), 0, s,
                   static_cast<const __nv_bfloat16*>(mem_bf16), dst, (long)batch * C, K, pitch));
    count_launch();
    mem_bf16 = dst;
  }
  int st = make_map_A(t, &mA, mem_bf16, K, C, batch, pitch);
  if (st != CGG_OK) return st;
  TcPairP p = {};
  p.N_TILE = 256;
  if (N % p.N_TILE != 0) return tc_fail(t, CGG_ERR_BAD_SHAPE, "K/V width not a multiple of 256");
  st = make_map_B(t, &mB, t->wkv[level], N, C, p.N_TILE / 2);     // each CTA of the pair loads half of a B chunk
  if (st != CGG_OK) return st;
  p.NT = N / p.N_TILE;
  // the key-bias table (pos / level / bk through Wk) is NOT added here: the attention kernel adds Q R^T
  p.bias = t->bkv[level];
  CUtensorMap mC;
  {
    const cuuint64_t dims[3] = {(cuuint64_t)N, (cuuint64_t)K, (cuuint64_t)batch};
    const cuuint64_t strides[2] = {(cuuint64_t)N * 2, (cuuint64_t)K * N * 2};
    const cuuint32_t box[3] = {64, (cuuint32_t)TC_BM, 1};
    if (!encode_tensor_map(&mC, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, kv_bf16, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B,
                           CU_TENSOR_MAP_L2_PROMOTION_NONE, "kv out", &t->err))
      return CGG_ERR_CUDA;
  }
  p.acc_stride = tmem_cols_for(p.N_TILE); p.tmem_cols = 2 * p.acc_stride;
  const size_t stage_bytes = (size_t)p.N_TILE * TC_BM * 2, bias_bytes = (size_t)p.NT * p.N_TILE * 4;
  const size_t b_stage = (size_t)(p.N_TILE / 2) * 128;
  int stages = (int)((224 * 1024 - 4 * A_CHUNK_BYTES - stage_bytes - bias_bytes - 512) / b_stage);
  if (stages > 8) stages = 8;
  if (stages < 3) return tc_fail(t, CGG_ERR_BAD_SHAPE, "K/V projection: weight ring does not fit shared memory");
  p.stages = stages;
  const size_t smem = 1024 + 4 * A_CHUNK_BYTES + stages * b_stage + stage_bytes + bias_bytes + (8 + 2 * stages + 4) * 8 + 64;
  return launch_pairs(t, tc_kv_pair_kernel, smem, s, mA, mB, mC, p, K, batch, cta_cap);
}

int tc_downsample(TcState* t, int batch, const void* mask_features_bf16, void* ws, cudaStream_t s) {
  TcWs w;
  w.carve(t, batch);
  if ((t->H4 % 8) || (t->W4 % 8)) return tc_fail(t, CGG_ERR_UNSUPPORTED, "mask feature size must be a multiple of 8");
  const int planes = batch * t->cfg.embed_dim;
  const long total = (long)planes * (t->H4 / 8) * (t->W4 / 8);
  char* base = static_cast<char*>(ws);
  TCU(launch_pdl(downsample3_kernel, dim3((unsigned)((total + 255) / 256)), dim3(256), 0, s,
      static_cast<const __nv_bfloat16*>(mask_features_bf16), planes, t->cfg.embed_dim, t->H4, t->W4,
      reinterpret_cast<__half*>(base + w.fds[0]), reinterpret_cast<__half*>(base + w.fds[1]),
      reinterpret_cast<__half*>(base + w.fds[2]), pitch8(t->lh[0] * t->lw[0]), pitch8(t->lh[1] * t->lw[1]),
      pitch8(t->lh[2] * t->lw[2])));
  count_launch();
  TCU(cudaGetLastError());
  return CGG_OK;
}

int tc_store_mask_embed(TcState* t, int batch, int call_idx, const float* me_f32, void* ws, cudaStream_t s) {
  TcWs w;
  w.carve(t, batch);
  const int C = t->cfg.embed_dim, Q = t->cfg.num_queries;
  const long total = (long)batch * Q * C;
  TCU(launch_pdl(store_me_kernel, dim3((unsigned)((total + 255) / 256)), dim3(256), 0, s,
      me_f32, reinterpret_cast<__nv_bfloat16*>(static_cast<char*>(ws) + w.me_all), batch, Q, C, t->rows_per_batch,
      call_idx * t->q_pad));
  count_launch();
  TCU(cudaGetLastError());
  return CGG_OK;
}

int tc_mask_bits(TcState* t, int batch, int call_idx, int level, uint32_t* bitmap, uint8_t* all_masked, void* ws,
                 cudaStream_t s) {
  TcWs w;
  w.carve(t, batch);
  const int C = t->cfg.embed_dim, Q = t->cfg.num_queries, K = t->lh[level] * t->lw[level];
  char* base = static_cast<char*>(ws);
  CUtensorMap mA, mB;
  // logits = F_ds . me with both operands in IEEE half (fp32 accumulate)
  int st = make_map_A(t, &mA, base + w.fds[level], K, C, batch, pitch8(K));
  if (st != CGG_OK) return st;
  TcBitsP bp = {};
  bp.N_TILE = t->bits_ntile; bp.m_tiles = (K + TC_BM - 1) / TC_BM; bp.K_valid = K; bp.Q = Q;
  bp.W32 = (K + 31) / 32; bp.C = C; bp.bitmap = bitmap;
  bp.acc_stride = tmem_cols_for(bp.N_TILE);
  bp.tmem_cols = 2 * bp.acc_stride;
  bp.stages = (int)((225 * 1024 - 4 * bp.N_TILE * 128) / (2 * A_CHUNK_BYTES));   // stages of two feature chunks
  if (bp.stages > 4) bp.stages = 4;
  bp.b_row = call_idx * t->q_pad;
  const size_t smem = 1024 + 4 * (size_t)bp.N_TILE * 128 + (size_t)bp.stages * 2 * A_CHUNK_BYTES + (1 + 2 * bp.stages + 4) * 8 + 64;
  // about one wave: (key-tile walkers) x images x query slices
  int gx = t->num_sms / (batch * t->bits_nt);
  if (gx < 1) gx = 1;
  if (gx > bp.m_tiles) gx = bp.m_tiles;
  // B map (k, row in image, image): the image's row block is selected by blockIdx.y; rows past the image's
  // block (the last call's second slice) load as zeros and their queries are not stored
  {
    const cuuint64_t dims[3] = {(cuuint64_t)(2 * C), (cuuint64_t)t->rows_per_batch, (cuuint64_t)batch};
    const cuuint64_t strides[2] = {(cuuint64_t)(2 * C) * 2, (cuuint64_t)t->rows_per_batch * (2 * C) * 2};
    const cuuint32_t box[3] = {64, (cuuint32_t)bp.N_TILE, 1};
    if (!encode_tensor_map(&mB, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, base + w.me_all, dims, strides, box,
                           CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, "me", &t->err))
      return CGG_ERR_CUDA;
  }
  TCU(launch_pdl(tc_bits_kernel, dim3(gx, batch, t->bits_nt), dim3(TC_THREADS), smem, s, mA, mB, bp));
  count_launch();
  TCU(cudaGetLastError());
  const int rows = batch * Q;
  TCU(launch_pdl(all_masked_kernel, dim3((rows + 7) / 8), dim3(256), 0, s, (const uint32_t*)bitmap, rows, bp.W32, K, all_masked));
  count_launch();
  TCU(cudaGetLastError());
  return CGG_OK;
}

int tc_mask_einsum(TcState* t, int batch, int first_call, int num_calls, const void* mask_features_bf16,
                   void* mask_bf16, long call_stride, void* ws, cudaStream_t s) {
  TcWs w;
  w.carve(t, batch);
  const int C = t->cfg.embed_dim, Q = t->cfg.num_queries;
  const long HW = (long)t->H4 * t->W4;
  char* base = static_cast<char*>(ws);
  if (num_calls > 1 && call_stride != (long)batch * Q * HW)
    return tc_fail(t, CGG_ERR_BAD_SHAPE, "mask outputs of consecutive head calls must be contiguous");
  CUtensorMap mA, mB, mC;
  int st = make_map_A(t, &mA, mask_features_bf16, (int)HW, C, batch);
  if (st != CGG_OK) return st;
  TcPairP p = {};
  p.b_row0 = first_call * t->q_pad; p.b_rows_per_batch = t->rows_per_batch;
  p.q_pad = t->q_pad; p.n_calls = num_calls;
  // B rows up to 128 past the last call of the last image fall in the slack of me_all (finite, never stored)
  const long b_rows = (long)batch * t->rows_per_batch + 128;
  // output map (pixels, q, call*B + image): rows q >= Q and pixels >= HW of a store box are clipped
  const cuuint64_t dims[3] = {(cuuint64_t)HW, (cuuint64_t)Q, (cuuint64_t)num_calls * batch};
  const cuuint64_t strides[2] = {(cuuint64_t)HW * 2, (cuuint64_t)Q * HW * 2};
  if (t->ein_ntile == 0) {
    // transposed CTA-pair kernel: queries on the TMEM lanes, pixels on the columns
    p.ein_split = t->q_pad > 104 ? 1 : 0;     // one head call per step, its rows split over the CTA pair
    p.q_rows = p.ein_split ? t->q_pad / 2 : t->q_pad;
    st = make_map_B(t, &mB, base + w.me_all, b_rows, 2 * C, p.q_rows);
    if (st != CGG_OK) return st;
    const cuuint32_t box[3] = {64, (cuuint32_t)p.q_rows, 1};
    if (!encode_tensor_map(&mC, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, mask_bf16, dims, strides, box,
                           CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE, "mask out, swizzled", &t->err))
      return CGG_ERR_CUDA;
    const size_t e_chunk = (size_t)p.q_rows * 128;
    // The MMA reads 128 rows of every E chunk (rows past q_rows land in TMEM lanes that are never stored).  From the
    // last ring chunk that read ends 7 e_chunk + 16 KB past the ring's start; below ~26 rows per chunk (Q <= 24) it
    // would run past the staging tiles and barriers out of the allocation, which is extended to cover it.
    const size_t e_read_end = 7 * e_chunk + 128 * 128, e_alloc = 12 * e_chunk + 24 * 8 + 64;
    const size_t smem = 1024 + 4 * A_CHUNK_BYTES + (e_read_end > e_alloc ? e_read_end : e_alloc);
    return launch_pairs(t, tc_einsum_t_kernel, smem, s, mA, mB, mC, p, HW, batch);
  }
  // pixel-on-lane CTA-pair kernel: q_pad / N_TILE tiles per head call, each CTA loads N_TILE/2 rows of every B chunk
  p.N_TILE = t->ein_ntile; p.NT = num_calls * (t->q_pad / t->ein_ntile);
  p.acc_stride = tmem_cols_for(p.N_TILE); p.tmem_cols = 2 * p.acc_stride;
  st = make_map_B(t, &mB, base + w.me_all, b_rows, 2 * C, p.N_TILE / 2);
  if (st != CGG_OK) return st;
  const cuuint32_t box[3] = {(cuuint32_t)TC_BM, (cuuint32_t)p.N_TILE, 1};
  if (!encode_tensor_map(&mC, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, mask_bf16, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_NONE,
                         CU_TENSOR_MAP_L2_PROMOTION_NONE, "mask out", &t->err))
    return CGG_ERR_CUDA;
  const size_t stage_bytes = (size_t)p.N_TILE * TC_BM * 2 + 1024;
  const size_t b_chunk = (size_t)(p.N_TILE / 2) * 128;
  const size_t smem = 1024 + 4 * A_CHUNK_BYTES + 8 * b_chunk + 24 * 8 + 64 + stage_bytes;
  return launch_pairs(t, tc_einsum_pair_kernel, smem, s, mA, mB, mC, p, HW, batch);
}

// ------------------------------------------------------------------ small-M linear layers
// y = A[M,K] W[N,K]^T (+ bias ...) with both operands bf16 K-major through TMA.  Rows are the
// flattened (image, query) pairs, in tiles of <= 128; 128 output features per CTA.
namespace {
int make_map_act(TcState* t, CUtensorMap* m, const void* base, long rows, int K) {
  const cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)rows};
  const cuuint64_t strides[1] = {(cuuint64_t)K * 2};
  const cuuint32_t box[2] = {64, 128};
  if (!encode_tensor_map(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, base, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B,
                         CU_TENSOR_MAP_L2_PROMOTION_L2_128B, "act", &t->err))
    return CGG_ERR_CUDA;
  return CGG_OK;
}

}  // namespace

int tc_linear(TcState* t, const __nv_bfloat16* A, int M, int K, const __nv_bfloat16* W, int n_padded, const float* bias,
              const TcSeg* segs, int nsegs, cudaStream_t s, bool split_k, int kparts, long kpart_stride, bool f16) {
  if (kparts < 1) kparts = 1;
  if (kparts > 1 && (nsegs != 1 || segs[0].is_bf16 || segs[0].relu || (K / TC_BK) % kparts != 0))
    return tc_fail(t, CGG_ERR_BAD_SHAPE, "K-parts need one plain fp32 output segment");
  // swap-AB: the WEIGHTS are the UMMA A operand (128 output features per CTA on the TMEM lanes), the
  // activations the B operand (a tile of <= 256 tokens on the columns); grid = feature tiles x token tiles.
  if (K % TC_BK != 0 || n_padded % TC_BM != 0 || nsegs < 1 || nsegs > 3)
    return tc_fail(t, CGG_ERR_BAD_SHAPE, "tc_linear shape (features must be padded to 128)");
  for (int i = 0; i < nsegs; ++i)
    if (segs[i].col0 % 32 != 0) return tc_fail(t, CGG_ERR_BAD_SHAPE, "segment start must be a multiple of 32");
  const int row_len = split_k ? 2 * K : K;
  TcLinP p = {};
  // token tile: as few CTAs-worth of padding as possible with N <= 128 (multiple of 16)
  const int tok_cap = 128;   // tokens per tile; measured best (3.93 vs 4.29 ms/step at 256)
  const int n_tok_tiles = (M + tok_cap - 1) / tok_cap;
  p.N_TILE = ((M + n_tok_tiles - 1) / n_tok_tiles + 15) / 16 * 16;
  CUtensorMap mW, mX;
  int st = make_map_act(t, &mW, W, n_padded, row_len);      // A operand: (64 k x 128 features) boxes
  if (st != CGG_OK) return st;
  st = make_map_B(t, &mX, A, M, row_len, p.N_TILE);          // B operand: (64 k x N_TILE tokens) boxes
  if (st != CGG_OK) return st;
  p.KC = K / TC_BK / kparts; p.kpart_stride = kpart_stride;
  if (split_k) { p.split_cpc = p.KC; p.split_K = K; p.KC = 3 * p.split_cpc; }
  p.n_tokens = M;
  p.f16 = f16 ? 1 : 0;
  p.nseg = nsegs; p.lin_bias = bias;
  for (int i = 0; i < nsegs; ++i) p.seg[i] = segs[i];
  p.tmem_cols = tmem_cols_for(p.N_TILE);
  const size_t stage_bytes = A_CHUNK_BYTES + (size_t)p.N_TILE * 128;
  p.stages = (int)(204 * 1024 / stage_bytes);
  if (p.stages > 8) p.stages = 8;
  if (p.stages > p.KC) p.stages = p.KC;
  const size_t smem = 1024 + p.stages * stage_bytes + (2 * p.stages + 1) * 8 + 64;
  TCU(launch_pdl(tc_gemm_kernel, dim3(n_padded / TC_BM, n_tok_tiles, kparts), dim3(TC_THREADS), smem, s, mW, mX, p));
  count_launch();
  TCU(cudaGetLastError());
  return CGG_OK;
}

}  // namespace cgg

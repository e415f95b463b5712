// K5 on tensor cores (throughput mode): masked multi-head cross-attention, flash-style, sm_100a.
//
// One CTA per (image, head, 128-query tile).  Keys stream in 128-key tiles:
//   S = Q K^T (+ Q R^T)  tcgen05.mma  M=128 (queries) x N=128 (keys) x K=32 (head dim), S in TMEM (three buffers)
//   softmax   16 warps, thread = query row (TMEM lane) x one 32-key quarter of the tile: the scores are read with
//             tcgen05.ld, the row's attention-mask word for those 32 keys is applied (bit = 1 -> -inf), max / sum
//             are thread-local (no shuffles), P is packed to bf16 and written with tcgen05.st over the scores it
//             came from
//   O += P V  tcgen05.mma  M=128 x N=32 x K=32 per key quarter, A = P from TMEM, into one O accumulator per key
//             quarter that stays in TMEM (lazy rescale of the running maximum)
// Warp 0 is the producer: one lane issues TMA for the K, V (and key-bias R) tiles, the whole warp copies the tile's
// 128 rows x 4 attention-mask words into the same stage, so the softmax loop has no global load.  Key tiles that are
// masked for EVERY query of the CTA are skipped; the flags come from attention_live_kernel, computed once per
// (image, query tile) for all heads.  Rows with all_masked set ignore the bitmap (the reference's all-masked-row
// fallback, head.py:825-826).
//   warp 0: producer   warp 1: MMA issuer (1 thread)   warps 2-17: softmax / epilogue -- four groups of 4 warps,
//   each owning 32 of the tile's 128 key columns with its OWN running max / sum / output accumulator (merged once
//   at the end), so the groups never synchronise per tile.
// The MMA thread issues P V of tile j and Q K^T of tile j+3 back to back and commits ONCE: phase n of step[b] means
// "S(3n+b) ready" and "P V(3(n-1)+b) done" (a tcgen05.commit costs the issuing thread several hundred cycles).
#include <cuda_fp16.h>
#include "kernels.h"
#include "tc_ptx.cuh"
#include "tc_state.h"

namespace cgg {

namespace {

constexpr int AT_THREADS = 64 + 512;       // producer warp + MMA warp + 16 softmax warps (four key-column quarters)
constexpr int AT_KT = 128;                   // keys per tile
constexpr int AT_STAGES = 6;                 // K/V ring
constexpr int AT_KV_TILE_BYTES = AT_KT * 64; // 128 keys x 32 dims x bf16 = 8 KB
constexpr int AT_STAGE_BYTES = 4 * AT_KV_TILE_BYTES;   // K tile, V tile, key-bias (R) tile as hi + lo
constexpr int AT_MASK_BYTES = 128 * 4 * 4;   // per stage: 128 query rows x 4 mask words, stored [key quarter][row]
constexpr int AT_Q_BYTES = 128 * 64;         // 128 queries x 32 dims bf16, core-matrix layout
constexpr int AT_MAX_TILES = 512;
constexpr float LOG2E = 1.4426950408889634f;
constexpr float AT_TAU = 8.0f;               // lazy-rescale threshold on the running maximum, in log2 units
constexpr size_t AT_SMEM = 1024 + AT_Q_BYTES + AT_STAGES * (AT_STAGE_BYTES + AT_MASK_BYTES) + AT_MAX_TILES +
                           (2 * AT_STAGES + 6) * 8 + 16;
static_assert(AT_SMEM <= 227 * 1024, "attention stage budget");

struct AttnP {
  const float* q; float* out; __nv_bfloat16* out_bf16;
  const uint32_t* bitmap; const uint8_t* all_masked;
  const uint8_t* live;           // [image][query tile][key tile] from attention_live_kernel; nullptr: every tile live
  int Q, K, heads, W32, ntiles, nqt;
  int has_r, r_col0, r_lo_off;   // key-bias table term: S += Q (R_hi + R_lo)^T, R columns r_col0 + head*32
  int out_hl;                    // out_bf16: 0 = bf16 rows of C, 1 = [hi(C) | lo(C)] bf16 pairs, 2 = IEEE half rows of C
};


// row (b, qi), head h of the attention output: o[32] * inv as fp32 and / or as a 16-bit GEMM operand (AttnP::out_hl)
__device__ __forceinline__ void store_attn_out(const AttnP& p, int b, int qi, int h, int C, const float* o, float inv) {
  if (p.out) {
    float4* dst = reinterpret_cast<float4*>(p.out + ((long)b * p.Q + qi) * C + h * 32);
#pragma unroll
    for (int i = 0; i < 8; ++i)
      dst[i] = make_float4(o[4 * i] * inv, o[4 * i + 1] * inv, o[4 * i + 2] * inv, o[4 * i + 3] * inv);
  }
  if (p.out_bf16) {
    const long ld = p.out_hl == 1 ? 2 * C : C;
    uint4* dst = reinterpret_cast<uint4*>(p.out_bf16 + ((long)b * p.Q + qi) * ld + h * 32);
    uint4* dst_lo = reinterpret_cast<uint4*>(p.out_bf16 + ((long)b * p.Q + qi) * ld + C + h * 32);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      uint4 pk, pl;
      uint32_t* w = reinterpret_cast<uint32_t*>(&pk);
      uint32_t* wl = reinterpret_cast<uint32_t*>(&pl);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float a0 = o[8 * i + 2 * j] * inv, a1 = o[8 * i + 2 * j + 1] * inv;
        if (p.out_hl == 2) {
          const __half2 h2 = __floats2half2_rn(a0, a1);
          w[j] = *reinterpret_cast<const uint32_t*>(&h2);
        } else {
          __nv_bfloat162 v2 = __floats2bfloat162_rn(a0, a1);
          w[j] = *reinterpret_cast<uint32_t*>(&v2);
          const float2 back = __bfloat1622float2(v2);
          __nv_bfloat162 l2 = __floats2bfloat162_rn(a0 - back.x, a1 - back.y);
          wl[j] = *reinterpret_cast<uint32_t*>(&l2);
        }
      }
      dst[i] = pk;
      if (p.out_hl == 1) dst_lo[i] = pl;
    }
  }
}

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float* v) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

__device__ __forceinline__ int next_live(const uint8_t* live, int t, int n) {
  while (t < n && !live[t]) ++t;
  return t;
}

// 32 lanes x 32 fp32 columns without the wait: the registers are written asynchronously, tmem_ld32_wait() before use
__device__ __forceinline__ void tmem_ld32_issue(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
}
// tcgen05.wait::ld; the registers are in/out operands so that no use of them is scheduled above the wait
__device__ __forceinline__ void tmem_ld32_wait(uint32_t* r) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                 "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]),
                 "+r"(r[16]), "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]),
                 "+r"(r[23]), "+r"(r[24]), "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]),
                 "+r"(r[30]), "+r"(r[31])
               :: "memory");
}
// 32 lanes x 16 columns store without the wait, and the wait; the source registers stay allocated until the wait
__device__ __forceinline__ void tmem_st16_issue(uint32_t taddr, const uint32_t* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
        "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st16_wait(uint32_t* r) {
  asm volatile("tcgen05.wait::st.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                 "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15])
               :: "memory");
}

// packed fp32 pairs (FFMA2 / FADD2 on sm_100a): a * b + c and a + b
__device__ __forceinline__ float2 fma2(float2 a, float2 b, float2 c) {
  float2 d;
  asm("{\n\t.reg .b64 ra, rb, rc, rd;\n\t"
      "mov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\tmov.b64 rc, {%6, %7};\n\t"
      "fma.rn.f32x2 rd, ra, rb, rc;\n\tmov.b64 {%0, %1}, rd;\n\t}"
      : "=f"(d.x), "=f"(d.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y), "f"(c.x), "f"(c.y));
  return d;
}
__device__ __forceinline__ float2 add2(float2 a, float2 b) {
  float2 d;
  asm("{\n\t.reg .b64 ra, rb, rd;\n\t"
      "mov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\t"
      "add.rn.f32x2 rd, ra, rb;\n\tmov.b64 {%0, %1}, rd;\n\t}"
      : "=f"(d.x), "=f"(d.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
  return d;
}

// raises the transaction count of the barrier's current phase without an arrival
__device__ __forceinline__ void mbar_expect_tx_only(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.expect_tx.relaxed.cta.shared::cta.b64 [%0], %1;" ::"r"(ptx::smem_u32(bar)), "r"(bytes) : "memory");
}

// D[tmem] (+)= A[tmem] * B[smem desc]: the A operand (M = 128 rows on the TMEM lanes, K-major, two bf16 per column)
// comes from tensor memory
__device__ __forceinline__ void mma_bf16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}\n"
      ::"r"(d_tmem), "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}

// live[(b * nqt + qt) * ntiles + t] = 1 when some query row of tile qt of image b attends to a key of key tile t: a
// row under the all-masked fallback attends everywhere, any other row where its bitmap has a 0 bit below K.  One CTA
// per (query tile, image); a warp reads one bitmap row at a time, coalesced.  The flags serve all heads.
__global__ void __launch_bounds__(512) attention_live_kernel(const uint32_t* __restrict__ bitmap,
                                                             const uint8_t* __restrict__ all_masked, int Q, int K,
                                                             int W32, int ntiles, int nqt, uint8_t* __restrict__ live) {
  __shared__ int s_tile[AT_MAX_TILES];
  __shared__ int s_fallback;
  const int qt = blockIdx.x, b = blockIdx.y, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int t = threadIdx.x; t < ntiles; t += blockDim.x) s_tile[t] = 0;
  if (threadIdx.x == 0) s_fallback = 0;
  ptx::grid_dep_launch();
  ptx::grid_dep_wait();
  __syncthreads();
  const int q0 = qt * 128, nrows = min(128, Q - q0);
  for (int r = warp; r < nrows; r += blockDim.x / 32) {
    const long row = (long)b * Q + q0 + r;
    if (all_masked && all_masked[row]) { s_fallback = 1; continue; }
    const uint32_t* brow = bitmap + row * W32;
#pragma unroll 4
    for (int w = lane; w < W32; w += 32) {
      const int k0 = w * 32;     // < K: W32 = ceil(K / 32)
      const uint32_t valid = (k0 + 32 > K) ? ((1u << (K - k0)) - 1u) : 0xffffffffu;
      if ((~__ldg(brow + w)) & valid) s_tile[w >> 2] = 1;
    }
  }
  __syncthreads();
  for (int t = threadIdx.x; t < ntiles; t += blockDim.x)
    live[((long)b * nqt + qt) * ntiles + t] = (s_fallback || s_tile[t]) ? 1 : 0;
}

__global__ void __launch_bounds__(AT_THREADS, 1)
masked_attention_tc_kernel(const __grid_constant__ CUtensorMap tmK, const __grid_constant__ CUtensorMap tmV,
                           const __grid_constant__ CUtensorMap tmR, const __grid_constant__ AttnP p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* sQ = smem;                                   // 8 KB
  uint8_t* sKV = sQ + AT_Q_BYTES;                       // AT_STAGES x (K, V, R_hi, R_lo tiles)
  uint8_t* sX = sKV;                                    // exchange area of the final merge (the ring is idle by then)
  uint32_t* sMask = reinterpret_cast<uint32_t*>(sKV + AT_STAGES * AT_STAGE_BYTES);   // AT_STAGES x [4][128] words
  uint8_t* sLive = reinterpret_cast<uint8_t*>(sMask) + AT_STAGES * AT_MASK_BYTES;    // this CTA's live-tile flags
  uint64_t* bars = reinterpret_cast<uint64_t*>(sLive + AT_MAX_TILES);
  uint64_t* kv_full = bars;                 // [AT_STAGES] K/V/R bytes landed and the stage's mask words stored
  uint64_t* kv_empty = kv_full + AT_STAGES;
  uint64_t* step = kv_empty + AT_STAGES;    // [3] commit n of step[b]: S(3n+b) ready and (n > 0) P.V(3(n-1)+b) done
  uint64_t* p_full = step + 3;              // [3] P tile written (512 arrivals)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(p_full + 3);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int h = blockIdx.x % p.heads, qt = blockIdx.x / p.heads, b = blockIdx.y;
  const uint8_t* live = sLive;
  const int C = p.heads * 32;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmK);
    ptx::prefetch_tmap(&tmV);
    if (p.has_r) ptx::prefetch_tmap(&tmR);
    for (int i = 0; i < AT_STAGES; ++i) { ptx::mbar_init(&kv_full[i], 32); ptx::mbar_init(&kv_empty[i], 1); }
    for (int i = 0; i < 3; ++i) { ptx::mbar_init(&step[i], 1); ptx::mbar_init(&p_full[i], 512); }
    ptx::fence_mbar_init();
  }
  if (warp == 1) {
    ptx::tmem_alloc(tmem_slot, 512);
    ptx::tmem_relinquish();
  }
  // barrier init / TMEM allocation above overlapped the previous kernel's tail
  ptx::grid_dep_launch();
  ptx::grid_dep_wait();
  {
    const uint8_t* src = p.live ? p.live + ((long)b * p.nqt + qt) * p.ntiles : nullptr;
    for (int t = threadIdx.x; t < p.ntiles; t += AT_THREADS) sLive[t] = src ? src[t] : 1;
  }
  if (warp >= 2 && warp < 6) {
    // Q tile -> bf16, core-matrix (no-swizzle) K-major layout: element (row, d) at
    // (row/8)*512 + (d/8)*128 + (row%8)*16 + (d%8)*2
    const int row = (warp & 3) * 32 + lane, qi = qt * 128 + row;
    float qv[32];
    if (qi < p.Q) {
      const float4* src = reinterpret_cast<const float4*>(p.q + ((long)b * p.Q + qi) * C + h * 32);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float4 x = __ldg(src + i);
        qv[4 * i] = x.x; qv[4 * i + 1] = x.y; qv[4 * i + 2] = x.z; qv[4 * i + 3] = x.w;
      }
    } else {
#pragma unroll
      for (int i = 0; i < 32; ++i) qv[i] = 0.f;
    }
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      uint4 pk;
      uint32_t* w = reinterpret_cast<uint32_t*>(&pk);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        __nv_bfloat162 v2 = __floats2bfloat162_rn(qv[8 * c + 2 * j], qv[8 * c + 2 * j + 1]);
        w[j] = *reinterpret_cast<uint32_t*>(&v2);
      }
      *reinterpret_cast<uint4*>(sQ + (row >> 3) * 512 + c * 128 + (row & 7) * 16) = pk;
    }
    ptx::fence_proxy_async_smem();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tmem_S = tmem_base;          // 3 x 128 columns (fp32 scores); P(j) overwrites the first 16 columns of each
                                              // key quarter of S(j) (a thread only overwrites scores it has already read)
  const uint32_t tmem_O = tmem_base + 384;    // 4 key quarters x 32 columns

  if (warp == 0) {
    // ------------- producer: lane 0 issues the TMA loads of K, V, R; every lane copies the mask words of query rows
    // lane, lane + 32, lane + 64, lane + 96.  A row >= Q, a fallback row or a call without a bitmap masks only the
    // keys >= K, like every row.
    const uint32_t* brow[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int qi = qt * 128 + lane + 32 * i;
      const bool use = p.bitmap && qi < p.Q && !(p.all_masked && p.all_masked[(long)b * p.Q + qi]);
      brow[i] = use ? p.bitmap + ((long)b * p.Q + qi) * p.W32 : nullptr;
    }
    const bool vec = (p.W32 & 3) == 0 && (reinterpret_cast<uintptr_t>(p.bitmap) & 15) == 0;   // a tile's 4 words = one uint4
    const uint32_t tx_bytes = (p.has_r ? (p.has_r > 1 ? 4 : 3) : 2) * AT_KV_TILE_BYTES;
    int it = 0;
    for (int t = next_live(live, 0, p.ntiles); t < p.ntiles; t = next_live(live, t + 1, p.ntiles), ++it) {
      const int s = it % AT_STAGES;
      // stage s was last used by live tile it-AT_STAGES: a softmax thread releases it once that tile's P V has completed
      ptx::mbar_wait(&kv_empty[s], ((uint32_t)(it / AT_STAGES) & 1u) ^ 1u);
      if (lane == 0) {
        mbar_expect_tx_only(&kv_full[s], tx_bytes);
        uint8_t* st = sKV + s * AT_STAGE_BYTES;
        if (p.has_r) {
          ptx::tma_load_2d(st + 2 * AT_KV_TILE_BYTES, &tmR, &kv_full[s], p.r_col0 + h * 32, t * AT_KT);
          if (p.has_r > 1) ptx::tma_load_2d(st + 3 * AT_KV_TILE_BYTES, &tmR, &kv_full[s], p.r_lo_off + p.r_col0 + h * 32, t * AT_KT);
        }
        ptx::tma_load_3d(st, &tmK, &kv_full[s], h * 32, t * AT_KT, b);
        ptx::tma_load_3d(st + AT_KV_TILE_BYTES, &tmV, &kv_full[s], h * 32, t * AT_KT, b);
      }
      uint32_t w[4][4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        if (brow[i] && vec) {
          const uint4 x = __ldg(reinterpret_cast<const uint4*>(brow[i] + t * 4));
          w[i][0] = x.x; w[i][1] = x.y; w[i][2] = x.z; w[i][3] = x.w;
        } else {
#pragma unroll
          for (int c = 0; c < 4; ++c) w[i][c] = (brow[i] && t * 4 + c < p.W32) ? __ldg(brow[i] + t * 4 + c) : 0u;
        }
      }
      uint32_t* sm = sMask + s * (AT_MASK_BYTES / 4);
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const int k0 = t * AT_KT + c * 32;
        const uint32_t tail = (k0 + 32 <= p.K) ? 0u : (k0 >= p.K) ? 0xffffffffu : ~((1u << (p.K - k0)) - 1u);
#pragma unroll
        for (int i = 0; i < 4; ++i) sm[c * 128 + lane + 32 * i] = w[i][c] | tail;
      }
      ptx::mbar_arrive(&kv_full[s]);
    }
  } else if (warp == 1) {
    // ------------- MMA issuer: the whole warp walks the loop (uniform control flow), one elected lane issues
    const uint32_t idesc_s = ptx::umma_idesc_bf16(128, AT_KT, false, false);   // S = Q K^T
    const uint32_t idesc_o = ptx::umma_idesc_bf16(128, 32, false, true);       // O = P V (A from TMEM, N-major B)
    int n_live = 0;
    for (int t = 0; t < p.ntiles; ++t) n_live += live[t] ? 1 : 0;
    // descriptors: base + constant increments of the 14-bit address field (16-byte units); the smem window is
    // < 256 KB so the field never carries
    const uint64_t qd0 = ptx::umma_desc(ptx::smem_u32(sQ), 128, 512, ptx::UMMA_INTERLEAVE);             // Q: core matrices
    const uint64_t kd0 = ptx::umma_desc(ptx::smem_u32(sKV), 16, 512, ptx::UMMA_SW64);                   // K / R tiles, K-major
    const uint64_t vd0 = ptx::umma_desc(ptx::smem_u32(sKV + AT_KV_TILE_BYTES), 1024, 512, ptx::UMMA_SW64);  // V, N-major (one N group)
    auto wait_kv = [&](int j) {
      ptx::mbar_wait(&kv_full[j % AT_STAGES], (uint32_t)(j / AT_STAGES) & 1u);
      ptx::tc_fence_after();
    };
    auto issue_qk = [&](int j) {                // elected lane only
      const uint64_t kd = kd0 + (uint64_t)((j % AT_STAGES) * (AT_STAGE_BYTES >> 4));
      const uint32_t d = tmem_S + (uint32_t)((j % 3) * 128);
#pragma unroll
      for (int k = 0; k < 2; ++k) ptx::mma_bf16_ss(d, qd0 + (uint64_t)(k * 16), kd + (uint64_t)(k * 2), idesc_s, k);
      if (p.has_r) {
        // + Q R^T: positional / level / bias part of the keys, a batch-independent table that the K/V
        // projection therefore never has to add (K = Wk x + R  =>  q.K = q.(Wk x) + q.R)
        // (R is kept as a bf16 hi/lo pair so that the table itself carries no bf16 rounding)
#pragma unroll
        for (int k = 0; k < 4; ++k)
          if (k < 2 || p.has_r > 1)      // has_r == 1: hi part of the table only
            ptx::mma_bf16_ss(d, qd0 + (uint64_t)((k & 1) * 16),
                             kd + (uint64_t)((((2 + (k >> 1)) * AT_KV_TILE_BYTES) >> 4) + (k & 1) * 2), idesc_s, 1u);
      }
    };
    for (int j = 0; j < 3 && j < n_live; ++j) {
      wait_kv(j);
      if (ptx::elect_one()) { issue_qk(j); ptx::mma_commit(&step[j]); }
      __syncwarp();
    }
    for (int j = 0; j < n_live; ++j) {
      const int s = j % AT_STAGES;
      ptx::mbar_wait(&p_full[j % 3], (uint32_t)(j / 3) & 1u);
      if (j + 3 < n_live) wait_kv(j + 3);
      ptx::tc_fence_after();
      if (ptx::elect_one()) {
        const uint64_t vd = vd0 + (uint64_t)(s * (AT_STAGE_BYTES >> 4));
        const uint32_t pa = tmem_S + (uint32_t)((j % 3) * 128);
#pragma unroll
        for (int cq = 0; cq < 4; ++cq) {
          // O_quarter += P[:, 32 keys of this quarter] . V[those keys, :]   (two K-steps of 16 keys = 8 TMEM columns)
#pragma unroll
          for (int k = 0; k < 2; ++k)
            mma_bf16_ts(tmem_O + (uint32_t)(cq * 32), pa + (uint32_t)(cq * 32 + k * 8),
                        vd + (uint64_t)((cq * 2048 + k * 1024) >> 4), idesc_o, (j > 0 || k > 0) ? 1u : 0u);
        }
        // S(j) has been consumed and P(j) is read by the P.V MMAs just issued (same thread: executed in order), so
        // the buffer takes Q K^T of tile j+3 right behind them
        if (j + 3 < n_live) issue_qk(j + 3);
        ptx::mma_commit(&step[j % 3]);
      }
      __syncwarp();
    }
  } else {
    // ------------- softmax: thread = query row x key quarter cq of every tile
    const int quarter = warp & 3;
    const int cq = (warp - 2) >> 2;
    const int row = quarter * 32 + lane, qi = qt * 128 + row;
    const bool row_ok = qi < p.Q;
    const uint32_t lane_off = (uint32_t)(quarter * 32) << 16;
    const uint32_t taddr_o = tmem_O + (uint32_t)(cq * 32) + lane_off;
    const uint32_t* mrow = sMask + cq * 128 + row;
    float m_ref = -INFINITY, l_run = 0.f;       // m_ref in log2 units (score * LOG2E)
    int it = 0;
    for (int t = next_live(live, 0, p.ntiles); t < p.ntiles; ++it) {
      const int buf = it % 3, s = it % AT_STAGES;
      const int t_next = next_live(live, t + 1, p.ntiles);
      ptx::mbar_wait(&kv_full[s], (uint32_t)(it / AT_STAGES) & 1u);     // this tile's mask words are in the stage
      const uint32_t mw = mrow[s * (AT_MASK_BYTES / 4)];
      ptx::mbar_wait(&step[buf], (uint32_t)(it / 3) & 1u);               // S(it) ready (and P.V(it-3) done)
      ptx::tc_fence_after();
      uint32_t sv[32];
      tmem_ld32_issue(tmem_S + (uint32_t)(buf * 128 + cq * 32) + lane_off, sv);
      tmem_ld32_wait(sv);
      float v[32];
#pragma unroll
      for (int i = 0; i < 32; ++i) v[i] = ((mw >> i) & 1u) ? -INFINITY : __uint_as_float(sv[i]);
      // tile maximum as a tree (short dependency chains)
      float mt[16];
#pragma unroll
      for (int i = 0; i < 16; ++i) mt[i] = fmaxf(v[i], v[i + 16]);
#pragma unroll
      for (int n = 8; n > 0; n >>= 1)
#pragma unroll
        for (int i = 0; i < n; ++i) mt[i] = fmaxf(mt[i], mt[i + n]);
      const float mx = mt[0] * LOG2E;
      // lazy rescale: move the reference only when the tile maximum exceeds it by more than 2^TAU
      const bool move = mx > m_ref + AT_TAU;      // (false for mx = -inf; true for m_ref = -inf and finite mx)
      const bool fix = move && m_ref != -INFINITY;                  // something has been accumulated at the old reference
      if (__any_sync(0xffffffffu, fix)) {
        // P.V(it-1) accumulates into the same O tile: it must have completed before the row is rescaled in place
        ptx::mbar_wait(&step[(it - 1) % 3], (uint32_t)(((it - 1) / 3) + 1) & 1u);
        ptx::tc_fence_after();
        const float sc = fix ? fast_exp2(m_ref - mx) : 1.f;
#pragma unroll
        for (int hf = 0; hf < 2; ++hf) {      // in halves: the scores of this tile stay in registers meanwhile
          float ov[16];
          uint32_t ou[16];
          ptx::tmem_ld16(taddr_o + (uint32_t)(hf * 16), ov);
#pragma unroll
          for (int i = 0; i < 16; ++i) ou[i] = __float_as_uint(ov[i] * sc);
          tmem_st16_issue(taddr_o + (uint32_t)(hf * 16), ou);
          tmem_st16_wait(ou);
        }
        l_run *= sc;
      }
      if (move) m_ref = mx;
      const float mneg = (m_ref == -INFINITY) ? 0.f : -m_ref;
      // p = exp2(s * log2e - m_ref) as bf16 pairs straight into the TMEM P tile of this buffer; the row sum adds the
      // fp32 values as a tree of packed pairs
      uint32_t pk[16];
      float2 e[16];
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        e[j] = fma2(make_float2(v[2 * j], v[2 * j + 1]), make_float2(LOG2E, LOG2E), make_float2(mneg, mneg));
        e[j].x = fast_exp2(e[j].x);
        e[j].y = fast_exp2(e[j].y);
        __nv_bfloat162 v2 = __floats2bfloat162_rn(e[j].x, e[j].y);
        pk[j] = *reinterpret_cast<uint32_t*>(&v2);
      }
      tmem_st16_issue(tmem_S + (uint32_t)(buf * 128 + cq * 32) + lane_off, pk);
#pragma unroll
      for (int n = 8; n > 0; n >>= 1)
#pragma unroll
        for (int j = 0; j < n; ++j) e[j] = add2(e[j], e[j + n]);
      l_run += e[0].x + e[0].y;
      tmem_st16_wait(pk);
      ptx::tc_fence_before();
      ptx::mbar_arrive(&p_full[buf]);
      // hand the previous tile's K/V stage back once its P.V has completed (long done by now)
      if (it > 0 && warp == 2) {
        ptx::mbar_wait(&step[(it - 1) % 3], (uint32_t)(((it - 1) / 3) + 1) & 1u);
        if (lane == 0) ptx::mbar_arrive(&kv_empty[(it - 1) % AT_STAGES]);
      }
      t = t_next;
    }
    float o[32];
    if (it > 0) {
      ptx::mbar_wait(&step[(it - 1) % 3], (uint32_t)(((it - 1) / 3) + 1) & 1u);      // the last P.V
      ptx::tc_fence_after();
      tmem_ld32(taddr_o, o);
    } else {
#pragma unroll
      for (int i = 0; i < 32; ++i) o[i] = 0.f;
    }
    // merge the four key quarters of the row: quarters 1..3 publish (m, l, o) through shared memory (the K/V ring:
    // every tile has been consumed once all 512 threads have seen the last commit)
    asm volatile("bar.sync 1, 512;" ::: "memory");
    float* xch = reinterpret_cast<float*>(sX);
    if (cq > 0) {
      float* dst = xch + ((cq - 1) * 128 + row) * 35;
      dst[0] = m_ref;
      dst[1] = l_run;
#pragma unroll
      for (int i = 0; i < 32; ++i) dst[2 + i] = o[i];
    }
    asm volatile("bar.sync 1, 512;" ::: "memory");
    if (cq == 0) {
      float m = m_ref;
#pragma unroll
      for (int c2 = 0; c2 < 3; ++c2) m = fmaxf(m, xch[(c2 * 128 + row) * 35]);
      const float a0 = (m_ref == -INFINITY) ? 0.f : fast_exp2(m_ref - m);
      l_run *= a0;
#pragma unroll
      for (int i = 0; i < 32; ++i) o[i] = (m_ref == -INFINITY) ? 0.f : o[i] * a0;
#pragma unroll
      for (int c2 = 0; c2 < 3; ++c2) {
        const float* src = xch + (c2 * 128 + row) * 35;
        const float m1 = src[0];
        if (m1 != -INFINITY) {           // (a quarter that never saw an unmasked key holds zeros / nothing useful)
          const float a1 = fast_exp2(m1 - m);
          l_run += src[1] * a1;
#pragma unroll
          for (int i = 0; i < 32; ++i) o[i] += src[2 + i] * a1;
        }
      }
      // (image, head and row recomputed from the block index rather than kept live across the tile loop)
      if (row_ok)
        store_attn_out(p, blockIdx.y, (blockIdx.x / p.heads) * 128 + row, blockIdx.x % p.heads, p.heads * 32, o,
                       l_run > 0.f ? 1.0f / l_run : 0.f);
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    ptx::tmem_dealloc(tmem_base, 512);
  }
}

int make_map_kv(TcState* t, CUtensorMap* m, const void* base, int K, long kv_stride, long kv_bstride, int B, int C) {
  if ((kv_stride * 2) % 16 != 0 || (kv_bstride * 2) % 16 != 0 || (reinterpret_cast<uintptr_t>(base) & 15))
    return tc_fail(t, CGG_ERR_UNSUPPORTED, "K/V rows must be 16-byte aligned");
  const cuuint64_t dims[3] = {(cuuint64_t)C, (cuuint64_t)K, (cuuint64_t)B};
  const cuuint64_t strides[2] = {(cuuint64_t)kv_stride * 2, (cuuint64_t)kv_bstride * 2};
  const cuuint32_t box[3] = {32, AT_KT, 1};
  if (!encode_tensor_map(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, base, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_64B,
                         CU_TENSOR_MAP_L2_PROMOTION_L2_128B, "KV", &t->err))
    return CGG_ERR_CUDA;
  return CGG_OK;
}

}  // namespace

cudaError_t tc_attention_setup() {
  return cudaFuncSetAttribute(masked_attention_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)AT_SMEM);
}

int tc_attention(TcState* t, int batch, int num_keys, const float* q, const void* k, const void* v, long kv_stride,
                 long kv_bstride, const uint32_t* bitmap, const uint8_t* all_masked, float* out, __nv_bfloat16* out_bf16,
                 cudaStream_t s, const void* r_table, long r_cols, int r_col0, int out_mode) {
  // r_table: (num_keys, r_cols) bf16 with columns [hi (r_cols/2) | lo (r_cols/2)]
  const int Q = t->cfg.num_queries, heads = t->cfg.num_heads, C = t->cfg.embed_dim;
  const int ntiles = (num_keys + AT_KT - 1) / AT_KT, nqt = (Q + 127) / 128;
  if (ntiles > AT_MAX_TILES) return tc_fail(t, CGG_ERR_BAD_SHAPE, "more than 512 key tiles");
  CUtensorMap mK, mV;
  int st = make_map_kv(t, &mK, k, num_keys, kv_stride, kv_bstride, batch, C);
  if (st != CGG_OK) return st;
  st = make_map_kv(t, &mV, v, num_keys, kv_stride, kv_bstride, batch, C);
  if (st != CGG_OK) return st;
  CUtensorMap mR = mK;
  if (r_table) {
    const cuuint64_t dims[2] = {(cuuint64_t)r_cols, (cuuint64_t)num_keys};
    const cuuint64_t strides[1] = {(cuuint64_t)r_cols * 2};
    const cuuint32_t box[2] = {32, AT_KT};
    if (!encode_tensor_map(&mR, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, r_table, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_64B,
                           CU_TENSOR_MAP_L2_PROMOTION_L2_128B, "R", &t->err))
      return CGG_ERR_CUDA;
  }
  const int W32 = (num_keys + 31) / 32;
  AttnP p;
  p.q = q; p.out = out; p.out_bf16 = out_bf16; p.bitmap = bitmap; p.all_masked = all_masked; p.live = nullptr;
  p.Q = Q; p.K = num_keys; p.heads = heads; p.W32 = W32; p.ntiles = ntiles; p.nqt = nqt;
  p.has_r = r_table ? 2 : 0;      // hi + lo halves of the key-bias table
  p.r_col0 = r_col0; p.r_lo_off = (int)(r_cols / 2);
  p.out_hl = out_mode;
  if (bitmap) {
    // live-tile flags of this bitmap, once per (image, query tile); the handle's attention calls run in stream order
    if ((size_t)batch * nqt * ntiles > t->live_bytes) return tc_fail(t, CGG_ERR_BAD_SHAPE, "live-tile flags exceed their buffer");
    TCU(launch_pdl(attention_live_kernel, dim3(nqt, batch), dim3(512), 0, s, bitmap, all_masked, Q, num_keys, W32, ntiles,
                   nqt, t->live_buf));
    count_launch();
    TCU(cudaGetLastError());
    p.live = t->live_buf;
  }
  TCU(launch_pdl(masked_attention_tc_kernel, dim3(heads * nqt, batch), dim3(AT_THREADS), AT_SMEM, s, mK, mV, mR, p));
  count_launch();
  TCU(cudaGetLastError());
  return CGG_OK;
}

}  // namespace cgg

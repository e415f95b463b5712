// Training-step contractions on tcgen05 tensor cores, straight from the fp32 tensors autograd hands over.
//
//   C[b,m,n] = epi( sum_k A[b,m,k] * W[b,n,k] )      (the GemmF32 contract of kernels.h, A2 excluded)
//
// kind::tf32 MMAs read fp32 words from shared memory and use their upper 19 bits (10-bit mantissa), fp32 accumulate in
// TMEM: no cast pass, no transposed copy.  Either operand may be K-major (k contiguous: activations x weights) or
// MN-major (m / n contiguous: the NCHW feature map of the mask einsum, the transposed operands of every dX / dW
// product) -- TMA delivers 128-byte-swizzled tiles of both kinds from the strided tensor and the operand-major bits of
// the instruction descriptor do the transposition.  (32-bit MN-major operands exist in one shared-memory layout only:
// the 128-byte swizzle with 32-byte atoms, 4 k-rows per swizzle period -- CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B on the
// TMA side, layout type 1 in the matrix descriptor.)  Shapes whose strides TMA cannot describe (row pitch not a multiple
// of 16 bytes: the 118-class rows) are reported as ineligible and run on the SIMT kernel.
//
// Persistent CTAs (one per SM) walk the (128 x n_tile) output tiles, n fastest (CTAs running side by side share an A tile
// through L2): warp 0 = TMA producer, warp 1 = MMA issuer, warps 2-5 = epilogue (one TMEM lane quarter each); two TMEM
// accumulators, so the epilogue of one tile overlaps the main loop of the next.  Products with few output tiles and a long
// contraction (dW of the K/V projections, d mask_embed of the mask einsum: K = 65 536) are split over K into a dense fp32
// partial buffer and summed, in a fixed order, by splitk_reduce_kernel, which also applies the epilogue.
//
// Epilogue forms (chosen per launch): row-major C without a residual goes through a per-warp XOR-swizzled shared-memory
// tile and leaves as whole 128-byte lines; with a residual / C += the thread keeps its accumulator row and the residual of
// the next 32-column chunk is requested one chunk ahead (the first before the accumulator barrier); m-contiguous C (NCHW
// outputs, the mask einsum) writes one line per column, with an optional bias; the tile's bias lives in a per-warp
// shared-memory row.  conv_cin turns the A loads into the nine taps of a 3x3 convolution over a token-major image (the TMA
// unit's out-of-bounds zero fill is the padding); a weight matrix shared by every batch entry is a tensor map without
// batch dimensions.
#include "common.cuh"
#include "tc_ptx.cuh"
#include "kernels.h"
#include "gemm_tf32.h"

#include <string>

namespace cgg {
namespace {

constexpr int BM = 128, BK = 32;                       // BK fp32 = one 128-byte swizzle row
constexpr int A_STAGE_BYTES = BM * BK * 4;             // 16 KB
// epilogue warps: 4 = one per TMEM lane quarter; 8 = two per quarter taking alternate 32-column chunks of a tile.  Measured
// with 8 (344 k-row products of the pixel decoder): residual products 0.41 -> 0.34 ms, but the FFN1 product 0.54 -> 0.75 ms
// (three TMA stages instead of four: the staging tiles take the shared memory; 168 registers with spills) and the
// training step 17.5 -> 18.9 ms -- so 4 it stays.
constexpr int EPI_WARPS = 4;
constexpr int THREADS = 64 + 32 * EPI_WARPS;
constexpr int EPI_STEP = 32 * (EPI_WARPS / 4);

struct Tf32P {
  int M, N, K, batch;
  int a_mn, b_mn;              // 1: operand is MN-major
  int n_tile;                  // UMMA N (multiple of 16, <= 256)
  int b_groups;                // MN-major B: 32-column groups loaded per stage
  int stages;
  int chunks, chunks_per_split, splits;
  int mt, nt;                  // output tiles along m / n
  int tmem_cols;               // 2 accumulators of tmem_cols / 2 columns
  int batch_inner;             // z -> (z / batch_inner, z % batch_inner): TMA coordinates 3 / 2, C offsets sCb / sCb2
  float* C; long sCb, sCb2, sCm, sCn;
  const float* bias; float alpha;
  const float* R; long sRb, sRm, sRn; int r_mod, r_ncols;
  int relu_from;
  float* partial;              // != nullptr: raw accumulators to partial[((split*batch + b)*M + m)*N + n]
  int epi_mode;                // 1: float4 rows, 2: m-contiguous C, 0: scalar
  int accumulate;              // C += result
  int conv_cpt;                // > 0: implicit 3x3 convolution, 32-channel chunks per tap (GemmF32::conv_cin / 32)
  int w_shared;                // the W operand has no batch stride (one weight matrix for every batch entry)
};

// kind::tf32 instruction descriptor: c_format F32 (1) at [4,6), a/b format TF32 (2) at [7,10)/[10,13), operand majors at
// 15 / 16 (1 = MN-major), N>>3 at [17,23), M>>4 at [24,29)  (cute::UMMA::InstrDescriptor).
__host__ __device__ constexpr uint32_t umma_idesc_tf32(int M, int N, bool a_mn, bool b_mn) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((a_mn ? 1u : 0u) << 15) | ((b_mn ? 1u : 0u) << 16) |
         ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

__device__ __forceinline__ float epi_value(const Tf32P& p, float acc, int b, int gm, int gn) {
  float v = acc;
  if (p.bias) v += p.bias[gn];
  v *= p.alpha;
  if (p.R && gn < p.r_ncols) v += p.R[(long)b * p.sRb + (long)(gm % p.r_mod) * p.sRm + (long)gn * p.sRn];
  if (gn >= p.relu_from) v = fmaxf(v, 0.f);
  return v;
}

__global__ void __launch_bounds__(THREADS) gemm_tf32_kernel(const __grid_constant__ CUtensorMap mA,
                                                        const __grid_constant__ CUtensorMap mB, const Tf32P p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int b_stage_bytes = (p.b_mn ? p.b_groups * 32 : p.n_tile) * BK * 4;
  const int stage_bytes = A_STAGE_BYTES + ((b_stage_bytes + 1023) & ~1023);
  __shared__ uint64_t full[4], empty[4], acc_full[2], acc_empty[2];
  __shared__ uint32_t tmem_slot;
  __shared__ __align__(16) float bias_s[EPI_WARPS][256];     // per epilogue warp: the bias of the current tile's columns
  __shared__ __align__(16) float stage_s[EPI_WARPS][1024];   // per epilogue warp: a 32 x 32 chunk on its way from row-per-thread to coalesced rows

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int acc_cols = p.tmem_cols >> 1;                 // two accumulators: the epilogue of tile i overlaps tile i + 1

  if (threadIdx.x == 0) {
    for (int i = 0; i < p.stages; ++i) { ptx::mbar_init(&full[i], 1); ptx::mbar_init(&empty[i], 1); }
    for (int i = 0; i < 2; ++i) { ptx::mbar_init(&acc_full[i], 1); ptx::mbar_init(&acc_empty[i], EPI_WARPS); }
    ptx::fence_mbar_init();
    ptx::prefetch_tmap(&mA);
    ptx::prefetch_tmap(&mB);
  }
  if (warp == 2) { ptx::tmem_alloc(&tmem_slot, (uint32_t)p.tmem_cols); ptx::tmem_relinquish(); }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem = tmem_slot;

  // persistent tile loop (all three roles walk the same sequence): tile -> (n tile fastest, m tile, batch, K split): the
  // CTAs that run side by side share one A tile (fetched from HBM once, re-read through L2) and the weights stay in L2
  const long tiles = (long)p.mt * p.nt * p.batch * p.splits;
  auto decode = [&](long t, int& m0, int& n0, int& b, int& split) {
    n0 = (int)(t % p.nt) * p.n_tile; t /= p.nt;
    m0 = (int)(t % p.mt) * BM; t /= p.mt;
    split = (int)(t % p.splits);
    b = (int)(t / p.splits);
  };

  if (warp == 0) {
    if (ptx::elect_one()) {
      const uint32_t tx = (uint32_t)(A_STAGE_BYTES + b_stage_bytes);
      uint32_t it = 0;
      for (long t = blockIdx.x; t < tiles; t += gridDim.x) {
        int m0, n0, b, split;
        decode(t, m0, n0, b, split);
        const int c0 = split * p.chunks_per_split, c1 = min(p.chunks, c0 + p.chunks_per_split);
        for (int c = c0; c < c1; ++c, ++it) {
          const int st = (int)(it % (uint32_t)p.stages);
          ptx::mbar_wait(&empty[st], ((it / (uint32_t)p.stages) & 1u) ^ 1u);
          uint8_t* sA = smem + (size_t)st * stage_bytes;
          uint8_t* sB = sA + A_STAGE_BYTES;
          ptx::mbar_expect_tx(&full[st], tx);
          const int bi = b % p.batch_inner, bo = b / p.batch_inner;
          if (p.conv_cpt > 0) {        // tap (dy, dx) of the 3x3 window: the TMA unit zero-fills rows / columns outside the image
            const int tap = c / p.conv_cpt;
            ptx::tma_load_4d(sA, &mA, &full[st], (c - tap * p.conv_cpt) * BK, m0 + tap % 3 - 1, bi + tap / 3 - 1, bo);
          } else if (!p.a_mn) ptx::tma_load_4d(sA, &mA, &full[st], c * BK, m0, bi, bo);                // (32 k, 128 rows)
          else
            for (int g = 0; g < 4; ++g) ptx::tma_load_4d(sA + g * 4096, &mA, &full[st], m0 + g * 32, c * BK, bi, bo);   // (32 m, 32 k)
          const int wbi = p.w_shared ? 0 : bi, wbo = p.w_shared ? 0 : bo;
          if (!p.b_mn) ptx::tma_load_4d(sB, &mB, &full[st], c * BK, n0, wbi, wbo);
          else
            for (int g = 0; g < p.b_groups; ++g) ptx::tma_load_4d(sB + g * 4096, &mB, &full[st], n0 + g * 32, c * BK, wbi, wbo);
        }
      }
    }
  } else if (warp == 1) {
    if (ptx::elect_one()) {
      const uint32_t idesc = umma_idesc_tf32(BM, p.n_tile, p.a_mn != 0, p.b_mn != 0);
      // K-major SW128: 8 tf32 = 32 B along the swizzled row per MMA, 8-row groups 1 KB apart (SBO).
      // MN-major SW128/32B-atom: 8 k-rows of 128 B = 1 KB per MMA; 32-wide m/n groups 4 KB apart (LBO), 4-row swizzle
      // periods 512 B apart (SBO).
      const uint32_t a_step = p.a_mn ? (1024u >> 4) : (32u >> 4);
      const uint32_t b_step = p.b_mn ? (1024u >> 4) : (32u >> 4);
      uint32_t it = 0, lt = 0;
      for (long t = blockIdx.x; t < tiles; t += gridDim.x, ++lt) {
        int m0, n0, b, split;
        decode(t, m0, n0, b, split);
        const int c0 = split * p.chunks_per_split, c1 = min(p.chunks, c0 + p.chunks_per_split);
        const uint32_t buf = lt & 1u;
        ptx::mbar_wait(&acc_empty[buf], ((lt >> 1) & 1u) ^ 1u);
        ptx::tc_fence_after();
        const uint32_t d_tmem = tmem + buf * (uint32_t)acc_cols;
        for (int c = c0; c < c1; ++c, ++it) {
          const int st = (int)(it % (uint32_t)p.stages);
          ptx::mbar_wait(&full[st], (it / (uint32_t)p.stages) & 1u);
          ptx::tc_fence_after();
          const uint32_t sA = ptx::smem_u32(smem + (size_t)st * stage_bytes);
          const uint64_t ad = p.a_mn ? ptx::umma_desc(sA, 4096, 512, ptx::UMMA_SW128_BASE32B)
                                     : ptx::umma_desc(sA, 16, 1024, ptx::UMMA_SW128);
          const uint64_t bd = p.b_mn ? ptx::umma_desc(sA + A_STAGE_BYTES, 4096, 512, ptx::UMMA_SW128_BASE32B)
                                     : ptx::umma_desc(sA + A_STAGE_BYTES, 16, 1024, ptx::UMMA_SW128);
#pragma unroll
          for (int kk = 0; kk < BK / 8; ++kk)
            ptx::mma_tf32_ss(d_tmem, ad + (uint64_t)(kk * a_step), bd + (uint64_t)(kk * b_step), idesc, (c > c0 || kk > 0) ? 1u : 0u);
          ptx::mma_commit(&empty[st]);
        }
        ptx::mma_commit(&acc_full[buf]);
      }
    }
  } else {
    // ---- epilogue: warp w owns TMEM lanes [32 (w & 3), +32) = output rows m0 + 32 (w & 3) + lane.
    // A single warp per lane quarter walks the whole tile, so the instruction count per element is what bounds it:
    // mode 1 (row-major C, 16-byte aligned rows) writes float4s straight from the registers, mode 2 (m-contiguous C:
    // the mask einsum and d mask_features) writes one 128-byte line per column; mode 0 is the scalar catch-all.
    const int quarter = warp & 3, ew = warp - 2;
    const int j0 = (ew >> 2) * 32;                         // this warp's first chunk of a tile
    const float* __restrict__ bias = p.bias;
    const float* __restrict__ R = p.R;
    const bool plain = !p.partial && !bias && !R && p.alpha == 1.0f && p.relu_from >= p.N && !p.accumulate;
    const bool plain_acc = !p.partial && !bias && !R && p.alpha == 1.0f && p.relu_from >= p.N && p.accumulate;
    uint32_t lt = 0;
    for (long t = blockIdx.x; t < tiles; t += gridDim.x, ++lt) {
      int m0, n0, b, split;
      decode(t, m0, n0, b, split);
      const uint32_t buf = lt & 1u;
      const int gm = m0 + quarter * 32 + lane;
      const bool rowok = gm < p.M;
      float* crow = p.partial ? p.partial + (((long)split * p.batch + b) * p.M + gm) * p.N
                              : p.C + (long)(b / p.batch_inner) * p.sCb + (long)(b % p.batch_inner) * p.sCb2 + (long)gm * p.sCm;
      // Row-major C (mode 1).  Everything the epilogue reads from memory is requested BEFORE the accumulator is waited for:
      // the tile's bias goes to the warp's shared-memory row, the residual / old-C values of a 32-column chunk ride in
      // registers one chunk ahead (a serial load -> add -> store chain per chunk was the top stall of the first version).
      // A thread owns an accumulator ROW, so stores straight from the registers touch 32 different lines per instruction,
      // 16 bytes each.  Products WITHOUT a residual therefore send each 32 x 32 chunk through the warp's shared-memory tile
      // (float4 index XOR row: conflict-free both ways) and store whole 128-byte lines, 4 rows per instruction (measured on
      // the 344 k x 1024 x 256 FFN product: 0.68 -> 0.57 ms); with a residual the row-per-thread form is the faster one
      // (0.38 vs 0.43 ms on 344 k x 256 x 256 + residual) and is kept.
      const bool add = R || p.accumulate;
      const bool rich = p.epi_mode == 1 && !p.partial;
      const bool staged = rich && !add;
      const bool rich2 = p.epi_mode == 2 && !p.partial && !plain && !R && !p.accumulate;   // m-contiguous C with bias / alpha / relu
      const int rsub = lane >> 3, cq = lane & 7;
      const int gm0 = m0 + quarter * 32;                     // first row of this warp
      float* cbase = p.C + (long)(b / p.batch_inner) * p.sCb + (long)(b % p.batch_inner) * p.sCb2;
      const float* rrow = (R && !p.partial) ? R + (long)b * p.sRb + (long)(p.r_mod >= p.M ? gm : gm % p.r_mod) * p.sRm : nullptr;
      const int col_end = min(p.N, n0 + p.n_tile);
      auto prefetch = [&](float4* rv, int j) {
        const int nq = min(8, (col_end - (n0 + j)) >> 2);
#pragma unroll
        for (int c4 = 0; c4 < 8; ++c4) {
          rv[c4] = (rrow && rowok && c4 < nq && n0 + j < p.r_ncols) ? __ldg(reinterpret_cast<const float4*>(rrow + n0 + j) + c4)
                                                                    : make_float4(0.f, 0.f, 0.f, 0.f);
          if (p.accumulate && rowok && c4 < nq) {          // C += ...: the old values ride in the residual registers
            const float4 ov = reinterpret_cast<const float4*>(crow + n0 + j)[c4];
            rv[c4].x += ov.x; rv[c4].y += ov.y; rv[c4].z += ov.z; rv[c4].w += ov.w;
          }
        }
      };
      float4 va[8], vb[8];
      if (rich || rich2) {
        if (bias) {
          __syncwarp();
#pragma unroll
          for (int t = 0; t < 2; ++t) {
            const int c = lane * 4 + 128 * t;
            *reinterpret_cast<float4*>(&bias_s[ew][c]) =
                (c < p.n_tile && n0 + c < p.N) ? __ldg(reinterpret_cast<const float4*>(bias + n0 + c)) : make_float4(0.f, 0.f, 0.f, 0.f);
          }
          __syncwarp();
        }
        if (rich && add && j0 < p.n_tile) prefetch(va, j0);
      }
      ptx::mbar_wait(&acc_full[buf], (lt >> 1) & 1u);
      ptx::tc_fence_after();
      // The accumulator is read 32 columns at a time; the tcgen05.ld of the next chunk is in flight while the current
      // chunk's stores are issued (two register sets, loop unrolled by two so that both stay in registers).
      const uint32_t tbase = tmem + buf * (uint32_t)acc_cols + ((uint32_t)(quarter * 32) << 16);
      auto issue = [&](uint32_t* r, int j) {
        ptx::tmem_ld16_issue(tbase + (uint32_t)j, r);
        if (j + 16 < p.n_tile) ptx::tmem_ld16_issue(tbase + (uint32_t)j + 16, r + 16);
        else
#pragma unroll
          for (int i = 16; i < 32; ++i) r[i] = 0u;
      };
      auto waitr = [&](uint32_t* r) { ptx::tmem_ld_wait16(r); ptx::tmem_ld_wait16(r + 16); };
      auto process = [&](const uint32_t* r, const float4* rv, int j) {
        if (!rowok && !staged) return;                   // (the staged path is warp-collective)
        float v[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
          if (staged) {
            float* stg = stage_s[ew];
#pragma unroll
            for (int c4 = 0; c4 < 8; ++c4)
              *reinterpret_cast<float4*>(stg + lane * 32 + ((c4 ^ (lane & 7)) << 2)) =
                  make_float4(v[4 * c4], v[4 * c4 + 1], v[4 * c4 + 2], v[4 * c4 + 3]);
            __syncwarp();
            const int col = n0 + j + cq * 4;
            const bool colok = col < col_end;
            const float4 bv = bias ? *reinterpret_cast<const float4*>(&bias_s[ew][j + cq * 4]) : make_float4(0.f, 0.f, 0.f, 0.f);
            const bool relu = n0 + j >= p.relu_from;               // relu_from is a multiple of 32 here (0 or "never")
#pragma unroll
            for (int it = 0; it < 8; ++it) {
              const int rr = it * 4 + rsub;
              const float4 a = *reinterpret_cast<const float4*>(stg + rr * 32 + ((cq ^ (rr & 7)) << 2));
              float4 o;
              o.x = (a.x + bv.x) * p.alpha; o.y = (a.y + bv.y) * p.alpha; o.z = (a.z + bv.z) * p.alpha; o.w = (a.w + bv.w) * p.alpha;
              if (relu) { o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f); }
              if (colok && gm0 + rr < p.M) *reinterpret_cast<float4*>(cbase + (long)(gm0 + rr) * p.sCm + col) = o;
            }
            __syncwarp();
          } else if (rich) {                                 // with a residual / C +=: row per thread
            if (rowok) {
              const int nq = min(8, (col_end - (n0 + j)) >> 2);
              float4* dst = reinterpret_cast<float4*>(crow + n0 + j);
              float4 bv[8];
#pragma unroll
              for (int c4 = 0; c4 < 8; ++c4)
                bv[c4] = bias ? *reinterpret_cast<const float4*>(&bias_s[ew][j + 4 * c4]) : make_float4(0.f, 0.f, 0.f, 0.f);
              const bool relu = n0 + j >= p.relu_from;
#pragma unroll
              for (int c4 = 0; c4 < 8; ++c4) {
                float4 o;
                o.x = (v[4 * c4] + bv[c4].x) * p.alpha + rv[c4].x;
                o.y = (v[4 * c4 + 1] + bv[c4].y) * p.alpha + rv[c4].y;
                o.z = (v[4 * c4 + 2] + bv[c4].z) * p.alpha + rv[c4].z;
                o.w = (v[4 * c4 + 3] + bv[c4].w) * p.alpha + rv[c4].w;
                if (relu) { o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f); }
                if (c4 < nq) dst[c4] = o;
              }
            }
          } else if (p.epi_mode == 1) {                    // split-K partial sums: raw accumulator rows
            const int nq = min(8, min(p.N - (n0 + j), p.n_tile - j) >> 2);
            float4* dst = reinterpret_cast<float4*>(crow + n0 + j);
#pragma unroll
            for (int c4 = 0; c4 < 8; ++c4)
              if (c4 < nq) dst[c4] = make_float4(v[4 * c4], v[4 * c4 + 1], v[4 * c4 + 2], v[4 * c4 + 3]);
          } else if (p.epi_mode == 2 && plain) {
            float* cp = crow + (long)(n0 + j) * p.sCn;
            const int nc = min(32, min(p.N - (n0 + j), p.n_tile - j));
#pragma unroll
            for (int i = 0; i < 32; ++i) {
              if (i < nc) *cp = v[i];
              cp += p.sCn;
            }
          } else if (rich2) {                              // one 128-byte line per column; the column's bias is warp-uniform
            float* cp = crow + (long)(n0 + j) * p.sCn;
            const int nc = min(32, min(p.N - (n0 + j), p.n_tile - j));
            const bool relu = n0 + j >= p.relu_from;
#pragma unroll
            for (int i = 0; i < 32; ++i) {
              float o = (v[i] + (bias ? bias_s[ew][j + i] : 0.f)) * p.alpha;
              if (relu) o = fmaxf(o, 0.f);
              if (i < nc) *cp = o;
              cp += p.sCn;
            }
          } else if (p.epi_mode == 2 && plain_acc) {       // C += acc: the chunk's 32 old values are read before any store
            float* cp = crow + (long)(n0 + j) * p.sCn;
            const int nc = min(32, min(p.N - (n0 + j), p.n_tile - j));
            float old[32];
#pragma unroll
            for (int i = 0; i < 32; ++i) old[i] = (i < nc) ? cp[(long)i * p.sCn] : 0.f;
#pragma unroll
            for (int i = 0; i < 32; ++i)
              if (i < nc) cp[(long)i * p.sCn] = old[i] + v[i];
          } else {
#pragma unroll
            for (int i = 0; i < 32; ++i) {
              const int gn = n0 + j + i;
              if (gn < p.N) {
                if (p.partial) crow[gn] = v[i];
                else crow[(long)gn * p.sCn] = epi_value(p, v[i], b, gm, gn) + (p.accumulate ? crow[(long)gn * p.sCn] : 0.f);
              }
            }
          }
      };
      auto more_after = [&](int j) { return j + EPI_STEP < p.n_tile && n0 + j + EPI_STEP < p.N; };
      uint32_t ra[32], rb[32];
      int j = j0;
      if (j < p.n_tile && n0 + j < p.N) {
        issue(ra, j);
        waitr(ra);
        while (true) {
          bool more = more_after(j);
          if (more) { issue(rb, j + EPI_STEP); if (rich && add) prefetch(vb, j + EPI_STEP); }
          process(ra, va, j);
          if (!more) break;
          waitr(rb);
          j += EPI_STEP;
          more = more_after(j);
          if (more) { issue(ra, j + EPI_STEP); if (rich && add) prefetch(va, j + EPI_STEP); }
          process(rb, vb, j);
          if (!more) break;
          waitr(ra);
          j += EPI_STEP;
        }
      }
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&acc_empty[buf]);
    }
  }
  __syncthreads();
  if (warp == 2) { ptx::tc_fence_after(); ptx::tmem_dealloc(tmem, (uint32_t)p.tmem_cols); }
}

__global__ void __launch_bounds__(256) splitk_reduce_kernel(const Tf32P p) {
  const long per = (long)p.batch * p.M * p.N;
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= per) return;
  float acc = 0.f;
  for (int s = 0; s < p.splits; ++s) acc += p.partial[(long)s * per + i];
  const int gn = (int)(i % p.N);
  const long bm = i / p.N;
  const int gm = (int)(bm % p.M);
  const int b = (int)(bm / p.M);
  float* c = p.C + (long)(b / p.batch_inner) * p.sCb + (long)(b % p.batch_inner) * p.sCb2 + (long)gm * p.sCm + (long)gn * p.sCn;
  *c = epi_value(p, acc, b, gm, gn) + (p.accumulate ? *c : 0.f);
}

// operand X[b, r, k] with element strides (sb, sr, sk): 0 = K-major, 1 = MN-major, -1 = TMA cannot describe it
int operand_major(const float* base, long sb, long sb2, long sr, long sk, int rows, int K, int batch, int batch_inner) {
  if (reinterpret_cast<uintptr_t>(base) & 15) return -1;
  if (batch > batch_inner && (sb <= 0 || sb % 4 != 0)) return -1;
  if (batch_inner > 1 && (sb2 <= 0 || sb2 % 4 != 0)) return -1;
  if (sk == 1 && sr > 0 && sr % 4 == 0) return 0;
  if (sr == 1 && sk > 0 && sk % 4 == 0) return 1;
  if (sk == 1 && rows == 1) return 0;
  (void)K;
  return -1;
}

}  // namespace

struct Tf32Ctx {
  // split-K partial sums: one buffer per workspace slot (GemmF32::slot) -- products issued on two streams at once (the
  // weight-gradient products run on a side stream) must not share one
  float* partial[2] = {nullptr, nullptr};
  size_t partial_bytes[2] = {0, 0};
  int sm_count = 148;
  std::string err;
};

Tf32Ctx* tf32_create() {
  Tf32Ctx* t = new (std::nothrow) Tf32Ctx();
  if (!t) return nullptr;
  int dev = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&t->sm_count, cudaDevAttrMultiProcessorCount, dev);
  if (cudaFuncSetAttribute(gemm_tf32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                           227 * 1024 - (EPI_WARPS > 4 ? 44 : 24) * 1024) != cudaSuccess) {
    delete t;
    return nullptr;
  }
  return t;
}
void tf32_destroy(Tf32Ctx* t) {
  if (!t) return;
  for (int i = 0; i < 2; ++i) if (t->partial[i]) cudaFree(t->partial[i]);
  delete t;
}
const char* tf32_last_error(const Tf32Ctx* t) { return t ? t->err.c_str() : ""; }

static int make_map(Tf32Ctx* t, CUtensorMap* m, const float* base, int major, long sb, long sb2, long sr, long sk, int rows,
                    int K, int batch, int batch_inner, int box_rows) {
  cuuint64_t dims[4], strides[3];
  cuuint32_t box[4];
  if (major == 0) {      // K-major: (k, row, batch), box (32 k, box_rows rows)
    dims[0] = (cuuint64_t)K; dims[1] = (cuuint64_t)rows;
    strides[0] = (cuuint64_t)(rows > 1 ? sr : ((K + 3) & ~3)) * 4;
    box[0] = BK; box[1] = (cuuint32_t)box_rows;
  } else {               // MN-major: (row, k, batch), box (32 rows, 32 k)
    dims[0] = (cuuint64_t)rows; dims[1] = (cuuint64_t)K;
    strides[0] = (cuuint64_t)(K > 1 ? sk : ((rows + 3) & ~3)) * 4;
    box[0] = 32; box[1] = BK;
  }
  // (inner batch, outer batch); a stride is unused when its extent is 1, but must still be a valid stride
  const int outer = batch / batch_inner;
  dims[2] = (cuuint64_t)batch_inner; dims[3] = (cuuint64_t)outer;
  box[2] = box[3] = 1;
  strides[1] = batch_inner > 1 ? (cuuint64_t)sb2 * 4 : strides[0] * dims[1];
  strides[2] = outer > 1 ? (cuuint64_t)sb * 4 : strides[0] * dims[1];
  return encode_tensor_map(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, base, dims, strides, box,
                           major == 0 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B,
                           CU_TENSOR_MAP_L2_PROMOTION_L2_128B, "tf32 operand", &t->err) ? 0 : -1;
}

// 0 = launched, 1 = not eligible (caller runs the SIMT kernel), < 0 = error (tf32_last_error)
int launch_gemm_tf32(Tf32Ctx* t, const GemmF32& g, cudaStream_t s) {
  if (g.M <= 0 || g.N <= 0 || g.batch <= 0) return 0;
  if (g.A2 || g.K <= 0) return 1;
  if ((reinterpret_cast<uintptr_t>(g.C) & 3)) return 1;
  const int a_major = operand_major(g.A, g.sAb, g.sAb2, g.sAm, g.sAk, g.M, g.K, g.batch, g.batch_inner);
  const bool w_shared = g.batch > 1 && g.sWb == 0 && g.sWb2 == 0;
  const int b_major = w_shared ? operand_major(g.W, 0, 0, g.sWn, g.sWk, g.N, g.K, 1, 1)
                               : operand_major(g.W, g.sWb, g.sWb2, g.sWn, g.sWk, g.N, g.K, g.batch, g.batch_inner);
  if (a_major < 0 || b_major < 0) return 1;
  if (g.batch_inner > 1 && g.R) return 1;
  if (g.conv_cin > 0 && (a_major != 0 || g.conv_cin % BK != 0 || g.K != 9 * g.conv_cin)) return 1;
  Tf32P p = {};
  p.conv_cpt = g.conv_cin > 0 ? g.conv_cin / BK : 0;
  p.M = g.M; p.N = g.N; p.K = g.K; p.batch = g.batch;
  p.a_mn = a_major; p.b_mn = b_major;
  p.w_shared = w_shared ? 1 : 0;
  // N <= 256: one tile of the whole width; wider: the fewest tiles of <= 256 columns, evenly sized (544 -> 3 x 192, 288 -> 2 x 144)
  // (several column tiles: multiples of 32, the epilogue's chunk width, so that no chunk straddles two tiles)
  { const int nt0 = (g.N + 255) / 256; p.n_tile = round_up((g.N + nt0 - 1) / nt0, nt0 > 1 ? 32 : 16); }
  p.b_groups = (p.n_tile + 31) / 32;
  const int b_stage = ((p.b_mn ? p.b_groups * 32 : p.n_tile) * BK * 4 + 1023) & ~1023;
  const int stage_bytes = A_STAGE_BYTES + b_stage;
  p.stages = (EPI_WARPS > 4 && stage_bytes > 32 * 1024) ? 3 : 4;   // (with 8 epilogue warps 40 KB of static shared memory go to the staging tiles)
  p.tmem_cols = 2 * (p.n_tile <= 32 ? 32 : p.n_tile <= 64 ? 64 : p.n_tile <= 128 ? 128 : 256);
  p.chunks = (g.K + BK - 1) / BK;
  const long mt = (g.M + BM - 1) / BM, nt = (g.N + p.n_tile - 1) / p.n_tile;
  const long tiles = mt * nt * g.batch;
  int splits = 1;
  if (tiles * 2 <= t->sm_count && p.chunks >= 16) {
    const int want = (int)((t->sm_count + tiles - 1) / tiles);
    splits = want < p.chunks / 8 ? want : p.chunks / 8;
    if (splits < 1) splits = 1;
  }
  p.chunks_per_split = (p.chunks + splits - 1) / splits;
  p.splits = (p.chunks + p.chunks_per_split - 1) / p.chunks_per_split;
  if (mt * nt * g.batch * p.splits > 0x7fffffffL) return 1;
  p.mt = (int)mt; p.nt = (int)nt;
  p.batch_inner = g.batch_inner > 1 ? g.batch_inner : 1;
  p.C = g.C; p.sCb = g.sCb; p.sCb2 = g.sCb2; p.sCm = g.sCm; p.sCn = g.sCn;
  p.bias = g.bias; p.alpha = g.alpha;
  p.R = g.R; p.sRb = g.sRb; p.sRm = g.sRm; p.sRn = g.sRn; p.r_mod = g.r_mod > 0 ? g.r_mod : 1; p.r_ncols = g.r_ncols;
  p.relu_from = g.relu_from;
  p.accumulate = g.accumulate ? 1 : 0;
  if (p.splits > 1) {
    const size_t need = (size_t)p.splits * g.batch * g.M * g.N * sizeof(float);
    const int slot = g.slot ? 1 : 0;
    if (need > t->partial_bytes[slot]) {
      cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
      cudaStreamIsCapturing(s, &cs);
      if (cs != cudaStreamCaptureStatusNone) { t->err = "split-K buffer must be sized by an eager step before graph capture"; return -1; }
      if (t->partial[slot]) { cudaDeviceSynchronize(); cudaFree(t->partial[slot]); t->partial[slot] = nullptr; t->partial_bytes[slot] = 0; }
      if (cudaMalloc(&t->partial[slot], need) != cudaSuccess) { t->err = "cudaMalloc(split-K partials) failed"; return -1; }
      t->partial_bytes[slot] = need;
    }
    p.partial = t->partial[slot];
  }
  CUtensorMap mA, mB;
  if (make_map(t, &mA, g.A, a_major, g.sAb, g.sAb2, g.sAm, g.sAk, g.M, g.conv_cin > 0 ? g.conv_cin : g.K, g.batch, p.batch_inner, BM)) return -1;
  if (w_shared ? make_map(t, &mB, g.W, b_major, 0, 0, g.sWn, g.sWk, g.N, g.K, 1, 1, p.n_tile)
               : make_map(t, &mB, g.W, b_major, g.sWb, g.sWb2, g.sWn, g.sWk, g.N, g.K, g.batch, p.batch_inner, p.n_tile)) return -1;
  const size_t smem = (size_t)p.stages * stage_bytes + 1024;
  auto al16 = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15) == 0; };
  if (p.partial) p.epi_mode = (g.N % 4 == 0) ? 1 : 0;
  else if (g.sCn == 1 && g.sCm % 4 == 0 && g.sCb % 4 == 0 && g.sCb2 % 4 == 0 && g.N % 4 == 0 && al16(g.C) && (!g.bias || al16(g.bias)) &&
           (!g.R || (g.sRn == 1 && g.sRm % 4 == 0 && g.sRb % 4 == 0 && al16(g.R) && (g.r_ncols >= g.N || g.r_ncols % 32 == 0))) &&
           (g.relu_from % 32 == 0))
    p.epi_mode = 1;
  else if (g.sCm == 1 && (g.relu_from % 32 == 0 || g.relu_from >= g.N) && (!g.bias || al16(g.bias)) && (!g.bias || g.N % 4 == 0)) p.epi_mode = 2;
  else p.epi_mode = 0;
  const long total = mt * nt * g.batch * p.splits;
  gemm_tf32_kernel<<<(unsigned)(total < t->sm_count ? total : t->sm_count), THREADS, smem, s>>>(mA, mB, p);
  count_launch();
  if (p.splits > 1) {
    const long per = (long)g.batch * g.M * g.N;
    splitk_reduce_kernel<<<(unsigned)((per + 255) / 256), 256, 0, s>>>(p);
    count_launch();
  }
  if (cudaGetLastError() != cudaSuccess) { t->err = "gemm_tf32 launch failed"; return -1; }
  return 0;
}

}  // namespace cgg

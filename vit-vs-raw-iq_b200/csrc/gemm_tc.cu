// bf16 GEMM on the 5th-generation tensor cores (tcgen05) for the AMC_BF16 path.
//
//   D[M,N] = A * B^T, fp32 accumulation in TMEM, fused epilogue (gemm_common.cuh).
//
// One persistent CTA per SM, 320 threads, warp-specialised:
//   warp 0      TMA producer   cp.async.bulk.tensor (128B-swizzled tiles) -> 4..6 stage smem ring
//   warp 1      MMA issuer     one elected thread issues tcgen05.mma (M=128, N=BN, K=16) per k-step,
//                              tcgen05.commit releases smem stages / publishes the accumulator
//   warps 2..9  epilogue       tcgen05.ld (32 lanes x 32 columns per warp) -> smem transpose -> fused
//                              bias/ReLU/mask/dropout/residual -> coalesced global stores
// The accumulator is double-buffered in TMEM (2 x BN columns) so the epilogue of tile i overlaps the
// main loop of tile i+1 -- with K as small as d_model=128..256 the epilogue is as long as the MMAs.
//
// Operand layouts
//   MODE_K  (forward, dgrad): A [M,K] and B [N,K] row-major (K contiguous)  -> K-major UMMA operands
//   MODE_MN (wgrad): A [K,M] and B [K,N] row-major (token-major activations) -> MN-major UMMA operands,
//           split-K over the token dimension with fp32 atomics into the gradient.
// TMA zero-fills out-of-bounds rows / columns, so M, N, K need no padding (row pitch % 16 B == 0).
#include <cuda.h>

#include <algorithm>
#include <cstdlib>
#include <initializer_list>

#include "gemm_common.cuh"
#include "ptx.cuh"

namespace amc {
namespace {

constexpr int BM = 128;        // UMMA M (cta_group::1)
constexpr int BK = 64;         // one 128-byte swizzle atom of bf16 per row
constexpr int UMMA_K = 16;
constexpr int NEPI_WARPS = 8;     // two warps per TMEM lane quadrant, each takes half of the columns
constexpr int NTHREADS = 64 + 32 * NEPI_WARPS;
constexpr int EPI_WARP0 = 2;
constexpr int STG_LD = 32;      // floats per staging row; 16-byte chunks are XOR-swizzled by (row & 7)

template <int BN> struct Cfg {
  static constexpr int A_BYTES = BM * BK * 2;              // 16 KB
  static constexpr int B_BYTES = BN * BK * 2;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int STAGES = (BN == 256) ? 4 : (BN == 128 ? 6 : 8);
  static constexpr int TMEM_COLS = 2 * BN;                 // double-buffered accumulator
  static constexpr int STG_BYTES = NEPI_WARPS * 32 * STG_LD * 4;   // per-epilogue-warp transpose tiles
  static constexpr int AUX_BYTES = 1024;                   // barriers, TMEM slot, bias-gradient reduction buffer
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 /*align slack*/ + AUX_BYTES + STG_BYTES;
};

struct TcParams {
  int M, N, K;
  int tiles_m, tiles_n, splits, kb_per_split, kb_total;
  int vec_ok;
};

// ---- roles shared by both kernels ---------------------------------------------------------------
template <int BN, int MODE_MN, int STAGES>
__device__ __forceinline__ void producer_loop(const CUtensorMap* mapA, const CUtensorMap* mapB, const TcParams& p,
                                              unsigned char* smem, uint64_t* full_bar, uint64_t* empty_bar) {
  constexpr int A_BYTES = BM * BK * 2, STAGE_BYTES = A_BYTES + BN * BK * 2;
  const int total_tiles = p.tiles_m * p.tiles_n * p.splits;
  int stage = 0;
  uint32_t phase = 0;
  for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
    const int split = tile % p.splits, mn = tile / p.splits;
    const int tn = mn % p.tiles_n, tm = mn / p.tiles_n;
    const int m0 = tm * BM, n0 = tn * BN;
    const int kb0 = split * p.kb_per_split, kb1 = min(p.kb_total, kb0 + p.kb_per_split);
    for (int kb = kb0; kb < kb1; ++kb) {
      mbar_wait(empty_bar + stage, phase ^ 1);
      unsigned char* sa = smem + stage * STAGE_BYTES;
      unsigned char* sb = sa + A_BYTES;
      mbar_expect_tx(full_bar + stage, STAGE_BYTES);
      if (MODE_MN == 0) {
        tma_load_2d(mapA, full_bar + stage, smem_u32(sa), kb * BK, m0);   // box {64 k, 128 rows}
        tma_load_2d(mapB, full_bar + stage, smem_u32(sb), kb * BK, n0);   // box {64 k, min(BN, 256) rows}
        if (BN > 256) tma_load_2d(mapB, full_bar + stage, smem_u32(sb + 256 * BK * 2), kb * BK, n0 + 256);
      } else {
#pragma unroll
        for (int j = 0; j < BM / 64; ++j)                            // boxes {64 m, 64 tokens}
          tma_load_2d(mapA, full_bar + stage, smem_u32(sa + j * 8192), m0 + 64 * j, kb * BK);
#pragma unroll
        for (int j = 0; j < BN / 64; ++j)
          tma_load_2d(mapB, full_bar + stage, smem_u32(sb + j * 8192), n0 + 64 * j, kb * BK);
      }
      if (++stage == STAGES) { stage = 0; phase ^= 1; }
    }
  }
}

template <int BN, int MODE_MN, int STAGES>
__device__ __forceinline__ void mma_loop(const TcParams& p, unsigned char* smem, uint64_t* full_bar,
                                         uint64_t* empty_bar, uint64_t* tfull_bar, uint64_t* tempty_bar,
                                         uint32_t tmem_base) {
  constexpr int A_BYTES = BM * BK * 2, STAGE_BYTES = A_BYTES + BN * BK * 2;
  constexpr int UN = BN > 256 ? 256 : BN;          // UMMA N (<= 256): a 512-column tile is two MMAs per k-step
  constexpr int NACC = BN > 256 ? 1 : 2;           // accumulator stages in TMEM (512 columns in all)
  constexpr uint32_t idesc = make_idesc(BM, UN, MODE_MN, MODE_MN);
  const int total_tiles = p.tiles_m * p.tiles_n * p.splits;
  int stage = 0;
  uint32_t phase = 0;
  int as = 0;
  uint32_t aphase = 0;
  for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
    const int split = tile % p.splits;
    const int kb0 = split * p.kb_per_split, kb1 = min(p.kb_total, kb0 + p.kb_per_split);
    mbar_wait(tempty_bar + as, aphase ^ 1);      // epilogue has drained this accumulator stage
    tc_fence_after();
    const uint32_t tmem_d = tmem_base + (uint32_t)(as * BN);
    for (int kb = kb0; kb < kb1; ++kb) {
      mbar_wait(full_bar + stage, phase);        // TMA bytes have landed
      tc_fence_after();
      const uint32_t sa = smem_u32(smem + stage * STAGE_BYTES);
      const uint32_t sb = sa + A_BYTES;
#pragma unroll
      for (int k = 0; k < BK / UMMA_K; ++k) {
        uint64_t adesc, bdesc;
        if (MODE_MN == 0) {
          adesc = make_smem_desc(sa + k * (UMMA_K * 2), 16, 1024, 2);
          bdesc = make_smem_desc(sb + k * (UMMA_K * 2), 16, 1024, 2);
        } else {
          adesc = make_smem_desc(sa + k * (UMMA_K * 128), 8192, 1024, 2);
          bdesc = make_smem_desc(sb + k * (UMMA_K * 128), 8192, 1024, 2);
        }
        umma_bf16(tmem_d, adesc, bdesc, idesc, (kb > kb0 || k > 0) ? 1u : 0u);
        if (BN > 256)          // (K-major only: the row kernel) second half of the N columns: B rows 256.. of the stage
          umma_bf16(tmem_d + 256u, adesc, make_smem_desc(sb + 256 * BK * 2 + k * (UMMA_K * 2), 16, 1024, 2), idesc,
                    (kb > kb0 || k > 0) ? 1u : 0u);
      }
      umma_commit(empty_bar + stage);            // frees the smem stage when the MMAs retire
      if (++stage == STAGES) { stage = 0; phase ^= 1; }
    }
    umma_commit(tfull_bar + as);                 // accumulator complete -> epilogue
    if (++as == NACC) { as = 0; aphase ^= 1; }
  }
}

// =================================================================================================
// Kernel 1: generic epilogue (any flag combination, ragged N, split-K atomics).  The accumulator chunk
// is transposed through shared memory so that global accesses are coalesced.
// =================================================================================================
// CS = 1 (weight-gradient mode only): also emit colsum_out[m] += sum_k A[k, m] from the staged A tiles.  It is a
// compile-time switch: the extra shared-memory reads compete with the tensor core's operand fetches, and even the
// dormant code path costs the main loop ~25 %, so the hot weight-gradient calls use CS = 0.
template <int BN, int MODE_MN, int CS>
__global__ void __launch_bounds__(NTHREADS, 1) gemm_tc_kernel(const __grid_constant__ CUtensorMap mapA,
                                                              const __grid_constant__ CUtensorMap mapB,
                                                              const TcParams p, const Epi epi) {
  using C = Cfg<BN>;
  extern __shared__ unsigned char smem_dyn[];
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023) &
                                                         ~(uintptr_t)1023);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + C::STAGES * C::STAGE_BYTES);
  uint64_t* empty_bar = full_bar + C::STAGES;
  uint64_t* tfull_bar = empty_bar + C::STAGES;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);
  float* sred = reinterpret_cast<float*>(smem + C::STAGES * C::STAGE_BYTES + 512);      // [128]
  float* stage_base = reinterpret_cast<float*>(smem + C::STAGES * C::STAGE_BYTES + C::AUX_BYTES);
  constexpr bool do_cs = (MODE_MN == 1) && (CS == 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int total_tiles = p.tiles_m * p.tiles_n * p.splits;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&mapA);
    tma_prefetch_desc(&mapB);
    for (int s = 0; s < C::STAGES; ++s) {
      mbar_init(full_bar + s, 1);
      mbar_init(empty_bar + s, do_cs ? 1 + NEPI_WARPS : 1);   // MMA commit (+ the column-sum readers)
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(tfull_bar + s, 1);
      mbar_init(tempty_bar + s, NEPI_WARPS);   // one arrive per epilogue warp
    }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, C::TMEM_COLS);
  if (threadIdx.x >= 64 && threadIdx.x < 64 + 128) sred[threadIdx.x - 64] = 0.f;
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) producer_loop<BN, MODE_MN, C::STAGES>(&mapA, &mapB, p, smem, full_bar, empty_bar);
  } else if (warp == 1) {
    if (lane == 0) mma_loop<BN, MODE_MN, C::STAGES>(p, smem, full_bar, empty_bar, tfull_bar, tempty_bar, tmem_base);
  } else {
    // ===================== epilogue warps =====================
    const int quad = warp & 3;                       // TMEM lane quadrant this warp may access
    int as = 0;
    uint32_t aphase = 0;
    int cs_stage = 0;
    uint32_t cs_phase = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
      const int mn = tile / p.splits;
      const int tn = mn % p.tiles_n, tm = mn / p.tiles_n;
      const int m_base = tm * BM + quad * 32;
      const int n0 = tn * BN;
      if (MODE_MN == 1 && do_cs) {
        // Bias gradient for free: while the MMAs consume a stage, the (otherwise idle) epilogue warps add up
        // the columns of its A tile (the gradient matrix, [64 tokens][128 outputs], 128B-swizzled rows).
        // Only the first N tile of each M block does the sums; every warp still releases every stage.
        const int split = tile % p.splits;
        const int kb0 = split * p.kb_per_split, kb1 = min(p.kb_total, kb0 + p.kb_per_split);
        const bool mine = (tn == 0);
        const int et = threadIdx.x - 64;              // 0..255
        const int q = et & 15, grp = et >> 4;         // 16-byte chunk of the 128 columns, group of 4 tokens
        float acc[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[j] = 0.f;
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(full_bar + cs_stage, cs_phase);
          if (mine) {
            const uint32_t sa = smem_u32(smem + cs_stage * C::STAGE_BYTES) + (uint32_t)(q >> 3) * 8192u;
#pragma unroll
            for (int t = 0; t < 4; ++t) {
              const int k = grp * 4 + t;
              const uint4 w = lds128(sa + (uint32_t)k * 128u + (uint32_t)(((q & 7) ^ (k & 7)) << 4));
              acc[0] += bf_lo(w.x); acc[1] += bf_hi(w.x);
              acc[2] += bf_lo(w.y); acc[3] += bf_hi(w.y);
              acc[4] += bf_lo(w.z); acc[5] += bf_hi(w.z);
              acc[6] += bf_lo(w.w); acc[7] += bf_hi(w.w);
            }
          }
          __syncwarp();
          if (lane == 0) mbar_arrive(empty_bar + cs_stage);
          if (++cs_stage == C::STAGES) { cs_stage = 0; cs_phase ^= 1; }
        }
        if (mine) {
#pragma unroll
          for (int j = 0; j < 8; ++j) atomicAdd(sred + q * 8 + j, acc[j]);
          bar_sync(1, 256);
          if (et < 128) {
            const float v = sred[et];
            sred[et] = 0.f;
            const int mrow = tm * BM + et;
            if (mrow < p.M && v != 0.f) atomicAdd(epi.colsum_out + mrow, v);
          }
          bar_sync(1, 256);
        }
      }
      mbar_wait(tfull_bar + as, aphase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(as * BN);
      // TMEM gives each thread one accumulator ROW (32 columns per load).  Row-per-thread global
      // accesses would touch 32 different rows per instruction, so each 32x32 chunk is transposed through
      // a per-warp smem tile: afterwards 8 lanes cover 128 contiguous bytes of one row and every epilogue
      // load (bias, residual, ReLU mask) and store is fully coalesced.
      const uint32_t stg = smem_u32(stage_base + (warp - EPI_WARP0) * (32 * STG_LD));
      const int sub_r = lane >> 3, sub_c = (lane & 7) * 4;
      const int half = (warp - EPI_WARP0) >> 2;       // which half of the tile's columns this warp drains
      const int c_begin = half * (BN / 2), c_end = min((half + 1) * (BN / 2), p.N - n0);
      uint32_t r[32];
      if (c_begin < c_end) tmem_ld32(taddr + c_begin, r);
#pragma unroll 1
      for (int c = c_begin; c < c_end; c += 32) {
        tmem_ld_wait(r);
#pragma unroll
        for (int j = 0; j < 32; j += 4)
          sts128(stg + (uint32_t)(lane * STG_LD + (((j >> 2) ^ (lane & 7)) << 2)) * 4, r[j], r[j + 1], r[j + 2],
                 r[j + 3]);
        if (c + 32 < c_end) tmem_ld32(taddr + c + 32, r);   // next chunk streams out of TMEM meanwhile
        __syncwarp();
        float4 v[8];
#pragma unroll
        for (int it = 0; it < 8; ++it) {
          const int rr = it * 4 + sub_r;
          v[it] = lds128f(stg + (uint32_t)(rr * STG_LD + ((((lane & 7)) ^ (rr & 7)) << 2)) * 4);
        }
#pragma unroll
        for (int it = 0; it < 8; ++it)
          epi_apply4<bf16>(epi, m_base + it * 4 + sub_r, n0 + c + sub_c, v[it], p.M, p.N, p.vec_ok != 0);
        __syncwarp();
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar + as);
      if (++as == 2) { as = 0; aphase ^= 1; }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, C::TMEM_COLS);
  }
}

// =================================================================================================
// Kernel 2: row-domain epilogue, all global traffic through TMA.
//   Each epilogue thread owns one accumulator row (its TMEM lane).  Per 32-column chunk the warp's
//   32x32 slab of the residual / ReLU-mask arrives by TMA into swizzled shared memory, the math runs
//   on registers with no per-element address arithmetic, and the results leave through swizzled
//   staging tiles and TMA stores (hardware-coalesced, out-of-bounds rows clipped).
//   RE_BF16  : D16 = [relu](acc + bias) [* dropout]                       (QKV, FFN1, dgrad out-proj)
//   RE_MASK  : D16 = acc * (mask > 0 ? scale : 0)                         (dgrad FFN2: ReLU/dropout mask)
//   RE_RES32 : D32 = (acc + bias) [* dropout] + res32                     (dgrad FFN1 / dgrad QKV skips)
//   RE_LN    : u = (acc + bias)[* dropout] + res32 ; LayerNorm(u) over the row (N <= BN) ->
//              y16, y32, xhat, rstd.  u is parked in TMEM between the passes (mean, variance, write).
// =================================================================================================
enum { RE_BF16 = 0, RE_MASK = 1, RE_RES32 = 2, RE_LN = 3 };

struct RowParams {
  const float* bias;
  int relu;
  DropoutCfg drop;
  uint32_t drop_site;
  float mask_scale;
  const float* gamma;
  const float* beta;
  float ln_eps;
  float* rstd;
  int has_xhat;
  float* colsum_out;   // RE_MASK / RE_BF16: += column sums of the values written (bias gradient of the producer layer)
  int n_cols;          // N (size of the shared-memory column accumulator)
};

template <int BN, int RE, int W = 8> struct RowCfg {
  // (the two-warps-per-quadrant LayerNorm epilogue pays for its second set of slabs with one operand stage)
  static constexpr bool LN8 = (RE == RE_LN && W == 8);
  static constexpr int STAGES = BN > 256 ? 2 : (LN8 ? ((BN == 256) ? 2 : (BN == 128 ? 3 : 4)) : ((BN == 256) ? 3 : (BN == 128 ? 4 : 6)));
  static constexpr int STAGE_BYTES = BM * BK * 2 + BN * BK * 2;
  // bf16-output epilogues are instruction-heavy (dropout hash, mask tests, packing): two warps per TMEM
  // lane quadrant alternate over the 32-column chunks; the fp32 / LayerNorm epilogues keep one warp per
  // quadrant (the row statistics stay thread-local).
  // The bf16 epilogue with ReLU / dropout (FFN1) runs W = 16 warps, four per quadrant: it needs no input slab (4 KB of
  // staging per warp), and with 2 warps per scheduler its TMEM-load -> bias / ReLU / dropout hash -> stage -> TMA-store chain
  // left the issue slots two thirds idle (FFN1 0.283 -> 0.248 ms at the bench size).  Without the elementwise work (QKV,
  // dgrad out-proj) 16 warps only add barrier / store-issue overhead (+5 %), so those keep W = 8.
  // The ReLU-mask epilogue (dgrad FFN2: mask test + bias-gradient column sums per element) takes 16 warps too, with its
  // 2 KB mask slab and its output staging SINGLE-buffered (16 x 4 KB next to three operand stages): the next slab is
  // requested as soon as the current one is in registers, four warps per scheduler cover its latency.
  // The LayerNorm epilogue (three passes over the row) takes W = 8 = two warps per quadrant for K <= 256 (out-proj): each
  // warp owns every other 32-column chunk of its rows through all three passes and the two partial row sums / sums of
  // squares are exchanged through the partner's (idle until pass C) staging area around a 64-thread named barrier.
  static constexpr bool WIDE = (RE == RE_RES32 || RE == RE_LN);        // fp32 slabs: 4 KB in, 4 + 2 + 2 KB out
  static constexpr int NEPI = WIDE ? (LN8 ? 8 : 4) : W;
  static constexpr int EPW = WIDE ? 16384 : ((NEPI == 16) ? 4096 : 8192);   // epilogue bytes per warp
  static constexpr int IN_STRIDE = WIDE ? 4096 : 2048;
  static constexpr int IN_BUFS = (!WIDE && NEPI == 16) ? 1 : 2;
  static constexpr int OUT_BUFS = (NEPI == 16 && RE == RE_MASK) ? 1 : 2;
  static constexpr int OUT_OFF = WIDE ? 8192 : ((NEPI == 16) ? (RE == RE_MASK ? 2048 : 0) : 4096);
  static constexpr int EPI_OFF = STAGES * STAGE_BYTES;
  static constexpr int BAR_OFF = EPI_OFF + NEPI * EPW;
  static constexpr int CS_OFF = BAR_OFF + 512;             // fp32 column accumulator (N <= 2048), bf16-output variants
  static constexpr int CS_BYTES = WIDE ? 0 : 8192;
  static constexpr int SMEM_BYTES = CS_OFF + CS_BYTES + 1024;
  static constexpr int TMEM_COLS = BN > 256 ? BN : 2 * BN;      // 512-column tiles: single-buffered accumulator
  static constexpr int THREADS = 64 + 32 * NEPI;
};

// thread-row access to a TMA-swizzled slab: 32 rows; fp32 rows are 128 B (SWIZZLE_128B: chunk ^= row & 7),
// bf16 rows are 64 B (SWIZZLE_64B: chunk ^= (row >> 1) & 3)
__device__ __forceinline__ uint32_t slab32_addr(uint32_t base, int row, int chunk) {
  return base + row * 128 + ((chunk ^ (row & 7)) << 4);
}
__device__ __forceinline__ uint32_t slab16_addr(uint32_t base, int row, int chunk) {
  return base + row * 64 + ((chunk ^ ((row >> 1) & 3)) << 4);
}

template <int BN, int RE, int W = 8>
__global__ void __launch_bounds__((RowCfg<BN, RE, W>::THREADS), 1)
gemm_tc_row_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB,
                   const __grid_constant__ CUtensorMap mapIn, const __grid_constant__ CUtensorMap mapO16,
                   const __grid_constant__ CUtensorMap mapO32, const __grid_constant__ CUtensorMap mapXh,
                   const TcParams p, const RowParams rp) {
  using C = RowCfg<BN, RE, W>;
  extern __shared__ unsigned char smem_dyn[];
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023) &
                                                         ~(uintptr_t)1023);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + C::BAR_OFF);
  uint64_t* empty_bar = full_bar + C::STAGES;
  uint64_t* tfull_bar = empty_bar + C::STAGES;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint64_t* in_bar = tempty_bar + 2;               // [NEPI warps][2 buffers]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(in_bar + 2 * C::NEPI);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int total_tiles = p.tiles_m * p.tiles_n;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&mapA);
    tma_prefetch_desc(&mapB);
    for (int s = 0; s < C::STAGES; ++s) {
      mbar_init(full_bar + s, 1);
      mbar_init(empty_bar + s, 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(tfull_bar + s, 1);
      mbar_init(tempty_bar + s, C::NEPI);
    }
    for (int s = 0; s < 2 * C::NEPI; ++s) mbar_init(in_bar + s, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, C::TMEM_COLS);
  float* sacc = reinterpret_cast<float*>(smem + C::CS_OFF);
  const bool do_cs = C::CS_BYTES > 0 && rp.colsum_out != nullptr;
  if (do_cs)
    for (int i = threadIdx.x; i < rp.n_cols; i += blockDim.x) sacc[i] = 0.f;
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) producer_loop<BN, 0, C::STAGES>(&mapA, &mapB, p, smem, full_bar, empty_bar);
  } else if (warp == 1) {
    if (lane == 0) mma_loop<BN, 0, C::STAGES>(p, smem, full_bar, empty_bar, tfull_bar, tempty_bar, tmem_base);
  } else {
    // ===================== epilogue: thread = accumulator row =====================
    constexpr bool HAS_IN = (RE != RE_BF16);
    constexpr int IN_BYTES = (RE == RE_MASK) ? 2048 : 4096;
    constexpr int NSPLIT = C::NEPI / 4;               // warps sharing one lane quadrant
    const int ew = warp - 2, quad = warp & 3, half = ew >> 2;
    unsigned char* egen = smem + C::EPI_OFF + ew * C::EPW;
    const uint32_t ebase = smem_u32(egen);
    uint64_t* my_in_bar = in_bar + ew * 2;
    const int nchunks_full = BN / 32;
    uint32_t g = 0;                                   // running chunk counter (input double buffer + phases)
    int as = 0;
    uint32_t aphase = 0;
    // (tile, chunk) this warp processes next, starting the search at (t, c); false when there is none
    auto next_chunk = [&](int& t, int& c) -> bool {
      while (t < total_tiles) {
        const int nc = min(nchunks_full, (p.N - (t % p.tiles_n) * BN) >> 5);
        if (c < nc) return true;
        t += gridDim.x;
        c = half;
      }
      return false;
    };
    auto issue_in = [&](int t, int c, uint32_t gi) {
      uint64_t* nb = my_in_bar + (gi & 1);
      mbar_expect_tx(nb, IN_BYTES);
      tma_load_2d(&mapIn, nb, smem_u32(egen + (C::IN_BUFS == 2 ? (gi & 1) : 0) * C::IN_STRIDE),
                  (t % p.tiles_n) * BN + c * 32, (t / p.tiles_n) * BM + quad * 32);
    };
    if (HAS_IN && lane == 0) {                        // first input slab
      int t = blockIdx.x, c = half;
      if (next_chunk(t, c)) issue_in(t, c, 0);
    }
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
      const int tn = tile % p.tiles_n, tm = tile / p.tiles_n;
      const int m_slab = tm * BM + quad * 32, m = m_slab + lane;
      const int n0 = tn * BN;
      const int nchunks = min(nchunks_full, (p.N - n0) >> 5);
      mbar_wait(tfull_bar + as, aphase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(as * BN);
      float sum = 0.f;

      // ---------------- pass A: finish the accumulator (bias, dropout, mask, residual) -------------
#pragma unroll 1
      for (int ci = half; ci < nchunks; ci += NSPLIT, ++g) {
        const int n = n0 + ci * 32;
        uint32_t r[32];
        tmem_ld32(taddr + ci * 32, r);
        float4 bv[8];
        if (RE != RE_MASK && rp.bias) {               // issue the bias loads before waiting on TMEM
#pragma unroll
          for (int k = 0; k < 8; ++k) bv[k] = __ldg(reinterpret_cast<const float4*>(rp.bias + n) + k);
        }
        if (HAS_IN) {
          // prefetch this warp's next input slab (same tile, or the first chunk of its next tile)
          if (C::IN_BUFS == 2 && lane == 0) {
            int t = tile, c = ci + NSPLIT;
            if (next_chunk(t, c)) issue_in(t, c, g + 1);
          }
          mbar_wait(my_in_bar + (g & 1), (g >> 1) & 1);
        }
        uint4 mw[4];                                    // RE_MASK: this thread's 32 mask values (bf16 pairs)
        if (RE == RE_MASK) {
          const uint32_t ib = ebase + (C::IN_BUFS == 2 ? (g & 1) : 0) * C::IN_STRIDE;
#pragma unroll
          for (int k = 0; k < 4; ++k) mw[k] = lds128(slab16_addr(ib, lane, k));
        }
        tmem_ld_wait(r);
        float v[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
        if (RE != RE_MASK && rp.bias) {
#pragma unroll
          for (int k = 0; k < 8; ++k) {
            v[4 * k] += bv[k].x; v[4 * k + 1] += bv[k].y; v[4 * k + 2] += bv[k].z; v[4 * k + 3] += bv[k].w;
          }
        }
        if (RE == RE_BF16 && rp.relu) {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = fmaxf(v[j], 0.f);
        }
        if (RE != RE_MASK && rp.drop.p > 0.f) {
          const uint64_t e0 = ((uint64_t)m * (uint64_t)p.N + (uint64_t)n) >> 2;
#pragma unroll
          for (int k = 0; k < 8; ++k) {
            const float4 d = dropout_mult4(rp.drop, rp.drop_site, e0 + k);
            v[4 * k] *= d.x; v[4 * k + 1] *= d.y; v[4 * k + 2] *= d.z; v[4 * k + 3] *= d.w;
          }
        }
        if (RE == RE_MASK) {
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const uint32_t w[4] = {mw[k].x, mw[k].y, mw[k].z, mw[k].w};
#pragma unroll
            for (int t = 0; t < 4; ++t) {
              // bf16 > 0  <=>  sign bit clear and magnitude non-zero
              const uint32_t lo = w[t] & 0xFFFFu, hi = w[t] >> 16;
              const bool plo = (lo & 0x8000u) == 0 && (lo & 0x7FFFu) != 0;
              const bool phi = (hi & 0x8000u) == 0 && (hi & 0x7FFFu) != 0;
              v[8 * k + 2 * t] = plo ? v[8 * k + 2 * t] * rp.mask_scale : 0.f;
              v[8 * k + 2 * t + 1] = phi ? v[8 * k + 2 * t + 1] * rp.mask_scale : 0.f;
            }
          }
          if (C::IN_BUFS == 1) {
            // single slab buffer: every lane has consumed its mask words (the selects above depend on them), so the
            // buffer can take this warp's next slab; the column sums, packing and the store below cover its latency
            __syncwarp();
            if (lane == 0) {
              int t = tile, c = ci + NSPLIT;
              if (next_chunk(t, c)) issue_in(t, c, g + 1);
            }
          }
        }
        if (RE == RE_RES32 || RE == RE_LN) {
          const uint32_t ib = ebase + (g & 1) * C::IN_STRIDE;
#pragma unroll
          for (int k = 0; k < 8; ++k) {
            const float4 q = lds128f(slab32_addr(ib, lane, k));
            v[4 * k] += q.x; v[4 * k + 1] += q.y; v[4 * k + 2] += q.z; v[4 * k + 3] += q.w;
          }
        }
        if ((RE == RE_MASK || RE == RE_BF16) && do_cs) {
          // column sums over the warp's 32 rows: transpose-reduce butterfly (31 shuffles), lane j ends up
          // with the sum of column n + j; rows beyond M hold zeros (TMA zero fill) and add nothing
          float t[32];
#pragma unroll
          for (int j = 0; j < 32; ++j) t[j] = (m < p.M) ? v[j] : 0.f;
#pragma unroll
          for (int sft = 16; sft >= 1; sft >>= 1) {
            const bool up = (lane & sft) != 0;
#pragma unroll
            for (int j = 0; j < sft; ++j) {
              const float send = up ? t[j] : t[j + sft];
              const float recv = __shfl_xor_sync(0xffffffffu, send, sft);
              t[j] = (up ? t[j + sft] : t[j]) + recv;
            }
          }
          atomicAdd(sacc + n + lane, t[0]);
        }
        if (RE == RE_LN) {
          uint32_t w[32];
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            sum += v[j];
            w[j] = __float_as_uint(v[j]);
          }
          tmem_st32(taddr + ci * 32, w);              // park u in TMEM for the statistics passes
          __syncwarp();
        } else if (RE == RE_RES32) {
          const uint32_t ob = ebase + C::OUT_OFF + (g & 1) * 4096;
          if (lane == 0) bulk_wait_read<1>();         // the store that last used this buffer has read it
          __syncwarp();
#pragma unroll
          for (int k = 0; k < 8; ++k)
            sts128(slab32_addr(ob, lane, k), __float_as_uint(v[4 * k]), __float_as_uint(v[4 * k + 1]),
                   __float_as_uint(v[4 * k + 2]), __float_as_uint(v[4 * k + 3]));
          fence_proxy_async();
          __syncwarp();
          if (lane == 0) {
            tma_store_2d(&mapO32, ob, n, m_slab);
            bulk_commit();
          }
        } else {
          const uint32_t ob = ebase + C::OUT_OFF + (C::OUT_BUFS == 2 ? (g & 1) : 0) * 2048;
          if (lane == 0) {
            if (C::OUT_BUFS == 2) bulk_wait_read<1>();
            else bulk_wait_read<0>();
          }
          __syncwarp();
#pragma unroll
          for (int k = 0; k < 4; ++k)
            sts128(slab16_addr(ob, lane, k), pack2(v[8 * k], v[8 * k + 1]), pack2(v[8 * k + 2], v[8 * k + 3]),
                   pack2(v[8 * k + 4], v[8 * k + 5]), pack2(v[8 * k + 6], v[8 * k + 7]));
          fence_proxy_async();
          __syncwarp();
          if (lane == 0) {
            tma_store_2d(&mapO16, ob, n, m_slab);
            bulk_commit();
          }
        }
      }

      if (RE == RE_LN) {
        // ---------------- pass B: variance around the exact mean (layers_norm.py:12-13) --------------
        tmem_st_wait();
        // two warps per quadrant: each has summed its own chunks; swap the partial sums through the staging areas (the
        // xhat staging of each warp: idle until pass C, its last TMA store has long read it -- confirmed, not assumed)
        const uint32_t xch_mine = ebase + 14336, xch_peer = smem_u32(smem + C::EPI_OFF + (ew ^ 4) * C::EPW) + 14336;
        auto swap_partial = [&](float mine, int slot) -> float {
          if (lane == 0) bulk_wait_read<0>();
          __syncwarp();
          sts32(xch_mine + (uint32_t)((slot * 32 + lane) * 4), __float_as_uint(mine));
          bar_sync(1 + quad, 64);
          return mine + lds32f(xch_peer + (uint32_t)((slot * 32 + lane) * 4));
        };
        if (NSPLIT == 2) sum = swap_partial(sum, 0);
        const float inv_n = 1.f / (float)p.N;
        const float mean = sum * inv_n;
        float sq = 0.f;
#pragma unroll 1
        for (int ci = half; ci < nchunks; ci += NSPLIT) {
          uint32_t r[32];
          tmem_ld32(taddr + ci * 32, r);
          tmem_ld_wait(r);
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const float t = __uint_as_float(r[j]) - mean;
            sq = fmaf(t, t, sq);
          }
        }
        if (NSPLIT == 2) sq = swap_partial(sq, 1);
        const float rstd = rsqrtf(sq * inv_n + rp.ln_eps);
        if (rp.rstd && m < p.M && half == 0) rp.rstd[m] = rstd;
        // ---------------- pass C: normalise, scale/shift, write y32 / y16 / xhat ---------------------
        const uint32_t o32 = ebase + 8192, o16 = ebase + 12288, oxh = ebase + 14336;
        if (NSPLIT == 2) bar_sync(1 + quad, 64);   // the peer has read slot 1: staging may be reused
#pragma unroll 1
        for (int ci = half; ci < nchunks; ci += NSPLIT) {
          const int n = n0 + ci * 32;
          uint32_t r[32];
          tmem_ld32(taddr + ci * 32, r);
          tmem_ld_wait(r);
          float xh[32], y[32];
#pragma unroll
          for (int k = 0; k < 8; ++k) {
            const float4 gm = __ldg(reinterpret_cast<const float4*>(rp.gamma + n) + k);
            const float4 bt = __ldg(reinterpret_cast<const float4*>(rp.beta + n) + k);
            xh[4 * k] = (__uint_as_float(r[4 * k]) - mean) * rstd;
            xh[4 * k + 1] = (__uint_as_float(r[4 * k + 1]) - mean) * rstd;
            xh[4 * k + 2] = (__uint_as_float(r[4 * k + 2]) - mean) * rstd;
            xh[4 * k + 3] = (__uint_as_float(r[4 * k + 3]) - mean) * rstd;
            y[4 * k] = fmaf(gm.x, xh[4 * k], bt.x);
            y[4 * k + 1] = fmaf(gm.y, xh[4 * k + 1], bt.y);
            y[4 * k + 2] = fmaf(gm.z, xh[4 * k + 2], bt.z);
            y[4 * k + 3] = fmaf(gm.w, xh[4 * k + 3], bt.w);
          }
          if (lane == 0) bulk_wait_read<0>();         // single-buffered staging: previous stores have read it
          __syncwarp();
#pragma unroll
          for (int k = 0; k < 8; ++k)
            sts128(slab32_addr(o32, lane, k), __float_as_uint(y[4 * k]), __float_as_uint(y[4 * k + 1]),
                   __float_as_uint(y[4 * k + 2]), __float_as_uint(y[4 * k + 3]));
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            sts128(slab16_addr(o16, lane, k), pack2(y[8 * k], y[8 * k + 1]), pack2(y[8 * k + 2], y[8 * k + 3]),
                   pack2(y[8 * k + 4], y[8 * k + 5]), pack2(y[8 * k + 6], y[8 * k + 7]));
            if (rp.has_xhat)
              sts128(slab16_addr(oxh, lane, k), pack2(xh[8 * k], xh[8 * k + 1]),
                     pack2(xh[8 * k + 2], xh[8 * k + 3]), pack2(xh[8 * k + 4], xh[8 * k + 5]),
                     pack2(xh[8 * k + 6], xh[8 * k + 7]));
          }
          fence_proxy_async();
          __syncwarp();
          if (lane == 0) {
            tma_store_2d(&mapO32, o32, n, m_slab);
            tma_store_2d(&mapO16, o16, n, m_slab);
            if (rp.has_xhat) tma_store_2d(&mapXh, oxh, n, m_slab);
            bulk_commit();
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar + as);
      if (++as == (BN > 256 ? 1 : 2)) { as = 0; aphase ^= 1; }
    }
    if (lane == 0) bulk_wait_all();
  }
  tc_fence_before();
  __syncthreads();
  if (do_cs)
    for (int i = threadIdx.x; i < rp.n_cols; i += blockDim.x) {
      const float vsum = sacc[i];
      if (vsum != 0.f) atomicAdd(rp.colsum_out + i, vsum);
    }
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, C::TMEM_COLS);
  }
}

// ---- host side ------------------------------------------------------------------------------------
// 2-D tensor [rows, cols] row-major with pitch ld (elements); box = {box_cols, box_rows}; the box's inner
// extent in bytes equals the swizzle span (128 B, or 64 B for 32-column bf16 epilogue slabs)
int make_map_ex(CUtensorMap* map, const void* base, int rows, int cols, int ld, int box_cols, int box_rows,
                bool is_f32, bool swz64) {
  const int esz = is_f32 ? 4 : 2;
  AMC_CHECK_ARG((reinterpret_cast<uintptr_t>(base) & 15) == 0, "GEMM tensor must be 16-byte aligned");
  AMC_CHECK_ARG(((size_t)ld * esz) % 16 == 0, "GEMM tensor pitch (%d elements) must be a multiple of 16 bytes", ld);
  const cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  const cuuint64_t strides[1] = {(cuuint64_t)ld * esz};
  const cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
  return encode_tiled_map(map, is_f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, base,
                          dims, strides, box, swz64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B,
                          CU_TENSOR_MAP_L2_PROMOTION_L2_256B);
}
int make_map(CUtensorMap* map, const void* base, int rows, int cols, int ld, int box_cols, int box_rows) {
  return make_map_ex(map, base, rows, cols, ld, box_cols, box_rows, false, false);
}

template <int BN, int MODE_MN, int CS = 0>
int launch(const GemmArgs& g, cudaStream_t st) {
  using C = Cfg<BN>;
  CUtensorMap mapA, mapB;
  if (MODE_MN == 0) {
    AMC_TRY(make_map(&mapA, g.A, g.M, g.K, g.lda, BK, BM));
    AMC_TRY(make_map(&mapB, g.B, g.N, g.K, g.ldb, BK, BN));
  } else {
    AMC_TRY(make_map(&mapA, g.A, g.K, g.M, g.lda, 64, BK));
    AMC_TRY(make_map(&mapB, g.B, g.K, g.N, g.ldb, 64, BK));
  }
  TcParams p;
  p.M = g.M; p.N = g.N; p.K = g.K;
  p.tiles_m = ceil_div(g.M, BM);
  p.tiles_n = ceil_div(g.N, BN);
  p.kb_total = ceil_div(g.K, BK);
  int splits = std::max(1, std::min(g.split_k, p.kb_total));
  p.kb_per_split = ceil_div(p.kb_total, splits);
  p.splits = ceil_div(p.kb_total, p.kb_per_split);
  p.vec_ok = epi_vec_ok<bf16>(g.epi, g.N) ? 1 : 0;
  const long long tiles = (long long)p.tiles_m * p.tiles_n * p.splits;
  AMC_CHECK_ARG(tiles < (1ll << 30), "gemm_bf16: too many tiles");
  const int grid = (int)std::min<long long>(tiles, device_sm_count());
  auto kern = gemm_tc_kernel<BN, MODE_MN, CS>;
  AMC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES));
  kern<<<grid, NTHREADS, C::SMEM_BYTES, st>>>(mapA, mapB, p, g.epi);
  AMC_LAUNCH_CHECK();
  return 0;
}

template <int BN, int RE, int W = 8>
int launch_row(const GemmArgs& g, cudaStream_t st) {
  using C = RowCfg<BN, RE, W>;
  const Epi& e = g.epi;
  CUtensorMap mapA, mapB, mapIn, mapO16, mapO32, mapXh;
  AMC_TRY(make_map(&mapA, g.A, g.M, g.K, g.lda, BK, BM));
  AMC_TRY(make_map(&mapB, g.B, g.N, g.K, g.ldb, BK, BN > 256 ? 256 : BN));
  mapIn = mapA; mapO16 = mapA; mapO32 = mapA; mapXh = mapA;      // placeholders for unused descriptors
  if (RE == RE_MASK) AMC_TRY(make_map_ex(&mapIn, e.mask_src, g.M, g.N, e.ldmask, 32, 32, false, true));
  if (RE == RE_RES32 || RE == RE_LN) AMC_TRY(make_map_ex(&mapIn, e.res32, g.M, g.N, e.ldres, 32, 32, true, false));
  if (e.D16) AMC_TRY(make_map_ex(&mapO16, e.D16, g.M, g.N, e.ldd16, 32, 32, false, true));
  if (e.D32) AMC_TRY(make_map_ex(&mapO32, e.D32, g.M, g.N, e.ldd32, 32, 32, true, false));
  if (RE == RE_LN && e.ln_xhat) AMC_TRY(make_map_ex(&mapXh, e.ln_xhat, g.M, g.N, g.N, 32, 32, false, true));
  TcParams p;
  p.M = g.M; p.N = g.N; p.K = g.K;
  p.tiles_m = ceil_div(g.M, BM);
  p.tiles_n = ceil_div(g.N, BN);
  p.kb_total = ceil_div(g.K, BK);
  p.kb_per_split = p.kb_total;
  p.splits = 1;
  p.vec_ok = 1;
  RowParams rp;
  rp.bias = e.bias; rp.relu = e.relu; rp.drop = e.drop; rp.drop_site = e.drop_site; rp.mask_scale = e.mask_scale;
  rp.gamma = e.ln_gamma; rp.beta = e.ln_beta; rp.ln_eps = e.ln_eps; rp.rstd = e.ln_rstd;
  rp.has_xhat = e.ln_xhat ? 1 : 0;
  rp.colsum_out = (C::CS_BYTES > 0 && g.N * 4 <= C::CS_BYTES) ? e.colsum_out : nullptr;
  rp.n_cols = g.N;
  AMC_CHECK_ARG(e.colsum_out == nullptr || rp.colsum_out != nullptr,
                "gemm_bf16: fused column sums need a bf16-output epilogue and N <= 2048");
  const long long tiles = (long long)p.tiles_m * p.tiles_n;
  AMC_CHECK_ARG(tiles < (1ll << 30), "gemm_bf16: too many tiles");
  const int grid = (int)std::min<long long>(tiles, device_sm_count());
  auto kern = gemm_tc_row_kernel<BN, RE, W>;
  AMC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES));
  kern<<<grid, C::THREADS, C::SMEM_BYTES, st>>>(mapA, mapB, mapIn, mapO16, mapO32, mapXh, p, rp);
  AMC_LAUNCH_CHECK();
  return 0;
}

template <int RE, int W = 8>
int launch_row_bn(int bn, const GemmArgs& g, cudaStream_t st) {
  if (bn == 256) return launch_row<256, RE, W>(g, st);
  if (bn == 128) return launch_row<128, RE, W>(g, st);
  return launch_row<64, RE, W>(g, st);
}

inline bool al16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

}  // namespace

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

int encode_tiled_map(CUtensorMap* map, CUtensorMapDataType dtype, int rank, const void* base, const cuuint64_t* dims,
                     const cuuint64_t* strides, const cuuint32_t* box, CUtensorMapSwizzle swizzle,
                     CUtensorMapL2promotion l2) {
  static const EncodeTiledFn enc = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess) {
      (void)cudaGetLastError();
      p = nullptr;
    }
    return reinterpret_cast<EncodeTiledFn>(p);
  }();
  AMC_CHECK_ARG(enc != nullptr, "cuTensorMapEncodeTiled not available");
  const cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  const CUresult r = enc(map, dtype, (cuuint32_t)rank, const_cast<void*>(base), dims, strides, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, l2, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  AMC_CHECK_ARG(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed (%d): rank %d, inner dim %llu, box %u x %u", (int)r,
                rank, (unsigned long long)dims[0], box[0], box[1]);
  return 0;
}

int gemm_bf16(const GemmArgs& g, cudaStream_t st) {
  AMC_CHECK_ARG(g.M > 0 && g.N > 0 && g.K > 0, "gemm_bf16: empty problem M=%d N=%d K=%d", g.M, g.N, g.K);
  AMC_CHECK_ARG(g.transA == g.transB, "gemm_bf16: operands must both be K-major (forward/dgrad) or both "
                "token-major (wgrad); mixed layouts are not built");
  AMC_CHECK_ARG(g.split_k == 1 || (g.epi.accumulate && !g.epi.bias && !g.epi.res32 && !g.epi.D16),
                "gemm_bf16: split-K needs an accumulate-only epilogue");
  AMC_CHECK_ARG(g.epi.drop.p == 0.f || g.N % 4 == 0, "gemm_bf16: dropout epilogue needs N %% 4 == 0");
  const Epi& e = g.epi;
  // N tile: least padding, ties -> larger tile
  int best = 256;
  long long best_pad = (long long)ceil_div(g.N, 256) * 256;
  for (int bn : {128, 64}) {
    const long long pad = (long long)ceil_div(g.N, bn) * bn;
    if (pad < best_pad) { best = bn; best_pad = pad; }
  }
  // ---- row-domain TMA epilogue for the hot call sites ----
  const bool row_ok = !g.transA && g.split_k == 1 && !e.accumulate && !e.pos && e.map_Ttok == 0 && g.N % 32 == 0 &&
                      (!e.D16 || (al16(e.D16) && e.ldd16 % 8 == 0)) && (!e.D32 || (al16(e.D32) && e.ldd32 % 4 == 0)) &&
                      (!e.res32 || (al16(e.res32) && e.ldres % 4 == 0)) &&
                      (!e.mask_src || (al16(e.mask_src) && e.ldmask % 8 == 0)) && (!e.bias || al16(e.bias));
  if (e.ln_gamma) {
    AMC_CHECK_ARG(row_ok && e.res32 && e.D16 && e.D32 && !e.mask_src && !e.relu && g.N <= 512 && al16(e.ln_gamma) &&
                      al16(e.ln_beta) && (!e.ln_xhat || al16(e.ln_xhat)),
                  "gemm_bf16: fused LayerNorm epilogue needs N %% 32 == 0, N <= 512, residual, D16 and D32");
    // d in (256, 512]: the row spans two N = 256 MMAs and all 512 TMEM columns (accumulator single-buffered: the epilogue of
    // a tile no longer overlaps the next tile's main loop, still cheaper than a separate LayerNorm pass over HBM)
    if (g.N > 256) return launch_row<512, RE_LN, 4>(g, st);
    const int bn_ln = g.N <= 64 ? 64 : (g.N <= 128 ? 128 : 256);
    // two epilogue warps per quadrant where the main loop is short (out-proj: K = d); FFN2 (K = F) keeps its third stage
    static const int ln8_maxk = [] { const char* e = getenv("AMC_LN8_MAXK"); return e ? atoi(e) : 256; }();
    return g.K <= ln8_maxk ? launch_row_bn<RE_LN, 8>(bn_ln, g, st) : launch_row_bn<RE_LN, 4>(bn_ln, g, st);
  }
  if (row_ok) {
    if (e.mask_src && !e.res32 && e.D16 && !e.D32 && !e.bias && !e.relu && e.drop.p == 0.f)
      return launch_row_bn<RE_MASK, 16>(best, g, st);
    if (e.res32 && !e.mask_src && e.D32 && !e.D16 && !e.relu) return launch_row_bn<RE_RES32, 4>(best, g, st);
    if (!e.res32 && !e.mask_src && e.D16 && !e.D32)
      return (e.relu || e.drop.p > 0.f) ? launch_row_bn<RE_BF16, 16>(best, g, st) : launch_row_bn<RE_BF16, 8>(best, g, st);
  }
  const int mn = g.transA ? 1 : 0;
  AMC_CHECK_ARG(e.colsum_out == nullptr || mn, "gemm_bf16: fused column sums are not available for this epilogue");
  if (mn && e.colsum_out) {
    if (best == 256) return launch<256, 1, 1>(g, st);
    if (best == 128) return launch<128, 1, 1>(g, st);
    return launch<64, 1, 1>(g, st);
  }
  if (best == 256) return mn ? launch<256, 1>(g, st) : launch<256, 0>(g, st);
  if (best == 128) return mn ? launch<128, 1>(g, st) : launch<128, 0>(g, st);
  return mn ? launch<64, 1>(g, st) : launch<64, 0>(g, st);
}

}  // namespace amc

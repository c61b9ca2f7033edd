// Fused short-sequence attention on the 5th-generation tensor cores (tcgen05 + TMEM), bf16, head dim 16 / 32 / 64,
// 49 <= T <= 272 tokens per frame (scale_dot_product_attention.py:26-37 + the head split / concat of
// multi_head_attention.py:34-47; backward per SURVEY Appendix B).
//
// Work unit = one (frame, head).  Its [T, dh] slices of q, k, v arrive as 3-D TMA tensor copies (dims = column, token,
// frame) into swizzled shared-memory tiles (swizzle span = the row: 32 / 64 / 128 B); rows past T are zero-filled by
// the TMA unit.  The same tiles are the UMMA operands: Q and K as K-major operands of S = Q K^T, V as the MN-major B
// operand of O = P V -- nothing is transposed or re-laid-out in shared memory.
//
// Every reference sequence length is 2^k + 1 (CLS token), so a unit is split into MAIN rows -- 128-row query tiles
// (64 rows for T <= 80) that fill the TMEM lanes exactly -- and up to 16 LEFTOVER rows (the +1) that one extra warp
// runs through the mma.sync 16-row block of attn_mma.cuh against the same K / V tiles.
//
// Forward, per main tile (one CTA = RM/32 softmax warps + 1 issuer warp + 1 leftover warp, two CTAs per SM):
//   issuer thread : TMA loads (2-stage ring over units) ; S[128, Tk] = Q K^T by tcgen05.mma into TMEM ;
//                   after the softmax: O[128, dh] = P V with P read from TMEM (A operand) ; TMA store of the output
//   softmax warps : thread = query row = TMEM lane.  Pass 1 over the row (tcgen05.ld) for the max, pass 2 for
//                   p = exp2(s c - m c), the row sum and the bf16 P written back over the S columns (tcgen05.st);
//                   then O is read back, scaled by 1 / sum and staged for the TMA store (the Q tile is dead by then
//                   and serves as the staging buffer); log2-domain row statistics lse2 = m c + log2(sum) are saved.
//   No shuffles, no ldmatrix, no per-element shared-memory traffic on the main rows.
// TMEM columns: S at [0, Tk), P aliases S at [0, Tk/2) (bf16 pairs), O at [OC, OC + dh) inside the dead S columns:
// 128 / 256 columns per CTA for T <= 80 / <= 144, so 4 / 2 CTAs share an SM and one CTA's MMA and copy phases overlap
// the other's softmax.  Two-tile units (T > 144) take all 512 columns -- one CTA per SM -- and run TWO threads per query
// row (SP = 2: 8 softmax warps; partial maxima / sums swapped through shared memory, P stores ordered against the
// partner's S reads by a 64-thread named barrier per chunk pair).
#ifdef TC5_BACKOFF
#define AMC_MBAR_BACKOFF_NS TC5_BACKOFF
#endif
#include <map>
#include <mutex>

#include "attention.cuh"
#include "attn_mma.cuh"
#include "ptx.cuh"

namespace amc {
namespace {

struct Tc5Geom {
  int T, Tk, NT, rem, Tmain;      // tokens, keys padded to 16, 128-row main tiles per unit, leftover rows, main rows
  int h, d, units;
  int kbox_rows, kbox_n;          // K / V tile = kbox_n TMA boxes of kbox_rows rows
  int q_bytes, qlo_bytes, kv_bytes, stage_bytes;
  int oc, tmem_cols, o_sep;       // O column offset, TMEM allocation (power of two), 1 = O outside the S columns
  int nst;                        // input stages (2..4)
  int nch;                        // 32-column chunks per score row
  float sl2;                      // log2(e) / sqrt(dh)
};

constexpr int TC5_HDR = 4096;     // mbarriers + TMEM slot (256 B), then the split-row exchange: [max | sum][half][128 rows] floats

// UMMA swizzle layout of a tile whose rows are 32 * KD bytes (make_smem_desc: 6 = 32B, 4 = 64B, 2 = 128B)
template <int KD> __device__ __forceinline__ constexpr uint32_t sw_layout() { return KD == 1 ? 6u : (KD == 2 ? 4u : 2u); }

// ===============================================================================================================
// Forward
// ===============================================================================================================
constexpr int TC5_MAXST = 4;
struct FwdBars {
  uint64_t full[TC5_MAXST], empty[TC5_MAXST];   // input ring: TMA -> MMA / leftover warp ; MMA commit (+ leftover warp) -> TMA
  uint64_t o_staged[TC5_MAXST];                 // the unit's output rows are staged in its (dead) Q tile -> TMA store
  uint64_t s_full, p_full, o_full, t_empty;
  uint32_t tmem_slot;
};

// kernel-study trace (AMC_TC5_TRACE=1): clock64 stamps of CTA 0, [role][unit][event]
constexpr int TR_UNITS = 8, TR_EV = 16;
__device__ __forceinline__ void tr(long long* trace, int role, int it, int ev) {
  if (trace != nullptr && blockIdx.x == 0 && it < TR_UNITS) trace[(role * TR_UNITS + it) * TR_EV + ev] = clock64();
}

// threads: SP * RM/32 softmax warps | MMA issuer warp | leftover warp | TMA warp
// SP = 2 (two-tile units, T > 144: one CTA per SM anyway -- its S tile takes all of TMEM): two threads per query row, each
// every other 32-column chunk of it through both passes; the partial row maxima / sums are swapped through shared memory
// around a 64-thread named barrier.  Four softmax warps alone left the MUFU pipe 31 % busy there.
template <int KD, int RM, int SP>
__global__ void __launch_bounds__(RM * SP + 96, SP == 2 ? 1 : ((RM == 64) ? (KD == 4 ? 3 : 4) : 2))
attn_tc5_fwd_kernel(const __grid_constant__ CUtensorMap mQ, const __grid_constant__ CUtensorMap mQlo,
                    const __grid_constant__ CUtensorMap mKV, const __grid_constant__ CUtensorMap mO, const Tc5Geom gm,
                    bf16* __restrict__ out, float* __restrict__ lse, long long* __restrict__ trace) {
  constexpr int dh = 16 * KD, RB = 32 * KD, NSQ = RM / 32, NSW = NSQ * SP;      // lane quadrants in use, softmax warps
  constexpr uint32_t LAY = sw_layout<KD>(), SBO = 8 * RB;
  extern __shared__ unsigned char smem_dyn[];
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023) & ~(uintptr_t)1023);
  FwdBars* bars = reinterpret_cast<FwdBars*>(smem);
  float* xch = reinterpret_cast<float*>(smem + 256);                   // [2 = max | sum][SP][128]
  const uint32_t stage0 = smem_u32(smem + TC5_HDR);
  const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0), lane = tid & 31;
  const int T = gm.T, Tk = gm.Tk, NT = gm.NT, NST = gm.nst;
  const bool has_lo = gm.rem > 0;
  auto q_tile = [&](int s) { return stage0 + (uint32_t)(s * gm.stage_bytes); };
  auto qlo_tile = [&](int s) { return q_tile(s) + (uint32_t)gm.q_bytes; };
  auto k_tile = [&](int s) { return qlo_tile(s) + (uint32_t)gm.qlo_bytes; };
  auto v_tile = [&](int s) { return k_tile(s) + (uint32_t)gm.kv_bytes; };

  if (tid == 0) {
    tma_prefetch_desc(&mQ); tma_prefetch_desc(&mQlo); tma_prefetch_desc(&mKV); tma_prefetch_desc(&mO);
    for (int s = 0; s < NST; ++s) {
      mbar_init(bars->full + s, 1);
      mbar_init(bars->empty + s, has_lo ? 2 : 1);
      mbar_init(bars->o_staged + s, NSW * NT);
    }
    mbar_init(&bars->s_full, 1);
    mbar_init(&bars->p_full, RM * SP);
    mbar_init(&bars->o_full, 1);
    mbar_init(&bars->t_empty, NSW);
    fence_barrier_init();
  }
  if (warp == NSW) tmem_alloc(&bars->tmem_slot, (uint32_t)gm.tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = bars->tmem_slot;

  if (warp == NSW) {
    // ============================ MMA issuer warp (all lanes run the loop, one elected lane issues) ============================
    {
      // descriptors differ only in the 14-bit start-address field: build the constant halves once
      constexpr uint32_t idPV = make_idesc(128, dh, 0, 1);
      const uint64_t hiK = make_smem_desc(0, 16, SBO, LAY), hiV = make_smem_desc(0, SBO, SBO, LAY);
      const uint32_t idS0 = make_idesc(128, min(256, Tk), 0, 0), idS1 = make_idesc(128, max(16, Tk - 256), 0, 0);
      const int npv = Tk / 16;
      const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
      int it = 0, s = 0;
      uint32_t ph = 0;
      for (int u = blockIdx.x; u < gm.units; u += gridDim.x, ++it) {
        mbar_wait(bars->full + s, ph);
        tc_fence_after();
        if (lane == 0) tr(trace, 0, it, 0);
        const uint32_t kb = k_tile(s) >> 4, vb = v_tile(s) >> 4;
        for (int t = 0; t < NT; ++t) {
          const int n = it * NT + t;
          if (!gm.o_sep) {                                           // O aliases the S columns: wait until it has been read
            mbar_wait(&bars->t_empty, (uint32_t)((n & 1) ^ 1));
            tc_fence_after();
          }
          // S[128, Tk] = Q_tile K^T : K-major operands, one MMA per 16 head-dim columns and per <= 256 keys
          const uint32_t qa = (q_tile(s) + (uint32_t)(t * 128 * RB)) >> 4;
          if (elect_one()) {
#pragma unroll
            for (int ks = 0; ks < KD; ++ks)
              umma_bf16(tmem_u, hiK | (uint64_t)(qa + 2 * ks), hiK | (uint64_t)(kb + 2 * ks), idS0, ks > 0 ? 1u : 0u);
            if (Tk > 256) {
#pragma unroll
              for (int ks = 0; ks < KD; ++ks)
                umma_bf16(tmem_u + 256u, hiK | (uint64_t)(qa + 2 * ks), hiK | (uint64_t)(kb + 16 * RB + 2 * ks), idS1,
                          ks > 0 ? 1u : 0u);
            }
            umma_commit(&bars->s_full);
          }
          __syncwarp();
          if (lane == 0 && t == 0) tr(trace, 0, it, 1);
          mbar_wait(&bars->p_full, (uint32_t)(n & 1));
          tc_fence_after();
          if (lane == 0 && t == 0) tr(trace, 0, it, 2);
          // O[128, dh] = P V : A = bf16 P in TMEM (8 columns per 16 keys), B = V tile read MN-major (16 keys = RB * 16 bytes)
          const uint32_t to = tmem_u + (uint32_t)gm.oc;
          if (elect_one()) {
            umma_bf16_ts(to, tmem_u, hiV | (uint64_t)vb, idPV, 0u);
#pragma unroll 4
            for (int j = 1; j < npv; ++j)
              umma_bf16_ts(to, tmem_u + (uint32_t)(j * 8), hiV | (uint64_t)(vb + j * RB), idPV, 1u);
            umma_commit(&bars->o_full);
          }
          __syncwarp();
        }
        if (elect_one()) umma_commit(bars->empty + s);
        __syncwarp();
        if (lane == 0) tr(trace, 0, it, 3);
        if (++s == NST) { s = 0; ph ^= 1; }
      }
    }
  } else if (warp == NSW + 2) {
    // ============================ TMA: loads run NST - 1 units ahead, stores trail the epilogue ============================
    if (lane == 0) {
      auto issue_loads = [&](int u, int s) {
        const int b = u / gm.h, hh = u - b * gm.h;
        const int col = hh * dh;
        mbar_expect_tx(bars->full + s, (uint32_t)(NT * RM * RB + 2 * Tk * RB + (has_lo ? 16 * RB : 0)));
        for (int t = 0; t < NT; ++t)
          tma_load_3d(&mQ, bars->full + s, q_tile(s) + (uint32_t)(t * 128 * RB), col, t * 128, b);
        if (has_lo) tma_load_3d(&mQlo, bars->full + s, qlo_tile(s), col, gm.Tmain, b);
        for (int bx = 0; bx < gm.kbox_n; ++bx) {
          const uint32_t off = (uint32_t)(bx * gm.kbox_rows * RB);
          tma_load_3d(&mKV, bars->full + s, k_tile(s) + off, gm.d + col, bx * gm.kbox_rows, b);
          tma_load_3d(&mKV, bars->full + s, v_tile(s) + off, 2 * gm.d + col, bx * gm.kbox_rows, b);
        }
      };
      for (int k = 0; k < NST; ++k)
        if ((int)blockIdx.x + k * (int)gridDim.x < gm.units) issue_loads(blockIdx.x + k * gridDim.x, k);
      int it = 0, s = 0;
      uint32_t ph = 0;
      for (int u = blockIdx.x; u < gm.units; u += gridDim.x, ++it) {
        const int b = u / gm.h, hh = u - b * gm.h;
        mbar_wait(bars->o_staged + s, ph);                    // every softmax warp has staged its rows of this unit
        tr(trace, 1, it, 0);
        for (int t = 0; t < NT; ++t) tma_store_3d(&mO, q_tile(s) + (uint32_t)(t * 128 * RB), hh * dh, t * 128, b);
        bulk_commit();
        const int un = u + NST * (int)gridDim.x;
        if (un < gm.units) {
          bulk_wait_read<0>();                              // the store has read the staging rows
          tr(trace, 1, it, 1);
          mbar_wait(bars->empty + s, ph);                     // MMAs (and the leftover warp) are done with K / V
          tr(trace, 1, it, 2);
          issue_loads(un, s);
        }
        if (++s == NST) { s = 0; ph ^= 1; }
      }
      bulk_wait_all();
    }
  } else if (warp == NSW + 1) {
    // ============================ leftover rows: one mma.sync 16-row block per unit ============================
    if (has_lo) {
      constexpr int NBC = 3;
      const int g = lane >> 2, cb = (lane & 3) * 2;
      const int NQ = Tk / 16, last_k0 = ((NQ - 1) / NBC) * NBC;
      int it = 0, s = 0;
      uint32_t ph = 0;
      for (int u = blockIdx.x; u < gm.units; u += gridDim.x, ++it) {
        const int b = u / gm.h, hh = u - b * gm.h;
        mbar_wait(bars->full + s, ph);
        if (lane == 0) tr(trace, 3, it, 0);
        const uint32_t qb = qlo_tile(s), kb = k_tile(s), vb = v_tile(s);
        uint32_t aq[KD][4];
#pragma unroll
        for (int ks = 0; ks < KD; ++ks) ldsm_x4(aq[ks], addrA<KD>(qb, 0, ks, lane));
        float o[2 * KD][4];
#pragma unroll
        for (int n = 0; n < 2 * KD; ++n) { o[n][0] = 0.f; o[n][1] = 0.f; o[n][2] = 0.f; o[n][3] = 0.f; }
        float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f;
        for (int k0 = 0; k0 < last_k0; k0 += NBC)
          fwd_chunk<KD, NBC, false>(kb, vb, k0, NBC, T, aq, o, m0, m1, l0, l1, gm.sl2, lane);
        fwd_chunk<KD, NBC, true>(kb, vb, last_k0, NQ - last_k0, T, aq, o, m0, m1, l0, l1, gm.sl2, lane);
        __syncwarp();
        if (lane == 0) mbar_arrive(bars->empty + s);       // this warp is done with the stage's tiles
        if (lane == 0) tr(trace, 3, it, 1);
        l0 += __shfl_xor_sync(0xffffffffu, l0, 1); l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
        l1 += __shfl_xor_sync(0xffffffffu, l1, 1); l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
        const float i0 = 1.f / l0, i1 = 1.f / l1;
        const int r0 = gm.Tmain + g, r1 = r0 + 8;
        bf16* ob = out + ((size_t)b * T) * gm.d + hh * dh + cb;
#pragma unroll
        for (int n = 0; n < 2 * KD; ++n) {
          if (r0 < T) *reinterpret_cast<uint32_t*>(ob + (size_t)r0 * gm.d + n * 8) = pack2(o[n][0] * i0, o[n][1] * i0);
          if (r1 < T) *reinterpret_cast<uint32_t*>(ob + (size_t)r1 * gm.d + n * 8) = pack2(o[n][2] * i1, o[n][3] * i1);
        }
        if (lse != nullptr && (lane & 3) == 0) {
          float* lp = lse + ((size_t)b * gm.h + hh) * T;
          if (r0 < T) lp[r0] = fmaf(m0, gm.sl2, __log2f(l0));
          if (r1 < T) lp[r1] = fmaf(m1, gm.sl2, __log2f(l1));
        }
        if (++s == NST) { s = 0; ph ^= 1; }
      }
    }
  } else {
    // ============================ softmax warps: thread = (half of a) query row = TMEM lane ============================
    const int q = warp % NSQ, hf = warp / NSQ;                // lane quadrant ; which chunks / output columns (SP = 2)
    const int row = q * 32 + lane;
    const uint32_t trow = tmem_base + ((uint32_t)(q * 32) << 16);
    const float sl2 = gm.sl2;
    const int nch = gm.nch;
    const int nmine = (nch - hf + SP - 1) / SP;               // this thread's chunks: hf, hf + SP, ...
    // swap a partial row statistic with the thread that holds the other half of the row
    auto swap_half = [&](int which, float mine) -> float {
      xch[(which * SP + hf) * 128 + row] = mine;
      bar_sync(1 + q, 64);
      return xch[(which * SP + (hf ^ 1)) * 128 + row];
    };
    int it = 0, s = 0;
    for (int u = blockIdx.x; u < gm.units; u += gridDim.x, ++it) {
      const int b = u / gm.h, hh = u - b * gm.h;
      for (int t = 0; t < NT; ++t) {
        const int n = it * NT + t;
        mbar_wait(&bars->s_full, (uint32_t)(n & 1));
        tc_fence_after();
        if (tid == 0 && t == 0) tr(trace, 2, it, 0);
        uint32_t ra[32], rb[32];
        // ---- pass 1: row maximum (columns >= T are padding) ----
        float mx = -INFINITY;
        auto max32 = [&](uint32_t (&r)[32], int c) {
          const int tv = T - c * 32;                           // valid columns of this chunk (warp-uniform)
          if (tv < 32) {
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (j >= tv) r[j] = 0xff800000u;
          }
          float a0 = __uint_as_float(r[0]), a1 = __uint_as_float(r[1]), a2 = __uint_as_float(r[2]), a3 = __uint_as_float(r[3]);
#pragma unroll
          for (int j = 4; j < 32; j += 4) {
            a0 = fmaxf(a0, __uint_as_float(r[j])); a1 = fmaxf(a1, __uint_as_float(r[j + 1]));
            a2 = fmaxf(a2, __uint_as_float(r[j + 2])); a3 = fmaxf(a3, __uint_as_float(r[j + 3]));
          }
          mx = fmaxf(mx, fmaxf(fmaxf(a0, a1), fmaxf(a2, a3)));
        };
        auto col = [&](int k) { return (uint32_t)((hf + SP * k) * 32); };      // first S column of this thread's k-th chunk
        if (nmine > 0) tmem_ld32(trow + col(0), ra);
        for (int k = 0; k < nmine; k += 2) {
          tmem_ld_wait(ra);
          if (k + 1 < nmine) tmem_ld32(trow + col(k + 1), rb);
          max32(ra, hf + SP * k);
          if (k + 1 < nmine) {
            tmem_ld_wait(rb);
            if (k + 2 < nmine) tmem_ld32(trow + col(k + 2), ra);
            max32(rb, hf + SP * (k + 1));
          }
        }
        if (SP == 2) mx = fmaxf(mx, swap_half(0, mx));
        if (tid == 0 && t == 0) tr(trace, 2, it, 1);
        // ---- pass 2: p = exp2(s c - m c), row sum, bf16 P back into TMEM over the S columns ----
        // (with SP = 2 a thread overwrites only the S columns of its OWN chunks' first halves ... P of chunk c lands in
        //  columns [16 c, 16 c + 16), which belong to chunk c / 2 of S: possibly the partner's, still unread.  So the
        //  partner must have finished pass 1 -- the barrier inside swap_half above -- and pass 2 reads a chunk before any P
        //  that overlaps a LATER chunk of either thread is stored: see the ordering note below.)
        const float ms = mx * sl2;
        float sum0 = 0.f, sum1 = 0.f;
        auto exp32 = [&](uint32_t (&r)[32], int c, uint32_t (&pk)[16]) {
          const int tv = T - c * 32;
          if (tv < 32) {
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (j >= tv) r[j] = 0xff800000u;
          }
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const float p0 = ex2(fmaf(__uint_as_float(r[2 * j]), sl2, -ms));
            const float p1 = ex2(fmaf(__uint_as_float(r[2 * j + 1]), sl2, -ms));
            sum0 += p0; sum1 += p1;
            pk[j] = pack2(p0, p1);
          }
        };
        if (SP == 1) {
          uint32_t pk[16];
          if (nmine > 0) tmem_ld32(trow, ra);
          for (int c = 0; c < nch; c += 2) {
            tmem_ld_wait(ra);
            if (c + 1 < nch) tmem_ld32(trow + (uint32_t)((c + 1) * 32), rb);
            exp32(ra, c, pk);
            tmem_st16(trow + (uint32_t)(c * 16), pk);
            if (c + 1 < nch) {
              tmem_ld_wait(rb);
              if (c + 2 < nch) tmem_ld32(trow + (uint32_t)((c + 2) * 32), ra);
              exp32(rb, c + 1, pk);
              tmem_st16(trow + (uint32_t)((c + 1) * 16), pk);
            }
          }
        } else {
          // Two threads per row.  P of chunk c overwrites S columns [16 c, 16 c + 16) = the first (c even) or second (c odd)
          // half of S chunk c / 2.  Chunks are taken in ascending order by both threads, a thread reads chunk c (and the
          // partner chunk c +- 1) before either stores P(c) or P(c +- 1), and P(c) can only land on chunks <= c / 2, i.e. on
          // chunks both threads have already read once c >= 2; for the first pair (c = 0, 1 -> S chunk 0) the store waits
          // for a barrier after both threads have their first chunk in registers.
          // (the chunk after next is requested before the barrier: it lies above every column a P store of this step can
          //  touch -- chunk hf + 2k + 2 > k)
          uint32_t pk[16];
          if (nmine > 0) tmem_ld32(trow + col(0), ra);
          for (int k = 0; k < nmine; k += 2) {
            tmem_ld_wait(ra);
            if (k + 1 < nmine) tmem_ld32(trow + col(k + 1), rb);
            // every chunk pair (2k, 2k + 1) is in registers on both sides before its P -- which overlaps S chunk k <= 2k --
            // is stored: one 64-thread barrier per pair (the partner may have one chunk less: it still takes the barrier)
            bar_sync(1 + q, 64);
            exp32(ra, hf + SP * k, pk);
            tmem_st16(trow + (uint32_t)((hf + SP * k) * 16), pk);
            if (k + 1 < nmine) {
              tmem_ld_wait(rb);
              if (k + 2 < nmine) tmem_ld32(trow + col(k + 2), ra);
              bar_sync(1 + q, 64);
              exp32(rb, hf + SP * (k + 1), pk);
              tmem_st16(trow + (uint32_t)((hf + SP * (k + 1)) * 16), pk);
            }
          }
          if (nmine < (nch + SP - 1) / SP) bar_sync(1 + q, 64);   // odd chunk count: keep the pair's barrier count equal
        }
        tmem_st_wait();
        tc_fence_before();
        mbar_arrive(&bars->p_full);
        if (tid == 0 && t == 0) tr(trace, 2, it, 2);
        float sum = sum0 + sum1;
        if (SP == 2) sum += swap_half(1, sum);
        const float inv = 1.f / sum;
        const int rg = t * 128 + row;                         // row inside the frame
        if (lse != nullptr && rg < T && hf == 0) lse[((size_t)b * gm.h + hh) * T + rg] = ms + __log2f(sum);
        // ---- epilogue: O / sum -> bf16 -> staging (the dead Q tile) -> TMA store by the TMA warp ----
        mbar_wait(&bars->o_full, (uint32_t)(n & 1));
        tc_fence_after();
        if (tid == 0 && t == 0) tr(trace, 2, it, 3);
        const uint32_t ot = q_tile(s) + (uint32_t)(t * 128 * RB);
        // this thread's output columns: all dh (SP = 1) or half of them (SP = 2): CW 32-bit accumulator columns from c0
        constexpr int CW = dh / SP, NCH = CW / 8;             // NCH 16-byte chunks of the staged row
        const uint32_t oc0 = (uint32_t)(gm.oc + hf * CW);
        uint32_t o[CW];
        if (CW == 8) {
          uint32_t t8[8];
          tmem_ld8(trow + oc0, t8);
          tmem_ld_wait(t8);
#pragma unroll
          for (int j = 0; j < CW; ++j) o[j] = t8[j % 8];
        } else if (CW == 16) {
          uint32_t t16[16];
          tmem_ld16(trow + oc0, t16);
          tmem_ld_wait(t16);
#pragma unroll
          for (int j = 0; j < CW; ++j) o[j] = t16[j % 16];
        } else {
          tmem_ld32(trow + oc0, ra);
          if (CW == 64) tmem_ld32(trow + oc0 + 32u, rb);
          tmem_ld_wait(ra);
          if (CW == 64) tmem_ld_wait(rb);
#pragma unroll
          for (int j = 0; j < CW; ++j) o[j] = j < 32 ? ra[j % 32] : rb[j % 32];
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&bars->t_empty);
#pragma unroll
        for (int ch = 0; ch < NCH; ++ch)
          sts128(chunk_addr<KD>(ot, row, hf * NCH + ch),
                 pack2(__uint_as_float(o[8 * ch]) * inv, __uint_as_float(o[8 * ch + 1]) * inv),
                 pack2(__uint_as_float(o[8 * ch + 2]) * inv, __uint_as_float(o[8 * ch + 3]) * inv),
                 pack2(__uint_as_float(o[8 * ch + 4]) * inv, __uint_as_float(o[8 * ch + 5]) * inv),
                 pack2(__uint_as_float(o[8 * ch + 6]) * inv, __uint_as_float(o[8 * ch + 7]) * inv));
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) mbar_arrive(bars->o_staged + s);
        if (tid == 0 && t == 0) tr(trace, 2, it, 4);
      }
      if (++s == NST) s = 0;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == NSW) {
    tc_fence_after();
    tmem_dealloc(tmem_base, (uint32_t)gm.tmem_cols);
  }
}

// ===============================================================================================================
// Backward (49 <= T <= 272)
// ===============================================================================================================
// One CTA per SM, 384 threads.  Queries are the TMEM lanes; a unit is walked as ITEMS = (key chunk of 64, query tile of
// 128), tile fastest.  Per item i
//   MMA threads  : S = Q_t K_c^T and dP = dO_t V_c^T   (M = 128, N = chunk, K = dh)  -> TMEM buffer i & 1
//   row threads  : P = exp2(S c - lse2), dS = P * (dP - delta) / sqrt(dh) -> bf16 tiles [query][key] in shared memory
//                  (buffer i & 1); two threads per row, 32 of the chunk's columns each
//   MMA threads  : dV_c (+)= P^T dO_t, dK_c (+)= dS^T Q_t  (M = 64 keys, K = the tile's queries: tiles read MN-major)
//                  dQ_t (+)= dS K_c                        (M = 128, K = chunk: the same dS tile read K-major)
//   row threads  : (one item later, so the sums never stall them) dV_c / dK_c rows after the chunk's last tile and
//                  dQ_t rows after the unit's last chunk -> global
// The S / dP MMAs of item i + 1 are issued before the gradient MMAs of item i, so the row threads go from one item's
// elementwise pass straight into the next; two issuer threads (S, dV, dQ | dP, dK) halve the issue latency chain.
// delta = rowsum(dO * O) is taken once per unit by the row's threads (dO from the staged tile, O from global memory).
// Leftover query rows (T = 128 k + 1): one mma.sync warp computes their S / dP blocks, writes its P / dS rows into
// rows 128.. of the same tiles (the tensor-core dV / dK sums then cover them) and keeps its dQ rows in registers.
// TMEM: [S | dP] x 2 at columns 0 / 128, dV_c 256, dK_c 320, dQ_t 384 + 64 t.
constexpr int CK = 64;                 // keys per chunk
struct BwdBars {
  uint64_t full[TC5_MAXST], empty[TC5_MAXST];
  uint64_t sdp_full[2], ps_full, g_full;
  uint64_t o_full, o_empty;                     // the unit's O slice (for delta = rowsum(dO * O)) in its own single buffer
  uint64_t lo_full[2], lo_free[2];              // per leftover warp: its P / dS rows are staged ; the MMAs that read them retired
  uint32_t tmem_slot;
};
// shared-memory header: barriers (1 KB) + the leftover warps' dQ exchange (16 x 64 floats, only with two leftover warps)
inline int bwd_hdr_bytes(int NT, int rem) { return 1024 + ((NT == 1 && rem > 0) ? 4096 : 0); }
struct Tc5BwdGeom {
  int T, Tk, NT, rem, h, d, units;
  int kbox_rows, kbox_n;
  int tile_bytes, stage_bytes, ps_bytes, hdr_bytes, nst, NC;
  float scale, sl2;
  int ablate;      // kernel-study switches (AMC_TC5_ABLATE): 1 no dVdK MMAs, 2 no dQ MMAs, 4 no S/dP MMAs, 8 no P/dS stores, 16 no exp math,
                   // 32 no dQ stores, 64 no dK / dV stores, 128 no bias sums
};
constexpr int BWD_THREADS = 352;       // 8 row warps | MMA issuer + TMA | leftover 0 | leftover 1

template <int KD>
__global__ void __launch_bounds__(BWD_THREADS, 1)
attn_tc5_bwd_kernel(const __grid_constant__ CUtensorMap mQKV, const __grid_constant__ CUtensorMap mDO,
                    const __grid_constant__ CUtensorMap mOut, const Tc5BwdGeom gm,
                    const bf16* __restrict__ out, const bf16* __restrict__ dout, const float* __restrict__ lse,
                    bf16* __restrict__ dqkv, float* __restrict__ dbias, long long* __restrict__ trace) {
  constexpr int dh = 16 * KD, RB = 32 * KD, NRW = 8;
  constexpr uint32_t LAY = sw_layout<KD>(), SBO = 8 * RB;
  constexpr uint32_t C_DVK = 256, C_DQ = 384;      // [dK_c | dV_c] accumulator (2 dh columns), dQ_t at C_DQ + 64 t
  extern __shared__ unsigned char smem_dyn[];
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023) & ~(uintptr_t)1023);
  BwdBars* bars = reinterpret_cast<BwdBars*>(smem);
  float* s_dqlo = reinterpret_cast<float*>(smem + 1024);              // [16][dh] leftover dQ partial sums
  const uint32_t ps0 = smem_u32(smem + gm.hdr_bytes);                  // [buffer][P | dS]
  const uint32_t o_ring = ps0 + 4u * (uint32_t)gm.ps_bytes;            // O slice of the current unit
  const uint32_t stage0 = o_ring + (uint32_t)gm.tile_bytes;
  const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0), lane = tid & 31;
  const int T = gm.T, Tk = gm.Tk, NT = gm.NT, NST = gm.nst, NC = gm.NC, NI = gm.NC * gm.NT;
  const bool has_lo = gm.rem > 0;
  auto p_tile = [&](int buf) { return ps0 + (uint32_t)(buf * 2) * (uint32_t)gm.ps_bytes; };
  auto ds_tile = [&](int buf) { return p_tile(buf) + (uint32_t)gm.ps_bytes; };
  auto q_tile = [&](int s) { return stage0 + (uint32_t)(s * gm.stage_bytes); };
  auto k_tile = [&](int s) { return q_tile(s) + (uint32_t)gm.tile_bytes; };
  auto v_tile = [&](int s) { return q_tile(s) + 2u * (uint32_t)gm.tile_bytes; };
  auto do_tile = [&](int s) { return q_tile(s) + 3u * (uint32_t)gm.tile_bytes; };

  if (tid == 0) {
    tma_prefetch_desc(&mQKV); tma_prefetch_desc(&mDO); tma_prefetch_desc(&mOut);
    for (int s = 0; s < NST; ++s) {
      mbar_init(bars->full + s, 1);
      mbar_init(bars->empty + s, has_lo ? 2 : 1);
    }
    mbar_init(bars->sdp_full + 0, 1);
    mbar_init(bars->sdp_full + 1, 1);
    mbar_init(&bars->ps_full, NRW);
    mbar_init(&bars->g_full, 1);
    mbar_init(&bars->o_full, 1);
    mbar_init(&bars->o_empty, NRW + (has_lo ? (NT == 1 ? 2 : 1) : 0));
    for (int k = 0; k < 2; ++k) {
      mbar_init(bars->lo_full + k, 1);
      mbar_init(bars->lo_free + k, 1);
    }
    fence_barrier_init();
  }
  if (warp == NRW) tmem_alloc(&bars->tmem_slot, 512u);
  // rows 128..143 of the P / dS tiles belong to the leftover warps; the ones they never write must read as zero
  for (int k = tid; k < 4 * 16 * 8; k += BWD_THREADS)
    sts128(ps0 + (uint32_t)((k >> 7) * gm.ps_bytes + 128 * 128 + (k & 127) * 16), 0u, 0u, 0u, 0u);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = bars->tmem_slot;

  if (warp == NRW) {
    // ============================ MMA issuer warp (all lanes run the loop, one elected lane issues) ============================
    {
      const uint64_t hiK = make_smem_desc(0, 16, SBO, LAY);          // K-major view of an input tile (rows of RB bytes)
      const uint64_t hiM = make_smem_desc(0, SBO, SBO, LAY);         // MN-major view of an input tile
      // [Q | dO] as one MN-major B operand: two dh-wide atoms 3 tiles apart (stage order Q, K, V, dO)
      const uint64_t hiM2 = make_smem_desc(0, 3u * (uint32_t)gm.tile_bytes, SBO, LAY);
      const uint64_t hiPK = make_smem_desc(0, 16, 1024, 2u);         // dS tile (128-byte rows), K-major
      // [P ; dS] as one MN-major A operand: two 64-key atoms ps_bytes apart
      const uint64_t hiPM2 = make_smem_desc(0, (uint32_t)gm.ps_bytes, 1024, 2u);
      constexpr uint32_t idG = make_idesc(128, 2 * dh, 1, 1);     // [dK_c | . ; . | dV_c] : both operands MN-major
      constexpr uint32_t idQ = make_idesc(128, dh, 0, 1);         // dQ : A = dS K-major, B = K MN-major
      const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
      // S and dP of item (c, t) of the unit staged in s -> TMEM buffer gi & 1
      auto issue_sdp = [&](int s, int c, int t, int gi) {
        const int k0 = c * CK, wc = min(CK, Tk - k0);
        const uint32_t idS = make_idesc(128, wc, 0, 0);
        const uint32_t qa = (q_tile(s) + (uint32_t)(t * 128 * RB)) >> 4, da = (do_tile(s) + (uint32_t)(t * 128 * RB)) >> 4;
        const uint32_t kb = (k_tile(s) + (uint32_t)(k0 * RB)) >> 4, vb = (v_tile(s) + (uint32_t)(k0 * RB)) >> 4;
        const uint32_t td = tmem_u + (uint32_t)((gi & 1) * 128);
        if (elect_one()) {
          if (!(gm.ablate & 4)) {
#pragma unroll
            for (int ks = 0; ks < KD; ++ks)
              umma_bf16(td, hiK | (uint64_t)(qa + 2 * ks), hiK | (uint64_t)(kb + 2 * ks), idS, ks > 0 ? 1u : 0u);
#pragma unroll
            for (int ks = 0; ks < KD; ++ks)
              umma_bf16(td + 64u, hiK | (uint64_t)(da + 2 * ks), hiK | (uint64_t)(vb + 2 * ks), idS, ks > 0 ? 1u : 0u);
          }
          umma_commit(bars->sdp_full + (gi & 1));
        }
        __syncwarp();
      };
      // TMA loads of unit u into stage s (one elected lane): Q, K, V, dO slices of the head
      auto issue_loads = [&](int u, int s) {
        const int b = u / gm.h, hh = u - b * gm.h;
        const int col = hh * dh;
        if (elect_one()) {
          mbar_expect_tx(bars->full + s, (uint32_t)(4 * Tk * RB));
          for (int bx = 0; bx < gm.kbox_n; ++bx) {
            const uint32_t off = (uint32_t)(bx * gm.kbox_rows * RB);
            const int r0 = bx * gm.kbox_rows;
            tma_load_3d(&mQKV, bars->full + s, q_tile(s) + off, col, r0, b);
            tma_load_3d(&mQKV, bars->full + s, k_tile(s) + off, gm.d + col, r0, b);
            tma_load_3d(&mQKV, bars->full + s, v_tile(s) + off, 2 * gm.d + col, r0, b);
            tma_load_3d(&mDO, bars->full + s, do_tile(s) + off, col, r0, b);
          }
        }
        __syncwarp();
      };
      // the O slice of unit u -> its single buffer (the readers free it early in the unit, so the next load has a unit's time)
      auto issue_o = [&](int u) {
        const int b = u / gm.h, hh = u - b * gm.h;
        if (elect_one()) {
          mbar_expect_tx(&bars->o_full, (uint32_t)(Tk * RB));
          for (int bx = 0; bx < gm.kbox_n; ++bx)
            tma_load_3d(&mOut, &bars->o_full, o_ring + (uint32_t)(bx * gm.kbox_rows * RB), hh * dh, bx * gm.kbox_rows, b);
        }
        __syncwarp();
      };
      issue_o(blockIdx.x);
      for (int k = 0; k < NST; ++k)
        if ((int)blockIdx.x + k * (int)gridDim.x < gm.units) issue_loads(blockIdx.x + k * gridDim.x, k);
      int it = 0, s = 0, gi = 0;
      int glo = 0, klo[2] = {0, 0};                                 // leftover items so far: all / per leftover warp
      const int NLW = NT == 1 ? 2 : 1;                              // leftover warps in use (they alternate over the items)
      uint32_t ph = 0;
      mbar_wait(bars->full + 0, 0);
      tc_fence_after();
      issue_sdp(0, 0, 0, 0);
      for (int u = blockIdx.x; u < gm.units; u += gridDim.x, ++it) {
        if (lane == 0) tr(trace, 0, it, 0);
        const uint32_t qa = q_tile(s) >> 4, ka = k_tile(s) >> 4;
        const bool has_next = u + (int)gridDim.x < gm.units;
        for (int i = 0; i < NI; ++i, ++gi) {
          const int c = i / NT, t = i - c * NT;
          // S / dP of the next item first: its TMEM buffer was released by ps_full(gi - 1), waited one iteration ago
          if (i + 1 < NI) {
            issue_sdp(s, (i + 1) / NT, (i + 1) % NT, gi + 1);
          } else if (has_next) {
            const int sn = (s + 1 == NST) ? 0 : s + 1;
            mbar_wait(bars->full + sn, (sn == 0) ? (ph ^ 1) : ph);
            tc_fence_after();
            issue_sdp(sn, 0, 0, gi + 1);
          }
          if (lane == 0 && i < 3) tr(trace, 0, it, 1 + 4 * i);
          mbar_wait(&bars->ps_full, (uint32_t)(gi & 1));            // P / dS of this item are in shared memory
          const bool lo_item = has_lo && t == NT - 1;
          const int lw = lo_item ? (NLW == 2 ? (glo & 1) : 0) : 0;
          if (lo_item) mbar_wait(bars->lo_full + lw, (uint32_t)(klo[lw] & 1));   // ... and the leftover rows too
          tc_fence_after();
          if (lane == 0 && i < 3) tr(trace, 0, it, 2 + 4 * i);
          const int k0 = c * CK, wc = min(CK, Tk - k0);
          const int nq = (t == NT - 1) ? (Tk - 128 * t) / 16 : 8;    // 16-row query steps (the last tile carries the leftover rows)
          const uint32_t pa = p_tile(gi & 1) >> 4, sa = ds_tile(gi & 1) >> 4;
          const uint32_t bb = qa + (uint32_t)(t * 8 * RB), kr = ka + (uint32_t)((k0 * RB) >> 4);
          if (elect_one()) {
            // rows 0..63 = P_c^T [Q_t | dO_t], rows 64..127 = dS_c^T [Q_t | dO_t]: dV_c = rows 0..63 x columns dh..2dh-1,
            // dK_c = rows 64..127 x columns 0..dh-1.  16 query rows per step = 2048 B of the tiles, 16 * RB of Q / dO.
#pragma unroll 3
            for (int j = 0; j < ((gm.ablate & 1) ? 0 : nq); ++j)
              umma_bf16(tmem_u + C_DVK, hiPM2 | (uint64_t)(pa + j * 128), hiM2 | (uint64_t)(bb + j * RB), idG,
                        (t > 0 || j > 0) ? 1u : 0u);
            // dQ_t [128, dh] (+)= dS K_c : 16 keys per step = 32 B inside the dS rows, 16 * RB of K
            for (int ks = 0; ks < ((gm.ablate & 2) ? 0 : wc / 16); ++ks)
              umma_bf16(tmem_u + C_DQ + (uint32_t)(t * 64), hiPK | (uint64_t)(sa + 2 * ks), hiM | (uint64_t)(kr + ks * RB), idQ,
                        (c > 0 || ks > 0) ? 1u : 0u);
            umma_commit(&bars->g_full);
            if (lo_item) umma_commit(bars->lo_free + lw);
          }
          __syncwarp();
          if (lo_item) { ++glo; ++klo[lw]; }
          if (lane == 0 && i < 3) tr(trace, 0, it, 3 + 4 * i);
          if (i == 0 && has_next) {
            mbar_wait(&bars->o_empty, (uint32_t)(it & 1));           // every row's delta of this unit has been taken
            issue_o(u + gridDim.x);
          }
          if (i == 0 && it > 0) {
            // refill the previous unit's stage (its MMAs retired while this item was prepared) NST - 1 units ahead
            const int un = u + (NST - 1) * (int)gridDim.x;
            if (un < gm.units) {
              const int sp = (s == 0 ? NST : s) - 1;
              mbar_wait(bars->empty + sp, s == 0 ? (ph ^ 1) : ph);
              issue_loads(un, sp);
            }
          }
        }
        if (elect_one()) umma_commit(bars->empty + s);
        __syncwarp();
        if (lane == 0) tr(trace, 0, it, 15);
        if (++s == NST) { s = 0; ph ^= 1; }
      }
    }
  } else if (warp == NRW + 1 || warp == NRW + 2) {
    // ============================ leftover query rows (128 NT ..): mma.sync 16-row blocks, two warps ============================
    // The two warps take alternate key chunks (each block is a long dependent chain: ldmatrix -> mma.sync -> exp -> stores,
    // about twice an item period), each keeps a partial dQ in registers; they are summed through shared memory per unit.
    const int lw = warp == NRW + 1 ? 0 : 1;
    const int NLW = NT == 1 ? 2 : 1;        // with two query tiles a leftover block comes every other item: one warp keeps up
    if (has_lo && lw < NLW) {
      const int g = lane >> 2, cb = (lane & 3) * 2;
      const int rbase = 128 * NT;
      const int r0 = rbase + g, r1 = r0 + 8;
      const int pr0 = 128 + g, pr1 = pr0 + 8;                       // rows inside the P / dS tiles
      const bool two = gm.rem > 8;                                  // rows 136.. of the tiles stay zero otherwise
      int it = 0, s = 0, glo = 0, k = 0;                            // leftover items so far: all / this warp's
      uint32_t ph = 0;
      for (int u = blockIdx.x; u < gm.units; u += gridDim.x, ++it) {
        const int b = u / gm.h, hh = u - b * gm.h;
        const float* lp = lse + ((size_t)b * gm.h + hh) * T;
        const float l0 = r0 < T ? __ldg(lp + r0) : INFINITY, l1 = r1 < T ? __ldg(lp + r1) : INFINITY;   // padded rows: P = 0
        mbar_wait(bars->full + s, ph);
        mbar_wait(&bars->o_full, (uint32_t)(it & 1));
        if (lane == 0 && lw == 0) tr(trace, 3, it, 0);
        const uint32_t qb = q_tile(s), kb = k_tile(s), vb = v_tile(s), db = do_tile(s);
        // Q and dO fragments of the leftover rows; delta = rowsum(dO * O) / sqrt(dh) from the same fragment layout of O
        uint32_t aq[KD][4], ad[KD][4];
        float d0 = 0.f, d1 = 0.f;
#pragma unroll
        for (int ks = 0; ks < KD; ++ks) {
          uint32_t ofr[4];
          ldsm_x4(aq[ks], addrA<KD>(qb, rbase, ks, lane));
          ldsm_x4(ad[ks], addrA<KD>(db, rbase, ks, lane));
          ldsm_x4(ofr, addrA<KD>(o_ring, rbase, ks, lane));
          d0 += bf_lo(ad[ks][0]) * bf_lo(ofr[0]) + bf_hi(ad[ks][0]) * bf_hi(ofr[0]) +
                bf_lo(ad[ks][2]) * bf_lo(ofr[2]) + bf_hi(ad[ks][2]) * bf_hi(ofr[2]);
          d1 += bf_lo(ad[ks][1]) * bf_lo(ofr[1]) + bf_hi(ad[ks][1]) * bf_hi(ofr[1]) +
                bf_lo(ad[ks][3]) * bf_lo(ofr[3]) + bf_hi(ad[ks][3]) * bf_hi(ofr[3]);
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&bars->o_empty);
        d0 += __shfl_xor_sync(0xffffffffu, d0, 1); d0 += __shfl_xor_sync(0xffffffffu, d0, 2);
        d1 += __shfl_xor_sync(0xffffffffu, d1, 1); d1 += __shfl_xor_sync(0xffffffffu, d1, 2);
        d0 *= gm.scale; d1 *= gm.scale;
        float dq[2 * KD][4];
#pragma unroll
        for (int n = 0; n < 2 * KD; ++n) { dq[n][0] = 0.f; dq[n][1] = 0.f; dq[n][2] = 0.f; dq[n][3] = 0.f; }
        for (int c = 0; c < NC; ++c, ++glo) {
          if (NLW == 2 && (glo & 1) != lw) continue;                 // the other warp's chunk
          const int gi = it * NI + c * NT + NT - 1;                  // the item this block belongs to (last query tile of chunk c)
          const int k0 = c * CK, wc = min(CK, Tk - k0);
          float st[8][4], dp[8][4];
#pragma unroll
          for (int n = 0; n < 8; ++n) {
            st[n][0] = 0.f; st[n][1] = 0.f; st[n][2] = 0.f; st[n][3] = 0.f;
            dp[n][0] = 0.f; dp[n][1] = 0.f; dp[n][2] = 0.f; dp[n][3] = 0.f;
          }
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            if (16 * j < wc) {
#pragma unroll
              for (int ks = 0; ks < KD; ++ks) {
                uint32_t bfr[4];
                ldsm_x4(bfr, addrB<KD>(kb, k0 + 16 * j, ks, lane));
                mma_bf16(st[2 * j], aq[ks], bfr[0], bfr[1]);
                mma_bf16(st[2 * j + 1], aq[ks], bfr[2], bfr[3]);
                ldsm_x4(bfr, addrB<KD>(vb, k0 + 16 * j, ks, lane));
                mma_bf16(dp[2 * j], ad[ks], bfr[0], bfr[1]);
                mma_bf16(dp[2 * j + 1], ad[ks], bfr[2], bfr[3]);
              }
            }
          }
          // rows 128.. of tile buffer gi & 1 were last read by the gradient MMAs of this warp's previous block (the two
          // warps of the one-tile case own one buffer each; with two tiles every block is on buffer 1)
          if (k > 0) mbar_wait(bars->lo_free + lw, (uint32_t)((k - 1) & 1));
          const uint32_t pt = p_tile(gi & 1), dt = ds_tile(gi & 1);
          uint32_t sa[8][2];
#pragma unroll
          for (int n = 0; n < 8; ++n) {
            const float p0 = ex2(fmaf(st[n][0], gm.sl2, -l0)), p1 = ex2(fmaf(st[n][1], gm.sl2, -l0));
            sa[n][0] = pack2(p0 * fmaf(dp[n][0], gm.scale, -d0), p1 * fmaf(dp[n][1], gm.scale, -d0));
            sts32(chunk_addr<4>(pt, pr0, n) + cb * 2, pack2(p0, p1));
            sts32(chunk_addr<4>(dt, pr0, n) + cb * 2, sa[n][0]);
            sa[n][1] = 0u;
            if (two) {
              const float p2 = ex2(fmaf(st[n][2], gm.sl2, -l1)), p3 = ex2(fmaf(st[n][3], gm.sl2, -l1));
              sa[n][1] = pack2(p2 * fmaf(dp[n][2], gm.scale, -d1), p3 * fmaf(dp[n][3], gm.scale, -d1));
              sts32(chunk_addr<4>(pt, pr1, n) + cb * 2, pack2(p2, p3));
              sts32(chunk_addr<4>(dt, pr1, n) + cb * 2, sa[n][1]);
            }
          }
          fence_proxy_async();
          __syncwarp();
          if (lane == 0) mbar_arrive(bars->lo_full + lw);
          ++k;
          if (lane == 0 && lw == 0 && c < 6) tr(trace, 3, it, 1 + c);
          // dQ rows += dS K_c
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            if (16 * j < wc) {
              const uint32_t a4[4] = {sa[2 * j][0], sa[2 * j][1], sa[2 * j + 1][0], sa[2 * j + 1][1]};
#pragma unroll
              for (int np = 0; np < KD; ++np) {
                uint32_t bfr[4];
                ldsm_x4_t(bfr, addrA<KD>(kb, k0 + 16 * j, np, lane));
                mma_bf16(dq[2 * np], a4, bfr[0], bfr[1]);
                mma_bf16(dq[2 * np + 1], a4, bfr[2], bfr[3]);
              }
            }
          }
        }
        // sum the two warps' dQ rows: warp 1 -> shared memory -> warp 0 -> global
        if (NLW == 2) {
          if (lw == 1) {
#pragma unroll
            for (int n = 0; n < 2 * KD; ++n) {
              *reinterpret_cast<float2*>(s_dqlo + g * dh + n * 8 + cb) = make_float2(dq[n][0], dq[n][1]);
              *reinterpret_cast<float2*>(s_dqlo + (g + 8) * dh + n * 8 + cb) = make_float2(dq[n][2], dq[n][3]);
            }
          }
          bar_sync(1, 64);
        }
        if (lw == 0) {
          __syncwarp();
          if (lane == 0) mbar_arrive(bars->empty + s);       // the leftover warps are done with the stage's tiles
          bf16* gp = dqkv + ((size_t)b * T) * (3 * gm.d) + hh * dh + cb;
#pragma unroll
          for (int n = 0; n < 2 * KD; ++n) {
            float2 a0 = make_float2(0.f, 0.f), a1 = make_float2(0.f, 0.f);
            if (NLW == 2) {
              a0 = *reinterpret_cast<const float2*>(s_dqlo + g * dh + n * 8 + cb);
              a1 = *reinterpret_cast<const float2*>(s_dqlo + (g + 8) * dh + n * 8 + cb);
            }
            if (r0 < T) *reinterpret_cast<uint32_t*>(gp + (size_t)r0 * (3 * gm.d) + n * 8) = pack2(dq[n][0] + a0.x, dq[n][1] + a0.y);
            if (r1 < T) *reinterpret_cast<uint32_t*>(gp + (size_t)r1 * (3 * gm.d) + n * 8) = pack2(dq[n][2] + a1.x, dq[n][3] + a1.y);
            if (dbias != nullptr) {        // q-bias gradient: column sums over the block's real rows
              float c0 = (r0 < T ? dq[n][0] + a0.x : 0.f) + (r1 < T ? dq[n][2] + a1.x : 0.f);
              float c1 = (r0 < T ? dq[n][1] + a0.y : 0.f) + (r1 < T ? dq[n][3] + a1.y : 0.f);
#pragma unroll
              for (int o = 4; o < 32; o <<= 1) {
                c0 += __shfl_xor_sync(0xffffffffu, c0, o);
                c1 += __shfl_xor_sync(0xffffffffu, c1, o);
              }
              if (g == 0) {
                atomicAdd(dbias + hh * dh + n * 8 + cb, c0);
                atomicAdd(dbias + hh * dh + n * 8 + cb + 1, c1);
              }
            }
          }
        }
        if (NLW == 2) bar_sync(2, 64);   // warp 0 has read the partial sums
        if (++s == NST) { s = 0; ph ^= 1; }
      }
    }
  } else {
    // ============================ row threads: lane quadrant q, column half hf of every chunk ============================
    const int q = warp & 3, hf = warp >> 2;
    const int row = q * 32 + lane;
    const uint32_t trow = tmem_base + ((uint32_t)(q * 32) << 16);
    const float sl2 = gm.sl2, scale = gm.scale;
    const int sw = row & 7;
    // deferred epilogue of the previous item: which accumulators it completed and where they go
    bool pend = false, p_kv = false, p_dq = false;
    int p_b = 0, p_hh = 0, p_k0 = 0, p_t = 0, p_gi = 0;
    // The fused accumulator holds dV_c in lanes 0..63 (columns dh..2dh-1) and dK_c in lanes 64..127 (columns 0..dh-1):
    // quadrants 0, 1 drain dV rows, quadrants 2, 3 dK rows; the two warps of a quadrant take half of the columns each
    // (of dQ as well).
    constexpr int HC = 8 * KD;                              // columns per thread = dh / 2
    auto ld_half = [&](uint32_t ta, uint32_t (&v)[HC]) {
      if (KD == 4) {
        uint32_t a[32];
        tmem_ld32(ta, a);
        tmem_ld_wait(a);
#pragma unroll
        for (int j = 0; j < HC; ++j) v[j] = a[j % 32];
      } else if (KD == 2) {
        uint32_t a[16];
        tmem_ld16(ta, a);
        tmem_ld_wait(a);
#pragma unroll
        for (int j = 0; j < HC; ++j) v[j] = a[j % 16];
      } else {
        uint32_t a[8];
        tmem_ld8(ta, a);
        tmem_ld_wait(a);
#pragma unroll
        for (int j = 0; j < HC; ++j) v[j] = a[j % 8];
      }
    };
    auto st_half = [&](bf16* g, const uint32_t (&v)[HC]) {
#pragma unroll
      for (int ch = 0; ch < KD; ++ch)
        *reinterpret_cast<uint4*>(g + ch * 8) =
            make_uint4(pack2(__uint_as_float(v[8 * ch]), __uint_as_float(v[8 * ch + 1])),
                       pack2(__uint_as_float(v[8 * ch + 2]), __uint_as_float(v[8 * ch + 3])),
                       pack2(__uint_as_float(v[8 * ch + 4]), __uint_as_float(v[8 * ch + 5])),
                       pack2(__uint_as_float(v[8 * ch + 6]), __uint_as_float(v[8 * ch + 7])));
    };
    // column sums over the warp's 32 rows (rows that do not exist contribute 0): halving exchange, lane l ends with the
    // sum of column (l mod HC) over half (HC = 16) or a quarter (HC = 8) of the rows ... one global reduction per column
    auto colsum_half = [&](const uint32_t (&v)[HC], bool live, float* dst) {
      float a[HC];
#pragma unroll
      for (int j = 0; j < HC; ++j) a[j] = live ? __uint_as_float(v[j]) : 0.f;
      // after the loop lane l holds column (l % HC) summed over the lanes that share l % HC's bits
#pragma unroll
      for (int w = HC / 2, o = 16; w >= 1; w >>= 1, o >>= 1) {
        const bool up = (lane & o) != 0;
#pragma unroll
        for (int j = 0; j < w; ++j) {
          const float mine = up ? a[j + w] : a[j], other = up ? a[j] : a[j + w];
          a[j] = mine + __shfl_xor_sync(0xffffffffu, other, o);
        }
      }
      // HC = 16: 4 steps used offsets 16, 8, 4, 2 -> lanes l and l ^ 1 hold the same column's two half sums; HC = 32: all 5
      float r = a[0];
      int col;
      if (HC == 32) {
        col = ((lane >> 4) & 1) * 16 + ((lane >> 3) & 1) * 8 + ((lane >> 2) & 1) * 4 + ((lane >> 1) & 1) * 2 + (lane & 1);
      } else if (HC == 16) {
        r += __shfl_xor_sync(0xffffffffu, r, 1);
        col = ((lane >> 4) & 1) * 8 + ((lane >> 3) & 1) * 4 + ((lane >> 2) & 1) * 2 + ((lane >> 1) & 1);
      } else {
        r += __shfl_xor_sync(0xffffffffu, r, 1);
        r += __shfl_xor_sync(0xffffffffu, r, 2);
        col = ((lane >> 4) & 1) * 4 + ((lane >> 3) & 1) * 2 + ((lane >> 2) & 1);
      }
      const bool writer = HC == 32 ? true : (HC == 16 ? (lane & 1) == 0 : (lane & 3) == 0);
      if (writer) atomicAdd(dst + col, r);
    };
    auto epilogue_load = [&](uint32_t (&kv)[HC], uint32_t (&dq)[HC]) {
      mbar_wait(&bars->g_full, (uint32_t)(p_gi & 1));
      tc_fence_after();
      if (p_kv) ld_half(trow + C_DVK + (uint32_t)((q < 2 ? dh : 0) + hf * HC), kv);
      if (p_dq) ld_half(trow + C_DQ + (uint32_t)(p_t * 64 + hf * HC), dq);
      tc_fence_before();
    };
    auto epilogue_store = [&](const uint32_t (&kv)[HC], const uint32_t (&dq)[HC]) {
      if (p_kv) {
        const int key = p_k0 + (q & 1) * 32 + lane;
        if (key < T && !(gm.ablate & 64))
          st_half(dqkv + ((size_t)p_b * T + key) * (3 * gm.d) + (q < 2 ? 2 * gm.d : gm.d) + p_hh * dh + hf * HC, kv);
        // (the k-bias gradient is exactly zero -- rows of dS sum to zero, SURVEY Appendix B -- so only dV is summed)
        if (dbias != nullptr && q < 2 && !(gm.ablate & 128)) colsum_half(kv, key < T, dbias + 2 * gm.d + p_hh * dh + hf * HC);
      }
      if (p_dq) {
        const int rg = p_t * 128 + row;
        if (rg < T && !(gm.ablate & 32)) st_half(dqkv + ((size_t)p_b * T + rg) * (3 * gm.d) + p_hh * dh + hf * HC, dq);
        if (dbias != nullptr && !(gm.ablate & 128)) colsum_half(dq, rg < T, dbias + p_hh * dh + hf * HC);
      }
    };
    auto load_lse = [&](int u, float (&l)[2]) {
      const int b = u / gm.h, hh = u - b * gm.h;
#pragma unroll
      for (int t = 0; t < 2; ++t) {
        const int rg = t * 128 + row;
        l[t] = (t < NT && rg < T) ? __ldg(lse + ((size_t)b * gm.h + hh) * T + rg) : INFINITY;
      }
    };
    float l2n[2];
    load_lse(blockIdx.x, l2n);
    int it = 0, s = 0, gi = 0;
    uint32_t ph = 0;
    for (int u = blockIdx.x; u < gm.units; u += gridDim.x, ++it) {
      const int b = u / gm.h, hh = u - b * gm.h;
      // lse2 (loaded during the previous unit's last item) and delta = rowsum(dO * O) / sqrt(dh) of this thread's row in
      // every query tile, from the staged dO tile and the unit's O buffer; rows >= T: lse2 = +inf -> P = 0
      float l2[2] = {l2n[0], l2n[1]}, dls[2] = {0.f, 0.f};
      mbar_wait(bars->full + s, ph);
      mbar_wait(&bars->o_full, (uint32_t)(it & 1));
#pragma unroll
      for (int t = 0; t < 2; ++t) {
        if (t < NT) {
          float dl = 0.f;
#pragma unroll
          for (int ch = 0; ch < 2 * KD; ++ch) {
            const uint4 a = lds128(chunk_addr<KD>(do_tile(s), t * 128 + row, ch));
            const uint4 o4 = lds128(chunk_addr<KD>(o_ring, t * 128 + row, ch));
            dl += bf_lo(a.x) * bf_lo(o4.x) + bf_hi(a.x) * bf_hi(o4.x) + bf_lo(a.y) * bf_lo(o4.y) +
                  bf_hi(a.y) * bf_hi(o4.y) + bf_lo(a.z) * bf_lo(o4.z) + bf_hi(a.z) * bf_hi(o4.z) +
                  bf_lo(a.w) * bf_lo(o4.w) + bf_hi(a.w) * bf_hi(o4.w);
          }
          dls[t] = dl * scale;
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&bars->o_empty);
      if (tid == 0) tr(trace, 2, it, 0);
      for (int i = 0; i < NI; ++i, ++gi) {
        const int c = i / NT, t = i - c * NT;
        const int k0 = c * CK, wc = min(CK, Tk - k0);
        const float l2t = t ? l2[1] : l2[0], dlt = t ? dls[1] : dls[0];
        if (i == NI - 1 && u + (int)gridDim.x < gm.units) load_lse(u + gridDim.x, l2n);
        mbar_wait(bars->sdp_full + (gi & 1), (uint32_t)((gi >> 1) & 1));
        tc_fence_after();
        if (tid == 0 && i < 3) tr(trace, 2, it, 1 + 4 * i);
        // (the P / dS tiles of buffer gi & 1 are free: item gi - 2's gradient MMAs were waited for in item gi - 1)
        const int ncol = wc - hf * 32;                        // columns of this chunk that belong to this thread's half
        const uint32_t tb = trow + (uint32_t)((gi & 1) * 128 + hf * 32);
        const uint32_t prow = p_tile(gi & 1) + (uint32_t)(row * 128), srow = ds_tile(gi & 1) + (uint32_t)(row * 128);
        auto emit8 = [&](const uint32_t* rs, const uint32_t* rd, int q4) {   // 8 keys = one 16-byte chunk of the tile rows
          uint32_t pw[4], dw[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float p0 = ex2(fmaf(__uint_as_float(rs[2 * e]), sl2, -l2t));
            const float p1 = ex2(fmaf(__uint_as_float(rs[2 * e + 1]), sl2, -l2t));
            pw[e] = pack2(p0, p1);
            dw[e] = pack2(p0 * fmaf(__uint_as_float(rd[2 * e]), scale, -dlt), p1 * fmaf(__uint_as_float(rd[2 * e + 1]), scale, -dlt));
          }
          const uint32_t off = (uint32_t)(((hf * 4 + q4) ^ sw) << 4);
          if (!(gm.ablate & 8)) {
            sts128(prow + off, pw[0], pw[1], pw[2], pw[3]);
            sts128(srow + off, dw[0], dw[1], dw[2], dw[3]);
          }
        };
        if (gm.ablate & 16) {
        } else if (ncol > 16) {
          uint32_t rs[32], rd[32];
          tmem_ld32(tb, rs);
          tmem_ld32(tb + 64u, rd);
          tmem_ld_wait(rs);
          tmem_ld_wait(rd);
#pragma unroll
          for (int q4 = 0; q4 < 4; ++q4) emit8(rs + 8 * q4, rd + 8 * q4, q4);
        } else if (ncol > 0) {
          uint32_t rs[16], rd[16];
          tmem_ld16(tb, rs);
          tmem_ld16(tb + 64u, rd);
          tmem_ld_wait(rs);
          tmem_ld_wait(rd);
#pragma unroll
          for (int q4 = 0; q4 < 2; ++q4) emit8(rs + 8 * q4, rd + 8 * q4, q4);
        }
        tc_fence_before();
        fence_proxy_async();
        if (tid == 0 && i < 3) tr(trace, 2, it, 2 + 4 * i);
        // drain what the previous item completed (its MMAs had this whole pass to retire), then release this item
        uint32_t kv[HC], dqr[HC];
        const bool had = pend;
        if (had) epilogue_load(kv, dqr);
        __syncwarp();
        if (lane == 0) mbar_arrive(&bars->ps_full);
        if (tid == 0 && i < 3) tr(trace, 2, it, 3 + 4 * i);
        if (had) epilogue_store(kv, dqr);
        if (tid == 0 && i < 3) tr(trace, 2, it, 4 + 4 * i);
        pend = true; p_kv = (t == NT - 1); p_dq = (c == NC - 1);
        p_b = b; p_hh = hh; p_k0 = k0; p_t = t; p_gi = gi;
      }
      if (++s == NST) { s = 0; ph ^= 1; }
    }
    if (pend) {
      uint32_t kv[HC], dqr[HC];
      epilogue_load(kv, dqr);
      epilogue_store(kv, dqr);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == NRW) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512u);
  }
}

// ---- host side -------------------------------------------------------------------------------------------------
constexpr size_t TC5_SMEM_MAX = 227 * 1024;

inline int up1024(int v) { return (v + 1023) / 1024 * 1024; }

// RM = main-tile rows (64 | 128); false = shape outside this kernel's envelope
bool tc5_plan(int B, int T, int h, int dh, Tc5Geom& g, int& RM) {
  if (!(dh == 16 || dh == 32 || dh == 64) || T < 49 || T > 272 || h < 1) return false;
  const int RB = 2 * dh;
  g.T = T; g.Tk = (T + 15) / 16 * 16; g.h = h; g.d = h * dh; g.units = B * h;
  if (T <= 80) { RM = 64; g.NT = 1; g.Tmain = std::min(T, 64); }
  else if (T <= 144) { RM = 128; g.NT = 1; g.Tmain = std::min(T, 128); }
  else { RM = 128; g.NT = 2; g.Tmain = std::min(T, 256); }
  g.rem = T - g.Tmain;
  g.kbox_n = g.Tk > 256 ? 2 : 1;
  g.kbox_rows = g.Tk / g.kbox_n;
  g.q_bytes = g.NT * 128 * RB;
  g.qlo_bytes = g.rem > 0 ? up1024(16 * RB) : 0;
  g.kv_bytes = up1024(g.Tk * RB);
  g.stage_bytes = g.q_bytes + g.qlo_bytes + 2 * g.kv_bytes;
  g.nch = (g.Tk + 31) / 32;
  // O outside the S columns (the next tile's S MMA need not wait for the epilogue) when that costs no larger allocation
  auto pow2 = [](int need) { return need <= 128 ? 128 : (need <= 256 ? 256 : 512); };
  const int alias_cols = pow2(std::max(32 * g.nch, 16 * g.nch + dh)), sep_cols = pow2(32 * g.nch + dh);
  g.o_sep = sep_cols == alias_cols ? 1 : 0;
  g.oc = g.o_sep ? 32 * g.nch : 16 * g.nch;
  g.tmem_cols = alias_cols;
  g.sl2 = 1.4426950408889634f / sqrtf((float)dh);
  // CTAs per SM allowed by TMEM (and the warp budget), then as many input stages as their shared-memory share holds
  int ctas = std::min(512 / g.tmem_cols, RM == 64 ? 4 : 2);
  for (;; --ctas) {
    const int budget = (228 * 1024 - ctas * 1024) / ctas - 1024 - TC5_HDR;
    g.nst = std::min(TC5_MAXST, budget / g.stage_bytes);
    if (g.nst >= 2 || ctas == 1) break;
  }
  return g.nst >= 2;
}
size_t tc5_fwd_bytes(const Tc5Geom& g) { return 1024 + TC5_HDR + (size_t)g.nst * g.stage_bytes; }


bool tc5_bwd_plan(int B, int T, int h, int dh, Tc5BwdGeom& g) {
  if (!(dh == 16 || dh == 32 || dh == 64) || T < 49 || T > 272 || h < 1) return false;
  const int RB = 2 * dh;
  g.T = T; g.Tk = (T + 15) / 16 * 16; g.h = h; g.d = h * dh; g.units = B * h;
  g.NT = T <= 144 ? 1 : 2;
  g.rem = std::max(0, T - 128 * g.NT);
  g.kbox_n = g.Tk > 256 ? 2 : 1;
  g.kbox_rows = g.Tk / g.kbox_n;
  // every tile holds at least the 128 rows per query tile that an M = 128 operand descriptor (and the row threads) touch
  g.tile_bytes = up1024(std::max(g.Tk, 128 * g.NT) * RB);
  g.stage_bytes = 4 * g.tile_bytes;
  g.ps_bytes = up1024(144 * 128);
  g.NC = (g.Tk + CK - 1) / CK;
  g.scale = 1.f / sqrtf((float)dh);
  g.sl2 = 1.4426950408889634f * g.scale;
  g.ablate = getenv("AMC_TC5_ABLATE") ? atoi(getenv("AMC_TC5_ABLATE")) : 0;
  g.hdr_bytes = bwd_hdr_bytes(g.NT, g.rem);
  const int budget = 227 * 1024 - 1024 - g.hdr_bytes - 4 * g.ps_bytes - g.tile_bytes;
  g.nst = std::min(TC5_MAXST, budget / g.stage_bytes);
  return g.nst >= 2;       // the next unit's first S / dP MMAs are issued before this unit's last gradient MMAs
}
size_t tc5_bwd_bytes(const Tc5BwdGeom& g) {
  return 1024 + (size_t)g.hdr_bytes + (size_t)4 * g.ps_bytes + (size_t)g.tile_bytes + (size_t)g.nst * g.stage_bytes;
}

// CTAs of one kernel an SM can hold: TMEM columns, shared memory (1 KB reserved per CTA), registers (allocated per warp
// in units of 256, 64 K per SM and 16 K per sub-partition), 2048 threads.
int tc5_ctas_per_sm(const void* kern, int threads, size_t smem, int tmem_cols) {
  static std::mutex mu;
  static std::map<const void*, int> regs_of;
  int regs;
  {
    std::lock_guard<std::mutex> lk(mu);
    auto f = regs_of.find(kern);
    if (f == regs_of.end()) {
      cudaFuncAttributes fa;
      if (cudaFuncGetAttributes(&fa, kern) != cudaSuccess) return 1;
      f = regs_of.emplace(kern, fa.numRegs).first;
    }
    regs = f->second;
  }
  const int warps = (threads + 31) / 32, regs_warp = (regs * 32 + 255) / 256 * 256;
  const int by_regs = (4 * (16384 / regs_warp)) / ((warps + 3) / 4 * 4);
  const int by_smem = (int)((228 * 1024) / (smem + 1024));
  return std::max(1, std::min(std::min(512 / tmem_cols, by_smem), std::min(by_regs, 2048 / threads)));
}

// ---- kernel-study trace: AMC_TC5_TRACE=1 prints the clock64 stamps of CTA 0 after every launch (debug only) ----
long long* tc5_trace_begin() {
  static const bool on = [] { const char* e = getenv("AMC_TC5_TRACE"); return e && e[0] == '1'; }();
  if (!on) return nullptr;
  static long long* buf = nullptr;
  const size_t n = 4 * TR_UNITS * TR_EV * sizeof(long long);
  if (!buf && cudaMalloc(&buf, n) != cudaSuccess) return nullptr;
  cudaMemset(buf, 0, n);
  return buf;
}
void tc5_trace_end(long long* buf, const char* what, int T, int dh, cudaStream_t st) {
  long long h[4 * TR_UNITS * TR_EV];
  cudaStreamSynchronize(st);
  cudaMemcpy(h, buf, sizeof(h), cudaMemcpyDeviceToHost);
  long long t0 = 0;
  for (size_t i = 0; i < sizeof(h) / sizeof(h[0]); ++i)
    if (h[i] && (!t0 || h[i] < t0)) t0 = h[i];
  static const char* roles[4] = {"mma ", "tma ", "smx0", "left"};
  fprintf(stderr, "[tc5 trace %s T=%d dh=%d] cycles since the first stamp, per unit of CTA 0\n", what, T, dh);
  for (int r = 0; r < 4; ++r)
    for (int u = 0; u < TR_UNITS; ++u) {
      bool any = false;
      for (int e = 0; e < TR_EV; ++e) any |= h[(r * TR_UNITS + u) * TR_EV + e] != 0;
      if (!any) continue;
      fprintf(stderr, "  %s u%-2d:", roles[r], u);
      for (int e = 0; e < TR_EV; ++e) {
        const long long v = h[(r * TR_UNITS + u) * TR_EV + e];
        if (v) fprintf(stderr, " e%d=%lld", e, v - t0);
      }
      fprintf(stderr, "\n");
    }
}

}  // namespace

// Where the tcgen05 kernels are the faster ones (B200, tools/probes/attn_tc5_check.py --bwd --time; profiles/
// r2_attn_tc5_check_and_timing.txt), per direction -- both forward kernels write the same log2-domain lse, so a tcgen05
// forward pairs with either backward:
//   forward : T > 80, and head dim 64 at any T (T = 65, dh = 64: 141 vs 196 us)
//   backward: head dim 32 at T > 80 (T = 129: 298 vs 373 us, T = 257: 393 vs 598 us) and head dim 64 (inside a training
//             step of the d512 / h8 grid corner, T = 65: 295 vs 311 us per layer -- the isolated probe, cold inputs, says the
//             opposite, 897 vs 551 us at twice the batch; the step is what counts); at head dim 16 the item's fixed
//             barrier / MMA cost is spread over half the bytes (T = 129: 263 vs 212 us isolated, 257 vs 214 us inside the
//             production-ViT step): the mma.sync tile kernels keep that.
// AMC_ATTN_TC5=all|none overrides for kernel studies.
bool tc5_preferred(int T, int dh, bool bwd) {
  static const int mode = [] {
    const char* e = getenv("AMC_ATTN_TC5");
    return e == nullptr ? 0 : (e[0] == 'a' ? 1 : (e[0] == 'n' ? 2 : 0));
  }();
  if (mode == 1) return true;
  if (mode == 2) return false;
  return bwd ? (dh == 64 || (T > 80 && dh == 32)) : (T > 80 || dh == 64);
}

bool attn_tc5_supported(int T, int h, int dh) {
  Tc5Geom g;
  int RM;
  return tc5_plan(1, T, h, dh, g, RM) && tc5_fwd_bytes(g) <= TC5_SMEM_MAX;
}

int attn_tc5_fwd(int B, int T, int h, int dh, const bf16* qkv, bf16* out, float* lse, bool* handled, cudaStream_t st) {
  *handled = false;
  Tc5Geom g;
  int RM = 0;
  if (!tc5_plan(B, T, h, dh, g, RM) || !tc5_preferred(T, dh, false)) return 0;
  const size_t sm = tc5_fwd_bytes(g);
  if (sm > TC5_SMEM_MAX || (g.d * 2) % 16 != 0) return 0;
  CUtensorMap mQ, mQlo, mKV, mO;
  AMC_TRY(attn_make_map3(&mQ, qkv, B, T, 3 * g.d, dh, RM));
  AMC_TRY(attn_make_map3(&mQlo, qkv, B, T, 3 * g.d, dh, 16));
  AMC_TRY(attn_make_map3(&mKV, qkv, B, T, 3 * g.d, dh, g.kbox_rows));
  AMC_TRY(attn_make_map3(&mO, out, B, T, g.d, dh, RM));
  long long* trace = tc5_trace_begin();
#define AMC_TC5_FWD(KD, RM_, SP_)                                                                                     \
  do {                                                                                                                \
    auto kern = attn_tc5_fwd_kernel<KD, RM_, SP_>;                                                                     \
    constexpr int threads = RM_ * SP_ + 96;                                                                           \
    AMC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TC5_SMEM_MAX));             \
    /* (cudaOccupancyMaxActiveBlocksPerMultiprocessor answers 1 for every kernel that allocates TMEM, whatever its    \
       resources; the hardware does co-schedule such CTAs -- measured -- so the limits are applied here) */           \
    int occ = tc5_ctas_per_sm((const void*)kern, threads, sm, g.tmem_cols);                                           \
    if (getenv("AMC_TC5_OCC")) occ = atoi(getenv("AMC_TC5_OCC"));                                                     \
    const int grid = std::min(g.units, device_sm_count() * occ);                                                      \
    if (trace) {                                                                                                      \
      cudaFuncAttributes fa;                                                                                          \
      cudaFuncGetAttributes(&fa, kern);                                                                               \
      fprintf(stderr, "[tc5 fwd] grid %d occ %d threads %d smem %zu nst %d tmem %d o_sep %d units %d | regs %d static smem %zu local %zu maxdyn %d\n", \
              grid, occ, threads, sm, g.nst, g.tmem_cols, g.o_sep, g.units, fa.numRegs, fa.sharedSizeBytes, fa.localSizeBytes, fa.maxDynamicSharedSizeBytes); \
    }                                                                                                                 \
    kern<<<grid, threads, sm, st>>>(mQ, mQlo, mKV, mO, g, out, lse, trace);                                           \
  } while (0)
  /* two threads per row where a unit has two query tiles (T > 144: all of TMEM, one CTA per SM); AMC_TC5_SPLIT=0 off */ \
  static const bool split_ok = [] { const char* e = getenv("AMC_TC5_SPLIT"); return !(e && e[0] == '0'); }();
#define AMC_TC5_FWD_KD(KD)                                   \
  do {                                                       \
    if (RM == 64) AMC_TC5_FWD(KD, 64, 1);                    \
    else if (g.NT == 2 && split_ok) AMC_TC5_FWD(KD, 128, 2); \
    else AMC_TC5_FWD(KD, 128, 1);                            \
  } while (0)
  if (dh == 16) AMC_TC5_FWD_KD(1);
  else if (dh == 32) AMC_TC5_FWD_KD(2);
  else AMC_TC5_FWD_KD(4);
#undef AMC_TC5_FWD_KD
#undef AMC_TC5_FWD
  AMC_LAUNCH_CHECK();
  if (trace) tc5_trace_end(trace, "fwd", T, dh, st);
  *handled = true;
  return 0;
}

int attn_tc5_bwd(int B, int T, int h, int dh, const bf16* qkv, const bf16* out, const float* lse, const bf16* dout,
                 bf16* dqkv, float* dbias, bool* handled, cudaStream_t st) {
  *handled = false;
  Tc5BwdGeom g;
  if (out == nullptr || lse == nullptr || !tc5_bwd_plan(B, T, h, dh, g) || !tc5_preferred(T, dh, true)) return 0;
  const size_t sm = tc5_bwd_bytes(g);
  if (sm > TC5_SMEM_MAX || (g.d * 2) % 16 != 0) return 0;
  CUtensorMap mQKV, mDO, mOut;
  AMC_TRY(attn_make_map3(&mQKV, qkv, B, T, 3 * g.d, dh, g.kbox_rows));
  AMC_TRY(attn_make_map3(&mDO, dout, B, T, g.d, dh, g.kbox_rows));
  AMC_TRY(attn_make_map3(&mOut, out, B, T, g.d, dh, g.kbox_rows));
  long long* trace = tc5_trace_begin();
#define AMC_TC5_BWD(KD)                                                                                               \
  do {                                                                                                                \
    auto kern = attn_tc5_bwd_kernel<KD>;                                                                               \
    AMC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TC5_SMEM_MAX));             \
    const int occ = 1;                                                                                                \
    const int grid = std::min(g.units, device_sm_count() * occ);                                                      \
    if (trace) fprintf(stderr, "[tc5 bwd] grid %d occ %d smem %zu nst %d units %d\n", grid, occ, sm, g.nst, g.units); \
    kern<<<grid, BWD_THREADS, sm, st>>>(mQKV, mDO, mOut, g, out, dout, lse, dqkv, dbias, trace);                                                 \
  } while (0)
  if (dh == 16) AMC_TC5_BWD(1);
  else if (dh == 32) AMC_TC5_BWD(2);
  else AMC_TC5_BWD(4);
#undef AMC_TC5_BWD
  AMC_LAUNCH_CHECK();
  if (trace) tc5_trace_end(trace, "bwd", T, dh, st);
  *handled = true;
  return 0;
}

}  // namespace amc

// Single-CTA fused attention for 16 < T <= 288 tokens (bf16, head dim 16 / 32 / 64), forward and backward.
// (scale_dot_product_attention.py:26-37 + the head split / concat of multi_head_attention.py:34-47; backward per
// SURVEY Appendix B.)
//
// A CTA owns one (frame, group of G heads) at a time and loops persistently over such units.  Every operand of a
// head -- the [T, dh] slices of q, k, v (and dO, O in backward) -- arrives as ONE 3-D TMA tensor copy
// (dims = column, token, frame; box = dh x Tpad x 1) into a swizzled shared-memory tile; rows T..Tpad-1 of the box
// lie outside the token dimension and are zero-filled by the TMA unit, so the MMA loops need no row clamping and
// results leave through TMA stores that clip the same rows.  Swizzle mode = row bytes (32 / 64 / 128 B): ldmatrix
// reads are bank-conflict free without padding.
//
// Math is mma.sync m16n8k16 (bf16 in, fp32 accumulate): with dh = 16..64 the tensor pipe is not the limiter --
// the exp / scale / pack work per score element is (SURVEY §8d: "issue/SMEM-bound in practice at dh=16") -- so
// the kernels minimise instructions per score element rather than chase tcgen05:
//   forward : a warp owns 16 query rows and walks the keys in chunks of 48 (or 80) with an online-softmax rescale, so
//             the score fragment stays small enough for two CTAs per SM; exp2 with the 1/sqrt(dh)*log2(e) factor
//             folded into one FFMA; normalisation is applied to O (dh columns), not to P (T columns);
//             log2-domain row statistics lse2 = max*c + log2(sum) are saved for the backward; the inputs arrive
//             through an n-stage TMA ring, the output leaves through double-buffered staging tiles.
//   backward: a warp owns 16 KEY rows and walks the query blocks: S^T = K Q^T and dP^T = V dO^T come out
//             transposed, P^T = exp2(S^T c - lse2) needs no row reduction, delta = rowsum(dO * O) is computed once
//             from the staged tiles.  dV += P^T dO and dK += dS^T Q accumulate in registers; dQ += dS K uses
//             movmatrix to turn the dS^T fragments into an A operand and accumulates in an fp32 shared tile.  The
//             warps visit the query blocks in rotated order (block (kt + step) mod NQ) with one CTA barrier per
//             step, so no two warps touch the same dQ rows at once: no atomics, deterministic sums.
//             The q/k/v bias gradients (column sums of dQ, dK, dV) are taken from the staged results.
#include "attention.cuh"
#include "attn_mma.cuh"

namespace amc {
namespace {

struct TileGeom {
  int T, Tpad, NQ, h, d, G, ngrp, units;
  int BR, nbox;          // TMA box rows and boxes per tile (Tpad = BR * nbox)
  int tile_bytes;        // Tpad * 32 * KD
  int nst, nso;          // forward: input stages (1|2), output stagings (1|2)
  float scale, sl2;      // 1/sqrt(dh), scale * log2(e)
};

constexpr int SMEM_HDR = 1024;   // mbarriers

// ===============================================================================================================
// Forward
// ===============================================================================================================
template <int KD, int NBC, int MINB>
__global__ void __launch_bounds__(320, MINB)
attn_tile_fwd_kernel(const __grid_constant__ CUtensorMap mQKV, const __grid_constant__ CUtensorMap mO,
                     const TileGeom gm, float* __restrict__ lse) {
  constexpr int dh = 16 * KD, RB = 32 * KD;
  extern __shared__ unsigned char smem_dyn[];
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023) & ~(uintptr_t)1023);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem);
  const uint32_t tiles = smem_u32(smem + SMEM_HDR);
  const uint32_t tb = (uint32_t)gm.tile_bytes, stage_bytes = 3u * gm.G * tb;
  const uint32_t so_base = tiles + gm.nst * stage_bytes;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, nw = blockDim.x >> 5;
  const int g = lane >> 2, cb = (lane & 3) * 2;
  const int T = gm.T, NQ = gm.NQ, items = gm.G * NQ;
  if (tid == 0) {
    tma_prefetch_desc(&mQKV);
    tma_prefetch_desc(&mO);
    for (int k = 0; k < gm.nst; ++k) mbar_init(full + k, 1);
    fence_barrier_init();
  }
  __syncthreads();
  auto issue = [&](int u, int s) {       // one thread
    const int b = u / gm.ngrp, hg = u - b * gm.ngrp;
    mbar_expect_tx(full + s, stage_bytes);
    for (int hh = 0; hh < gm.G; ++hh) {
      const int col = (hg * gm.G + hh) * dh;
      for (int w3 = 0; w3 < 3; ++w3)
        for (int bx = 0; bx < gm.nbox; ++bx)
          tma_load_3d(&mQKV, full + s, tiles + s * stage_bytes + (hh * 3 + w3) * tb + bx * gm.BR * RB, w3 * gm.d + col,
                      bx * gm.BR, b);
    }
  };
  // input ring of nst stages: the copies of unit i + nst - 1 are issued at the top of iteration i, into the stage
  // iteration i - 1 has just finished reading (nst = 1: after this iteration's own barrier instead)
  const int ahead = gm.nst - 1;
  if (tid == 0)
    for (int k = 0; k < max(ahead, 1); ++k)
      if ((int)blockIdx.x + k * (int)gridDim.x < gm.units) issue(blockIdx.x + k * gridDim.x, k);
  const int last_k0 = ((NQ - 1) / NBC) * NBC;      // first block of the final chunk
  int i = 0, s = 0;
  uint32_t ph = 0;
  for (int u = blockIdx.x; u < gm.units; u += gridDim.x, ++i) {
    const int b = u / gm.ngrp, hg = u - b * gm.ngrp;
    if (ahead > 0 && tid == 0 && u + ahead * (int)gridDim.x < gm.units) issue(u + ahead * gridDim.x, (s + ahead) % gm.nst);
    mbar_wait(full + s, ph);
    const uint32_t so = so_base + (gm.nso == 2 ? (i & 1) : 0) * gm.G * tb;
    for (int item = warp; item < items; item += nw) {
      const int hh = item / NQ, qt = item - hh * NQ;
      const uint32_t qb = tiles + s * stage_bytes + (hh * 3) * tb, kb = qb + tb, vb = kb + tb;
      uint32_t aq[KD][4];
#pragma unroll
      for (int ks = 0; ks < KD; ++ks) ldsm_x4(aq[ks], addrA<KD>(qb, qt * 16, ks, lane));
      float o[2 * KD][4];
#pragma unroll
      for (int n = 0; n < 2 * KD; ++n) { o[n][0] = 0.f; o[n][1] = 0.f; o[n][2] = 0.f; o[n][3] = 0.f; }
      float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f;
      for (int k0 = 0; k0 < last_k0; k0 += NBC)
        fwd_chunk<KD, NBC, false>(kb, vb, k0, NBC, T, aq, o, m0, m1, l0, l1, gm.sl2, lane);
      fwd_chunk<KD, NBC, true>(kb, vb, last_k0, NQ - last_k0, T, aq, o, m0, m1, l0, l1, gm.sl2, lane);
      l0 += __shfl_xor_sync(0xffffffffu, l0, 1); l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
      l1 += __shfl_xor_sync(0xffffffffu, l1, 1); l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
      const float i0 = 1.f / l0, i1 = 1.f / l1;
      const int r0 = qt * 16 + g, r1 = r0 + 8;
      const uint32_t ot = so + hh * tb;
#pragma unroll
      for (int n = 0; n < 2 * KD; ++n) {
        sts32(chunk_addr<KD>(ot, r0, n) + cb * 2, pack2(o[n][0] * i0, o[n][1] * i0));
        sts32(chunk_addr<KD>(ot, r1, n) + cb * 2, pack2(o[n][2] * i1, o[n][3] * i1));
      }
      if (lse != nullptr && (lane & 3) == 0) {
        float* lp = lse + ((size_t)b * gm.h + hg * gm.G + hh) * T;
        if (r0 < T) lp[r0] = fmaf(m0, gm.sl2, __log2f(l0));
        if (r1 < T) lp[r1] = fmaf(m1, gm.sl2, __log2f(l1));
      }
    }
    fence_proxy_async();
    if (tid == 0) bulk_wait_read<0>();      // the previous unit's output tiles have left shared memory
    __syncthreads();
    if (tid == 0) {
      for (int hh = 0; hh < gm.G; ++hh)
        for (int bx = 0; bx < gm.nbox; ++bx)
          tma_store_3d(&mO, so + hh * tb + bx * gm.BR * RB, (hg * gm.G + hh) * dh, bx * gm.BR, b);
      bulk_commit();
      if (gm.nso == 1) bulk_wait_read<0>();
      if (gm.nst == 1 && u + (int)gridDim.x < gm.units) issue(u + gridDim.x, 0);
    }
    if (gm.nso == 1) __syncthreads();
    if (++s == gm.nst) { s = 0; ph ^= 1; }
  }
  if (tid == 0) bulk_wait_all();
}

// ===============================================================================================================
// Backward
// ===============================================================================================================
// shared memory: per head the tiles Q K V dO O(-> dQ staging) dKst dVst ; fp32 dQ accumulator [G][Tpad][dh+8] ;
// row statistics {lse2, delta*scale} [G][Tpad] ; column-sum slots for the bias gradients.  One input stage; the
// next unit's Q K V dO copies are issued as soon as the MMA loop is over, its O copy after the gradient stores
// have left the staging tiles.  Two CTAs per SM overlap one's copy / store phases with the other's MMA loop.
template <int KD, int MINB>
__global__ void __launch_bounds__(320, MINB)
attn_tile_bwd_kernel(const __grid_constant__ CUtensorMap mQKV, const __grid_constant__ CUtensorMap mOut,
                     const __grid_constant__ CUtensorMap mDO, const __grid_constant__ CUtensorMap mDQKV,
                     const TileGeom gm, const float* __restrict__ lse, float* __restrict__ dbias) {
  constexpr int dh = 16 * KD, RB = 32 * KD, DQP = dh + 8;
  extern __shared__ unsigned char smem_dyn[];
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023) & ~(uintptr_t)1023);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem);
  const uint32_t tiles = smem_u32(smem + SMEM_HDR);
  const uint32_t tb = (uint32_t)gm.tile_bytes;
  const int T = gm.T, Tpad = gm.Tpad, NQ = gm.NQ, G = gm.G, items = G * NQ;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, nt = blockDim.x, nw = nt >> 5;
  const int g = lane >> 2, cb = (lane & 3) * 2;
  float* sdq = reinterpret_cast<float*>(smem + SMEM_HDR + (size_t)7 * G * tb);     // [G][Tpad][DQP]
  float2* s_stat = reinterpret_cast<float2*>(sdq + (size_t)G * Tpad * DQP);         // [G][Tpad] {lse2, delta*scale}
  float* s_colkv = reinterpret_cast<float*>(s_stat + G * Tpad);                     // [items][2][dh]
  float* s_colq = s_colkv + (size_t)items * 2 * dh;                                 // [nw][G][dh]
  float* s_bias = s_colq + (size_t)nw * G * dh;                                     // [3d]
  const uint32_t sdq_u = smem_u32(sdq), stat_u = smem_u32(s_stat);
  auto tile = [&](int hh, int which) { return tiles + (uint32_t)(hh * 7 + which) * tb; };
  // lane-constant ldmatrix offsets inside a 16-row block (block bases are multiples of 16 rows, the swizzle term
  // depends on the row modulo 8 only)
  uint32_t offA[KD], offB[KD];
  {
    const int rA = (lane & 7) + ((lane >> 3) & 1) * 8, rB = (lane & 7) + (lane >> 4) * 8;
#pragma unroll
    for (int k = 0; k < KD; ++k) {
      offA[k] = (uint32_t)(rA * RB + (((2 * k + (lane >> 4)) ^ swz<KD>(rA)) << 4));
      offB[k] = (uint32_t)(rB * RB + (((2 * k + ((lane >> 3) & 1)) ^ swz<KD>(rB)) << 4));
    }
  }
  if (tid == 0) {
    tma_prefetch_desc(&mQKV); tma_prefetch_desc(&mOut); tma_prefetch_desc(&mDO); tma_prefetch_desc(&mDQKV);
    mbar_init(full, 1);
    fence_barrier_init();
  }
  if (dbias != nullptr)
    for (int c = tid; c < 3 * gm.d; c += nt) s_bias[c] = 0.f;
  __syncthreads();
  auto issue_main = [&](int u) {        // Q, K, V, dO of unit u (one thread); arms the barrier for all 5 tiles
    const int b = u / gm.ngrp, hg = u - b * gm.ngrp;
    mbar_expect_tx(full, 5u * G * tb);
    for (int hh = 0; hh < G; ++hh) {
      const int col = (hg * G + hh) * dh;
      for (int bx = 0; bx < gm.nbox; ++bx) {
        const uint32_t off = bx * gm.BR * RB;
        for (int w3 = 0; w3 < 3; ++w3) tma_load_3d(&mQKV, full, tile(hh, w3) + off, w3 * gm.d + col, bx * gm.BR, b);
        tma_load_3d(&mDO, full, tile(hh, 3) + off, col, bx * gm.BR, b);
      }
    }
  };
  auto issue_o = [&](int u) {
    const int b = u / gm.ngrp, hg = u - b * gm.ngrp;
    for (int hh = 0; hh < G; ++hh)
      for (int bx = 0; bx < gm.nbox; ++bx)
        tma_load_3d(&mOut, full, tile(hh, 4) + bx * gm.BR * RB, (hg * G + hh) * dh, bx * gm.BR, b);
  };
  if (tid == 0 && (int)blockIdx.x < gm.units) { issue_main(blockIdx.x); issue_o(blockIdx.x); }
  const int rounds = (items + nw - 1) / nw;
  int i = 0;
  for (int u = blockIdx.x; u < gm.units; u += gridDim.x, ++i) {
    const int b = u / gm.ngrp, hg = u - b * gm.ngrp;
    const bool has_next = u + (int)gridDim.x < gm.units;
    mbar_wait(full, i & 1);
    // row statistics: lse2 from the forward, delta = rowsum(dO * O) (pre-multiplied by the softmax scale)
    for (int idx = tid; idx < G * Tpad; idx += nt) {
      const int hh = idx / Tpad, r = idx - hh * Tpad;
      float dl = 0.f, l2 = INFINITY;            // padded query rows: P = exp2(s - inf) = 0
      if (r < T) {
        l2 = __ldg(lse + ((size_t)b * gm.h + hg * G + hh) * T + r);
#pragma unroll
        for (int ch = 0; ch < 2 * KD; ++ch) {
          const uint4 a = lds128(chunk_addr<KD>(tile(hh, 3), r, ch)), o4 = lds128(chunk_addr<KD>(tile(hh, 4), r, ch));
          dl += bf_lo(a.x) * bf_lo(o4.x) + bf_hi(a.x) * bf_hi(o4.x) + bf_lo(a.y) * bf_lo(o4.y) + bf_hi(a.y) * bf_hi(o4.y) +
                bf_lo(a.z) * bf_lo(o4.z) + bf_hi(a.z) * bf_hi(o4.z) + bf_lo(a.w) * bf_lo(o4.w) + bf_hi(a.w) * bf_hi(o4.w);
        }
      }
      s_stat[idx] = make_float2(l2, dl * gm.scale);
    }
    for (int idx = tid; idx < G * Tpad * DQP / 4; idx += nt) reinterpret_cast<float4*>(sdq)[idx] = make_float4(0.f, 0.f, 0.f, 0.f);
    __syncthreads();
    for (int rd = 0; rd < rounds; ++rd) {
      const int item = rd * nw + warp;
      const bool live = item < items;
      const int hh = live ? item / NQ : 0, kt = live ? item - hh * NQ : 0;
      const uint32_t qb = tile(hh, 0), kb = qb + tb, vb = kb + tb;
      uint32_t ak[KD][4], av[KD][4], kB[KD][4];
      float dk[2 * KD][4], dv[2 * KD][4];
#pragma unroll
      for (int ks = 0; ks < KD; ++ks) {
        const uint32_t ra = (uint32_t)(kt * 16 * RB) + offA[ks];
        ldsm_x4(ak[ks], kb + ra);
        ldsm_x4(av[ks], vb + ra);
        ldsm_x4_t(kB[ks], kb + ra);
      }
#pragma unroll
      for (int n = 0; n < 2 * KD; ++n) {
        dk[n][0] = 0.f; dk[n][1] = 0.f; dk[n][2] = 0.f; dk[n][3] = 0.f;
        dv[n][0] = 0.f; dv[n][1] = 0.f; dv[n][2] = 0.f; dv[n][3] = 0.f;
      }
      const uint32_t stat_h = stat_u + (uint32_t)((hh * Tpad + cb) * 8);
      const uint32_t dq_h = sdq_u + (uint32_t)(((hh * Tpad + g) * DQP + cb) * 4);
      int qbk = kt;
      for (int step = 0; step < NQ; ++step) {
        if (live) {
          const uint32_t qblk = qb + (uint32_t)(qbk * 16 * RB), oblk = qblk + 3u * tb;
          const uint32_t dqa = dq_h + (uint32_t)(qbk * 16 * DQP * 4);
          // this warp is the only one on query block qbk during this step: its dQ rows are the accumulator (C
          // operand) of the dS K product -- a plain read-modify-write, no atomics
          float dq[2 * KD][4];
#pragma unroll
          for (int n = 0; n < 2 * KD; ++n) {
            const float2 a0 = lds64f(dqa + n * 32), a1 = lds64f(dqa + 8 * DQP * 4 + n * 32);
            dq[n][0] = a0.x; dq[n][1] = a0.y; dq[n][2] = a1.x; dq[n][3] = a1.y;
          }
          float stt[2][4] = {}, dpt[2][4] = {};      // S^T and dP^T blocks: rows = keys, cols = queries
#pragma unroll
          for (int ks = 0; ks < KD; ++ks) {
            uint32_t bfr[4];
            ldsm_x4(bfr, qblk + offB[ks]);
            mma_bf16(stt[0], ak[ks], bfr[0], bfr[1]);
            mma_bf16(stt[1], ak[ks], bfr[2], bfr[3]);
            ldsm_x4(bfr, oblk + offB[ks]);
            mma_bf16(dpt[0], av[ks], bfr[0], bfr[1]);
            mma_bf16(dpt[1], av[ks], bfr[2], bfr[3]);
          }
          uint32_t pa[4], sa[4];
#pragma unroll
          for (int u2 = 0; u2 < 2; ++u2) {
            const float4 st4 = lds128f(stat_h + (uint32_t)(qbk * 16 * 8) + u2 * 64);   // {lse2, dls} of queries cb, cb+1
            const float p0 = ex2(fmaf(stt[u2][0], gm.sl2, -st4.x)), p1 = ex2(fmaf(stt[u2][1], gm.sl2, -st4.z));
            const float p2 = ex2(fmaf(stt[u2][2], gm.sl2, -st4.x)), p3 = ex2(fmaf(stt[u2][3], gm.sl2, -st4.z));
            pa[2 * u2] = pack2(p0, p1);
            pa[2 * u2 + 1] = pack2(p2, p3);
            sa[2 * u2] = pack2(p0 * fmaf(dpt[u2][0], gm.scale, -st4.y), p1 * fmaf(dpt[u2][1], gm.scale, -st4.w));
            sa[2 * u2 + 1] = pack2(p2 * fmaf(dpt[u2][2], gm.scale, -st4.y), p3 * fmaf(dpt[u2][3], gm.scale, -st4.w));
          }
#pragma unroll
          for (int np = 0; np < KD; ++np) {
            uint32_t bfr[4];
            ldsm_x4_t(bfr, oblk + offA[np]);     // B[k = query][n = c] = dO[query][c]
            mma_bf16(dv[2 * np], pa, bfr[0], bfr[1]);
            mma_bf16(dv[2 * np + 1], pa, bfr[2], bfr[3]);
            ldsm_x4_t(bfr, qblk + offA[np]);     // B[k = query][n = c] = Q[query][c]
            mma_bf16(dk[2 * np], sa, bfr[0], bfr[1]);
            mma_bf16(dk[2 * np + 1], sa, bfr[2], bfr[3]);
          }
          // dQ block += dS K_tile: A = dS = (dS^T)^T, one movmatrix per 8x8 sub-block
          const uint32_t da[4] = {movm_t(sa[0]), movm_t(sa[2]), movm_t(sa[1]), movm_t(sa[3])};
#pragma unroll
          for (int np = 0; np < KD; ++np) {
            mma_bf16(dq[2 * np], da, kB[np][0], kB[np][1]);
            mma_bf16(dq[2 * np + 1], da, kB[np][2], kB[np][3]);
          }
#pragma unroll
          for (int n = 0; n < 2 * KD; ++n) {
            sts64f(dqa + n * 32, dq[n][0], dq[n][1]);
            sts64f(dqa + 8 * DQP * 4 + n * 32, dq[n][2], dq[n][3]);
          }
        }
        if (++qbk == NQ) qbk = 0;
        __syncthreads();
      }
      if (live) {
        const int r0 = kt * 16 + g, r1 = r0 + 8;
        const uint32_t kt_ = tile(hh, 5), vt_ = tile(hh, 6);
#pragma unroll
        for (int n = 0; n < 2 * KD; ++n) {
          sts32(chunk_addr<KD>(kt_, r0, n) + cb * 2, pack2(dk[n][0], dk[n][1]));
          sts32(chunk_addr<KD>(kt_, r1, n) + cb * 2, pack2(dk[n][2], dk[n][3]));
          sts32(chunk_addr<KD>(vt_, r0, n) + cb * 2, pack2(dv[n][0], dv[n][1]));
          sts32(chunk_addr<KD>(vt_, r1, n) + cb * 2, pack2(dv[n][2], dv[n][3]));
        }
        if (dbias != nullptr) {           // column sums of this key tile's real rows -> slot [item][dK | dV][dh]
          const float w0 = r0 < T ? 1.f : 0.f, w1 = r1 < T ? 1.f : 0.f;
#pragma unroll
          for (int n = 0; n < 2 * KD; ++n)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
              float a = dk[n][e] * w0 + dk[n][2 + e] * w1, c2 = dv[n][e] * w0 + dv[n][2 + e] * w1;
#pragma unroll
              for (int o = 4; o < 32; o <<= 1) {
                a += __shfl_xor_sync(0xffffffffu, a, o);
                c2 += __shfl_xor_sync(0xffffffffu, c2, o);
              }
              if (g == 0) {
                s_colkv[(item * 2) * dh + n * 8 + cb + e] = a;
                s_colkv[(item * 2 + 1) * dh + n * 8 + cb + e] = c2;
              }
            }
        }
      }
    }
    __syncthreads();                        // every tile read and every dQ / dK / dV write of this unit is done
    if (tid == 0 && has_next) issue_main(u + gridDim.x);
    // dQ fp32 -> bf16 into the (now dead) O tile; a thread keeps one 8-column chunk, so its column sums stay in registers
    for (int hh = 0; hh < G; ++hh) {
      const int ch = tid % (2 * KD);
      float cs[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      for (int r = tid / (2 * KD); r < Tpad; r += nt / (2 * KD)) {
        const uint32_t pa_ = sdq_u + (uint32_t)((((hh * Tpad + r) * DQP) + ch * 8) * 4);
        const float4 a = lds128f(pa_), c4 = lds128f(pa_ + 16);
        sts128(chunk_addr<KD>(tile(hh, 4), r, ch), pack2(a.x, a.y), pack2(a.z, a.w), pack2(c4.x, c4.y), pack2(c4.z, c4.w));
        cs[0] += a.x; cs[1] += a.y; cs[2] += a.z; cs[3] += a.w; cs[4] += c4.x; cs[5] += c4.y; cs[6] += c4.z; cs[7] += c4.w;
      }
      if (dbias != nullptr) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
#pragma unroll
          for (int o = 2 * KD; o < 32; o <<= 1) cs[j] += __shfl_xor_sync(0xffffffffu, cs[j], o);
        }
        if (lane < 2 * KD) {
#pragma unroll
          for (int j = 0; j < 8; ++j) s_colq[(warp * G + hh) * dh + lane * 8 + j] = cs[j];
        }
      }
    }
    fence_proxy_async();
    __syncthreads();
    if (tid == 0) {
      for (int hh = 0; hh < G; ++hh) {
        const int col = (hg * G + hh) * dh;
        for (int bx = 0; bx < gm.nbox; ++bx) {
          const uint32_t off = bx * gm.BR * RB;
          tma_store_3d(&mDQKV, tile(hh, 4) + off, col, bx * gm.BR, b);
          tma_store_3d(&mDQKV, tile(hh, 5) + off, gm.d + col, bx * gm.BR, b);
          tma_store_3d(&mDQKV, tile(hh, 6) + off, 2 * gm.d + col, bx * gm.BR, b);
        }
      }
      bulk_commit();
      bulk_wait_read<0>();
      if (has_next) issue_o(u + gridDim.x);
    }
    if (dbias != nullptr) {                 // fold the slots into the CTA's running bias-gradient sums
      for (int c = tid; c < 3 * G * dh; c += nt) {
        const int w3 = c / (G * dh), rem = c - w3 * (G * dh), hh = rem / dh, cc = rem - hh * dh;
        float acc = 0.f;
        if (w3 == 0) {
          for (int w = 0; w < nw; ++w) acc += s_colq[(w * G + hh) * dh + cc];
        } else {
          for (int kt = 0; kt < NQ; ++kt) acc += s_colkv[((hh * NQ + kt) * 2 + (w3 - 1)) * dh + cc];
        }
        s_bias[w3 * gm.d + (hg * G + hh) * dh + cc] += acc;
      }
    }
  }
  if (tid == 0) bulk_wait_all();
  if (dbias != nullptr) {
    __syncthreads();
    for (int c = tid; c < 3 * gm.d; c += nt) {
      const float v = s_bias[c];
      if (v != 0.f) atomicAdd(dbias + c, v);
    }
  }
}

// ---- host side -------------------------------------------------------------------------------------------------
constexpr size_t SMEM_MAX = 227 * 1024;

size_t fwd_bytes(const TileGeom& g) { return 1024 + SMEM_HDR + (size_t)(3 * g.nst + g.nso) * g.G * g.tile_bytes; }
size_t bwd_bytes(const TileGeom& g, int dh) {
  return 1024 + SMEM_HDR + (size_t)7 * g.G * g.tile_bytes + (size_t)g.G * g.Tpad * (dh + 8) * 4 + (size_t)2 * g.G * g.Tpad * 4 +
         (size_t)g.G * g.NQ * 2 * dh * 4 + (size_t)10 * g.G * dh * 4 + (size_t)3 * g.d * 4;
}

void base_geom(TileGeom& g, int B, int T, int h, int dh) {
  g.T = T; g.NQ = (T + 15) / 16; g.Tpad = g.NQ * 16; g.h = h; g.d = h * dh;
  g.nbox = g.Tpad > 256 ? 2 : 1;
  g.BR = g.Tpad / g.nbox;
  g.tile_bytes = g.Tpad * dh * 2;
  g.scale = 1.f / sqrtf((float)dh);
  g.sl2 = g.scale * 1.4426950408889634f;
  g.nst = g.nso = 1;
  (void)B;
}
void set_group(TileGeom& g, int B, int G) { g.G = G; g.ngrp = g.h / G; g.units = B * g.ngrp; }
// warps for `items` equal work items: at most 10 warps, the fewest rounds, no idle warp in the last round if possible
int pick_warps(int items) {
  const int rounds = (items + 9) / 10;
  return (items + rounds - 1) / rounds;
}

}  // namespace

int attn_make_map3(CUtensorMap* map, const void* base, int B, int T, int cols, int dh, int box_rows) {
  AMC_CHECK_ARG((reinterpret_cast<uintptr_t>(base) & 15) == 0 && (cols * 2) % 16 == 0,
                "attention tensors must be 16-byte aligned with a 16-byte row pitch");
  const cuuint64_t dims[3] = {(cuuint64_t)cols, (cuuint64_t)T, (cuuint64_t)B};
  const cuuint64_t strides[2] = {(cuuint64_t)cols * 2, (cuuint64_t)T * cols * 2};
  const cuuint32_t box[3] = {(cuuint32_t)dh, (cuuint32_t)box_rows, 1};
  const CUtensorMapSwizzle sw = dh == 16 ? CU_TENSOR_MAP_SWIZZLE_32B : (dh == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B);
  return encode_tiled_map(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, base, dims, strides, box, sw,
                          CU_TENSOR_MAP_L2_PROMOTION_L2_128B);
}

bool attn_tiles_supported(int T, int h, int dh) {
  return T > 16 && T <= 288 && (dh == 16 || dh == 32 || dh == 64) && h >= 1;
}

int attn_tiles_fwd(int B, int T, int h, int dh, const bf16* qkv, bf16* out, float* lse, bool* handled, cudaStream_t st) {
  *handled = false;
  if (!attn_tiles_supported(T, h, dh)) return 0;
  TileGeom g;
  base_geom(g, B, T, h, dh);
  // heads per CTA: enough (about two per warp) work items per unit to amortise the per-unit barrier / copy issue,
  // while two input stages + two output stagings still let two CTAs share an SM; then as many input stages (<= 4) as fit
  const size_t budget = (SMEM_MAX - 2048) / 2;
  int G = 0;
  for (int c = 1; c <= h; ++c) {
    if (h % c) continue;
    set_group(g, B, c);
    g.nst = 2; g.nso = 2;
    if (G != 0 && (fwd_bytes(g) > budget || c * g.NQ > 20)) break;
    G = c;
  }
  set_group(g, B, G);
  g.nst = 2; g.nso = 2;
  if (fwd_bytes(g) > SMEM_MAX) { g.nso = 1; }
  if (fwd_bytes(g) > SMEM_MAX) { g.nst = 1; }
  if (fwd_bytes(g) > SMEM_MAX) return 0;
  while (g.nst < 4) {
    ++g.nst;
    if (fwd_bytes(g) > budget) { --g.nst; break; }
  }
  const size_t sm = fwd_bytes(g);
  const int threads = 32 * pick_warps(G * g.NQ);
  CUtensorMap mQKV, mO;
  AMC_TRY(attn_make_map3(&mQKV, qkv, B, T, 3 * g.d, dh, g.BR));
  AMC_TRY(attn_make_map3(&mO, out, B, T, g.d, dh, g.BR));
#define AMC_TILE_FWD(KD, NBC)                                                                                         \
  do {                                                                                                                \
    auto kern = attn_tile_fwd_kernel<KD, NBC, 2>;                                                                      \
    AMC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_MAX));                 \
    int occ = 1;                                                                                                      \
    AMC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, threads, sm));                                 \
    const int grid = std::min(g.units, device_sm_count() * std::max(occ, 1));                                         \
    kern<<<grid, threads, sm, st>>>(mQKV, mO, g, lse);                                                                \
  } while (0)
#define AMC_TILE_FWD_KD(KD)                            \
  do {                                                 \
    if ((g.NQ == 4 || g.NQ == 5) && KD < 4) AMC_TILE_FWD(KD, 5);   \
    else AMC_TILE_FWD(KD, 3);                          \
  } while (0)
  if (dh == 16) AMC_TILE_FWD_KD(1);
  else if (dh == 32) AMC_TILE_FWD_KD(2);
  else AMC_TILE_FWD_KD(4);
#undef AMC_TILE_FWD_KD
#undef AMC_TILE_FWD
  AMC_LAUNCH_CHECK();
  *handled = true;
  return 0;
}

int attn_tiles_bwd(int B, int T, int h, int dh, const bf16* qkv, const bf16* out, const float* lse, const bf16* dout,
                   bf16* dqkv, float* dbias, bool* handled, cudaStream_t st) {
  *handled = false;
  if (!attn_tiles_supported(T, h, dh) || out == nullptr || lse == nullptr) return 0;
  TileGeom g;
  base_geom(g, B, T, h, dh);
  const size_t budget = (SMEM_MAX - 2048) / 2;
  int G = 0;
  for (int c = 1; c <= h; ++c) {
    if (h % c) continue;
    set_group(g, B, c);
    if (bwd_bytes(g, dh) > SMEM_MAX) break;
    if (G != 0 && (bwd_bytes(g, dh) > budget || c * g.NQ > 20)) break;
    G = c;
  }
  if (G == 0) return 0;
  set_group(g, B, G);
  const size_t sm = bwd_bytes(g, dh);
  const int threads = 32 * pick_warps(G * g.NQ);
  CUtensorMap mQKV, mOut, mDO, mDQKV;
  AMC_TRY(attn_make_map3(&mQKV, qkv, B, T, 3 * g.d, dh, g.BR));
  AMC_TRY(attn_make_map3(&mOut, out, B, T, g.d, dh, g.BR));
  AMC_TRY(attn_make_map3(&mDO, dout, B, T, g.d, dh, g.BR));
  AMC_TRY(attn_make_map3(&mDQKV, dqkv, B, T, 3 * g.d, dh, g.BR));
#define AMC_TILE_BWD(KD, MINB)                                                                                        \
  do {                                                                                                                \
    auto kern = attn_tile_bwd_kernel<KD, MINB>;                                                                        \
    AMC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_MAX));                 \
    int occ = 1;                                                                                                      \
    AMC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, threads, sm));                                 \
    const int grid = std::min(g.units, device_sm_count() * std::max(occ, 1));                                         \
    kern<<<grid, threads, sm, st>>>(mQKV, mOut, mDO, mDQKV, g, lse, dbias);                                           \
  } while (0)
  const bool two = 2 * (sm + 1024) <= SMEM_MAX + 1024;      // two CTAs per SM fit: cap registers for it
  if (dh == 16) { if (two) AMC_TILE_BWD(1, 2); else AMC_TILE_BWD(1, 1); }
  else if (dh == 32) { if (two) AMC_TILE_BWD(2, 2); else AMC_TILE_BWD(2, 1); }
  else AMC_TILE_BWD(4, 1);
#undef AMC_TILE_BWD
  AMC_LAUNCH_CHECK();
  *handled = true;
  return 0;
}

}  // namespace amc

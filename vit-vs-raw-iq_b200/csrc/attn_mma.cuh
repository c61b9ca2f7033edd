// Building blocks of the mma.sync / TMA attention kernels (attn_tiles.cu, attn_long.cu, and the leftover rows of
// attn_tc5.cu): the swizzled-tile addressing and the forward chunk of a 16-query-row item.
#pragma once
#include "ptx.cuh"

namespace amc {
// bf16 tensor [B][T][cols] (row pitch = cols) as a 3-D TMA map, box = {dh, box_rows, 1}, swizzle span = dh * 2 bytes
int attn_make_map3(CUtensorMap* map, const void* base, int B, int T, int cols, int dh, int box_rows);

namespace {

// ---- swizzled tile addressing --------------------------------------------------------------------------------
// A tile is Tpad rows of RB = 32*KD bytes written by TMA with SWIZZLE_{32,64,128}B: the 16-byte chunk index is
// XORed with address bits [7, 7+log2(chunks per row)); tile bases are aligned to 1024 B so those bits are a
// function of the row alone.
template <int KD> __device__ __forceinline__ int swz(int r) {
  return KD == 1 ? ((r >> 2) & 1) : (KD == 2 ? ((r >> 1) & 3) : (r & 7));
}
template <int KD> __device__ __forceinline__ uint32_t chunk_addr(uint32_t tile, int r, int ch) {
  return tile + (uint32_t)(r * (32 * KD)) + (uint32_t)((ch ^ swz<KD>(r)) << 4);
}
// ldmatrix.x4 lane addresses over a 16-row x 16-column block (rows row0.., columns 16*ks..):
//  pattern A: matrices = (rows 0-7, cols 0-7), (rows 8-15, cols 0-7), (rows 0-7, cols 8-15), (rows 8-15, cols 8-15)
//             -> A operand (non-trans) / [k][n] B operand of two n-blocks (with .trans)
//  pattern B: matrices = (rows 0-7, cols 0-7), (rows 0-7, cols 8-15), (rows 8-15, cols 0-7), (rows 8-15, cols 8-15)
//             -> B operand pairs {b0,b1} for n-block rows 0-7 and {b2,b3} for n-block rows 8-15 (rows = n, cols = k)
template <int KD> __device__ __forceinline__ uint32_t addrA(uint32_t tile, int row0, int ks, int lane) {
  return chunk_addr<KD>(tile, row0 + (lane & 7) + ((lane >> 3) & 1) * 8, 2 * ks + (lane >> 4));
}
template <int KD> __device__ __forceinline__ uint32_t addrB(uint32_t tile, int row0, int ks, int lane) {
  return chunk_addr<KD>(tile, row0 + (lane & 7) + (lane >> 4) * 8, 2 * ks + ((lane >> 3) & 1));
}

// ---- forward building block --------------------------------------------------------------------------------
// One chunk of NBC key blocks (16 keys each) of a 16-query-row item: S = Q K^T, online-softmax update, O += P V.
// LAST = false: all NBC blocks exist and none needs masking -> straight-line code.
// LAST = true : the final chunk of the row: `nblk` (1..NBC) blocks exist and the zero-filled key rows >= T of the
//               very last block are masked to -inf.
template <int KD, int NBC, bool LAST>
__device__ __forceinline__ void fwd_chunk(uint32_t kb, uint32_t vb, int k0, int nblk, int T, const uint32_t (&aq)[KD][4],
                                          float (&o)[2 * KD][4], float& m0, float& m1, float& l0, float& l1, float sl2,
                                          int lane) {
  const int cb = (lane & 3) * 2;
  float c[2 * NBC][4];
#pragma unroll
  for (int n = 0; n < 2 * NBC; ++n) { c[n][0] = 0.f; c[n][1] = 0.f; c[n][2] = 0.f; c[n][3] = 0.f; }
#pragma unroll
  for (int j = 0; j < NBC; ++j) {
    if (!LAST || j < nblk) {
#pragma unroll
      for (int ks = 0; ks < KD; ++ks) {
        uint32_t bfr[4];
        ldsm_x4(bfr, addrB<KD>(kb, (k0 + j) * 16, ks, lane));
        mma_bf16(c[2 * j], aq[ks], bfr[0], bfr[1]);
        mma_bf16(c[2 * j + 1], aq[ks], bfr[2], bfr[3]);
      }
    }
  }
  if (LAST) {      // keys >= T (zero-filled rows of the last block, and blocks past the end) take no probability mass
#pragma unroll
    for (int n = 0; n < 2 * NBC; ++n) {
      const int key = k0 * 16 + n * 8 + cb;
      if (key >= T) { c[n][0] = -INFINITY; c[n][2] = -INFINITY; }
      if (key + 1 >= T) { c[n][1] = -INFINITY; c[n][3] = -INFINITY; }
    }
  }
  float x0 = -INFINITY, x1 = -INFINITY;
#pragma unroll
  for (int n = 0; n < 2 * NBC; ++n) {
    x0 = fmaxf(x0, fmaxf(c[n][0], c[n][1]));
    x1 = fmaxf(x1, fmaxf(c[n][2], c[n][3]));
  }
  x0 = fmaxf(x0, __shfl_xor_sync(0xffffffffu, x0, 1)); x0 = fmaxf(x0, __shfl_xor_sync(0xffffffffu, x0, 2));
  x1 = fmaxf(x1, __shfl_xor_sync(0xffffffffu, x1, 1)); x1 = fmaxf(x1, __shfl_xor_sync(0xffffffffu, x1, 2));
  const float n0 = fmaxf(m0, x0), n1 = fmaxf(m1, x1);
  const float al0 = ex2((m0 - n0) * sl2), al1 = ex2((m1 - n1) * sl2);   // first chunk: ex2(-inf) = 0
  m0 = n0; m1 = n1;
  const float ms0 = m0 * sl2, ms1 = m1 * sl2;
  float s0 = 0.f, s1 = 0.f;
#pragma unroll
  for (int n = 0; n < 2 * NBC; ++n) {
    c[n][0] = ex2(fmaf(c[n][0], sl2, -ms0)); c[n][1] = ex2(fmaf(c[n][1], sl2, -ms0));
    c[n][2] = ex2(fmaf(c[n][2], sl2, -ms1)); c[n][3] = ex2(fmaf(c[n][3], sl2, -ms1));
    s0 += c[n][0] + c[n][1];
    s1 += c[n][2] + c[n][3];
  }
  l0 = fmaf(l0, al0, s0);
  l1 = fmaf(l1, al1, s1);
#pragma unroll
  for (int n = 0; n < 2 * KD; ++n) { o[n][0] *= al0; o[n][1] *= al0; o[n][2] *= al1; o[n][3] *= al1; }
#pragma unroll
  for (int j = 0; j < NBC; ++j) {
    if (!LAST || j < nblk) {
      const uint32_t pa[4] = {pack2(c[2 * j][0], c[2 * j][1]), pack2(c[2 * j][2], c[2 * j][3]),
                              pack2(c[2 * j + 1][0], c[2 * j + 1][1]), pack2(c[2 * j + 1][2], c[2 * j + 1][3])};
#pragma unroll
      for (int np = 0; np < KD; ++np) {
        uint32_t bfr[4];
        ldsm_x4_t(bfr, addrA<KD>(vb, (k0 + j) * 16, np, lane));
        mma_bf16(o[2 * np], pa, bfr[0], bfr[1]);
        mma_bf16(o[2 * np + 1], pa, bfr[2], bfr[3]);
      }
    }
  }
}

}  // namespace
}  // namespace amc

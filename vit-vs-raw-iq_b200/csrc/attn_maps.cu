// Attention maps for analysing a trained model: the probabilities P = softmax(q k^T / sqrt(dh)) that the reference's
// ScaleDotProductAttention returns as `score` (R/models/layers/scale_dot_product_attention.py:26-39) and the fused
// forward kernels never write, and one attention-rollout step, which needs P only as a reduction and never writes it.
//
// Both kernels read the [B*T, 3d] qkv buffer of the forward (either dtype) and compute their own row statistics, so they
// work after every forward kernel, including the ones that keep no `lse`.  The unit of work is one warp on a tile of 16
// query rows of one (frame, head): S for 64 keys at a time, on mma.sync m16n8k16 for bf16 and on the FMA pipe for fp32,
// into the same accumulator layout (lane: rows g = lane/4 and g + 8, keys 8n + 2(lane%4) + {0,1}).  Pass 1 forms each
// row's max and sum over all keys; pass 2 uses them.  Warps never wait for each other inside a tile.
//
//   attn_probs_kernel    P as fp32 [B, h, T, T].  For T <= PROBS_ROW_MAX the tile's log2-domain logits are staged whole in
//                        shared memory by pass 1 and written out normalised; longer rows recompute S in pass 2, 64 keys at
//                        a time.  Each row segment leaves in 16-byte streaming stores (the staged copy sits at the same
//                        address modulo 16 as its destination, so rows of any length vectorise).
//   attn_rollout_kernel  v_out = 0.5 v_in + (0.5 / h) sum_hh v_in^T P_hh, one CTA per frame.  Each warp adds its tiles'
//                        column sums into its own shared-memory row; the CTA (up to 16 warps) then sums the warps in a
//                        fixed order: no atomics, bit-reproducible.  Tiles whose 16 v_in entries are all zero are
//                        skipped, so the top layer of a CLS model (v_in = e_0) costs one tile per head.
//                        With REL, one step of class-specific relevance (Chefer, Gur & Wolf, ICCV 2021):
//                        v_out = v_in + (1 / h) sum_hh v_in^T relu(dP_hh * P_hh), dP = dO V^T the gradient of the target
//                        score w.r.t. P.  The tile's dO rows sit next to its Q rows and each V chunk next to its K
//                        chunk; pass 2 forms dP with the same chunk product as S.  dO rows whose v_in is 0 are zero-filled
//                        on load, never read: under the CLS-row top layer only row 0 of each frame's dO is written.
#include "attention.cuh"
#include "ptx.cuh"

namespace amc {
namespace {

constexpr int KC = 64;                // keys per chunk
constexpr int PROBS_ROW_MAX = 512;    // probs: longest row staged whole (16 x 528 fp32 = 33 KB per warp)
constexpr int SMEM_CAP = 200 * 1024;  // dynamic shared memory per CTA the launchers plan with

// per-warp tile geometry: head dim padded to DHP = 16 KD, row pitch LDE elements (16-byte rows; for bf16 the 8-element pad
// makes the ldmatrix rows conflict-free, for fp32 the 4-element pad spreads the 8 query rows over distinct banks)
template <typename E, int KD> struct Geo {
  static constexpr int DHP = 16 * KD;
  static constexpr int LDE = std::is_same<E, bf16>::value ? DHP + 8 : DHP + 4;
  static constexpr int VEC = 16 / (int)sizeof(E);
  static constexpr size_t q_bytes = (size_t)16 * LDE * sizeof(E);
  static constexpr size_t k_bytes = (size_t)KC * LDE * sizeof(E);
};

// dst[r][c] = src[r * ld + c] for r < nvalid, c < dh and bit r % 32 of `live` set, zero elsewhere (r < nrows, c < DHP)
template <typename E, int KD>
__device__ __forceinline__ void load_rows(E* dst, const E* __restrict__ src, int ld, int nvalid, int nrows, int dh,
                                          bool vec, int lane, uint32_t live = 0xffffffffu) {
  using G = Geo<E, KD>;
  if (vec) {
    constexpr int CPR = G::DHP / G::VEC;
    for (int i = lane; i < nrows * CPR; i += 32) {
      const int r = i / CPR, c = (i - r * CPR) * G::VEC;
      uint4 v = make_uint4(0u, 0u, 0u, 0u);
      if (r < nvalid && c < dh && ((live >> (r & 31)) & 1u)) v = __ldg(reinterpret_cast<const uint4*>(src + (size_t)r * ld + c));
      *reinterpret_cast<uint4*>(dst + r * G::LDE + c) = v;
    }
  } else {
    for (int i = lane; i < nrows * G::DHP; i += 32) {
      const int r = i / G::DHP, c = i - r * G::DHP;
      dst[r * G::LDE + c] = (r < nvalid && c < dh && ((live >> (r & 31)) & 1u)) ? src[(size_t)r * ld + c] : from_f<E>(0.f);
    }
  }
}

// query-row A fragments of the tile (bf16 only; the fp32 path reads Qs directly)
template <typename E, int KD>
__device__ __forceinline__ void load_qfrag(const E* Qs, uint32_t (&aq)[KD][4], int lane) {
  if constexpr (std::is_same<E, bf16>::value) {
    using G = Geo<E, KD>;
    const int row = (lane & 7) + ((lane >> 3) & 1) * 8;
#pragma unroll
    for (int ks = 0; ks < KD; ++ks) ldsm_x4(aq[ks], smem_u32(Qs + row * G::LDE + ks * 16 + (lane >> 4) * 8));
  }
}

// c = Q K^T for the 16 rows and the 64 keys of the chunk in Ks (keys >= T are NOT masked here)
template <typename E, int KD>
__device__ __forceinline__ void chunk_scores(const E* Qs, const E* Ks, const uint32_t (&aq)[KD][4], float (&c)[8][4],
                                             int lane) {
  using G = Geo<E, KD>;
#pragma unroll
  for (int n = 0; n < 8; ++n) { c[n][0] = 0.f; c[n][1] = 0.f; c[n][2] = 0.f; c[n][3] = 0.f; }
  if constexpr (std::is_same<E, bf16>::value) {
    const int row = (lane & 7) + (lane >> 4) * 8, col = ((lane >> 3) & 1) * 8;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
#pragma unroll
      for (int ks = 0; ks < KD; ++ks) {
        uint32_t b[4];
        ldsm_x4(b, smem_u32(Ks + (j * 16 + row) * G::LDE + ks * 16 + col));
        mma_bf16(c[2 * j], aq[ks], b[0], b[1]);
        mma_bf16(c[2 * j + 1], aq[ks], b[2], b[3]);
      }
    }
  } else {
    const int g = lane >> 2, q2 = (lane & 3) * 2;
    const float* q0 = Qs + g * G::LDE;
    const float* q1 = q0 + 8 * G::LDE;
#pragma unroll 4
    for (int kk = 0; kk < G::DHP; ++kk) {
      const float a0 = q0[kk], a1 = q1[kk];
#pragma unroll
      for (int n = 0; n < 8; ++n) {
        const float k0 = Ks[(n * 8 + q2) * G::LDE + kk], k1 = Ks[(n * 8 + q2 + 1) * G::LDE + kk];
        c[n][0] = fmaf(a0, k0, c[n][0]); c[n][1] = fmaf(a0, k1, c[n][1]);
        c[n][2] = fmaf(a1, k0, c[n][2]); c[n][3] = fmaf(a1, k1, c[n][3]);
      }
    }
  }
}

// log2-domain logits x = s * log2(e) / sqrt(dh); keys >= T -> -inf
__device__ __forceinline__ void scale_mask(float (&c)[8][4], int k0, int T, float sl2, int lane) {
  const int q2 = (lane & 3) * 2;
#pragma unroll
  for (int n = 0; n < 8; ++n) {
    const int key = k0 + n * 8 + q2;
    c[n][0] = key < T ? c[n][0] * sl2 : -INFINITY;
    c[n][2] = key < T ? c[n][2] * sl2 : -INFINITY;
    c[n][1] = key + 1 < T ? c[n][1] * sl2 : -INFINITY;
    c[n][3] = key + 1 < T ? c[n][3] * sl2 : -INFINITY;
  }
}

// online max / sum over one chunk for rows g (m0, l0) and g + 8 (m1, l1); the max is kept equal across the quad of lanes
// that share a row (every chunk holds at least one key < T, so it is finite); the sums stay per lane until row_sums()
__device__ __forceinline__ void update_stats(const float (&c)[8][4], float& m0, float& m1, float& l0, float& l1) {
  float x0 = -INFINITY, x1 = -INFINITY;
#pragma unroll
  for (int n = 0; n < 8; ++n) {
    x0 = fmaxf(x0, fmaxf(c[n][0], c[n][1]));
    x1 = fmaxf(x1, fmaxf(c[n][2], c[n][3]));
  }
  x0 = fmaxf(x0, __shfl_xor_sync(0xffffffffu, x0, 1)); x0 = fmaxf(x0, __shfl_xor_sync(0xffffffffu, x0, 2));
  x1 = fmaxf(x1, __shfl_xor_sync(0xffffffffu, x1, 1)); x1 = fmaxf(x1, __shfl_xor_sync(0xffffffffu, x1, 2));
  const float n0 = fmaxf(m0, x0), n1 = fmaxf(m1, x1);
  float s0 = 0.f, s1 = 0.f;
#pragma unroll
  for (int n = 0; n < 8; ++n) {
    s0 += ex2(c[n][0] - n0) + ex2(c[n][1] - n0);
    s1 += ex2(c[n][2] - n1) + ex2(c[n][3] - n1);
  }
  l0 = fmaf(l0, ex2(m0 - n0), s0);   // first chunk: ex2(-inf) = 0
  l1 = fmaf(l1, ex2(m1 - n1), s1);
  m0 = n0; m1 = n1;
}
__device__ __forceinline__ void row_sums(float& l0, float& l1) {
  l0 += __shfl_xor_sync(0xffffffffu, l0, 1); l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 1); l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
}

// Pass 1 over every key chunk of the tile: row statistics (m in the log2 domain, l), and with `stage` != nullptr the logits
// themselves, row r at stage + r * ss + off[r], column k.
template <typename E, int KD>
__device__ __forceinline__ void tile_stats(const E* kbase, int ld, int T, int dh, bool vec, float sl2, E* Ks, const E* Qs,
                                           const uint32_t (&aq)[KD][4], float* stage, int ss, int off0, int off1,
                                           float& m0, float& m1, float& l0, float& l1, int lane) {
  const int g = lane >> 2, q2 = (lane & 3) * 2;
  m0 = m1 = -INFINITY;
  l0 = l1 = 0.f;
  for (int k0 = 0; k0 < T; k0 += KC) {
    __syncwarp();
    load_rows<E, KD>(Ks, kbase + (size_t)k0 * ld, ld, min(KC, T - k0), KC, dh, vec, lane);
    __syncwarp();
    float c[8][4];
    chunk_scores<E, KD>(Qs, Ks, aq, c, lane);
    scale_mask(c, k0, T, sl2, lane);
    update_stats(c, m0, m1, l0, l1);
    if (stage) {
      float* s0 = stage + g * ss + off0 + k0;
      float* s1 = stage + (g + 8) * ss + off1 + k0;
#pragma unroll
      for (int n = 0; n < 8; ++n) {
        const int k = n * 8 + q2;
        if (k0 + k < T) { s0[k] = c[n][0]; s1[k] = c[n][2]; }
        if (k0 + k + 1 < T) { s0[k + 1] = c[n][1]; s1[k + 1] = c[n][3]; }
      }
    }
  }
  row_sums(l0, l1);
}

// gdst[0..n) = ex2(src[i] - m) * inv, where src and gdst agree modulo 16 bytes: scalar head and tail, 16-byte streaming
// stores in between
__device__ __forceinline__ void store_row(float* gdst, int n, const float* src, float m, float inv, int lane) {
  const int head = min(n, (int)(((16u - ((uint32_t)reinterpret_cast<uintptr_t>(gdst) & 15u)) & 15u) >> 2));
  if (lane < head) __stcs(gdst + lane, ex2(src[lane] - m) * inv);
  const int nv = (n - head) >> 2;
  const float4* s4 = reinterpret_cast<const float4*>(src + head);
  float4* g4 = reinterpret_cast<float4*>(gdst + head);
  for (int v = lane; v < nv; v += 32) {
    float4 x = s4[v];
    x.x = ex2(x.x - m) * inv; x.y = ex2(x.y - m) * inv; x.z = ex2(x.z - m) * inv; x.w = ex2(x.w - m) * inv;
    __stcs(g4 + v, x);
  }
  const int t0 = head + 4 * nv;
  if (lane < n - t0) __stcs(gdst + t0 + lane, ex2(src[t0 + lane] - m) * inv);
}

template <typename E, int KD>
inline size_t probs_warp_bytes(int T) {
  using G = Geo<E, KD>;
  const int w = T <= PROBS_ROW_MAX ? T : KC;
  return G::q_bytes + G::k_bytes + (size_t)16 * ((w + 3) / 4 * 4 + 4) * 4 + 32 * 4;
}

template <typename E, int KD>
__global__ void __launch_bounds__(128) attn_probs_kernel(int T, int h, int dh, int64_t items, const E* __restrict__ qkv,
                                                         float* __restrict__ probs, float sl2, size_t warp_bytes,
                                                         int vec) {
  using G = Geo<E, KD>;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t item = (int64_t)blockIdx.x * (blockDim.x >> 5) + warp;
  if (item >= items) return;
  unsigned char* wsm = smem_raw + (size_t)warp * warp_bytes;
  E* Qs = reinterpret_cast<E*>(wsm);
  E* Ks = reinterpret_cast<E*>(wsm + G::q_bytes);
  float* stage = reinterpret_cast<float*>(wsm + G::q_bytes + G::k_bytes);
  const bool whole = T <= PROBS_ROW_MAX;
  const int ss = (whole ? (T + 3) / 4 * 4 : KC) + 4;
  float* rstat = stage + 16 * ss;   // [16] m, [16] 1/l

  const int ntile = (T + 15) / 16;
  const int64_t bh = item / ntile;
  const int i0 = (int)(item - bh * ntile) * 16;
  const int b = (int)(bh / h), hh = (int)(bh - (int64_t)b * h);
  const int d = h * dh, ld = 3 * d, nrow = min(16, T - i0);
  const E* qbase = qkv + ((size_t)b * T + i0) * ld + (size_t)hh * dh;
  const E* kbase = qkv + (size_t)b * T * ld + d + (size_t)hh * dh;
  float* pbase = probs + ((size_t)bh * T + i0) * T;   // row r of the tile at pbase + r * T

  load_rows<E, KD>(Qs, qbase, ld, nrow, 16, dh, vec != 0, lane);
  __syncwarp();
  uint32_t aq[KD][4];
  load_qfrag<E, KD>(Qs, aq, lane);
  const int g = lane >> 2, q2 = (lane & 3) * 2;
  // staged row r starts at the same address modulo 16 as its first destination element
  const uintptr_t pb = reinterpret_cast<uintptr_t>(pbase);
  auto off = [&](int r, int k0) { return (int)(((pb >> 2) + (size_t)r * T + k0) & 3); };
  float m0, m1, l0, l1;
  tile_stats<E, KD>(kbase, ld, T, dh, vec != 0, sl2, Ks, Qs, aq, whole ? stage : nullptr, ss, off(g, 0), off(g + 8, 0),
                    m0, m1, l0, l1, lane);
  if ((lane & 3) == 0) {
    rstat[g] = m0; rstat[g + 8] = m1;
    rstat[16 + g] = 1.f / l0; rstat[16 + g + 8] = 1.f / l1;
  }
  __syncwarp();
  if (whole) {
    for (int r = 0; r < nrow; ++r)
      store_row(pbase + (size_t)r * T, T, stage + r * ss + off(r, 0), rstat[r], rstat[16 + r], lane);
    return;
  }
  // pass 2 for long rows: S again, 64 keys at a time, each row segment staged and stored
  for (int k0 = 0; k0 < T; k0 += KC) {
    __syncwarp();
    load_rows<E, KD>(Ks, kbase + (size_t)k0 * ld, ld, min(KC, T - k0), KC, dh, vec != 0, lane);
    __syncwarp();
    float c[8][4];
    chunk_scores<E, KD>(Qs, Ks, aq, c, lane);
    scale_mask(c, k0, T, sl2, lane);
    float* s0 = stage + g * ss + off(g, k0);
    float* s1 = stage + (g + 8) * ss + off(g + 8, k0);
#pragma unroll
    for (int n = 0; n < 8; ++n) {
      const int k = n * 8 + q2;
      s0[k] = c[n][0]; s0[k + 1] = c[n][1];
      s1[k] = c[n][2]; s1[k + 1] = c[n][3];
    }
    __syncwarp();
    const int w = min(KC, T - k0);
    for (int r = 0; r < nrow; ++r)
      store_row(pbase + (size_t)r * T + k0, w, stage + r * ss + off(r, k0), rstat[r], rstat[16 + r], lane);
  }
}

// per warp: Q rows | K chunk | fp32 column sums [T] | (REL: dO rows | V chunk)
__host__ __device__ inline size_t rollout_acc_bytes(int T) { return (size_t)(T + 3) / 4 * 4 * 4; }
template <typename E, int KD, bool REL>
inline size_t rollout_warp_bytes(int T) {
  using G = Geo<E, KD>;
  return (REL ? 2 : 1) * (G::q_bytes + G::k_bytes) + rollout_acc_bytes(T);
}

template <typename E, int KD, bool REL>
__global__ void __launch_bounds__(512) attn_rollout_kernel(int T, int h, int dh, const E* __restrict__ qkv,
                                                           const float* __restrict__ v_in, float* __restrict__ v_out,
                                                           float sl2, size_t warp_bytes, int vec,
                                                           const E* __restrict__ dout) {
  using G = Geo<E, KD>;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int nw = blockDim.x >> 5, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  unsigned char* wsm = smem_raw + (size_t)warp * warp_bytes;
  E* Qs = reinterpret_cast<E*>(wsm);
  E* Ks = reinterpret_cast<E*>(wsm + G::q_bytes);
  float* colacc = reinterpret_cast<float*>(wsm + G::q_bytes + G::k_bytes);
  E* dOs = reinterpret_cast<E*>(wsm + G::q_bytes + G::k_bytes + rollout_acc_bytes(T));
  E* Vs = dOs + 16 * G::LDE;
  const int b = blockIdx.x, d = h * dh, ld = 3 * d;
  const float* vb = v_in + (size_t)b * T;
  for (int j = lane; j < T; j += 32) colacc[j] = 0.f;
  const int g = lane >> 2, q2 = (lane & 3) * 2;
  const int ntile = (T + 15) / 16;
  for (int item = warp; item < h * ntile; item += nw) {
    const int hh = item / ntile, i0 = (item - hh * ntile) * 16, nrow = min(16, T - i0);
    const float vr = lane < nrow ? vb[i0 + lane] : 0.f;
    if (!__any_sync(0xffffffffu, lane < 16 && vr != 0.f)) continue;   // rows with v_in = 0 contribute nothing
    const float v0 = __shfl_sync(0xffffffffu, vr, g), v1 = __shfl_sync(0xffffffffu, vr, g + 8);
    const E* kbase = qkv + (size_t)b * T * ld + d + (size_t)hh * dh;
    __syncwarp();
    load_rows<E, KD>(Qs, qkv + ((size_t)b * T + i0) * ld + (size_t)hh * dh, ld, nrow, 16, dh, vec != 0, lane);
    if constexpr (REL) {
      const uint32_t live = __ballot_sync(0xffffffffu, lane < 16 && vr != 0.f);
      load_rows<E, KD>(dOs, dout + ((size_t)b * T + i0) * d + (size_t)hh * dh, d, nrow, 16, dh, vec != 0, lane, live);
    }
    __syncwarp();
    uint32_t aq[KD][4];
    load_qfrag<E, KD>(Qs, aq, lane);
    float m0, m1, l0, l1;
    tile_stats<E, KD>(kbase, ld, T, dh, vec != 0, sl2, Ks, Qs, aq, nullptr, 0, 0, 0, m0, m1, l0, l1, lane);
    const float w0 = v0 / l0, w1 = v1 / l1;   // rows >= T have v = 0
    for (int k0 = 0; k0 < T; k0 += KC) {
      __syncwarp();
      load_rows<E, KD>(Ks, kbase + (size_t)k0 * ld, ld, min(KC, T - k0), KC, dh, vec != 0, lane);
      if constexpr (REL) load_rows<E, KD>(Vs, kbase + d + (size_t)k0 * ld, ld, min(KC, T - k0), KC, dh, vec != 0, lane);
      __syncwarp();
      float s[8][2];
      if constexpr (REL) {
        // dP first; the dO and Q fragments (bf16) are reloaded from shared memory per chunk, so that no fragment stays
        // live across chunks and every instantiation fits the 128 registers of a 512-thread CTA without spilling
        float dp[8][4];
        {
          uint32_t ado[KD][4];
          load_qfrag<E, KD>(dOs, ado, lane);
          chunk_scores<E, KD>(dOs, Vs, ado, dp, lane);   // unscaled; keys >= T meet zero-filled V rows: dP = 0
        }
        float c[8][4];
        {
          uint32_t aqc[KD][4];
          load_qfrag<E, KD>(Qs, aqc, lane);
          chunk_scores<E, KD>(Qs, Ks, aqc, c, lane);
        }
        scale_mask(c, k0, T, sl2, lane);
        // relu that keeps NaN (fmaxf would drop it): a NaN dO row, which an invalid target's NaN dlogits row produces,
        // must reach v_out.  Rows with v_in = 0 were zero-filled and keys >= T give 0 * 0, so neither makes a NaN.
        auto relu = [](float x) { return x < 0.f ? 0.f : x; };
#pragma unroll
        for (int n = 0; n < 8; ++n) {
          s[n][0] = fmaf(w0, relu(dp[n][0] * ex2(c[n][0] - m0)), w1 * relu(dp[n][2] * ex2(c[n][2] - m1)));
          s[n][1] = fmaf(w0, relu(dp[n][1] * ex2(c[n][1] - m0)), w1 * relu(dp[n][3] * ex2(c[n][3] - m1)));
        }
      } else {
        float c[8][4];
        chunk_scores<E, KD>(Qs, Ks, aq, c, lane);
        scale_mask(c, k0, T, sl2, lane);
#pragma unroll
        for (int n = 0; n < 8; ++n) {
          s[n][0] = fmaf(w0, ex2(c[n][0] - m0), w1 * ex2(c[n][2] - m1));
          s[n][1] = fmaf(w0, ex2(c[n][1] - m0), w1 * ex2(c[n][3] - m1));
        }
      }
      // sum over the 8 row pairs (lanes with equal lane % 4), in a fixed order
#pragma unroll
      for (int o = 4; o < 32; o <<= 1) {
#pragma unroll
        for (int n = 0; n < 8; ++n) {
          s[n][0] += __shfl_xor_sync(0xffffffffu, s[n][0], o);
          s[n][1] += __shfl_xor_sync(0xffffffffu, s[n][1], o);
        }
      }
      if (g == 0) {
#pragma unroll
        for (int n = 0; n < 8; ++n) {
          const int k = k0 + n * 8 + q2;
          if (k < T) colacc[k] += s[n][0];
          if (k + 1 < T) colacc[k + 1] += s[n][1];
        }
      }
    }
  }
  __syncthreads();
  const float hs = (REL ? 1.f : 0.5f) / (float)h;
  for (int j = threadIdx.x; j < T; j += blockDim.x) {
    float a = 0.f;
    for (int w = 0; w < nw; ++w) a += reinterpret_cast<const float*>(smem_raw + (size_t)w * warp_bytes + G::q_bytes + G::k_bytes)[j];
    v_out[(size_t)b * T + j] = REL ? fmaf(hs, a, vb[j]) : fmaf(0.5f, vb[j], hs * a);
  }
}

// v[b, t] = e_0 (CLS pooling) or 1/T (mean pooling): the head's read-out of the top layer
__global__ void rollout_init_kernel(int B, int T, int has_cls, float* __restrict__ v) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)B * T) return;
  const int t = (int)(i % T);
  v[i] = has_cls ? (t == 0 ? 1.f : 0.f) : 1.f / (float)T;
}

// dlogits[r] = w_k one_hot(t_b) for the n rows r = k * B + b: t_b = target[b], or with target NULL the first maximum of
// logits[b] (amc_argmax's rule); w_k = weight[k], or 1 with weight NULL (relevance: n = B).  A target outside [0, C)
// gives a NaN row.  One thread per row.
__global__ void relevance_seed_kernel(int n, int B, int C, const float* __restrict__ logits,
                                      const int64_t* __restrict__ target, const float* __restrict__ weight,
                                      float* __restrict__ dlogits) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  const int k = r / B, b = r - k * B;
  const int64_t t = target ? target[b] : row_argmax(logits + (size_t)b * C, C);
  const bool ok = t >= 0 && t < C;
  const float w = weight ? weight[k] : 1.f;
  for (int c = 0; c < C; ++c) dlogits[(size_t)r * C + c] = ok ? (c == t ? w : 0.f) : __int_as_float(0x7fffffff);
}

// warps per CTA (at most `cap`) whose shared memory fits the plan, or 0
inline int warps_for(size_t warp_bytes, int cap) { return (int)std::min<size_t>(cap, SMEM_CAP / warp_bytes); }

inline bool vec_ok(const void* qkv, int h, int dh, size_t esz) {
  const int v = 16 / (int)esz;
  return dh % v == 0 && (3 * h * dh) % v == 0 && (reinterpret_cast<uintptr_t>(qkv) & 15) == 0;
}

template <typename E, int KD>
int probs_launch(int B, int T, int h, int dh, const E* qkv, float* probs, cudaStream_t st) {
  const size_t wb = probs_warp_bytes<E, KD>(T);
  const int nw = warps_for(wb, 4);
  AMC_CHECK_ARG(nw >= 1, "attention_probs: T=%d dh=%d needs %zu bytes of shared memory per warp", T, dh, wb);
  const int64_t items = (int64_t)B * h * ((T + 15) / 16);
  const int64_t grid = (items + nw - 1) / nw;
  AMC_CHECK_ARG(grid < (1ll << 31), "attention_probs: grid too large");
  AMC_CUDA(cudaFuncSetAttribute(attn_probs_kernel<E, KD>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_CAP));
  attn_probs_kernel<E, KD><<<(unsigned)grid, nw * 32, nw * wb, st>>>(T, h, dh, items, qkv, probs,
                                                                     1.4426950408889634f / sqrtf((float)dh), wb,
                                                                     vec_ok(qkv, h, dh, sizeof(E)) ? 1 : 0);
  AMC_LAUNCH_CHECK();
  return 0;
}

template <typename E, int KD, bool REL = false>
int rollout_launch(int B, int T, int h, int dh, const E* qkv, const float* v_in, float* v_out, cudaStream_t st,
                   const E* dout = nullptr) {
  const char* what = REL ? "attention_relevance_step" : "attention_rollout_step";
  const size_t wb = rollout_warp_bytes<E, KD, REL>(T);
  // One CTA per frame of h * ceil(T / 16) tiles.  4 warps while the batch gives every SM two CTAs or more; 16 when it does
  // not, so that a small batch of long frames (conv1d: 128 frames, 520 tiles each) still fills the SMs (2.19 against
  // 6.28 ms per step).  With enough frames 16 warps lose 2-10 % to the longer cross-warp sum (DESIGN §5.8).  Never more
  // warps than half the frame's tiles.
  const int tiles = h * ((T + 15) / 16);
  const int cap = B >= 2 * device_sm_count() ? 4 : 16;
  const int nw = std::min(warps_for(wb, cap), std::max(1, (tiles + 1) / 2));
  AMC_CHECK_ARG(nw >= 1, "%s: T=%d dh=%d needs %zu bytes of shared memory per warp", what, T, dh, wb);
  AMC_CUDA(cudaFuncSetAttribute(attn_rollout_kernel<E, KD, REL>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_CAP));
  const bool vec = vec_ok(qkv, h, dh, sizeof(E)) && (reinterpret_cast<uintptr_t>(dout) & 15) == 0;
  attn_rollout_kernel<E, KD, REL><<<B, nw * 32, nw * wb, st>>>(T, h, dh, qkv, v_in, v_out,
                                                               1.4426950408889634f / sqrtf((float)dh), wb, vec ? 1 : 0,
                                                               dout);
  AMC_LAUNCH_CHECK();
  return 0;
}
template <typename E, int KD>
int relevance_launch(int B, int T, int h, int dh, const E* qkv, const E* dout, const float* v_in, float* v_out,
                     cudaStream_t st) {
  return rollout_launch<E, KD, true>(B, T, h, dh, qkv, v_in, v_out, st, dout);
}

int check_shape(const char* what, int B, int T, int h, int dh) {
  AMC_CHECK_ARG(B >= 0 && h >= 1, "%s: bad batch / head count", what);
  AMC_CHECK_ARG(T >= 1 && T <= ATTN_LONG_MAX_T, "%s: T=%d unsupported (1..%d tokens per frame)", what, T, ATTN_LONG_MAX_T);
  AMC_CHECK_ARG(dh >= 1 && dh <= 128, "%s: head dim %d unsupported (1..128)", what, dh);
  return 0;
}

#define AMC_MAPS_DISPATCH(FN, ...)                                     \
  switch ((dh + 15) / 16) {                                            \
    case 1: return FN<E, 1>(__VA_ARGS__);                              \
    case 2: return FN<E, 2>(__VA_ARGS__);                              \
    case 3: return FN<E, 3>(__VA_ARGS__);                              \
    case 4: return FN<E, 4>(__VA_ARGS__);                              \
    case 5: return FN<E, 5>(__VA_ARGS__);                              \
    case 6: return FN<E, 6>(__VA_ARGS__);                              \
    case 7: return FN<E, 7>(__VA_ARGS__);                              \
    default: return FN<E, 8>(__VA_ARGS__);                             \
  }

}  // namespace

template <typename E>
int attention_probs(int B, int T, int h, int dh, const E* qkv, float* probs, cudaStream_t st) {
  AMC_TRY(check_shape("attention_probs", B, T, h, dh));
  if (B == 0) return 0;
  AMC_MAPS_DISPATCH(probs_launch, B, T, h, dh, qkv, probs, st)
}
template int attention_probs<float>(int, int, int, int, const float*, float*, cudaStream_t);
template int attention_probs<bf16>(int, int, int, int, const bf16*, float*, cudaStream_t);

template <typename E>
int attention_rollout_step(int B, int T, int h, int dh, const E* qkv, const float* v_in, float* v_out, cudaStream_t st) {
  AMC_TRY(check_shape("attention_rollout_step", B, T, h, dh));
  if (B == 0) return 0;
  AMC_MAPS_DISPATCH(rollout_launch, B, T, h, dh, qkv, v_in, v_out, st)
}
template int attention_rollout_step<float>(int, int, int, int, const float*, const float*, float*, cudaStream_t);
template int attention_rollout_step<bf16>(int, int, int, int, const bf16*, const float*, float*, cudaStream_t);

template <typename E>
int attention_relevance_step(int B, int T, int h, int dh, const E* qkv, const E* dout, const float* v_in, float* v_out,
                             cudaStream_t st) {
  AMC_TRY(check_shape("attention_relevance_step", B, T, h, dh));
  if (B == 0) return 0;
  AMC_MAPS_DISPATCH(relevance_launch, B, T, h, dh, qkv, dout, v_in, v_out, st)
}
template int attention_relevance_step<float>(int, int, int, int, const float*, const float*, const float*, float*,
                                             cudaStream_t);
template int attention_relevance_step<bf16>(int, int, int, int, const bf16*, const bf16*, const float*, float*,
                                            cudaStream_t);

int rollout_init(int B, int T, int has_cls, float* v, cudaStream_t st) {
  const int64_t n = (int64_t)B * T;
  if (n == 0) return 0;
  rollout_init_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(B, T, has_cls, v);
  AMC_LAUNCH_CHECK();
  return 0;
}

int relevance_seed(int n, int B, int C, const float* logits, const int64_t* target, const float* weight, float* dlogits,
                   cudaStream_t st) {
  if (n == 0) return 0;
  relevance_seed_kernel<<<(n + 127) / 128, 128, 0, st>>>(n, B, C, logits, target, weight, dlogits);
  AMC_LAUNCH_CHECK();
  return 0;
}

}  // namespace amc

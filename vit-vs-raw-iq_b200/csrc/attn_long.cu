// Long-sequence multi-head attention (T > 288 tokens per frame), forward and backward: the `embedding_type='conv1d'`
// variant of the raw-IQ model makes every IQ sample a token (T = 1025; R/models/encoder.py:34-41), which is outside
// the single-CTA regime of attention.cu / attn_tiles.cu -- keys, values and the gradient accumulators of a whole
// head no longer fit in shared memory.  Same math as scale_dot_product_attention.py:26-37 (+ the head split / concat
// of multi_head_attention.py:34-47; backward per SURVEY Appendix B), tiled flash-style:
//
//   forward : a CTA owns a block of query rows of one (frame, head) and streams the keys / values through shared
//             memory in chunks with an online-softmax rescale; the log2-domain row statistics lse2 are saved.
//   backward: two passes, no atomics, deterministic: `dq` is query-block parallel (streams K, V), `dkdv` is key-block
//             parallel (streams Q, dO, O); both recompute P = exp2(S c - lse2) and delta = rowsum(dO * O).
//
// Two implementations behind one dispatcher:
//   * bf16, head dim 16 / 32 / 64: mma.sync m16n8k16 kernels; operand tiles arrive as 3-D TMA tensor copies into
//     swizzled shared memory (rows past T are zero-filled by the TMA unit), double-buffered on mbarriers.  The inner
//     steps are the ones of attn_tiles.cu (fwd_chunk, the S^T / dP^T step of its backward).
//   * fp32 (the 1e-4 parity mode) and every other head dim: SIMT kernels, one warp per query / key row.
#include "attention.cuh"
#include "attn_mma.cuh"

namespace amc {
namespace {

constexpr float LOG2E = 1.4426950408889634f;
constexpr float LN2 = 0.6931471805599453f;

// =================================================================================================================
// SIMT kernels (any element type, head dim <= 128)
// =================================================================================================================
constexpr int S_NW = 8;        // warps per CTA
constexpr int S_RPW = 4;       // rows (queries, or keys in dkdv) owned by a warp
constexpr int S_QB = S_NW * S_RPW;
constexpr int S_KT = 128;      // streamed rows per tile: 4 per lane
constexpr int S_CC = 4;        // head-dim columns per lane (dh <= 128)

template <typename S> struct LongPad;
template <> struct LongPad<float> { static constexpr int v = 1; };
template <> struct LongPad<bf16> { static constexpr int v = 2; };

template <typename E>
__device__ __forceinline__ void load_rows(E* dst, int stride, const E* __restrict__ src, int ld, int rows, int dh) {
  for (int i = threadIdx.x; i < rows * dh; i += blockDim.x) {
    const int t = i / dh, c = i - t * dh;
    dst[t * stride + c] = src[(size_t)t * ld + c];
  }
}

template <typename E>
__global__ void __launch_bounds__(S_NW * 32) attn_long_fwd_kernel(int T, int h, int dh, int nqb,
                                                                  const E* __restrict__ qkv, E* __restrict__ out,
                                                                  float* __restrict__ lse, float scale) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int d = h * dh, ld = 3 * d, stride = dh + LongPad<E>::v;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tile = (S_KT * stride + 1) & ~1;
  E* Ks = reinterpret_cast<E*>(smem_raw);
  E* Vs = Ks + tile;
  float* qs = reinterpret_cast<float*>(Vs + tile);     // [S_NW][S_RPW][dh], pre-scaled
  float* ps = qs + S_QB * dh;                           // [S_NW][S_KT]
  const int qb = blockIdx.x % nqb, bh = blockIdx.x / nqb;
  const int b = bh / h, hh = bh - b * h;
  const E* base = qkv + (size_t)b * T * ld + hh * dh;
  const int row0 = qb * S_QB + warp * S_RPW;
  float* myq = qs + warp * S_RPW * dh;
  float* myp = ps + warp * S_KT;
#pragma unroll
  for (int rr = 0; rr < S_RPW; ++rr) {
    const int i = row0 + rr;
    for (int c = lane; c < dh; c += 32) myq[rr * dh + c] = i < T ? to_f(base[(size_t)i * ld + c]) * scale : 0.f;
  }
  float m[S_RPW], l[S_RPW], o[S_RPW][S_CC];
#pragma unroll
  for (int rr = 0; rr < S_RPW; ++rr) {
    m[rr] = -INFINITY;
    l[rr] = 0.f;
#pragma unroll
    for (int cc = 0; cc < S_CC; ++cc) o[rr][cc] = 0.f;
  }
  for (int k0 = 0; k0 < T; k0 += S_KT) {
    const int nk = min(S_KT, T - k0);
    __syncthreads();                                    // the previous tile has been consumed (and myq is written)
    load_rows(Ks, stride, base + (size_t)k0 * ld + d, ld, nk, dh);
    load_rows(Vs, stride, base + (size_t)k0 * ld + 2 * d, ld, nk, dh);
    __syncthreads();
#pragma unroll
    for (int rr = 0; rr < S_RPW; ++rr) {
      if (row0 + rr >= T) continue;                     // warp-uniform
      const float* q = myq + rr * dh;
      float s[S_KT / 32];
      float mx = -INFINITY;
#pragma unroll
      for (int jj = 0; jj < S_KT / 32; ++jj) {
        const int j = lane + 32 * jj;
        float a = -INFINITY;
        if (j < nk) {
          a = 0.f;
          const E* kr = Ks + j * stride;
          for (int c = 0; c < dh; ++c) a = fmaf(q[c], to_f(kr[c]), a);
        }
        s[jj] = a;
        mx = fmaxf(mx, a);
      }
      mx = warp_max(mx);                                // nk >= 1: finite
      const float mn = fmaxf(m[rr], mx);
      const float al = __expf(m[rr] - mn);              // first tile: exp(-inf) = 0
      float sum = 0.f;
#pragma unroll
      for (int jj = 0; jj < S_KT / 32; ++jj) {
        const int j = lane + 32 * jj;
        const float e = j < nk ? __expf(s[jj] - mn) : 0.f;
        myp[j] = e;
        sum += e;
      }
      sum = warp_sum(sum);
      l[rr] = fmaf(l[rr], al, sum);
      m[rr] = mn;
      __syncwarp();
#pragma unroll
      for (int cc = 0; cc < S_CC; ++cc) {
        const int c = lane + 32 * cc;
        if (c < dh) {
          float a = 0.f;
          for (int j = 0; j < nk; ++j) a = fmaf(myp[j], to_f(Vs[j * stride + c]), a);
          o[rr][cc] = fmaf(o[rr][cc], al, a);
        }
      }
      __syncwarp();
    }
  }
#pragma unroll
  for (int rr = 0; rr < S_RPW; ++rr) {
    const int i = row0 + rr;
    if (i >= T) continue;
    const float inv = 1.f / l[rr];
#pragma unroll
    for (int cc = 0; cc < S_CC; ++cc) {
      const int c = lane + 32 * cc;
      if (c < dh) out[((size_t)b * T + i) * d + hh * dh + c] = from_f<E>(o[rr][cc] * inv);
    }
    if (lse != nullptr && lane == 0) lse[((size_t)b * h + hh) * T + i] = (m[rr] + __logf(l[rr])) * LOG2E;
  }
}

// dQ: query-block parallel.  dS = P * (dP - delta) * scale with P = exp(S - L), L = lse2 * ln 2.
template <typename E>
__global__ void __launch_bounds__(S_NW * 32) attn_long_dq_kernel(int T, int h, int dh, int nqb,
                                                                 const E* __restrict__ qkv, const E* __restrict__ out,
                                                                 const float* __restrict__ lse,
                                                                 const E* __restrict__ dout, E* __restrict__ dqkv,
                                                                 float scale) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int d = h * dh, ld = 3 * d, stride = dh + LongPad<E>::v;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tile = (S_KT * stride + 1) & ~1;
  E* Ks = reinterpret_cast<E*>(smem_raw);
  E* Vs = Ks + tile;
  float* qs = reinterpret_cast<float*>(Vs + tile);     // [S_QB][dh] q rows (unscaled)
  float* gs = qs + S_QB * dh;                           // [S_QB][dh] dO rows
  float* ps = gs + S_QB * dh;                           // [S_NW][S_KT]
  const int qb = blockIdx.x % nqb, bh = blockIdx.x / nqb;
  const int b = bh / h, hh = bh - b * h;
  const E* base = qkv + (size_t)b * T * ld + hh * dh;
  const int row0 = qb * S_QB + warp * S_RPW;
  float* myq = qs + warp * S_RPW * dh;
  float* myg = gs + warp * S_RPW * dh;
  float* myp = ps + warp * S_KT;
  float L[S_RPW], dl[S_RPW], dq[S_RPW][S_CC];
#pragma unroll
  for (int rr = 0; rr < S_RPW; ++rr) {
    const int i = row0 + rr;
    float part = 0.f;
    for (int c = lane; c < dh; c += 32) {
      float qv = 0.f, gv = 0.f, ov = 0.f;
      if (i < T) {
        qv = to_f(base[(size_t)i * ld + c]);
        gv = to_f(dout[((size_t)b * T + i) * d + hh * dh + c]);
        ov = to_f(out[((size_t)b * T + i) * d + hh * dh + c]);
      }
      myq[rr * dh + c] = qv;
      myg[rr * dh + c] = gv;
      part = fmaf(gv, ov, part);
    }
    dl[rr] = warp_sum(part);
    L[rr] = i < T ? lse[((size_t)b * h + hh) * T + i] * LN2 : 0.f;
#pragma unroll
    for (int cc = 0; cc < S_CC; ++cc) dq[rr][cc] = 0.f;
  }
  for (int k0 = 0; k0 < T; k0 += S_KT) {
    const int nk = min(S_KT, T - k0);
    __syncthreads();
    load_rows(Ks, stride, base + (size_t)k0 * ld + d, ld, nk, dh);
    load_rows(Vs, stride, base + (size_t)k0 * ld + 2 * d, ld, nk, dh);
    __syncthreads();
#pragma unroll
    for (int rr = 0; rr < S_RPW; ++rr) {
      if (row0 + rr >= T) continue;
      const float* q = myq + rr * dh;
      const float* gq = myg + rr * dh;
#pragma unroll
      for (int jj = 0; jj < S_KT / 32; ++jj) {
        const int j = lane + 32 * jj;
        if (j < nk) {
          const E* kr = Ks + j * stride;
          const E* vr = Vs + j * stride;
          float a = 0.f, g = 0.f;
          for (int c = 0; c < dh; ++c) {
            a = fmaf(q[c], to_f(kr[c]), a);
            g = fmaf(gq[c], to_f(vr[c]), g);
          }
          const float p = __expf(fmaf(a, scale, -L[rr]));
          myp[j] = p * (g - dl[rr]) * scale;            // dS[i, j]
        }
      }
      __syncwarp();
#pragma unroll
      for (int cc = 0; cc < S_CC; ++cc) {
        const int c = lane + 32 * cc;
        if (c < dh) {
          float a = 0.f;
          for (int j = 0; j < nk; ++j) a = fmaf(myp[j], to_f(Ks[j * stride + c]), a);
          dq[rr][cc] += a;
        }
      }
      __syncwarp();
    }
  }
#pragma unroll
  for (int rr = 0; rr < S_RPW; ++rr) {
    const int i = row0 + rr;
    if (i >= T) continue;
#pragma unroll
    for (int cc = 0; cc < S_CC; ++cc) {
      const int c = lane + 32 * cc;
      if (c < dh) dqkv[((size_t)b * T + i) * ld + hh * dh + c] = from_f<E>(dq[rr][cc]);
    }
  }
}

// dK, dV: key-block parallel, streams the query rows (Q, dO; delta from dO * O; L from lse2).
template <typename E>
__global__ void __launch_bounds__(S_NW * 32) attn_long_dkdv_kernel(int T, int h, int dh, int nkb,
                                                                   const E* __restrict__ qkv,
                                                                   const E* __restrict__ out,
                                                                   const float* __restrict__ lse,
                                                                   const E* __restrict__ dout, E* __restrict__ dqkv,
                                                                   float scale) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int d = h * dh, ld = 3 * d, stride = dh + LongPad<E>::v;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tile = (S_KT * stride + 1) & ~1;
  E* Qs = reinterpret_cast<E*>(smem_raw);
  E* Gs = Qs + tile;                                    // dO
  float* ks = reinterpret_cast<float*>(Gs + tile);     // [S_QB][dh] key rows of this CTA
  float* vs = ks + S_QB * dh;                           // [S_QB][dh] value rows
  float* stL = vs + S_QB * dh;                          // [S_KT]
  float* stD = stL + S_KT;                              // [S_KT]
  float* pA = stD + S_KT;                               // [S_NW][S_KT]  P[i, j]
  float* pB = pA + S_NW * S_KT;                         // [S_NW][S_KT]  dS[i, j]
  const int kb = blockIdx.x % nkb, bh = blockIdx.x / nkb;
  const int b = bh / h, hh = bh - b * h;
  const E* base = qkv + (size_t)b * T * ld + hh * dh;
  const E* gbase = dout + (size_t)b * T * d + hh * dh;
  const E* obase = out + (size_t)b * T * d + hh * dh;
  const float* lbase = lse + ((size_t)b * h + hh) * T;
  const int row0 = kb * S_QB + warp * S_RPW;
  float* myk = ks + warp * S_RPW * dh;
  float* myv = vs + warp * S_RPW * dh;
  float* myA = pA + warp * S_KT;
  float* myB = pB + warp * S_KT;
  float dk[S_RPW][S_CC], dv[S_RPW][S_CC];
#pragma unroll
  for (int rr = 0; rr < S_RPW; ++rr) {
    const int j = row0 + rr;
    for (int c = lane; c < dh; c += 32) {
      myk[rr * dh + c] = j < T ? to_f(base[(size_t)j * ld + d + c]) : 0.f;
      myv[rr * dh + c] = j < T ? to_f(base[(size_t)j * ld + 2 * d + c]) : 0.f;
    }
#pragma unroll
    for (int cc = 0; cc < S_CC; ++cc) { dk[rr][cc] = 0.f; dv[rr][cc] = 0.f; }
  }
  for (int i0 = 0; i0 < T; i0 += S_KT) {
    const int nq = min(S_KT, T - i0);
    __syncthreads();
    load_rows(Qs, stride, base + (size_t)i0 * ld, ld, nq, dh);
    load_rows(Gs, stride, gbase + (size_t)i0 * d, d, nq, dh);
    for (int r = warp; r < nq; r += S_NW) {             // row statistics of this tile
      float part = 0.f;
      for (int c = lane; c < dh; c += 32)
        part = fmaf(to_f(gbase[(size_t)(i0 + r) * d + c]), to_f(obase[(size_t)(i0 + r) * d + c]), part);
      part = warp_sum(part);
      if (lane == 0) {
        stD[r] = part;
        stL[r] = lbase[i0 + r] * LN2;
      }
    }
    __syncthreads();
#pragma unroll
    for (int rr = 0; rr < S_RPW; ++rr) {
      if (row0 + rr >= T) continue;
      const float* kq = myk + rr * dh;
      const float* vq = myv + rr * dh;
#pragma unroll
      for (int ii = 0; ii < S_KT / 32; ++ii) {
        const int i = lane + 32 * ii;
        if (i < nq) {
          const E* qr = Qs + i * stride;
          const E* gr = Gs + i * stride;
          float a = 0.f, g = 0.f;
          for (int c = 0; c < dh; ++c) {
            a = fmaf(to_f(qr[c]), kq[c], a);
            g = fmaf(to_f(gr[c]), vq[c], g);
          }
          const float p = __expf(fmaf(a, scale, -stL[i]));
          myA[i] = p;
          myB[i] = p * (g - stD[i]) * scale;
        }
      }
      __syncwarp();
#pragma unroll
      for (int cc = 0; cc < S_CC; ++cc) {
        const int c = lane + 32 * cc;
        if (c < dh) {
          float a = 0.f, g = 0.f;
          for (int i = 0; i < nq; ++i) {
            a = fmaf(myB[i], to_f(Qs[i * stride + c]), a);
            g = fmaf(myA[i], to_f(Gs[i * stride + c]), g);
          }
          dk[rr][cc] += a;
          dv[rr][cc] += g;
        }
      }
      __syncwarp();
    }
  }
#pragma unroll
  for (int rr = 0; rr < S_RPW; ++rr) {
    const int j = row0 + rr;
    if (j >= T) continue;
#pragma unroll
    for (int cc = 0; cc < S_CC; ++cc) {
      const int c = lane + 32 * cc;
      if (c < dh) {
        dqkv[((size_t)b * T + j) * ld + d + hh * dh + c] = from_f<E>(dk[rr][cc]);
        dqkv[((size_t)b * T + j) * ld + 2 * d + hh * dh + c] = from_f<E>(dv[rr][cc]);
      }
    }
  }
}

template <typename E> size_t simt_tile_bytes(int dh) {
  const int stride = dh + LongPad<E>::v;
  return (size_t)((S_KT * stride + 1) & ~1) * sizeof(E);
}

// =================================================================================================================
// mma.sync kernels (bf16, head dim 16 * KD)
// =================================================================================================================
constexpr int M_NW = 8;            // warps per CTA, 16 rows each
constexpr int M_QS = M_NW * 16;    // rows owned by a CTA (queries; keys in dkdv)
constexpr int M_CB = 9;            // 16-row blocks per streamed chunk
constexpr int M_CR = M_CB * 16;    // rows per streamed chunk (TMA box rows, <= 256)
constexpr int M_NBC = 3;           // key blocks per online-softmax step (fwd_chunk)
constexpr int M_HDR = 1024;        // mbarriers

struct LongGeom {
  int T, h, d, NQ;       // NQ = ceil(T / 16)
  int nsb;               // 128-row super-blocks per (frame, head)
  int nchunk;            // streamed chunks per (frame, head)
  float scale, sl2;      // 1/sqrt(dh), scale * log2(e)
};

// Forward.  shared memory: [barriers | Q tile 128 x RB | 2 stages x (K, V chunk tiles 144 x RB)]
template <int KD>
__global__ void __launch_bounds__(M_NW * 32)
attn_long_mma_fwd_kernel(const __grid_constant__ CUtensorMap mOwn, const __grid_constant__ CUtensorMap mStream,
                         const LongGeom gm, bf16* __restrict__ out, float* __restrict__ lse) {
  constexpr int dh = 16 * KD, RB = 32 * KD;
  constexpr uint32_t OWN_B = M_QS * RB, CH_B = M_CR * RB;
  extern __shared__ unsigned char smem_dyn[];
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023) & ~(uintptr_t)1023);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem);     // [0] own tile, [1], [2] stream stages
  const uint32_t qtile = smem_u32(smem + M_HDR), st0 = qtile + OWN_B;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int g = lane >> 2, cb = (lane & 3) * 2;
  const int T = gm.T;
  const int sb = blockIdx.x % gm.nsb, bh = blockIdx.x / gm.nsb;
  const int b = bh / gm.h, hh = bh - b * gm.h;
  const int col = hh * dh;
  if (tid == 0) {
    tma_prefetch_desc(&mOwn);
    tma_prefetch_desc(&mStream);
    mbar_init(bars, 1); mbar_init(bars + 1, 1); mbar_init(bars + 2, 1);
    fence_barrier_init();
  }
  __syncthreads();
  auto issue = [&](int c, int s) {        // one thread: K and V rows [c * M_CR, +M_CR) -> stage s
    mbar_expect_tx(bars + 1 + s, 2 * CH_B);
    tma_load_3d(&mStream, bars + 1 + s, st0 + s * 2 * CH_B, gm.d + col, c * M_CR, b);
    tma_load_3d(&mStream, bars + 1 + s, st0 + s * 2 * CH_B + CH_B, 2 * gm.d + col, c * M_CR, b);
  };
  if (tid == 0) {
    mbar_expect_tx(bars, OWN_B);
    tma_load_3d(&mOwn, bars, qtile, col, sb * M_QS, b);
    issue(0, 0);
    if (gm.nchunk > 1) issue(1, 1);
  }
  const int qrow = sb * M_QS + warp * 16;
  const bool live = qrow < T;
  mbar_wait(bars, 0);
  uint32_t aq[KD][4];
#pragma unroll
  for (int ks = 0; ks < KD; ++ks) ldsm_x4(aq[ks], addrA<KD>(qtile, warp * 16, ks, lane));
  float o[2 * KD][4];
#pragma unroll
  for (int n = 0; n < 2 * KD; ++n) { o[n][0] = 0.f; o[n][1] = 0.f; o[n][2] = 0.f; o[n][3] = 0.f; }
  float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f;
  for (int c = 0; c < gm.nchunk; ++c) {
    const int s = c & 1;
    mbar_wait(bars + 1 + s, (c >> 1) & 1);
    if (live) {
      const uint32_t kb = st0 + s * 2 * CH_B, vb = kb + CH_B;
      const int Trel = T - c * M_CR;
      if (c + 1 < gm.nchunk) {
#pragma unroll
        for (int k0 = 0; k0 < M_CB; k0 += M_NBC)
          fwd_chunk<KD, M_NBC, false>(kb, vb, k0, M_NBC, Trel, aq, o, m0, m1, l0, l1, gm.sl2, lane);
      } else {
        const int nblk = gm.NQ - c * M_CB;      // 1..M_CB blocks hold keys < T
        for (int k0 = 0; k0 < nblk; k0 += M_NBC)
          fwd_chunk<KD, M_NBC, true>(kb, vb, k0, min(M_NBC, nblk - k0), Trel, aq, o, m0, m1, l0, l1, gm.sl2, lane);
      }
    }
    __syncthreads();                        // every warp is done with stage s
    if (tid == 0 && c + 2 < gm.nchunk) issue(c + 2, s);
  }
  if (!live) return;
  l0 += __shfl_xor_sync(0xffffffffu, l0, 1); l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 1); l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
  const float i0 = 1.f / l0, i1 = 1.f / l1;
  const int r0 = qrow + g, r1 = r0 + 8;
  bf16* o0 = out + ((size_t)b * T + r0) * gm.d + col + cb;
  bf16* o1 = out + ((size_t)b * T + r1) * gm.d + col + cb;
#pragma unroll
  for (int n = 0; n < 2 * KD; ++n) {
    if (r0 < T) *reinterpret_cast<uint32_t*>(o0 + n * 8) = pack2(o[n][0] * i0, o[n][1] * i0);
    if (r1 < T) *reinterpret_cast<uint32_t*>(o1 + n * 8) = pack2(o[n][2] * i1, o[n][3] * i1);
  }
  if (lse != nullptr && (lane & 3) == 0) {
    float* lp = lse + ((size_t)b * gm.h + hh) * T;
    if (r0 < T) lp[r0] = fmaf(m0, gm.sl2, __log2f(l0));
    if (r1 < T) lp[r1] = fmaf(m1, gm.sl2, __log2f(l1));
  }
}

// one quad (4 lanes sharing a fragment row) sums dO[r, :] * O[r, :] of one head: delta of the softmax backward
template <int KD>
__device__ __forceinline__ float quad_delta(const bf16* __restrict__ g_row, const bf16* __restrict__ o_row, int lane) {
  constexpr int W = 2 * KD;                 // 32-bit words (bf16 pairs) per lane: dh / 4 elements
  const uint32_t* gp = reinterpret_cast<const uint32_t*>(g_row) + (lane & 3) * W;
  const uint32_t* op = reinterpret_cast<const uint32_t*>(o_row) + (lane & 3) * W;
  float a = 0.f;
#pragma unroll
  for (int w = 0; w < W; ++w) {
    const uint32_t x = __ldg(gp + w), y = __ldg(op + w);
    a = fmaf(bf_lo(x), bf_lo(y), a);
    a = fmaf(bf_hi(x), bf_hi(y), a);
  }
  a += __shfl_xor_sync(0xffffffffu, a, 1);
  a += __shfl_xor_sync(0xffffffffu, a, 2);
  return a;
}

// dQ.  shared memory: [barriers | Q tile | dO tile (128 x RB each) | 2 stages x (K, V chunk tiles)]
template <int KD>
__global__ void __launch_bounds__(M_NW * 32)
attn_long_mma_dq_kernel(const __grid_constant__ CUtensorMap mOwn, const __grid_constant__ CUtensorMap mOwnDO,
                        const __grid_constant__ CUtensorMap mStream, const LongGeom gm,
                        const bf16* __restrict__ out, const bf16* __restrict__ dout, const float* __restrict__ lse,
                        bf16* __restrict__ dqkv) {
  constexpr int dh = 16 * KD, RB = 32 * KD;
  constexpr uint32_t OWN_B = M_QS * RB, CH_B = M_CR * RB;
  extern __shared__ unsigned char smem_dyn[];
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023) & ~(uintptr_t)1023);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem);
  const uint32_t qtile = smem_u32(smem + M_HDR), gtile = qtile + OWN_B, st0 = gtile + OWN_B;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int g = lane >> 2, cb = (lane & 3) * 2;
  const int T = gm.T;
  const int sb = blockIdx.x % gm.nsb, bh = blockIdx.x / gm.nsb;
  const int b = bh / gm.h, hh = bh - b * gm.h;
  const int col = hh * dh;
  if (tid == 0) {
    tma_prefetch_desc(&mOwn);
    tma_prefetch_desc(&mOwnDO);
    tma_prefetch_desc(&mStream);
    mbar_init(bars, 1); mbar_init(bars + 1, 1); mbar_init(bars + 2, 1);
    fence_barrier_init();
  }
  __syncthreads();
  auto issue = [&](int c, int s) {
    mbar_expect_tx(bars + 1 + s, 2 * CH_B);
    tma_load_3d(&mStream, bars + 1 + s, st0 + s * 2 * CH_B, gm.d + col, c * M_CR, b);
    tma_load_3d(&mStream, bars + 1 + s, st0 + s * 2 * CH_B + CH_B, 2 * gm.d + col, c * M_CR, b);
  };
  if (tid == 0) {
    mbar_expect_tx(bars, 2 * OWN_B);
    tma_load_3d(&mOwn, bars, qtile, col, sb * M_QS, b);
    tma_load_3d(&mOwnDO, bars, gtile, col, sb * M_QS, b);
    issue(0, 0);
    if (gm.nchunk > 1) issue(1, 1);
  }
  const int qrow = sb * M_QS + warp * 16;
  const bool live = qrow < T;
  const int r0 = qrow + g, r1 = r0 + 8;
  // row statistics of this lane's two fragment rows; rows >= T: P = exp2(s - inf) = 0
  float ls0 = INFINITY, ls1 = INFINITY, dl0 = 0.f, dl1 = 0.f;
  if (live) {
    const float* lp = lse + ((size_t)b * gm.h + hh) * T;
    const int c0 = min(r0, T - 1), c1 = min(r1, T - 1);      // clamped addresses keep the quad shuffles uniform
    const float a0 = quad_delta<KD>(dout + ((size_t)b * T + c0) * gm.d + col, out + ((size_t)b * T + c0) * gm.d + col, lane);
    const float a1 = quad_delta<KD>(dout + ((size_t)b * T + c1) * gm.d + col, out + ((size_t)b * T + c1) * gm.d + col, lane);
    if (r0 < T) { ls0 = __ldg(lp + r0); dl0 = a0 * gm.scale; }
    if (r1 < T) { ls1 = __ldg(lp + r1); dl1 = a1 * gm.scale; }
  }
  mbar_wait(bars, 0);
  uint32_t aq[KD][4], ag[KD][4];
#pragma unroll
  for (int ks = 0; ks < KD; ++ks) {
    ldsm_x4(aq[ks], addrA<KD>(qtile, warp * 16, ks, lane));
    ldsm_x4(ag[ks], addrA<KD>(gtile, warp * 16, ks, lane));
  }
  float dq[2 * KD][4];
#pragma unroll
  for (int n = 0; n < 2 * KD; ++n) { dq[n][0] = 0.f; dq[n][1] = 0.f; dq[n][2] = 0.f; dq[n][3] = 0.f; }
  for (int c = 0; c < gm.nchunk; ++c) {
    const int s = c & 1;
    mbar_wait(bars + 1 + s, (c >> 1) & 1);
    if (live) {
      const uint32_t kb = st0 + s * 2 * CH_B, vb = kb + CH_B;
      const int nblk = min(M_CB, gm.NQ - c * M_CB);   // zero-filled key rows >= T give dS * 0: no masking needed
      for (int j = 0; j < nblk; ++j) {
        float sc[2][4] = {}, dp[2][4] = {};           // S and dP blocks: rows = queries, columns = 16 keys
#pragma unroll
        for (int ks = 0; ks < KD; ++ks) {
          uint32_t bfr[4];
          ldsm_x4(bfr, addrB<KD>(kb, j * 16, ks, lane));
          mma_bf16(sc[0], aq[ks], bfr[0], bfr[1]);
          mma_bf16(sc[1], aq[ks], bfr[2], bfr[3]);
          ldsm_x4(bfr, addrB<KD>(vb, j * 16, ks, lane));
          mma_bf16(dp[0], ag[ks], bfr[0], bfr[1]);
          mma_bf16(dp[1], ag[ks], bfr[2], bfr[3]);
        }
        uint32_t da[4];
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          const float p0 = ex2(fmaf(sc[u][0], gm.sl2, -ls0)), p1 = ex2(fmaf(sc[u][1], gm.sl2, -ls0));
          const float p2 = ex2(fmaf(sc[u][2], gm.sl2, -ls1)), p3 = ex2(fmaf(sc[u][3], gm.sl2, -ls1));
          da[2 * u] = pack2(p0 * fmaf(dp[u][0], gm.scale, -dl0), p1 * fmaf(dp[u][1], gm.scale, -dl0));
          da[2 * u + 1] = pack2(p2 * fmaf(dp[u][2], gm.scale, -dl1), p3 * fmaf(dp[u][3], gm.scale, -dl1));
        }
#pragma unroll
        for (int np = 0; np < KD; ++np) {
          uint32_t bfr[4];
          ldsm_x4_t(bfr, addrA<KD>(kb, j * 16, np, lane));      // B[k = key][n = c] = K[key][c]
          mma_bf16(dq[2 * np], da, bfr[0], bfr[1]);
          mma_bf16(dq[2 * np + 1], da, bfr[2], bfr[3]);
        }
      }
    }
    __syncthreads();
    if (tid == 0 && c + 2 < gm.nchunk) issue(c + 2, s);
  }
  if (!live) return;
  bf16* q0 = dqkv + ((size_t)b * T + r0) * (3 * gm.d) + col + cb;
  bf16* q1 = dqkv + ((size_t)b * T + r1) * (3 * gm.d) + col + cb;
#pragma unroll
  for (int n = 0; n < 2 * KD; ++n) {
    if (r0 < T) *reinterpret_cast<uint32_t*>(q0 + n * 8) = pack2(dq[n][0], dq[n][1]);
    if (r1 < T) *reinterpret_cast<uint32_t*>(q1 + n * 8) = pack2(dq[n][2], dq[n][3]);
  }
}

// dK, dV.  shared memory: [barriers | K tile | V tile (128 x RB each) | 2 stages x (Q, dO, O chunk tiles) | row stats]
template <int KD>
__global__ void __launch_bounds__(M_NW * 32)
attn_long_mma_dkdv_kernel(const __grid_constant__ CUtensorMap mOwn, const __grid_constant__ CUtensorMap mStreamQ,
                          const __grid_constant__ CUtensorMap mStreamDO, const __grid_constant__ CUtensorMap mStreamO,
                          const LongGeom gm, const float* __restrict__ lse, bf16* __restrict__ dqkv) {
  constexpr int dh = 16 * KD, RB = 32 * KD;
  constexpr uint32_t OWN_B = M_QS * RB, CH_B = M_CR * RB;
  extern __shared__ unsigned char smem_dyn[];
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023) & ~(uintptr_t)1023);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem);
  const uint32_t ktile = smem_u32(smem + M_HDR), vtile = ktile + OWN_B, st0 = vtile + OWN_B;
  float2* s_stat = reinterpret_cast<float2*>(smem + M_HDR + 2 * OWN_B + 6 * CH_B);    // [M_CR] {lse2, delta * scale}
  const uint32_t stat_u = smem_u32(s_stat);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, nt = blockDim.x;
  const int g = lane >> 2, cb = (lane & 3) * 2;
  const int T = gm.T;
  const int sb = blockIdx.x % gm.nsb, bh = blockIdx.x / gm.nsb;
  const int b = bh / gm.h, hh = bh - b * gm.h;
  const int col = hh * dh;
  // lane-constant ldmatrix offsets inside a 16-row block (see attn_tiles.cu)
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
    tma_prefetch_desc(&mOwn);
    tma_prefetch_desc(&mStreamQ);
    tma_prefetch_desc(&mStreamDO);
    tma_prefetch_desc(&mStreamO);
    mbar_init(bars, 1); mbar_init(bars + 1, 1); mbar_init(bars + 2, 1);
    fence_barrier_init();
  }
  __syncthreads();
  auto issue = [&](int c, int s) {        // Q, dO, O rows [c * M_CR, +M_CR) -> stage s
    const uint32_t base = st0 + s * 3 * CH_B;
    mbar_expect_tx(bars + 1 + s, 3 * CH_B);
    tma_load_3d(&mStreamQ, bars + 1 + s, base, col, c * M_CR, b);
    tma_load_3d(&mStreamDO, bars + 1 + s, base + CH_B, col, c * M_CR, b);
    tma_load_3d(&mStreamO, bars + 1 + s, base + 2 * CH_B, col, c * M_CR, b);
  };
  if (tid == 0) {
    mbar_expect_tx(bars, 2 * OWN_B);
    tma_load_3d(&mOwn, bars, ktile, gm.d + col, sb * M_QS, b);
    tma_load_3d(&mOwn, bars, vtile, 2 * gm.d + col, sb * M_QS, b);
    issue(0, 0);
    if (gm.nchunk > 1) issue(1, 1);
  }
  const int krow = sb * M_QS + warp * 16;
  const bool live = krow < T;
  mbar_wait(bars, 0);
  uint32_t ak[KD][4], av[KD][4];
#pragma unroll
  for (int ks = 0; ks < KD; ++ks) {
    ldsm_x4(ak[ks], ktile + (uint32_t)(warp * 16 * RB) + offA[ks]);
    ldsm_x4(av[ks], vtile + (uint32_t)(warp * 16 * RB) + offA[ks]);
  }
  float dk[2 * KD][4], dv[2 * KD][4];
#pragma unroll
  for (int n = 0; n < 2 * KD; ++n) {
    dk[n][0] = 0.f; dk[n][1] = 0.f; dk[n][2] = 0.f; dk[n][3] = 0.f;
    dv[n][0] = 0.f; dv[n][1] = 0.f; dv[n][2] = 0.f; dv[n][3] = 0.f;
  }
  const float* lp = lse + ((size_t)b * gm.h + hh) * T;
  for (int c = 0; c < gm.nchunk; ++c) {
    const int s = c & 1;
    const uint32_t qb = st0 + s * 3 * CH_B, gb = qb + CH_B, ob = gb + CH_B;
    mbar_wait(bars + 1 + s, (c >> 1) & 1);
    // row statistics of the chunk's query rows (rows >= T: zero-filled tiles, lse2 = +inf -> P = 0)
    for (int idx = tid; idx < M_CR; idx += nt) {
      const int r = c * M_CR + idx;
      float dl = 0.f, l2 = INFINITY;
      if (r < T) {
        l2 = __ldg(lp + r);
#pragma unroll
        for (int ch = 0; ch < 2 * KD; ++ch) {
          const uint4 a = lds128(chunk_addr<KD>(gb, idx, ch)), o4 = lds128(chunk_addr<KD>(ob, idx, ch));
          dl += bf_lo(a.x) * bf_lo(o4.x) + bf_hi(a.x) * bf_hi(o4.x) + bf_lo(a.y) * bf_lo(o4.y) + bf_hi(a.y) * bf_hi(o4.y) +
                bf_lo(a.z) * bf_lo(o4.z) + bf_hi(a.z) * bf_hi(o4.z) + bf_lo(a.w) * bf_lo(o4.w) + bf_hi(a.w) * bf_hi(o4.w);
        }
      }
      s_stat[idx] = make_float2(l2, dl * gm.scale);
    }
    __syncthreads();
    if (live) {
      const int nblk = min(M_CB, gm.NQ - c * M_CB);
      for (int qk = 0; qk < nblk; ++qk) {
        const uint32_t qblk = qb + (uint32_t)(qk * 16 * RB), oblk = gb + (uint32_t)(qk * 16 * RB);
        float stt[2][4] = {}, dpt[2][4] = {};      // S^T and dP^T blocks: rows = keys, columns = queries
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
          const float4 st4 = lds128f(stat_u + (uint32_t)((qk * 16 + cb) * 8) + u2 * 64);   // {lse2, dls} of queries cb, cb+1
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
      }
    }
    __syncthreads();                        // stage s and the statistics are free again
    if (tid == 0 && c + 2 < gm.nchunk) issue(c + 2, s);
  }
  if (!live) return;
  const int r0 = krow + g, r1 = r0 + 8;
  bf16* k0p = dqkv + ((size_t)b * T + r0) * (3 * gm.d) + gm.d + col + cb;
  bf16* k1p = dqkv + ((size_t)b * T + r1) * (3 * gm.d) + gm.d + col + cb;
#pragma unroll
  for (int n = 0; n < 2 * KD; ++n) {
    if (r0 < T) {
      *reinterpret_cast<uint32_t*>(k0p + n * 8) = pack2(dk[n][0], dk[n][1]);
      *reinterpret_cast<uint32_t*>(k0p + gm.d + n * 8) = pack2(dv[n][0], dv[n][1]);
    }
    if (r1 < T) {
      *reinterpret_cast<uint32_t*>(k1p + n * 8) = pack2(dk[n][2], dk[n][3]);
      *reinterpret_cast<uint32_t*>(k1p + gm.d + n * 8) = pack2(dv[n][2], dv[n][3]);
    }
  }
}

inline bool mma_ok(int h, int dh) { return (dh == 16 || dh == 32 || dh == 64) && (h * dh) % 8 == 0; }

LongGeom long_geom(int T, int h, int dh) {
  LongGeom g;
  g.T = T; g.h = h; g.d = h * dh; g.NQ = (T + 15) / 16;
  g.nsb = (T + M_QS - 1) / M_QS;
  g.nchunk = (T + M_CR - 1) / M_CR;
  g.scale = 1.f / sqrtf((float)dh);
  g.sl2 = g.scale * LOG2E;
  return g;
}

template <int KD>
int mma_fwd(int B, int T, int h, const bf16* qkv, bf16* out, float* lse, cudaStream_t st) {
  constexpr int dh = 16 * KD, RB = 32 * KD;
  const LongGeom g = long_geom(T, h, dh);
  CUtensorMap mOwn, mStream;
  AMC_TRY(attn_make_map3(&mOwn, qkv, B, T, 3 * g.d, dh, M_QS));
  AMC_TRY(attn_make_map3(&mStream, qkv, B, T, 3 * g.d, dh, M_CR));
  const size_t sm = 1024 + M_HDR + (size_t)M_QS * RB + (size_t)4 * M_CR * RB;
  auto kern = attn_long_mma_fwd_kernel<KD>;
  AMC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
  kern<<<B * h * g.nsb, M_NW * 32, sm, st>>>(mOwn, mStream, g, out, lse);
  AMC_LAUNCH_CHECK();
  return 0;
}

template <int KD>
int mma_bwd(int B, int T, int h, const bf16* qkv, const bf16* out, const float* lse, const bf16* dout, bf16* dqkv,
            cudaStream_t st) {
  constexpr int dh = 16 * KD, RB = 32 * KD;
  const LongGeom g = long_geom(T, h, dh);
  CUtensorMap mOwn, mOwnDO, mStream, mStreamDO, mStreamO;
  AMC_TRY(attn_make_map3(&mOwn, qkv, B, T, 3 * g.d, dh, M_QS));
  AMC_TRY(attn_make_map3(&mOwnDO, dout, B, T, g.d, dh, M_QS));
  AMC_TRY(attn_make_map3(&mStream, qkv, B, T, 3 * g.d, dh, M_CR));
  AMC_TRY(attn_make_map3(&mStreamDO, dout, B, T, g.d, dh, M_CR));
  AMC_TRY(attn_make_map3(&mStreamO, out, B, T, g.d, dh, M_CR));
  {
    const size_t sm = 1024 + M_HDR + (size_t)2 * M_QS * RB + (size_t)4 * M_CR * RB;
    auto kern = attn_long_mma_dq_kernel<KD>;
    AMC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
    kern<<<B * h * g.nsb, M_NW * 32, sm, st>>>(mOwn, mOwnDO, mStream, g, out, dout, lse, dqkv);
    AMC_LAUNCH_CHECK();
  }
  {
    const size_t sm = 1024 + M_HDR + (size_t)2 * M_QS * RB + (size_t)6 * M_CR * RB + (size_t)M_CR * 8;
    auto kern = attn_long_mma_dkdv_kernel<KD>;
    AMC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
    kern<<<B * h * g.nsb, M_NW * 32, sm, st>>>(mOwn, mStream, mStreamDO, mStreamO, g, lse, dqkv);
    AMC_LAUNCH_CHECK();
  }
  return 0;
}

}  // namespace

template <typename E>
int attn_long_fwd(int B, int T, int h, int dh, const E* qkv, E* out, float* lse, cudaStream_t st) {
  AMC_CHECK_ARG(T >= 1 && T <= ATTN_LONG_MAX_T, "attention: T=%d unsupported (1..%d tokens per frame)", T, ATTN_LONG_MAX_T);
  AMC_CHECK_ARG(dh >= 1 && dh <= 32 * S_CC, "attention: head dim %d unsupported (1..%d)", dh, 32 * S_CC);
  if (B == 0) return 0;
  AMC_CHECK_ARG((long long)B * h * ceil_div(T, S_QB) < (1ll << 31), "attention: grid too large");
  if constexpr (std::is_same<E, bf16>::value) {
    if (mma_ok(h, dh) && T > M_CR && (reinterpret_cast<uintptr_t>(qkv) & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 3) == 0) {
      if (dh == 16) return mma_fwd<1>(B, T, h, qkv, out, lse, st);
      if (dh == 32) return mma_fwd<2>(B, T, h, qkv, out, lse, st);
      return mma_fwd<4>(B, T, h, qkv, out, lse, st);
    }
  }
  const int nqb = ceil_div(T, S_QB);
  const size_t sm = 2 * simt_tile_bytes<E>(dh) + (size_t)(S_QB * dh + S_NW * S_KT) * sizeof(float);
  AMC_CUDA(cudaFuncSetAttribute(attn_long_fwd_kernel<E>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
  attn_long_fwd_kernel<E><<<B * h * nqb, S_NW * 32, sm, st>>>(T, h, dh, nqb, qkv, out, lse, 1.f / sqrtf((float)dh));
  AMC_LAUNCH_CHECK();
  return 0;
}
template int attn_long_fwd<float>(int, int, int, int, const float*, float*, float*, cudaStream_t);
template int attn_long_fwd<bf16>(int, int, int, int, const bf16*, bf16*, float*, cudaStream_t);

template <typename E>
int attn_long_bwd(int B, int T, int h, int dh, const E* qkv, const E* out, const float* lse, const E* dout, E* dqkv,
                  cudaStream_t st) {
  AMC_CHECK_ARG(T >= 1 && T <= ATTN_LONG_MAX_T, "attention_bwd: T=%d unsupported (1..%d tokens per frame)", T, ATTN_LONG_MAX_T);
  AMC_CHECK_ARG(dh >= 1 && dh <= 32 * S_CC, "attention_bwd: head dim %d unsupported (1..%d)", dh, 32 * S_CC);
  AMC_CHECK_ARG(out != nullptr && lse != nullptr,
                "attention_bwd: T=%d needs the forward's output and row statistics (out, lse)", T);
  if (B == 0) return 0;
  AMC_CHECK_ARG((long long)B * h * ceil_div(T, S_QB) < (1ll << 31), "attention_bwd: grid too large");
  if constexpr (std::is_same<E, bf16>::value) {
    const bool al = ((reinterpret_cast<uintptr_t>(qkv) | reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(dout)) & 15) == 0 &&
                    (reinterpret_cast<uintptr_t>(dqkv) & 3) == 0;
    if (mma_ok(h, dh) && T > M_CR && al) {
      if (dh == 16) return mma_bwd<1>(B, T, h, qkv, out, lse, dout, dqkv, st);
      if (dh == 32) return mma_bwd<2>(B, T, h, qkv, out, lse, dout, dqkv, st);
      return mma_bwd<4>(B, T, h, qkv, out, lse, dout, dqkv, st);
    }
  }
  const int nb = ceil_div(T, S_QB);
  const float sc = 1.f / sqrtf((float)dh);
  {
    const size_t sm = 2 * simt_tile_bytes<E>(dh) + (size_t)(2 * S_QB * dh + S_NW * S_KT) * sizeof(float);
    AMC_CUDA(cudaFuncSetAttribute(attn_long_dq_kernel<E>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
    attn_long_dq_kernel<E><<<B * h * nb, S_NW * 32, sm, st>>>(T, h, dh, nb, qkv, out, lse, dout, dqkv, sc);
    AMC_LAUNCH_CHECK();
  }
  {
    const size_t sm = 2 * simt_tile_bytes<E>(dh) + (size_t)(2 * S_QB * dh + 2 * S_KT + 2 * S_NW * S_KT) * sizeof(float);
    AMC_CUDA(cudaFuncSetAttribute(attn_long_dkdv_kernel<E>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
    attn_long_dkdv_kernel<E><<<B * h * nb, S_NW * 32, sm, st>>>(T, h, dh, nb, qkv, out, lse, dout, dqkv, sc);
    AMC_LAUNCH_CHECK();
  }
  return 0;
}
template int attn_long_bwd<float>(int, int, int, int, const float*, const float*, const float*, const float*, float*,
                                  cudaStream_t);
template int attn_long_bwd<bf16>(int, int, int, int, const bf16*, const bf16*, const float*, const bf16*, bf16*,
                                 cudaStream_t);

}  // namespace amc

// Short-sequence multi-head attention, forward and backward, one CTA per (frame, head).
// The whole sequence (T <= 257 tokens) of one head lives in shared memory; softmax statistics are
// warp-shuffle reductions in fp32; the [T,T] probability matrix is never written to HBM (the
// reference materialises [B,h,T,T] fp32: scale_dot_product_attention.py:26-37).
// Backward recomputes P from Q,K (SURVEY Appendix B "what to save"): phase 1 is query-row parallel
// (row statistics, dQ), phase 2 is key-row parallel (dK, dV) -- no atomics, deterministic.
//
// Dispatch (attention_fwd / attention_bwd below), first match wins; every branch is reachable and covered by
// tests/test_gpu_ops.py (the shape lists there name the branch each case exercises):
//   T > 288                                   attn_long.cu   flash-style tiles (conv1d embedding, T = 1025)
//   bf16, T <= 16, dh in {16,32,64}           attn_mma_*     frames x heads packed per CTA (ViT p16: T = 9)
//   bf16, 49 <= T <= 272, dh in {16,32,64}    attn_tc5.cu    tcgen05 / TMEM, where it is the faster kernel, per direction (forward: T > 80 or
//                                                            dh = 64; backward: dh = 32 at T > 80, dh = 64): tc5_preferred()
//   bf16, 16 < T <= 288, dh in {16,32,64}     attn_tiles.cu  mma.sync tiles (backward: while its tiles fit, i.e. not dh = 64, T > 176)
//   T <= 32, dh <= 32, h T <= 256             attn_frames_*  SIMT, several frames per CTA (fp32 parity path; bf16 odd head dims)
//   anything else (T <= 288, dh <= 128)       attn_fwd/bwd_kernel  SIMT, one CTA per (frame, head): fp32, head dims 48 / 96 / 128,
//                                             backward without the forward's out / lse
// (Round 2 removed a fourth generation -- the bulk-copy mma.sync "attn_tc" kernels -- that only dh = 64, 177 <= T <= 215
//  backward still reached; those shapes take the SIMT kernel now.)
#include <cstdlib>

#include "attention.cuh"
#include "ptx.cuh"
#include "rowops.cuh"

#include <type_traits>

namespace amc {
namespace {

template <typename S> struct SmemPad;
template <> struct SmemPad<float> { static constexpr int v = 1; };
template <> struct SmemPad<bf16> { static constexpr int v = 2; };

constexpr int MAXJ = 9;  // ceil(257 / 32) keys per lane

template <typename E>
__device__ __forceinline__ void load_head_tile(E* dst, int stride, const E* __restrict__ src, int ld, int T, int dh) {
  // dst[t][c] = src[t*ld + c]
  for (int i = threadIdx.x; i < T * dh; i += blockDim.x) {
    const int t = i / dh, c = i - t * dh;
    dst[t * stride + c] = src[(size_t)t * ld + c];
  }
}

template <typename E>
__global__ void __launch_bounds__(256) attn_fwd_kernel(int T, int h, int dh, const E* __restrict__ qkv,
                                                       E* __restrict__ out, float scale) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int d = h * dh, ld = 3 * d;
  const int stride = dh + SmemPad<E>::v;
  const int nw = blockDim.x >> 5, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tile = (T * stride + 1) & ~1;   // even element count keeps the float region aligned
  E* Ks = reinterpret_cast<E*>(smem_raw);
  E* Vs = Ks + tile;
  float* qs = reinterpret_cast<float*>(Vs + tile);
  float* ps = qs + nw * dh;
  const int b = blockIdx.x / h, hh = blockIdx.x - b * h;
  const E* base = qkv + (size_t)b * T * ld + hh * dh;
  load_head_tile(Ks, stride, base + d, ld, T, dh);
  load_head_tile(Vs, stride, base + 2 * d, ld, T, dh);
  __syncthreads();
  float* myq = qs + warp * dh;
  float* myp = ps + warp * T;
  for (int i = warp; i < T; i += nw) {
    for (int c = lane; c < dh; c += 32) myq[c] = to_f(base[(size_t)i * ld + c]) * scale;
    __syncwarp();
    float s[MAXJ];
    float mx = -INFINITY;
#pragma unroll
    for (int jj = 0; jj < MAXJ; ++jj) {
      const int j = lane + 32 * jj;
      float a = -INFINITY;
      if (j < T) {
        a = 0.f;
        const E* kr = Ks + j * stride;
        for (int c = 0; c < dh; ++c) a = fmaf(myq[c], to_f(kr[c]), a);
      }
      s[jj] = a;
      mx = fmaxf(mx, a);
    }
    mx = warp_max(mx);
    float l = 0.f;
#pragma unroll
    for (int jj = 0; jj < MAXJ; ++jj) {
      const int j = lane + 32 * jj;
      const float e = j < T ? __expf(s[jj] - mx) : 0.f;
      s[jj] = e;
      l += e;
    }
    l = warp_sum(l);
    const float inv = 1.f / l;
#pragma unroll
    for (int jj = 0; jj < MAXJ; ++jj) {
      const int j = lane + 32 * jj;
      if (j < T) myp[j] = s[jj] * inv;
    }
    __syncwarp();
    for (int c = lane; c < dh; c += 32) {
      float a = 0.f;
      for (int j = 0; j < T; ++j) a = fmaf(myp[j], to_f(Vs[j * stride + c]), a);
      out[((size_t)b * T + i) * d + hh * dh + c] = from_f<E>(a);
    }
    __syncwarp();
  }
}

template <typename E>
__global__ void __launch_bounds__(256) attn_bwd_kernel(int T, int h, int dh, const E* __restrict__ qkv,
                                                       const E* __restrict__ dout, E* __restrict__ dqkv,
                                                       float scale) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int d = h * dh, ld = 3 * d;
  const int stride = dh + SmemPad<E>::v;
  const int nw = blockDim.x >> 5, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tile = (T * stride + 1) & ~1;   // even element count keeps the float region aligned
  E* Qs = reinterpret_cast<E*>(smem_raw);
  E* Ks = Qs + tile;
  E* Vs = Ks + tile;
  E* Os = Vs + tile;                        // dO
  float* st_m = reinterpret_cast<float*>(Os + tile);
  float* st_il = st_m + T;
  float* st_dl = st_il + T;
  float* bufA = st_dl + T;                  // [nw][T]
  float* bufB = bufA + nw * T;              // [nw][T]
  const int b = blockIdx.x / h, hh = blockIdx.x - b * h;
  const E* base = qkv + (size_t)b * T * ld + hh * dh;
  load_head_tile(Qs, stride, base, ld, T, dh);
  load_head_tile(Ks, stride, base + d, ld, T, dh);
  load_head_tile(Vs, stride, base + 2 * d, ld, T, dh);
  load_head_tile(Os, stride, dout + (size_t)b * T * d + hh * dh, d, T, dh);
  __syncthreads();
  float* myA = bufA + warp * T;
  E* dbase = dqkv + (size_t)b * T * ld + hh * dh;

  // ---- phase 1: one warp per query row: statistics + dQ ---------------------------------
  for (int i = warp; i < T; i += nw) {
    const E* qr = Qs + i * stride;
    const E* orow = Os + i * stride;
    float s[MAXJ], dp[MAXJ];
    float mx = -INFINITY;
#pragma unroll
    for (int jj = 0; jj < MAXJ; ++jj) {
      const int j = lane + 32 * jj;
      float a = -INFINITY, g = 0.f;
      if (j < T) {
        a = 0.f;
        const E* kr = Ks + j * stride;
        const E* vr = Vs + j * stride;
        for (int c = 0; c < dh; ++c) {
          a = fmaf(to_f(qr[c]), to_f(kr[c]), a);
          g = fmaf(to_f(orow[c]), to_f(vr[c]), g);
        }
        a *= scale;
      }
      s[jj] = a;
      dp[jj] = g;
      mx = fmaxf(mx, a);
    }
    mx = warp_max(mx);
    float l = 0.f;
#pragma unroll
    for (int jj = 0; jj < MAXJ; ++jj) {
      const int j = lane + 32 * jj;
      const float e = j < T ? __expf(s[jj] - mx) : 0.f;
      s[jj] = e;
      l += e;
    }
    l = warp_sum(l);
    const float inv = 1.f / l;
    float dl = 0.f;
#pragma unroll
    for (int jj = 0; jj < MAXJ; ++jj) {
      s[jj] *= inv;
      dl = fmaf(s[jj], dp[jj], dl);
    }
    dl = warp_sum(dl);
    if (lane == 0) {
      st_m[i] = mx;
      st_il[i] = inv;
      st_dl[i] = dl;
    }
#pragma unroll
    for (int jj = 0; jj < MAXJ; ++jj) {
      const int j = lane + 32 * jj;
      if (j < T) myA[j] = s[jj] * (dp[jj] - dl) * scale;   // dS[i, j]
    }
    __syncwarp();
    for (int c = lane; c < dh; c += 32) {
      float a = 0.f;
      for (int j = 0; j < T; ++j) a = fmaf(myA[j], to_f(Ks[j * stride + c]), a);
      dbase[(size_t)i * ld + c] = from_f<E>(a);              // dQ
    }
    __syncwarp();
  }
  __syncthreads();

  // ---- phase 2: one warp per key row: dK, dV -------------------------------------------
  float* myB = bufB + warp * T;
  for (int j = warp; j < T; j += nw) {
    const E* kr = Ks + j * stride;
    const E* vr = Vs + j * stride;
#pragma unroll
    for (int ii = 0; ii < MAXJ; ++ii) {
      const int i = lane + 32 * ii;
      if (i < T) {
        const E* qr = Qs + i * stride;
        const E* orow = Os + i * stride;
        float a = 0.f, g = 0.f;
        for (int c = 0; c < dh; ++c) {
          a = fmaf(to_f(qr[c]), to_f(kr[c]), a);
          g = fmaf(to_f(orow[c]), to_f(vr[c]), g);
        }
        const float p = __expf(a * scale - st_m[i]) * st_il[i];
        myA[i] = p;                                         // P[i, j]
        myB[i] = p * (g - st_dl[i]) * scale;                // dS[i, j]
      }
    }
    __syncwarp();
    for (int c = lane; c < dh; c += 32) {
      float dk = 0.f, dv = 0.f;
      for (int i = 0; i < T; ++i) {
        dk = fmaf(myB[i], to_f(Qs[i * stride + c]), dk);
        dv = fmaf(myA[i], to_f(Os[i * stride + c]), dv);
      }
      dbase[(size_t)j * ld + d + c] = from_f<E>(dk);
      dbase[(size_t)j * ld + 2 * d + c] = from_f<E>(dv);
    }
    __syncwarp();
  }
}


// ---------------------------------------------------------------------------------------------
// Small-sequence variant (T <= 32 tokens, head dim <= 32 and % 4 == 0, e.g. ViT patch 16: T = 9).
// A CTA owns whole FRAMES: the [T, 3d] q|k|v rows of a frame are contiguous in HBM, so staging is a
// straight 16-byte-vector copy (no gather), kept in the storage dtype; rows get 16 B of padding so the
// per-thread row reads spread over the banks.  One THREAD per (frame, head, query row) keeps its q / dO /
// output rows in registers and streams K/V rows as broadcast vector loads.  Results are staged in shared
// memory and leave as 16-byte row copies.  The grid is persistent (a few CTAs per SM loop over frames).
// ---------------------------------------------------------------------------------------------
template <typename E> struct Vec16 { static constexpr int n = 16 / sizeof(E); };   // elements per 16 bytes

// copy `rows` rows of `row_elems` elements between a dense global block and a padded smem block
template <typename E, bool TO_SMEM>
__device__ __forceinline__ void rows_copy(E* smem_blk, int smem_stride, E* gmem_blk, int rows, int row_elems, int tid,
                                          int nt) {
  const int vpr = row_elems / Vec16<E>::n;      // vectors per row
  int r = tid / vpr, c = tid - r * vpr;
  const int dr = nt / vpr, dc = nt - dr * vpr;
  while (r < rows) {
    uint4* sp = reinterpret_cast<uint4*>(smem_blk + (size_t)r * smem_stride) + c;
    uint4* gp = reinterpret_cast<uint4*>(gmem_blk + (size_t)r * row_elems) + c;
    if (TO_SMEM) *sp = *gp;
    else *gp = *sp;
    r += dr;
    c += dc;
    if (c >= vpr) { c -= vpr; ++r; }
  }
}

// ---- 1-D bulk (TMA) row copies: one elected thread moves whole rows, completion on an mbarrier ----
// load `rows` dense global rows into padded smem rows (called by ONE thread)
template <typename E>
__device__ __forceinline__ void bulk_rows_in(E* smem_blk, int smem_stride, const E* gmem_blk, int rows, int row_elems,
                                             uint64_t* bar) {
  const uint32_t rb = (uint32_t)(row_elems * sizeof(E));
  mbar_expect_tx(bar, rb * (uint32_t)rows);
  for (int r = 0; r < rows; ++r)
    bulk_g2s(smem_u32(smem_blk + (size_t)r * smem_stride), gmem_blk + (size_t)r * row_elems, rb, bar);
}
template <typename E>
__device__ __forceinline__ void bulk_rows_out(E* gmem_blk, const E* smem_blk, int smem_stride, int rows, int row_elems) {
  const uint32_t rb = (uint32_t)(row_elems * sizeof(E));
  for (int r = 0; r < rows; ++r)
    bulk_s2g(gmem_blk + (size_t)r * row_elems, smem_u32(smem_blk + (size_t)r * smem_stride), rb);
  bulk_commit();
}

// row (<= 32 elements) <-> registers; only the first nq float4 are live
template <typename E>
__device__ __forceinline__ void row_load(float4 (&r)[8], const E* p, int nq) {
#pragma unroll
  for (int k = 0; k < 8; ++k) r[k] = k < nq ? load4(p + 4 * k) : make_float4(0, 0, 0, 0);
}
template <typename E>
__device__ __forceinline__ void row_store(E* p, const float4 (&r)[8], int nq) {
#pragma unroll
  for (int k = 0; k < 8; ++k)
    if (k < nq) store4(p + 4 * k, r[k]);
}
template <typename E>
__device__ __forceinline__ float row_dot(const float4 (&a)[8], const E* p, int nq) {
  float s = 0.f;
#pragma unroll
  for (int k = 0; k < 8; ++k)
    if (k < nq) {
      const float4 b = load4(p + 4 * k);
      s = fmaf(a[k].x, b.x, s); s = fmaf(a[k].y, b.y, s); s = fmaf(a[k].z, b.z, s); s = fmaf(a[k].w, b.w, s);
    }
  return s;
}
template <typename E>
__device__ __forceinline__ void row_axpy(float4 (&acc)[8], float w, const E* p, int nq) {
#pragma unroll
  for (int k = 0; k < 8; ++k)
    if (k < nq) {
      const float4 b = load4(p + 4 * k);
      acc[k].x = fmaf(w, b.x, acc[k].x); acc[k].y = fmaf(w, b.y, acc[k].y);
      acc[k].z = fmaf(w, b.z, acc[k].z); acc[k].w = fmaf(w, b.w, acc[k].w);
    }
}
__device__ __forceinline__ void row_zero(float4 (&r)[8]) {
#pragma unroll
  for (int k = 0; k < 8; ++k) r[k] = make_float4(0, 0, 0, 0);
}

template <typename E, int MAXT>
__global__ void __launch_bounds__(256) attn_frames_fwd_kernel(int B, int T, int h, int dh, int F,
                                                              const E* __restrict__ qkv, E* __restrict__ out,
                                                              float scale) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int d = h * dh, ld = 3 * d, nq = dh >> 2;
  const int s_in = ld + Vec16<E>::n, s_out = d + Vec16<E>::n;     // padded row strides (elements)
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw);          // [2] input buffers
  E* blk0 = reinterpret_cast<E*>(smem_raw + 128);
  const size_t in_elems = (size_t)F * T * s_in;
  E* oblk = blk0 + 2 * in_elems;
  const int tid = threadIdx.x;
  const int hT = h * T;
  const int f = tid / hT, rem = tid - f * hT, hh = rem / T, i = rem - hh * T;
  if (tid == 0) {
    mbar_init(bars, 1);
    fence_barrier_init();
    mbar_init(bars + 1, 1);
    fence_barrier_init();
  }
  __syncthreads();
  const int stride_f = gridDim.x * F;
  int f0 = blockIdx.x * F;
  if (tid == 0 && f0 < B) bulk_rows_in(blk0, s_in, qkv + (size_t)f0 * T * ld, min(F, B - f0) * T, ld, bars);
  for (uint32_t it = 0; f0 < B; f0 += stride_f, ++it) {
    const int nf = min(F, B - f0);
    E* blk = blk0 + (it & 1) * in_elems;
    if (tid == 0) {
      const int fn = f0 + stride_f;           // prefetch the next frames into the other buffer
      if (fn < B) bulk_rows_in(blk0 + ((it + 1) & 1) * in_elems, s_in, qkv + (size_t)fn * T * ld, min(F, B - fn) * T, ld,
                               bars + ((it + 1) & 1));
    }
    mbar_wait(bars + (it & 1), (it >> 1) & 1);
    float4 o[8];
    if (f < nf) {
      const E* fb = blk + (size_t)f * T * s_in + hh * dh;
      float4 q[8];
      row_load(q, fb + (size_t)i * s_in, nq);
      float s[MAXT];
      float mx = -INFINITY;
#pragma unroll
      for (int j = 0; j < MAXT; ++j) {
        s[j] = j < T ? row_dot(q, fb + (size_t)j * s_in + d, nq) * scale : -INFINITY;
        mx = fmaxf(mx, s[j]);
      }
      float l = 0.f;
#pragma unroll
      for (int j = 0; j < MAXT; ++j) {
        s[j] = j < T ? __expf(s[j] - mx) : 0.f;
        l += s[j];
      }
      const float inv = 1.f / l;
      row_zero(o);
#pragma unroll
      for (int j = 0; j < MAXT; ++j)
        if (j < T) row_axpy(o, s[j] * inv, fb + (size_t)j * s_in + 2 * d, nq);
    }
    if (tid == 0) bulk_wait_read<0>();          // previous iteration's output rows have left oblk
    __syncthreads();                          // ... and everyone is done reading blk (it may be refilled next iteration)
    if (f < nf) row_store(oblk + ((size_t)f * T + i) * s_out + hh * dh, o, nq);
    fence_proxy_async();
    __syncthreads();
    if (tid == 0) bulk_rows_out(out + (size_t)f0 * T * d, oblk, s_out, nf * T, d);
  }
  if (tid == 0) bulk_wait_all();
}

template <typename E, int MAXT>
__global__ void __launch_bounds__(256) attn_frames_bwd_kernel(int B, int T, int h, int dh, int F,
                                                              const E* __restrict__ qkv, const E* __restrict__ dout,
                                                              E* __restrict__ dqkv, float scale) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int d = h * dh, ld = 3 * d, nq = dh >> 2, pt = T * (T + 1);
  const int s_in = ld + Vec16<E>::n, s_do = d + Vec16<E>::n;
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem_raw);
  E* blk = reinterpret_cast<E*>(smem_raw + 128);
  E* doblk = blk + (size_t)F * T * s_in;
  E* oblk = doblk + (size_t)F * T * s_do;                          // dq|dk|dv staging
  float* pbase = reinterpret_cast<float*>(oblk + (size_t)F * T * s_in);   // [F*h][2][T][T+1]
  const int tid = threadIdx.x;
  const int hT = h * T;
  const int f = tid / hT, rem = tid - f * hT, hh = rem / T, i = rem - hh * T;
  if (tid == 0) {
    mbar_init(bar, 1);
    fence_barrier_init();
  }
  __syncthreads();
  const int stride_f = gridDim.x * F;
  int f0 = blockIdx.x * F;
  if (tid == 0 && f0 < B) {
    const int rows = min(F, B - f0) * T;
    mbar_expect_tx(bar, (uint32_t)(rows * (ld + d) * sizeof(E)));
    for (int r = 0; r < rows; ++r) {
      bulk_g2s(smem_u32(blk + (size_t)r * s_in), qkv + ((size_t)f0 * T + r) * ld, (uint32_t)(ld * sizeof(E)), bar);
      bulk_g2s(smem_u32(doblk + (size_t)r * s_do), dout + ((size_t)f0 * T + r) * d, (uint32_t)(d * sizeof(E)), bar);
    }
  }
  for (uint32_t it = 0; f0 < B; f0 += stride_f, ++it) {
    const int nf = min(F, B - f0);
    mbar_wait(bar, it & 1);
    const bool act = f < nf;
    const E* fb = blk + (size_t)(act ? f : 0) * T * s_in + hh * dh;          // q at +0, k at +d, v at +2d
    const E* fo = doblk + (size_t)(act ? f : 0) * T * s_do + hh * dh;
    float* P = pbase + (size_t)((act ? f : 0) * h + hh) * 2 * pt;
    float* dS = P + pt;
    if (act) {   // phase 1: row i of P and dS
      float4 q[8], o[8];
      row_load(q, fb + (size_t)i * s_in, nq);
      row_load(o, fo + (size_t)i * s_do, nq);
      float s[MAXT], dp[MAXT];
      float mx = -INFINITY;
#pragma unroll
      for (int j = 0; j < MAXT; ++j) {
        s[j] = j < T ? row_dot(q, fb + (size_t)j * s_in + d, nq) * scale : -INFINITY;
        dp[j] = j < T ? row_dot(o, fb + (size_t)j * s_in + 2 * d, nq) : 0.f;
        mx = fmaxf(mx, s[j]);
      }
      float l = 0.f;
#pragma unroll
      for (int j = 0; j < MAXT; ++j) {
        s[j] = j < T ? __expf(s[j] - mx) : 0.f;
        l += s[j];
      }
      const float inv = 1.f / l;
      float dl = 0.f;
#pragma unroll
      for (int j = 0; j < MAXT; ++j) {
        s[j] *= inv;
        dl = fmaf(s[j], dp[j], dl);
      }
#pragma unroll
      for (int j = 0; j < MAXT; ++j)
        if (j < T) {
          P[i * (T + 1) + j] = s[j];
          dS[i * (T + 1) + j] = s[j] * (dp[j] - dl) * scale;
        }
    }
    __syncthreads();
    float4 dq[8], dk[8], dv[8];
    row_zero(dq); row_zero(dk); row_zero(dv);
    if (act) {   // phase 2: dQ_i (as query row i) and dK_i, dV_i (as key row i)
      for (int j = 0; j < T; ++j) {
        row_axpy(dq, dS[i * (T + 1) + j], fb + (size_t)j * s_in + d, nq);    // query i, key j
        row_axpy(dk, dS[j * (T + 1) + i], fb + (size_t)j * s_in, nq);        // query j, key i
        row_axpy(dv, P[j * (T + 1) + i], fo + (size_t)j * s_do, nq);
      }
    }
    if (tid == 0) bulk_wait_read<0>();          // previous iteration's gradient rows have left oblk
    __syncthreads();                          // every read of q/k/v/dO is done: inputs may be refilled
    if (tid == 0) {
      const int fn = f0 + stride_f;
      if (fn < B) {
        const int rows = min(F, B - fn) * T;
        mbar_expect_tx(bar, (uint32_t)(rows * (ld + d) * sizeof(E)));
        for (int r = 0; r < rows; ++r) {
          bulk_g2s(smem_u32(blk + (size_t)r * s_in), qkv + ((size_t)fn * T + r) * ld, (uint32_t)(ld * sizeof(E)), bar);
          bulk_g2s(smem_u32(doblk + (size_t)r * s_do), dout + ((size_t)fn * T + r) * d, (uint32_t)(d * sizeof(E)), bar);
        }
      }
    }
    if (act) {
      E* ob = oblk + ((size_t)f * T + i) * s_in + hh * dh;
      row_store(ob, dq, nq);
      row_store(ob + d, dk, nq);
      row_store(ob + 2 * d, dv, nq);
    }
    fence_proxy_async();
    __syncthreads();
    if (tid == 0) bulk_rows_out(dqkv + (size_t)f0 * T * ld, oblk, s_in, nf * T, ld);
  }
  if (tid == 0) bulk_wait_all();
}

// ---------------------------------------------------------------------------------------------
// Tensor-core variant for T <= 16 tokens, bf16, head dim 16*KD (KD = 1, 2, 4): one WARP per (frame, head).
// The 16x16 score tile is two m16n8k16 MMAs per 16 head-dim columns; operands come straight from the staged
// frame rows with ldmatrix (row pitch 6d+16 bytes: the 8 rows of every 8x8 matrix hit 8 different 16-byte
// bank groups).  Softmax runs on the accumulator fragments (quad shuffles); P and dS are re-used as A
// fragments directly from registers, and go through a tiny per-warp smem tile only where the transpose is
// needed (dK = dS^T Q, dV = P^T dO).  Rows/keys >= T are padding: their addresses are clamped to row T-1,
// key columns are masked to -inf, query rows are zeroed in backward and never written.
// ---------------------------------------------------------------------------------------------
// A-operand address (rows r0.., 16 columns at col0) / "K-pattern" B address (rows = n, cols = k) for lane
__device__ __forceinline__ uint32_t addr_a(uint32_t base, int pitch_b, int T, int col0, int lane) {
  const int r = min((lane & 7) + ((lane >> 3) & 1) * 8, T - 1);
  return base + r * pitch_b + (col0 + (lane >> 4) * 8) * 2;
}
__device__ __forceinline__ uint32_t addr_bk(uint32_t base, int pitch_b, int T, int col0, int lane) {
  const int r = min((lane & 7) + (lane >> 4) * 8, T - 1);
  return base + r * pitch_b + (col0 + ((lane >> 3) & 1) * 8) * 2;
}
// "V-pattern" (transposed) B address: rows = k (tokens), cols = n (16 head-dim columns at col0)
__device__ __forceinline__ uint32_t addr_bv(uint32_t base, int pitch_b, int T, int col0, int lane) {
  const int r = min((lane & 7) + ((lane >> 3) & 1) * 8, T - 1);
  return base + r * pitch_b + (col0 + (lane >> 4) * 8) * 2;
}

// scores -> probabilities on the accumulator fragments; returns nothing, p[nt][*] normalised, masked
__device__ __forceinline__ void frag_softmax(float (&c)[2][4], int T, float scale, int lane) {
  const int cb = (lane & 3) * 2;
  float m0 = -INFINITY, m1 = -INFINITY;
#pragma unroll
  for (int nt = 0; nt < 2; ++nt)
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const bool ok = nt * 8 + cb + e < T;
      c[nt][e] = ok ? c[nt][e] * scale : -INFINITY;
      c[nt][2 + e] = ok ? c[nt][2 + e] * scale : -INFINITY;
      m0 = fmaxf(m0, c[nt][e]);
      m1 = fmaxf(m1, c[nt][2 + e]);
    }
  m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 1)); m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 2));
  m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 1)); m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 2));
  float s0 = 0.f, s1 = 0.f;
#pragma unroll
  for (int nt = 0; nt < 2; ++nt)
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      c[nt][e] = __expf(c[nt][e] - m0);
      c[nt][2 + e] = __expf(c[nt][2 + e] - m1);
      s0 += c[nt][e];
      s1 += c[nt][2 + e];
    }
  s0 += __shfl_xor_sync(0xffffffffu, s0, 1); s0 += __shfl_xor_sync(0xffffffffu, s0, 2);
  s1 += __shfl_xor_sync(0xffffffffu, s1, 1); s1 += __shfl_xor_sync(0xffffffffu, s1, 2);
  const float i0 = 1.f / s0, i1 = 1.f / s1;
#pragma unroll
  for (int nt = 0; nt < 2; ++nt)
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      c[nt][e] *= i0;
      c[nt][2 + e] *= i1;
    }
}

template <int KD>
__global__ void __launch_bounds__(256) attn_mma_fwd_kernel(int B, int T, int h, int F, const bf16* __restrict__ qkv,
                                                           bf16* __restrict__ out, float scale) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  constexpr int dh = 16 * KD;
  const int d = h * dh, ld = 3 * d;
  const int s_in = ld + 8, s_out = d + 8;
  const int pin = s_in * 2;                                        // row pitch in bytes
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw);
  bf16* blk0 = reinterpret_cast<bf16*>(smem_raw + 128);
  const size_t in_elems = (size_t)F * T * s_in;
  bf16* oblk = blk0 + 2 * in_elems;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, nw = blockDim.x >> 5;
  if (tid == 0) {
    mbar_init(bars, 1);
    fence_barrier_init();
    mbar_init(bars + 1, 1);
    fence_barrier_init();
  }
  __syncthreads();
  const int stride_f = gridDim.x * F;
  int f0 = blockIdx.x * F;
  // Row copies are dealt round-robin to lane 0 of every warp: issued by one thread, the ~60 bulk copies of an
  // iteration cost about a quarter of it.  Thread 0 arms the barrier with the byte count, the copies may land first.
  auto rows_in = [&](bf16* dst, int fs, uint64_t* bar) {      // called by lane 0 of each warp
    const int rows = min(F, B - fs) * T;
    if (warp == 0) mbar_expect_tx(bar, (uint32_t)(rows * ld * 2));
    for (int r = warp; r < rows; r += nw)
      bulk_g2s(smem_u32(dst + (size_t)r * s_in), qkv + ((size_t)fs * T + r) * ld, (uint32_t)(ld * 2), bar);
  };
  if (lane == 0 && f0 < B) rows_in(blk0, f0, bars);
  for (uint32_t it = 0; f0 < B; f0 += stride_f, ++it) {
    const int nf = min(F, B - f0);
    bf16* blk = blk0 + (it & 1) * in_elems;
    if (lane == 0) {
      const int fn = f0 + stride_f;
      if (fn < B) rows_in(blk0 + ((it + 1) & 1) * in_elems, fn, bars + ((it + 1) & 1));
      bulk_wait_read<0>();                       // this warp's output rows of the previous iteration have left oblk
    }
    mbar_wait(bars + (it & 1), (it >> 1) & 1);
    __syncthreads();
    for (int pr = warp; pr < nf * h; pr += nw) {
      const int f = pr / h, hh = pr - f * h;
      const uint32_t qb = smem_u32(blk + (size_t)f * T * s_in + hh * dh);
      const uint32_t kb = qb + d * 2, vb = qb + 2 * d * 2;
      float c[2][4] = {};
#pragma unroll
      for (int ks = 0; ks < KD; ++ks) {
        uint32_t a[4], b[4];
        ldsm_x4(a, addr_a(qb, pin, T, ks * 16, lane));
        ldsm_x4(b, addr_bk(kb, pin, T, ks * 16, lane));
        mma_bf16(c[0], a, b[0], b[1]);
        mma_bf16(c[1], a, b[2], b[3]);
      }
      frag_softmax(c, T, scale, lane);
      uint32_t pa[4] = {pack2(c[0][0], c[0][1]), pack2(c[0][2], c[0][3]), pack2(c[1][0], c[1][1]),
                        pack2(c[1][2], c[1][3])};
      float o[2 * KD][4] = {};
#pragma unroll
      for (int np = 0; np < KD; ++np) {
        uint32_t b[4];
        ldsm_x4_t(b, addr_bv(vb, pin, T, np * 16, lane));
        mma_bf16(o[2 * np], pa, b[0], b[1]);
        mma_bf16(o[2 * np + 1], pa, b[2], b[3]);
      }
      const int g = lane >> 2, cb = (lane & 3) * 2;
      bf16* ob = oblk + (size_t)f * T * s_out + hh * dh + cb;
#pragma unroll
      for (int nt = 0; nt < 2 * KD; ++nt) {
        if (g < T) *reinterpret_cast<uint32_t*>(ob + (size_t)g * s_out + nt * 8) = pack2(o[nt][0], o[nt][1]);
        if (g + 8 < T) *reinterpret_cast<uint32_t*>(ob + (size_t)(g + 8) * s_out + nt * 8) = pack2(o[nt][2], o[nt][3]);
      }
    }
    fence_proxy_async();
    __syncthreads();
    if (lane == 0) {
      for (int r = warp; r < nf * T; r += nw)
        bulk_s2g(out + ((size_t)f0 * T + r) * d, smem_u32(oblk + (size_t)r * s_out), (uint32_t)(d * 2));
      bulk_commit();
    }
  }
  if (lane == 0) bulk_wait_all();
}

template <int KD>
__global__ void __launch_bounds__(256) attn_mma_bwd_kernel(int B, int T, int h, int F, const bf16* __restrict__ qkv,
                                                           const bf16* __restrict__ dout, bf16* __restrict__ dqkv,
                                                           float* __restrict__ dbias, float scale) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  constexpr int dh = 16 * KD;
  constexpr int TP = 24;                                            // pitch (elements) of the 16x16 transpose tiles
  const int d = h * dh, ld = 3 * d;
  const int s_in = ld + 8, s_do = d + 8;
  const int pin = s_in * 2, pdo = s_do * 2;
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem_raw);
  bf16* blk = reinterpret_cast<bf16*>(smem_raw + 128);
  bf16* doblk = blk + (size_t)F * T * s_in;
  bf16* oblk = doblk + (size_t)F * T * s_do;
  bf16* tiles = oblk + (size_t)F * T * s_in;                        // [warps][2][16][TP]
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, nw = blockDim.x >> 5;
  bf16* tP = tiles + (size_t)warp * 2 * 16 * TP;
  bf16* tS = tP + 16 * TP;
  if (tid == 0) {
    mbar_init(bar, 1);
    fence_barrier_init();
  }
  __syncthreads();
  const int stride_f = gridDim.x * F;
  int f0 = blockIdx.x * F;
  // row copies dealt round-robin to lane 0 of every warp (see the forward kernel); thread 0 arms the barrier
  auto issue = [&](int fs) {                                  // called by lane 0 of each warp
    const int rows = min(F, B - fs) * T;
    if (warp == 0) mbar_expect_tx(bar, (uint32_t)(rows * (ld + d) * 2));
    for (int r = warp; r < rows; r += nw) {
      bulk_g2s(smem_u32(blk + (size_t)r * s_in), qkv + ((size_t)fs * T + r) * ld, (uint32_t)(ld * 2), bar);
      bulk_g2s(smem_u32(doblk + (size_t)r * s_do), dout + ((size_t)fs * T + r) * d, (uint32_t)(d * 2), bar);
    }
  };
  if (lane == 0 && f0 < B) issue(f0);
  // bias gradient of the QKV projection (Appendix B: db = sum of dQ|dK|dV rows): each thread owns up to two
  // 4-column groups of the staged gradient rows and keeps their sums in registers across all its frames
  float4 bsum[2] = {make_float4(0, 0, 0, 0), make_float4(0, 0, 0, 0)};
  const int ngroups = ld >> 2;
  for (uint32_t it = 0; f0 < B; f0 += stride_f, ++it) {
    const int nf = min(F, B - f0);
    if (lane == 0) bulk_wait_read<0>();         // this warp's gradient rows of the previous iteration have left oblk
    mbar_wait(bar, it & 1);
    __syncthreads();
    const int g = lane >> 2, cb = (lane & 3) * 2;
    for (int pr = warp; pr < nf * h; pr += nw) {
      const int f = pr / h, hh = pr - f * h;
      const uint32_t qb = smem_u32(blk + (size_t)f * T * s_in + hh * dh);
      const uint32_t kb = qb + d * 2, vb = qb + 2 * d * 2;
      const uint32_t ob = smem_u32(doblk + (size_t)f * T * s_do + hh * dh);
      float c[2][4] = {}, dp[2][4] = {};
#pragma unroll
      for (int ks = 0; ks < KD; ++ks) {
        uint32_t a[4], b[4];
        ldsm_x4(a, addr_a(qb, pin, T, ks * 16, lane));
        ldsm_x4(b, addr_bk(kb, pin, T, ks * 16, lane));
        mma_bf16(c[0], a, b[0], b[1]);
        mma_bf16(c[1], a, b[2], b[3]);
        ldsm_x4(a, addr_a(ob, pdo, T, ks * 16, lane));           // dO rows
        ldsm_x4(b, addr_bk(vb, pin, T, ks * 16, lane));          // V^T: B[k=c][n=j] = V[j][c]
        mma_bf16(dp[0], a, b[0], b[1]);
        mma_bf16(dp[1], a, b[2], b[3]);
      }
      frag_softmax(c, T, scale, lane);
      // delta_i = sum_j P dP ; dS = P (dP - delta) scale ; padded query rows are zeroed
      float d0 = 0.f, d1 = 0.f;
#pragma unroll
      for (int nt = 0; nt < 2; ++nt)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          d0 = fmaf(c[nt][e], dp[nt][e], d0);
          d1 = fmaf(c[nt][2 + e], dp[nt][2 + e], d1);
        }
      d0 += __shfl_xor_sync(0xffffffffu, d0, 1); d0 += __shfl_xor_sync(0xffffffffu, d0, 2);
      d1 += __shfl_xor_sync(0xffffffffu, d1, 1); d1 += __shfl_xor_sync(0xffffffffu, d1, 2);
      const bool r0 = g < T, r1 = g + 8 < T;
      float ds[2][4];
#pragma unroll
      for (int nt = 0; nt < 2; ++nt)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          c[nt][e] = r0 ? c[nt][e] : 0.f;
          c[nt][2 + e] = r1 ? c[nt][2 + e] : 0.f;
          ds[nt][e] = r0 ? c[nt][e] * (dp[nt][e] - d0) * scale : 0.f;
          ds[nt][2 + e] = r1 ? c[nt][2 + e] * (dp[nt][2 + e] - d1) * scale : 0.f;
        }
      uint32_t pa[4] = {pack2(c[0][0], c[0][1]), pack2(c[0][2], c[0][3]), pack2(c[1][0], c[1][1]),
                        pack2(c[1][2], c[1][3])};
      uint32_t sa[4] = {pack2(ds[0][0], ds[0][1]), pack2(ds[0][2], ds[0][3]), pack2(ds[1][0], ds[1][1]),
                        pack2(ds[1][2], ds[1][3])};
      // stage P and dS ([query][key], bf16) for the transposed products
      __syncwarp();
#pragma unroll
      for (int nt = 0; nt < 2; ++nt) {
        *reinterpret_cast<uint32_t*>(tP + g * TP + nt * 8 + cb) = pa[2 * nt];
        *reinterpret_cast<uint32_t*>(tP + (g + 8) * TP + nt * 8 + cb) = pa[2 * nt + 1];
        *reinterpret_cast<uint32_t*>(tS + g * TP + nt * 8 + cb) = sa[2 * nt];
        *reinterpret_cast<uint32_t*>(tS + (g + 8) * TP + nt * 8 + cb) = sa[2 * nt + 1];
      }
      __syncwarp();
      uint32_t pta[4], sta[4];     // A fragments of P^T and dS^T: rows = keys, k = queries
      {
        const int r = (lane & 7) + (lane >> 4) * 8, cc = ((lane >> 3) & 1) * 8;
        ldsm_x4_t(pta, smem_u32(tP + r * TP + cc));
        ldsm_x4_t(sta, smem_u32(tS + r * TP + cc));
      }
      bf16* og = oblk + (size_t)f * T * s_in + hh * dh + cb;
#pragma unroll
      for (int np = 0; np < KD; ++np) {
        uint32_t bk_[4], bq_[4], bo_[4];
        ldsm_x4_t(bk_, addr_bv(kb, pin, T, np * 16, lane));      // B[k=j][n=c] = K[j][c]
        ldsm_x4_t(bq_, addr_bv(qb, pin, T, np * 16, lane));      // B[k=i][n=c] = Q[i][c]
        ldsm_x4_t(bo_, addr_bv(ob, pdo, T, np * 16, lane));      // B[k=i][n=c] = dO[i][c]
        float dq[2][4] = {}, dk[2][4] = {}, dv[2][4] = {};
        mma_bf16(dq[0], sa, bk_[0], bk_[1]);
        mma_bf16(dq[1], sa, bk_[2], bk_[3]);
        mma_bf16(dk[0], sta, bq_[0], bq_[1]);
        mma_bf16(dk[1], sta, bq_[2], bq_[3]);
        mma_bf16(dv[0], pta, bo_[0], bo_[1]);
        mma_bf16(dv[1], pta, bo_[2], bo_[3]);
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          const int col = np * 16 + u * 8;
          if (r0) {
            *reinterpret_cast<uint32_t*>(og + (size_t)g * s_in + col) = pack2(dq[u][0], dq[u][1]);
            *reinterpret_cast<uint32_t*>(og + (size_t)g * s_in + d + col) = pack2(dk[u][0], dk[u][1]);
            *reinterpret_cast<uint32_t*>(og + (size_t)g * s_in + 2 * d + col) = pack2(dv[u][0], dv[u][1]);
          }
          if (r1) {
            *reinterpret_cast<uint32_t*>(og + (size_t)(g + 8) * s_in + col) = pack2(dq[u][2], dq[u][3]);
            *reinterpret_cast<uint32_t*>(og + (size_t)(g + 8) * s_in + d + col) = pack2(dk[u][2], dk[u][3]);
            *reinterpret_cast<uint32_t*>(og + (size_t)(g + 8) * s_in + 2 * d + col) = pack2(dv[u][2], dv[u][3]);
          }
        }
      }
    }
    fence_proxy_async();
    __syncthreads();                          // all reads of q/k/v/dO done, all gradient rows staged
    if (lane == 0) {
      for (int r = warp; r < nf * T; r += nw)
        bulk_s2g(dqkv + ((size_t)f0 * T + r) * ld, smem_u32(oblk + (size_t)r * s_in), (uint32_t)(ld * 2));
      bulk_commit();
      const int fn = f0 + stride_f;
      if (fn < B) issue(fn);
    }
    if (dbias) {
#pragma unroll
      for (int sl = 0; sl < 2; ++sl) {
        const int gi = tid + sl * 256;
        if (gi < ngroups)
          for (int r = 0; r < nf * T; ++r) {
            const float4 v = load4(oblk + (size_t)r * s_in + gi * 4);
            bsum[sl].x += v.x; bsum[sl].y += v.y; bsum[sl].z += v.z; bsum[sl].w += v.w;
          }
      }
    }
  }
  if (dbias) {
#pragma unroll
    for (int sl = 0; sl < 2; ++sl) {
      const int gi = tid + sl * 256;
      if (gi < ngroups) {
        atomicAdd(dbias + gi * 4 + 0, bsum[sl].x);
        atomicAdd(dbias + gi * 4 + 1, bsum[sl].y);
        atomicAdd(dbias + gi * 4 + 2, bsum[sl].z);
        atomicAdd(dbias + gi * 4 + 3, bsum[sl].w);
      }
    }
  }
  if (lane == 0) bulk_wait_all();
}

inline bool use_mma(int T, int h, int dh) {
  return T <= 16 && (dh == 16 || dh == 32 || dh == 64) && (h * dh) % 8 == 0 && 3 * h * dh <= 2048;
}
inline size_t mma_fwd_bytes(int T, int h, int dh, int F) {
  const int d = h * dh;
  return 128 + ((size_t)2 * F * T * (3 * d + 8) + (size_t)F * T * (d + 8)) * 2;
}
inline size_t mma_bwd_bytes(int T, int h, int dh, int F) {
  const int d = h * dh;
  return 128 + ((size_t)2 * F * T * (3 * d + 8) + (size_t)F * T * (d + 8)) * 2 + 8 * 2 * 16 * 24 * 2;
}
inline int mma_frames(int T, int h, int dh, bool bwd) {
  // AMC_MMA_SMEM_KB (kernel study): shared-memory target per CTA = how many CTAs share an SM
  static const int lim_fwd = [] { const char* e = getenv("AMC_MMA_SMEM_KB"); return (e ? atoi(e) : 100) * 1024; }();
  static const int lim_bwd = [] { const char* e = getenv("AMC_MMA_SMEM_KB_BWD"); const char* f = getenv("AMC_MMA_SMEM_KB");
                                  return (e ? atoi(e) : (f ? atoi(f) : 100)) * 1024; }();
  static const int fmin = [] { const char* e = getenv("AMC_MMA_FMIN"); return e ? atoi(e) : 0; }();
  int F = fmin > 0 ? fmin : std::max(1, ceil_div(16, h));                 // at least ~2 pairs per warp
  while (F < 8 && (bwd ? mma_bwd_bytes(T, h, dh, F + 1) : mma_fwd_bytes(T, h, dh, F + 1)) <= (size_t)(bwd ? lim_bwd : lim_fwd)) ++F;
  return F;
}
// resident CTAs per SM for a given dynamic shared-memory size (256 threads each)
inline int mma_ctas_per_sm(size_t sm) { return (int)std::max<size_t>(1, std::min<size_t>(8, (220 * 1024) / (sm + 1024))); }

// A/B switch for kernel studies (tools/probes/attn_tc5_check.py): AMC_ATTN_LEGACY=1 skips the tcgen05 kernels
inline bool attn_legacy_only() {
  static const bool v = [] { const char* e = getenv("AMC_ATTN_LEGACY"); return e && e[0] == '1'; }();
  return v;
}

// the frame kernels need 16-byte row copies: (3d, d) * sizeof(E) % 16 == 0
template <typename E>
inline bool use_small(int T, int h, int dh) {
  return T <= 32 && dh <= 32 && dh % 4 == 0 && (h * dh) % Vec16<E>::n == 0 && h * T <= 256;
}
template <typename E>
inline size_t small_fwd_bytes(int T, int h, int dh, int F) {
  const int d = h * dh;
  return 128 + ((size_t)2 * F * T * (3 * d + Vec16<E>::n) + (size_t)F * T * (d + Vec16<E>::n)) * sizeof(E);
}
template <typename E>
inline size_t small_bwd_bytes(int T, int h, int dh, int F) {
  const int d = h * dh;
  return 128 + ((size_t)2 * F * T * (3 * d + Vec16<E>::n) + (size_t)F * T * (d + Vec16<E>::n)) * sizeof(E) +
         (size_t)F * h * 2 * T * (T + 1) * sizeof(float);
}
// frames per CTA iteration: <= 256 threads and <= ~72 KB of shared memory (3 CTAs per SM)
template <typename E, typename BytesFn>
inline int small_frames(int T, int h, int dh, BytesFn bytes) {
  int F = std::max(1, 256 / (h * T));
  while (F > 1 && bytes(T, h, dh, F) > 100 * 1024) --F;
  return F;
}

inline int pick_warps(int T) { return std::max(1, std::min(8, (T + 7) / 8)); }

}  // namespace

template <typename E>
int attention_fwd(int B, int T, int h, int dh, const E* qkv, E* out, float* lse, cudaStream_t st) {
  if (T > 32 * MAXJ) return attn_long_fwd<E>(B, T, h, dh, qkv, out, lse, st);   // outside the single-CTA regime
  AMC_CHECK_ARG(T >= 1 && T <= 32 * MAXJ, "attention: T=%d unsupported (1..%d tokens per frame)", T, 32 * MAXJ);
  AMC_CHECK_ARG(dh >= 1 && dh <= 128, "attention: head dim %d unsupported (1..128)", dh);
  if (B == 0) return 0;
  if constexpr (std::is_same<E, bf16>::value) {
    if (use_mma(T, h, dh)) {
      const int F = mma_frames(T, h, dh, false);
      const size_t sm = mma_fwd_bytes(T, h, dh, F);
      const int grid = std::min(ceil_div(B, F), 148 * mma_ctas_per_sm(sm));
      const float sc = 1.f / sqrtf((float)dh);
#define AMC_LAUNCH_MMA_FWD(KD)                                                                                      \
  do {                                                                                                              \
    AMC_CUDA(cudaFuncSetAttribute(attn_mma_fwd_kernel<KD>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024)); \
    attn_mma_fwd_kernel<KD><<<grid, 256, sm, st>>>(B, T, h, F, qkv, out, sc);                                       \
  } while (0)
      if (dh == 16) AMC_LAUNCH_MMA_FWD(1);
      else if (dh == 32) AMC_LAUNCH_MMA_FWD(2);
      else AMC_LAUNCH_MMA_FWD(4);
#undef AMC_LAUNCH_MMA_FWD
      AMC_LAUNCH_CHECK();
      return 0;
    }
  }
  if constexpr (std::is_same<E, bf16>::value) {
    bool handled = false;
    if (!attn_legacy_only()) AMC_TRY(attn_tc5_fwd(B, T, h, dh, qkv, out, lse, &handled, st));
    if (handled) return 0;
    AMC_TRY(attn_tiles_fwd(B, T, h, dh, qkv, out, lse, &handled, st));
    if (handled) return 0;
  }
  if (use_small<E>(T, h, dh)) {
    const int F = small_frames<E>(T, h, dh, small_fwd_bytes<E>);
    const size_t sm = small_fwd_bytes<E>(T, h, dh, F);
    AMC_CHECK_ARG(sm <= 200 * 1024, "attention: frame tile needs %zu bytes of shared memory", sm);
    const int threads = ((F * h * T + 31) / 32) * 32;
    const int grid = std::min(ceil_div(B, F), 148 * 2);
    const float sc = 1.f / sqrtf((float)dh);
    if (T <= 16) {
      AMC_CUDA(cudaFuncSetAttribute(attn_frames_fwd_kernel<E, 16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
      attn_frames_fwd_kernel<E, 16><<<grid, threads, sm, st>>>(B, T, h, dh, F, qkv, out, sc);
    } else {
      AMC_CUDA(cudaFuncSetAttribute(attn_frames_fwd_kernel<E, 32>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
      attn_frames_fwd_kernel<E, 32><<<grid, threads, sm, st>>>(B, T, h, dh, F, qkv, out, sc);
    }
    AMC_LAUNCH_CHECK();
    return 0;
  }
  const int nw = pick_warps(T), stride = dh + SmemPad<E>::v;
  const int tile = (T * stride + 1) & ~1;
  const size_t smem = (size_t)2 * tile * sizeof(E) + (size_t)nw * (dh + T) * sizeof(float);
  AMC_CHECK_ARG(smem <= 227 * 1024, "attention: T=%d dh=%d needs %zu bytes of shared memory (> 227 KB)", T, dh, smem);
  if (smem > 48 * 1024)
    AMC_CUDA(cudaFuncSetAttribute(attn_fwd_kernel<E>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
  attn_fwd_kernel<E><<<B * h, nw * 32, smem, st>>>(T, h, dh, qkv, out, 1.f / sqrtf((float)dh));
  AMC_LAUNCH_CHECK();
  return 0;
}
template int attention_fwd<float>(int, int, int, int, const float*, float*, float*, cudaStream_t);
template int attention_fwd<bf16>(int, int, int, int, const bf16*, bf16*, float*, cudaStream_t);

template <typename E>
int attention_bwd_impl(int B, int T, int h, int dh, const E* qkv, const E* out, const float* lse, const E* dout, E* dqkv,
                       float* dbias, bool* fused, cudaStream_t st) {
  *fused = false;
  if (T > 32 * MAXJ) return attn_long_bwd<E>(B, T, h, dh, qkv, out, lse, dout, dqkv, st);
  AMC_CHECK_ARG(T >= 1 && T <= 32 * MAXJ, "attention_bwd: T=%d unsupported (1..%d tokens per frame)", T, 32 * MAXJ);
  AMC_CHECK_ARG(dh >= 1 && dh <= 128, "attention_bwd: head dim %d unsupported (1..128)", dh);
  if (B == 0) return 0;
  if constexpr (std::is_same<E, bf16>::value) {
    if (use_mma(T, h, dh)) {
      const int F = mma_frames(T, h, dh, true);
      const size_t sm = mma_bwd_bytes(T, h, dh, F);
      const int grid = std::min(ceil_div(B, F), 148 * mma_ctas_per_sm(sm));
      const float sc = 1.f / sqrtf((float)dh);
#define AMC_LAUNCH_MMA_BWD(KD)                                                                                      \
  do {                                                                                                              \
    AMC_CUDA(cudaFuncSetAttribute(attn_mma_bwd_kernel<KD>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024)); \
    attn_mma_bwd_kernel<KD><<<grid, 256, sm, st>>>(B, T, h, F, qkv, dout, dqkv, dbias, sc);                         \
  } while (0)
      if (dh == 16) AMC_LAUNCH_MMA_BWD(1);
      else if (dh == 32) AMC_LAUNCH_MMA_BWD(2);
      else AMC_LAUNCH_MMA_BWD(4);
#undef AMC_LAUNCH_MMA_BWD
      AMC_LAUNCH_CHECK();
      *fused = true;
      return 0;
    }
  }
  if constexpr (std::is_same<E, bf16>::value) {
    bool handled = false;
    if (!attn_legacy_only()) AMC_TRY(attn_tc5_bwd(B, T, h, dh, qkv, out, lse, dout, dqkv, dbias, &handled, st));
    if (handled) {
      *fused = true;
      return 0;
    }
    AMC_TRY(attn_tiles_bwd(B, T, h, dh, qkv, out, lse, dout, dqkv, dbias, &handled, st));
    if (handled) {
      *fused = true;
      return 0;
    }
  }
  if (use_small<E>(T, h, dh)) {
    const int F = small_frames<E>(T, h, dh, small_bwd_bytes<E>);
    const size_t sm = small_bwd_bytes<E>(T, h, dh, F);
    AMC_CHECK_ARG(sm <= 200 * 1024, "attention_bwd: frame tile needs %zu bytes of shared memory", sm);
    const int threads = ((F * h * T + 31) / 32) * 32;
    const int grid = std::min(ceil_div(B, F), 148 * 2);
    const float sc = 1.f / sqrtf((float)dh);
    if (T <= 16) {
      AMC_CUDA(cudaFuncSetAttribute(attn_frames_bwd_kernel<E, 16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
      attn_frames_bwd_kernel<E, 16><<<grid, threads, sm, st>>>(B, T, h, dh, F, qkv, dout, dqkv, sc);
    } else {
      AMC_CUDA(cudaFuncSetAttribute(attn_frames_bwd_kernel<E, 32>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
      attn_frames_bwd_kernel<E, 32><<<grid, threads, sm, st>>>(B, T, h, dh, F, qkv, dout, dqkv, sc);
    }
    AMC_LAUNCH_CHECK();
    return 0;
  }
  const int nw = pick_warps(T), stride = dh + SmemPad<E>::v;
  const int tile = (T * stride + 1) & ~1;
  size_t smem = (size_t)4 * tile * sizeof(E) + (size_t)(3 * T + 2 * nw * T) * sizeof(float);
  AMC_CHECK_ARG(smem <= 227 * 1024,
                "attention_bwd: T=%d dh=%d needs %zu bytes of shared memory (> 227 KB); unsupported shape", T, dh,
                smem);
  if (smem > 48 * 1024)
    AMC_CUDA(cudaFuncSetAttribute(attn_bwd_kernel<E>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
  attn_bwd_kernel<E><<<B * h, nw * 32, smem, st>>>(T, h, dh, qkv, dout, dqkv, 1.f / sqrtf((float)dh));
  AMC_LAUNCH_CHECK();
  return 0;
}
// dbias (nullable): += column sums of dqkv, i.e. the gradient of the q/k/v biases.  The tensor-core kernel
// produces it from its staged rows; the other kernels are followed by a column-sum pass.
template <typename E>
int attention_bwd(int B, int T, int h, int dh, const E* qkv, const E* out, const float* lse, const E* dout, E* dqkv,
                  float* dbias, cudaStream_t st) {
  bool fused = false;
  AMC_TRY(attention_bwd_impl<E>(B, T, h, dh, qkv, out, lse, dout, dqkv, dbias, &fused, st));
  if (dbias && !fused) AMC_TRY(colsum<E>(B * T, 3 * h * dh, dqkv, 3 * h * dh, dbias, st));
  return 0;
}
template int attention_bwd<float>(int, int, int, int, const float*, const float*, const float*, const float*, float*,
                                  float*, cudaStream_t);
template int attention_bwd<bf16>(int, int, int, int, const bf16*, const bf16*, const float*, const bf16*, bf16*, float*,
                                 cudaStream_t);

}  // namespace amc

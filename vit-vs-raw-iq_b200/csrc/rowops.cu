// Bandwidth-bound row kernels: LayerNorm fwd/bwd, column sums (bias gradients), IQ normalise +
// framing + patchify, CLS rows, classifier head fwd/bwd, cross-entropy, weight packing, AdamW.
// All reductions are warp-shuffle based (one warp per row); fp32 statistics in both dtypes.
#include "rowops.cuh"

namespace amc {
namespace {

constexpr int MAXV = 16;  // d <= 512 -> <= 16 values per lane

__device__ __forceinline__ float pick4(const float4& k, int j) {
  return j == 0 ? k.x : (j == 1 ? k.y : (j == 2 ? k.z : k.w));
}
__device__ __forceinline__ float dropout_mult1(const DropoutCfg& c, uint32_t site, uint64_t e) {
  return pick4(dropout_mult4(c, site, e >> 2), (int)(e & 3));
}

// ---------------------------------------------------------------------------------------
// LayerNorm forward: layers_norm.py:11-19 (biased variance, eps inside the sqrt)
// ---------------------------------------------------------------------------------------
template <typename E>
__global__ void __launch_bounds__(256) ln_fwd_kernel(int M, int d, const float* __restrict__ u,
                                                     const float* __restrict__ gamma,
                                                     const float* __restrict__ beta, float eps, E* __restrict__ y16,
                                                     float* __restrict__ y32, E* __restrict__ xhat,
                                                     float* __restrict__ rstd) {
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= M) return;
  const float* ur = u + (size_t)row * d;
  float v[MAXV];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    const int c = lane + 32 * i;
    v[i] = c < d ? ur[c] : 0.f;
    s += v[i];
  }
  const float mean = warp_sum(s) / (float)d;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    const int c = lane + 32 * i;
    const float t = c < d ? v[i] - mean : 0.f;
    q += t * t;
  }
  const float rs = rsqrtf(warp_sum(q) / (float)d + eps);
  if (rstd && lane == 0) rstd[row] = rs;
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    const int c = lane + 32 * i;
    if (c < d) {
      const float xh = (v[i] - mean) * rs;
      const float y = fmaf(__ldg(gamma + c), xh, __ldg(beta + c));
      const size_t o = (size_t)row * d + c;
      if (y16) y16[o] = from_f<E>(y);
      if (y32) y32[o] = y;
      if (xhat) xhat[o] = from_f<E>(xh);
    }
  }
}

// ---------------------------------------------------------------------------------------
// LayerNorm backward (SURVEY Appendix B).  Optionally regenerates the dropout mask of the
// sub-layer output so du16 (the operand of the following dgrad/wgrad GEMMs) is already
// mask * du / (1-p), while du32 (the skip path) stays unmasked.
// ---------------------------------------------------------------------------------------
template <typename E>
__global__ void __launch_bounds__(256) ln_bwd_kernel(int M, int d, const float* __restrict__ dy,
                                                     const E* __restrict__ xhat, const float* __restrict__ rstd,
                                                     const float* __restrict__ gamma, E* __restrict__ du16,
                                                     float* __restrict__ du32, float* __restrict__ dgamma,
                                                     float* __restrict__ dbeta, DropoutCfg drop, uint32_t site) {
  __shared__ float red[2][8][32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  float ag[MAXV], ab[MAXV], g[MAXV];
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    ag[i] = 0.f;
    ab[i] = 0.f;
    const int c = lane + 32 * i;
    g[i] = c < d ? __ldg(gamma + c) : 0.f;
  }
  for (int row = blockIdx.x * nw + warp; row < M; row += gridDim.x * nw) {
    const size_t base = (size_t)row * d;
    float dyv[MAXV], xh[MAXV];
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
      const int c = lane + 32 * i;
      dyv[i] = c < d ? dy[base + c] : 0.f;
      xh[i] = c < d ? to_f(xhat[base + c]) : 0.f;
      const float gg = dyv[i] * g[i];
      s1 += gg;
      s2 += gg * xh[i];
      ag[i] += dyv[i] * xh[i];
      ab[i] += dyv[i];
    }
    s1 = warp_sum(s1) / (float)d;
    s2 = warp_sum(s2) / (float)d;
    const float rs = rstd[row];
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
      const int c = lane + 32 * i;
      if (c < d) {
        const float du = rs * (dyv[i] * g[i] - s1 - xh[i] * s2);
        if (du32) du32[base + c] = du;
        if (du16) {
          float m = 1.f;
          if (drop.p > 0.f) m = dropout_mult1(drop, site, (uint64_t)base + (uint64_t)c);
          du16[base + c] = from_f<E>(du * m);
        }
      }
    }
  }
  // block reduction of the parameter gradients, then one atomic per column per block
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    if (i * 32 < d) {
      __syncthreads();
      red[0][warp][lane] = ag[i];
      red[1][warp][lane] = ab[i];
      __syncthreads();
      if (warp == 0) {
        float a = 0.f, b = 0.f;
        for (int w = 0; w < nw; ++w) {
          a += red[0][w][lane];
          b += red[1][w][lane];
        }
        const int c = lane + 32 * i;
        if (c < d) {
          if (dgamma) atomicAdd(dgamma + c, a);
          if (dbeta) atomicAdd(dbeta + c, b);
        }
      }
    }
  }
}

// Vectorised LayerNorm backward for d = 128 * NV (NV = 1..4): each lane owns 4*NV consecutive columns, so a
// row is one contiguous, fully coalesced warp transaction (16*NV B fp32 / 8*NV B bf16 per lane) and every
// lane is busy.  Besides dgamma/dbeta it also accumulates the column sums of the (dropout-masked) du16 it
// writes, i.e. the bias gradient of the sub-layer's output projection (Appendix B: db = sum d_out), saving
// a pass over du16.  R rows per warp iteration keep enough loads in flight.
template <typename E, int NV>
__global__ void __launch_bounds__(256) ln_bwd_vec_kernel(int M, int d, const float* __restrict__ dy,
                                                         const E* __restrict__ xhat, const float* __restrict__ rstd,
                                                         const float* __restrict__ gamma, E* __restrict__ du16,
                                                         float* __restrict__ du32, float* __restrict__ dgamma,
                                                         float* __restrict__ dbeta, float* __restrict__ dbias,
                                                         DropoutCfg drop, uint32_t site) {
  constexpr int CPL = 4 * NV;                     // columns per lane
  constexpr int R = (NV <= 2) ? 4 : 2;
  __shared__ float red[3][8][33];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const int c0 = lane * CPL;
  float g[CPL], ag[CPL], ab[CPL], ad[CPL];
#pragma unroll
  for (int j = 0; j < CPL; ++j) {
    g[j] = __ldg(gamma + c0 + j);
    ag[j] = 0.f; ab[j] = 0.f; ad[j] = 0.f;
  }
  const float inv_d = 1.f / (float)d;
  const int wstride = gridDim.x * nw;
  for (int row0 = (blockIdx.x * nw + warp) * R; row0 < M; row0 += wstride * R) {
    float dyv[R][CPL], xh[R][CPL], rs[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const int row = row0 + r;
      const bool rok = row < M;
      const size_t base = (size_t)(rok ? row : 0) * d + c0;
      rs[r] = rok ? rstd[row] : 0.f;
#pragma unroll
      for (int v = 0; v < NV; ++v) {
        float4 a = make_float4(0, 0, 0, 0), x = make_float4(0, 0, 0, 0);
        if (rok) {
          a = *reinterpret_cast<const float4*>(dy + base + 4 * v);
          x = load4(xhat + base + 4 * v);
        }
        dyv[r][4 * v] = a.x; dyv[r][4 * v + 1] = a.y; dyv[r][4 * v + 2] = a.z; dyv[r][4 * v + 3] = a.w;
        xh[r][4 * v] = x.x; xh[r][4 * v + 1] = x.y; xh[r][4 * v + 2] = x.z; xh[r][4 * v + 3] = x.w;
      }
    }
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const int row = row0 + r;
      if (row >= M) break;
      const size_t base = (size_t)row * d + c0;
      float s1 = 0.f, s2 = 0.f;
#pragma unroll
      for (int j = 0; j < CPL; ++j) {
        const float gg = dyv[r][j] * g[j];
        s1 += gg;
        s2 = fmaf(gg, xh[r][j], s2);
        ag[j] = fmaf(dyv[r][j], xh[r][j], ag[j]);
        ab[j] += dyv[r][j];
      }
      s1 = warp_sum(s1) * inv_d;
      s2 = warp_sum(s2) * inv_d;
      float du[CPL];
#pragma unroll
      for (int j = 0; j < CPL; ++j) du[j] = rs[r] * (dyv[r][j] * g[j] - s1 - xh[r][j] * s2);
      if (du32) {
#pragma unroll
        for (int v = 0; v < NV; ++v)
          *reinterpret_cast<float4*>(du32 + base + 4 * v) = make_float4(du[4 * v], du[4 * v + 1], du[4 * v + 2], du[4 * v + 3]);
      }
      if (drop.p > 0.f) {
#pragma unroll
        for (int v = 0; v < NV; ++v) {
          const float4 mk = dropout_mult4(drop, site, ((uint64_t)base >> 2) + v);
          du[4 * v] *= mk.x; du[4 * v + 1] *= mk.y; du[4 * v + 2] *= mk.z; du[4 * v + 3] *= mk.w;
        }
      }
      if (du16) {
#pragma unroll
        for (int v = 0; v < NV; ++v)
          store4(du16 + base + 4 * v, make_float4(du[4 * v], du[4 * v + 1], du[4 * v + 2], du[4 * v + 3]));
      }
#pragma unroll
      for (int j = 0; j < CPL; ++j) ad[j] += du[j];
    }
  }
  // block reduction (8 warps) then one atomic per column per block
#pragma unroll
  for (int j = 0; j < CPL; ++j) {
    __syncthreads();
    red[0][warp][lane] = ag[j];
    red[1][warp][lane] = ab[j];
    red[2][warp][lane] = ad[j];
    __syncthreads();
    if (warp < 3) {
      float t = 0.f;
      for (int w = 0; w < nw; ++w) t += red[warp][w][lane];
      float* dst = warp == 0 ? dgamma : (warp == 1 ? dbeta : dbias);
      if (dst) atomicAdd(dst + c0 + j, t);
    }
  }
}

// ---------------------------------------------------------------------------------------
// Column sums: out[n] += sum_m X[m, n]   (bias gradients: Appendix B "db = sum dY")
// ---------------------------------------------------------------------------------------
template <typename E>
__global__ void __launch_bounds__(256) colsum_kernel(int M, int N, const E* __restrict__ X, int ld,
                                                     float* __restrict__ out, int rows_per_block) {
  __shared__ float red[8][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int n = blockIdx.x * 32 + tx;
  const int r0 = blockIdx.y * rows_per_block, r1 = min(M, r0 + rows_per_block);
  float s = 0.f;
  if (n < N)
    for (int r = r0 + ty; r < r1; r += 8) s += to_f(X[(size_t)r * ld + n]);
  red[ty][tx] = s;
  __syncthreads();
  if (ty == 0) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) t += red[w][tx];
    if (n < N) atomicAdd(out + n, t);
  }
}

// ---------------------------------------------------------------------------------------
// Front end, step 1: dataset z-score + framing + patchify into the embedding GEMM's A operand.
//   A[b*Ttok + t, k]  (SURVEY §8 a1-a4)
// ---------------------------------------------------------------------------------------
template <typename E>
__global__ void __launch_bounds__(256) patchify_kernel(PatchP p, const float* __restrict__ src, E* __restrict__ A) {
  const size_t total = (size_t)p.B * p.Ttok * p.K;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int k = (int)(i % p.K);
    const size_t row = i / p.K;
    const int t = (int)(row % p.Ttok), b = (int)(row / p.Ttok);
    int ch;
    const float x = __ldg(src + patch_src_offset(p, b, t, k, &ch));
    A[i] = from_f<E>(ch < 0 ? x : (x - p.mean[ch]) * p.inv_std[ch]);
  }
}

// Input gradient, last step: the transpose of patchify.  d(x - mean) * inv_std / dx = inv_std in dataset layout.
__global__ void __launch_bounds__(256) patch_scatter_kernel(PatchP p, const float* __restrict__ dX,
                                                            float* __restrict__ dsrc) {
  const size_t total = (size_t)p.B * p.Ttok * p.K;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int k = (int)(i % p.K);
    const size_t row = i / p.K;
    const int t = (int)(row % p.Ttok), b = (int)(row / p.Ttok);
    int ch;
    const size_t o = patch_src_offset(p, b, t, k, &ch);
    const float g = dX[i];
    dsrc[o] = ch < 0 ? g : g * p.inv_std[ch];
  }
}

// Bandwidth-bound version (K % 8 == 0): one frame at a time is staged in shared memory as a planar,
// normalised [channel][sample] image with coalesced 128-bit loads (the dataset layout de-interleaves and
// z-scores on the way in); the patch / segment gather then runs out of shared memory and every thread writes
// 8 consecutive operand elements as 128-bit stores.  HBM sees each input byte and each output byte once.
template <typename E>
__global__ void __launch_bounds__(256) patchify_frames_kernel(PatchP p, const float* __restrict__ src,
                                                              E* __restrict__ A) {
  extern __shared__ __align__(16) float plane[];          // [in_ch_eff][n_per_ch]
  const int n_per_ch = p.kind == AMC_KIND_RAWIQ ? p.seq_len : p.img_h * p.img_w;
  const int raw = p.input_layout == AMC_INPUT_RAW;
  // dataset layout: 2 planes of L samples (raw-IQ: L = seq_len; ViT: L = H*W/2 and the image is cat(I, Q))
  const int L = raw ? (p.kind == AMC_KIND_RAWIQ ? p.seq_len : p.img_h * p.img_w / 2) : 0;
  const int total = raw ? 2 * L : p.in_ch * n_per_ch;    // floats per frame
  const int groups = p.Ttok * p.K / 8;                    // 8-element output groups per frame
  for (int b = blockIdx.x; b < p.B; b += gridDim.x) {
    const float* fsrc = src + (size_t)b * total;
    for (int i = threadIdx.x; i < total / 4; i += blockDim.x) {
      const float4 v = __ldg(reinterpret_cast<const float4*>(fsrc) + i);
      if (raw) {      // (I, Q, I, Q) -> planar + z-score (dataset.py:215-217)
        const int n = 2 * i;
        plane[n] = (v.x - p.mean[0]) * p.inv_std[0];
        plane[L + n] = (v.y - p.mean[1]) * p.inv_std[1];
        plane[n + 1] = (v.z - p.mean[0]) * p.inv_std[0];
        plane[L + n + 1] = (v.w - p.mean[1]) * p.inv_std[1];
      } else {
        *reinterpret_cast<float4*>(plane + 4 * i) = v;
      }
    }
    __syncthreads();
    E* arow = A + (size_t)b * p.Ttok * p.K;
    for (int gI = threadIdx.x; gI < groups; gI += blockDim.x) {
      const int e0 = gI * 8, t = e0 / p.K, k0 = e0 - t * p.K;
      float v[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int k = k0 + j;
        int idx;
        if (p.kind == AMC_KIND_RAWIQ) {
          const int c = k / p.seg, sidx = k - c * p.seg;
          idx = c * p.seq_len + t * p.seg + sidx;          // dataset layout: plane c == channel c
        } else {
          const int pp = p.patch * p.patch, wp = p.img_w / p.patch;
          const int c = k / pp, rem = k - c * pp, r = rem / p.patch, cc = rem - r * p.patch;
          const int ph = t / wp, pw = t - ph * wp;
          idx = c * p.img_h * p.img_w + (ph * p.patch + r) * p.img_w + pw * p.patch + cc;   // cat(I,Q) == planar
        }
        v[j] = plane[idx];
      }
      store4(arow + e0, make_float4(v[0], v[1], v[2], v[3]));
      store4(arow + e0 + 4, make_float4(v[4], v[5], v[6], v[7]));
    }
    __syncthreads();
  }
}

// CLS rows of x0: x0[b,0,:] = dropout(cls + pos[0])   (encoder.py:104-111)
template <typename E>
__global__ void cls_rows_kernel(int B, int T, int d, const float* __restrict__ cls, const float* __restrict__ pos,
                                E* __restrict__ y16, float* __restrict__ y32, DropoutCfg drop) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * d) return;
  const int b = i / d, c = i - b * d;
  float v = __ldg(cls + c) + __ldg(pos + c);
  const size_t o = (size_t)b * T * d + c;
  if (drop.p > 0.f) v *= dropout_mult1(drop, site_pe(), (uint64_t)o);
  if (y16) y16[o] = from_f<E>(v);
  if (y32) y32[o] = v;
}

// dcls[c] += sum_b mask * dx0[b,0,c]
__global__ void cls_grad_kernel(int B, int T, int d, const float* __restrict__ dx0, float* __restrict__ dcls,
                                DropoutCfg drop) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= d) return;
  float s = 0.f;
  for (int b = blockIdx.y; b < B; b += gridDim.y) {
    const size_t o = (size_t)b * T * d + c;
    float v = dx0[o];
    if (drop.p > 0.f) v *= dropout_mult1(drop, site_pe(), (uint64_t)o);
    s += v;
  }
  atomicAdd(dcls + c, s);
}

// gather the non-CLS rows of dx0 (with the PE-dropout mask) into a dense [B*Ttok, d] operand
template <typename E>
__global__ void __launch_bounds__(256) gather_tok_rows_kernel(int B, int T, int Ttok, int d, int has_cls,
                                                              const float* __restrict__ dx0, E* __restrict__ out,
                                                              DropoutCfg drop) {
  const size_t total = (size_t)B * Ttok * d;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % d);
    const size_t row = i / d;
    const int t = (int)(row % Ttok), b = (int)(row / Ttok);
    const size_t o = ((size_t)b * T + has_cls + t) * d + c;
    float v = dx0[o];
    if (drop.p > 0.f) v *= dropout_mult1(drop, site_pe(), (uint64_t)o);
    out[i] = from_f<E>(v);
  }
}

// ---------------------------------------------------------------------------------------
// Classifier head (transformer_rawIQ.py:67-70,88-96 ; amc_transformer.py:24,29-30)
// one warp per frame
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) head_fwd_kernel(int B, int T, int d, int C, int has_cls, int head_ln,
                                                       float eps, const float* __restrict__ x,
                                                       const float* __restrict__ lnw, const float* __restrict__ lnb,
                                                       const float* __restrict__ W, const float* __restrict__ bias,
                                                       float* __restrict__ logits, float* __restrict__ s_hl,
                                                       float* __restrict__ s_xhat, float* __restrict__ s_rstd) {
  const int lane = threadIdx.x & 31;
  const int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (b >= B) return;
  float v[MAXV];
  const float* xb = x + (size_t)b * T * d;
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    const int c = lane + 32 * i;
    float a = 0.f;
    if (c < d) {
      if (has_cls) {
        a = xb[c];
      } else {
        for (int t = 0; t < T; ++t) a += xb[(size_t)t * d + c];
        a /= (float)T;
      }
    }
    v[i] = a;
  }
  if (head_ln) {
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < MAXV; ++i) s += v[i];
    const float mean = warp_sum(s) / (float)d;
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
      const float t = (lane + 32 * i) < d ? v[i] - mean : 0.f;
      q += t * t;
    }
    const float rs = rsqrtf(warp_sum(q) / (float)d + eps);
    if (s_rstd && lane == 0) s_rstd[b] = rs;
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
      const int c = lane + 32 * i;
      if (c < d) {
        const float xh = (v[i] - mean) * rs;
        if (s_xhat) s_xhat[(size_t)b * d + c] = xh;
        v[i] = fmaf(__ldg(lnw + c), xh, __ldg(lnb + c));
      }
    }
  }
  if (s_hl) {
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
      const int c = lane + 32 * i;
      if (c < d) s_hl[(size_t)b * d + c] = v[i];
    }
  }
  for (int k = 0; k < C; ++k) {
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
      const int c = lane + 32 * i;
      if (c < d) s = fmaf(v[i], __ldg(W + (size_t)k * d + c), s);
    }
    s = warp_sum(s);
    if (lane == 0) logits[(size_t)b * C + k] = s + __ldg(bias + k);
  }
}

// head backward, part 1 (warp per frame): dhl = dlogits W ; LN bwd ; scatter into dxL [B,T,d]
__global__ void __launch_bounds__(128) head_bwd_rows_kernel(int B, int T, int d, int C, int has_cls, int head_ln,
                                                            const float* __restrict__ dlogits,
                                                            const float* __restrict__ W,
                                                            const float* __restrict__ lnw,
                                                            const float* __restrict__ s_xhat,
                                                            const float* __restrict__ s_rstd,
                                                            float* __restrict__ dxL, float* __restrict__ dhl_out) {
  const int lane = threadIdx.x & 31;
  const int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (b >= B) return;
  float g[MAXV];
#pragma unroll
  for (int i = 0; i < MAXV; ++i) g[i] = 0.f;
  for (int k = 0; k < C; ++k) {
    const float dl = __ldg(dlogits + (size_t)b * C + k);
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
      const int c = lane + 32 * i;
      if (c < d) g[i] = fmaf(dl, __ldg(W + (size_t)k * d + c), g[i]);
    }
  }
  if (dhl_out) {  // dhl, needed for the LN parameter gradients
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
      const int c = lane + 32 * i;
      if (c < d) dhl_out[(size_t)b * d + c] = g[i];
    }
  }
  if (head_ln) {
    float s1 = 0.f, s2 = 0.f, xh[MAXV];
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
      const int c = lane + 32 * i;
      xh[i] = c < d ? s_xhat[(size_t)b * d + c] : 0.f;
      g[i] = c < d ? g[i] * __ldg(lnw + c) : 0.f;
      s1 += g[i];
      s2 += g[i] * xh[i];
    }
    s1 = warp_sum(s1) / (float)d;
    s2 = warp_sum(s2) / (float)d;
    const float rs = s_rstd[b];
#pragma unroll
    for (int i = 0; i < MAXV; ++i) g[i] = rs * (g[i] - s1 - xh[i] * s2);
  }
  float* db = dxL + (size_t)b * T * d;
  const float invT = 1.f / (float)T;
  for (int t = 0; t < T; ++t) {
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
      const int c = lane + 32 * i;
      if (c < d) db[(size_t)t * d + c] = has_cls ? (t == 0 ? g[i] : 0.f) : g[i] * invT;
    }
  }
}

// head backward, part 2: dW[k,:] += sum_b dlogits[b,k] hl[b,:] ; db[k] += sum_b dlogits[b,k]
// and (head_ln) dlnw += sum_b dhl*xhat ; dlnb += sum_b dhl.
// grid (ceil(d/128), frame chunks); one thread per column keeps a register accumulator per class, so
// hl is read exactly once and dlogits rows are warp-uniform (broadcast) loads.
__global__ void __launch_bounds__(128) head_bwd_params_kernel(int B, int d, int C, int head_ln,
                                                              const float* __restrict__ dlogits,
                                                              const float* __restrict__ s_hl,
                                                              const float* __restrict__ dhl,
                                                              const float* __restrict__ s_xhat,
                                                              float* __restrict__ dW, float* __restrict__ dbias,
                                                              float* __restrict__ dlnw, float* __restrict__ dlnb) {
  constexpr int KG = 24, ROWS = 32;
  __shared__ float sdl[ROWS * 64];                  // this block's rows of dlogits (C <= 64), staged once
  const int c = blockIdx.x * 128 + threadIdx.x;
  const int per = min((B + gridDim.y - 1) / gridDim.y, ROWS);
  const int b0 = blockIdx.y * per, b1 = min(B, b0 + per);
  for (int i = threadIdx.x; i < (b1 - b0) * C; i += blockDim.x) sdl[i] = __ldg(dlogits + (size_t)b0 * C + i);
  __syncthreads();
  if (c < d) {
    for (int k0 = 0; k0 < C; k0 += KG) {
      float acc[KG];
#pragma unroll
      for (int k = 0; k < KG; ++k) acc[k] = 0.f;
      for (int b = b0; b < b1; ++b) {
        const float h = s_hl[(size_t)b * d + c];
        const float* dl = sdl + (b - b0) * C + k0;
#pragma unroll
        for (int k = 0; k < KG; ++k)
          if (k0 + k < C) acc[k] = fmaf(dl[k], h, acc[k]);
      }
#pragma unroll
      for (int k = 0; k < KG; ++k)
        if (k0 + k < C) atomicAdd(dW + (size_t)(k0 + k) * d + c, acc[k]);
    }
    if (head_ln) {
      float sg = 0.f, sb = 0.f;
      for (int b = b0; b < b1; ++b) {
        const float g = dhl[(size_t)b * d + c];
        sg = fmaf(g, s_xhat[(size_t)b * d + c], sg);
        sb += g;
      }
      atomicAdd(dlnw + c, sg);
      atomicAdd(dlnb + c, sb);
    }
  }
  if (blockIdx.x == 0 && (int)threadIdx.x < C) {
    float sbias = 0.f;
    for (int b = b0; b < b1; ++b) sbias += sdl[(b - b0) * C + threadIdx.x];
    atomicAdd(dbias + threadIdx.x, sbias);
  }
}

// ---------------------------------------------------------------------------------------
// CrossEntropyLoss(label_smoothing) + accuracy counters (train.py:260,274-277,504)
// ---------------------------------------------------------------------------------------
__global__ void ce_loss_kernel(int B, int C, const float* __restrict__ logits, const int64_t* __restrict__ labels,
                               float ls, float grad_scale, float loss_scale, float* __restrict__ dlogits,
                               float* __restrict__ stats) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  float loss = 0.f, correct = 0.f;
  if (b < B) {
    const float* z = logits + (size_t)b * C;
    float mx = z[0];
    int am = 0;
    for (int k = 1; k < C; ++k)
      if (z[k] > mx) {
        mx = z[k];
        am = k;
      }
    float se = 0.f;
    for (int k = 0; k < C; ++k) se += expf(z[k] - mx);
    const float lse = logf(se);
    const int64_t y64 = labels[b];
    // nn.CrossEntropyLoss raises on a target outside [0, C); an asynchronous kernel cannot, so the frame's loss becomes
    // NaN: the running loss statistic is NaN from then on and the host raises when it reads it (trainer.read_stats).
    // Such a frame matches no class (y = -1): it is never counted correct -- a label of 2^32 + 3 truncated to 32 bits
    // would otherwise read as class 3 -- and its gradient has the all-smoothing target.
    const bool valid = y64 >= 0 && y64 < (int64_t)C;
    const int y = valid ? (int)y64 : -1;
    const float poison = valid ? 0.f : __int_as_float(0x7fc00000);
    float sum_logp = 0.f;
    for (int k = 0; k < C; ++k) {
      const float logp = z[k] - mx - lse;
      sum_logp += logp;
      const float tgt = (k == y ? 1.f - ls : 0.f) + ls / (float)C;
      if (dlogits) dlogits[(size_t)b * C + k] = (expf(logp) - tgt) * grad_scale;
      if (k == y) loss -= (1.f - ls) * logp;
    }
    loss -= ls / (float)C * sum_logp;
    loss += poison;
    correct = (am == y) ? 1.f : 0.f;
  }
  loss = warp_sum(loss);
  correct = warp_sum(correct);
  if ((threadIdx.x & 31) == 0 && stats) {
    atomicAdd(stats + 0, loss * loss_scale);
    atomicAdd(stats + 1, correct);
  }
}

// ---------------------------------------------------------------------------------------
// weight packing for the bf16 path: cast the whole fp32 blob, plus batched cast+transpose
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) cast_blob_kernel(int64_t n4, const float4* __restrict__ src,
                                                        uint2* __restrict__ dst) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    const float4 v = __ldg(src + i);
    __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y), b = __floats2bfloat162_rn(v.z, v.w);
    uint2 r;
    r.x = *reinterpret_cast<uint32_t*>(&a);
    r.y = *reinterpret_cast<uint32_t*>(&b);
    dst[i] = r;
  }
}

__global__ void __launch_bounds__(256) transpose_batch_kernel(const __grid_constant__ TransposeBatch tb) {
  __shared__ float tile[32][33];
  int task = 0;
  while (task + 1 < tb.n && (int)blockIdx.x >= tb.t[task + 1].tile0) ++task;
  const TransposeTask tk = tb.t[task];
  const int local = blockIdx.x - tk.tile0;
  const int tiles_c = (tk.C + 31) / 32;
  const int tr = local / tiles_c, tc = local - tr * tiles_c;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int i = ty; i < 32; i += 8) {
    const int r = tr * 32 + i, c = tc * 32 + tx;
    tile[i][tx] = (r < tk.R && c < tk.C) ? __ldg(tk.src + (size_t)r * tk.C + c) : 0.f;
  }
  __syncthreads();
  for (int i = ty; i < 32; i += 8) {
    const int c = tc * 32 + i, r = tr * 32 + tx;  // dst[c, r]
    if (c < tk.C && r < tk.R) tk.dst[(size_t)c * tk.R + r] = __float2bfloat16_rn(tile[tx][i]);
  }
}

// ---------------------------------------------------------------------------------------
// clip_grad_norm_ + AdamW (train.py:266-271,506-511)
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) sqnorm_kernel(int64_t n, const float* __restrict__ g, float scale,
                                                     float* __restrict__ ws) {
  float s = 0.f;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float v = g[i] * scale;
    s = fmaf(v, v, s);
  }
  __shared__ float red[8];
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x < 32) {
    float t = threadIdx.x < 8 ? red[threadIdx.x] : 0.f;
    t = warp_sum(t);
    if (threadIdx.x == 0) atomicAdd(ws, t);
  }
}

__global__ void __launch_bounds__(256) adamw_kernel(int64_t n, float* __restrict__ p, const float* __restrict__ g,
                                                    float* __restrict__ m, float* __restrict__ v, float lr,
                                                    float b1, float b2, float eps, float wd, float max_norm,
                                                    float grad_scale, float bc1, float bc2_sqrt,
                                                    float* __restrict__ ws) {
  float coef = grad_scale;
  if (max_norm > 0.f) {
    const float norm = sqrtf(ws[0]);
    if (blockIdx.x == 0 && threadIdx.x == 0) ws[1] = norm;
    coef *= fminf(1.f, max_norm / (norm + 1e-6f));
  }
  const float step_size = lr / bc1;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float gi = g[i] * coef;
    float pi = p[i] * (1.f - lr * wd);
    const float mi = b1 * m[i] + (1.f - b1) * gi;
    const float vi = b2 * v[i] + (1.f - b2) * gi * gi;
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    pi -= step_size * (mi / denom);
    p[i] = pi;
    m[i] = mi;
    v[i] = vi;
  }
}

// the same update with the step number read from device memory (CUDA-graph replays): bias corrections per block
__global__ void __launch_bounds__(256) adamw_dev_kernel(int64_t n, float* __restrict__ p, const float* __restrict__ g,
                                                        float* __restrict__ m, float* __restrict__ v, float lr,
                                                        float b1, float b2, float eps, float wd, float max_norm,
                                                        float grad_scale, const uint32_t* __restrict__ step_counter,
                                                        float* __restrict__ ws) {
  __shared__ float s_bc[2];
  if (threadIdx.x == 0) {
    const double step = (double)(*step_counter) + 1.0;
    s_bc[0] = 1.f - (float)pow((double)b1, step);
    s_bc[1] = (float)sqrt(1.0 - pow((double)b2, step));
  }
  __syncthreads();
  const float bc1 = s_bc[0], bc2_sqrt = s_bc[1];
  float coef = grad_scale;
  if (max_norm > 0.f) {
    const float norm = sqrtf(ws[0]);
    if (blockIdx.x == 0 && threadIdx.x == 0) ws[1] = norm;
    coef *= fminf(1.f, max_norm / (norm + 1e-6f));
  }
  const float step_size = lr / bc1;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float gi = g[i] * coef;
    float pi = p[i] * (1.f - lr * wd);
    const float mi = b1 * m[i] + (1.f - b1) * gi;
    const float vi = b2 * v[i] + (1.f - b2) * gi * gi;
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    pi -= step_size * (mi / denom);
    p[i] = pi;
    m[i] = mi;
    v[i] = vi;
  }
}
__global__ void counter_inc_kernel(uint32_t* c) { *c += 1u; }

// ---------------------------------------------------------------------------------------
// Dataset normalisation statistics (R/dataloader/dataset.py:115-157): sums and sums of squares of the I and Q
// channels of interleaved frames, fp64 accumulation, one atomic per block.  acc = {sum I, sum I^2, sum Q, sum Q^2}
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) iq_stats_kernel(int64_t n_pairs, const float2* __restrict__ x,
                                                       double* __restrict__ acc) {
  double s[4] = {0.0, 0.0, 0.0, 0.0};
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_pairs; i += (int64_t)gridDim.x * blockDim.x) {
    const float2 v = __ldg(x + i);
    s[0] += v.x; s[1] += (double)v.x * v.x; s[2] += v.y; s[3] += (double)v.y * v.y;
  }
  __shared__ double red[4][8];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s[k] += __shfl_xor_sync(0xffffffffu, s[k], o);
    if ((threadIdx.x & 31) == 0) red[k][threadIdx.x >> 5] = s[k];
  }
  __syncthreads();
  if (threadIdx.x < 4) {
    double t = 0.0;
    for (int w = 0; w < 8; ++w) t += red[threadIdx.x][w];
    atomicAdd(acc + threadIdx.x, t);
  }
}

}  // namespace

// ---- host launchers ---------------------------------------------------------------------
template <typename E>
int ln_fwd(int M, int d, const float* u, const float* gamma, const float* beta, float eps, E* y16, float* y32,
           E* xhat, float* rstd, cudaStream_t st) {
  AMC_CHECK_ARG(d >= 1 && d <= 32 * MAXV, "layernorm: d=%d unsupported (1..512)", d);
  if (M == 0) return 0;
  ln_fwd_kernel<E><<<ceil_div(M, 8), 256, 0, st>>>(M, d, u, gamma, beta, eps, y16, y32, xhat, rstd);
  AMC_LAUNCH_CHECK();
  return 0;
}
template int ln_fwd<float>(int, int, const float*, const float*, const float*, float, float*, float*, float*,
                           float*, cudaStream_t);
template int ln_fwd<bf16>(int, int, const float*, const float*, const float*, float, bf16*, float*, bf16*, float*,
                          cudaStream_t);

template <typename E>
int colsum(int M, int N, const E* X, int ld, float* out, cudaStream_t st) {
  if (M == 0 || N == 0) return 0;
  const int cb = ceil_div(N, 32);
  int rb = std::max(1, std::min(ceil_div(M, 64), (148 * 8) / cb));
  const int rpb = ceil_div(M, rb);
  rb = ceil_div(M, rpb);
  colsum_kernel<E><<<dim3(cb, rb), 256, 0, st>>>(M, N, X, ld, out, rpb);
  AMC_LAUNCH_CHECK();
  return 0;
}
template int colsum<float>(int, int, const float*, int, float*, cudaStream_t);
template int colsum<bf16>(int, int, const bf16*, int, float*, cudaStream_t);

template <typename E>
int ln_bwd(int M, int d, const float* dy, const E* xhat, const float* rstd, const float* gamma, E* du16,
           float* du32, float* dgamma, float* dbeta, float* dbias, const DropoutCfg& drop, uint32_t site,
           cudaStream_t st) {
  AMC_CHECK_ARG(d >= 1 && d <= 32 * MAXV, "layernorm_bwd: d=%d unsupported (1..512)", d);
  if (M == 0) return 0;
  auto al = [](const void* p, size_t a) { return p == nullptr || (reinterpret_cast<uintptr_t>(p) % a) == 0; };
  if (d % 128 == 0 && al(dy, 16) && al(xhat, 16) && al(du16, 16) && al(du32, 16) && al(gamma, 4)) {
    const int nv = d / 128;
    const int blocks = std::min(ceil_div(M, 8 * (nv <= 2 ? 4 : 2)), 148 * 2);
#define AMC_LN_BWD(NV)                                                                                           \
  ln_bwd_vec_kernel<E, NV><<<blocks, 256, 0, st>>>(M, d, dy, xhat, rstd, gamma, du16, du32, dgamma, dbeta, dbias, \
                                                   drop, site)
    if (nv == 1) AMC_LN_BWD(1);
    else if (nv == 2) AMC_LN_BWD(2);
    else if (nv == 3) AMC_LN_BWD(3);
    else AMC_LN_BWD(4);
#undef AMC_LN_BWD
    AMC_LAUNCH_CHECK();
    return 0;
  }
  const int blocks = std::min(ceil_div(M, 8), 148 * 4);
  ln_bwd_kernel<E><<<blocks, 256, 0, st>>>(M, d, dy, xhat, rstd, gamma, du16, du32, dgamma, dbeta, drop, site);
  AMC_LAUNCH_CHECK();
  if (dbias && du16) AMC_TRY(colsum<E>(M, d, du16, d, dbias, st));
  return 0;
}
template int ln_bwd<float>(int, int, const float*, const float*, const float*, const float*, float*, float*,
                           float*, float*, float*, const DropoutCfg&, uint32_t, cudaStream_t);
template int ln_bwd<bf16>(int, int, const float*, const bf16*, const float*, const float*, bf16*, float*, float*,
                          float*, float*, const DropoutCfg&, uint32_t, cudaStream_t);


PatchP make_patchp(const AmcDesc& D, int Ttok, int K) {
  PatchP p;
  p.kind = D.kind;
  p.input_layout = D.input_layout;
  p.B = D.B;
  p.Ttok = Ttok;
  p.K = K;
  p.in_ch = D.in_ch;
  p.seq_len = D.seq_len;
  p.seg = D.seg;
  p.img_h = D.img_h;
  p.img_w = D.img_w;
  p.patch = D.patch;
  p.mean[0] = D.norm[0];
  p.inv_std[0] = 1.f / D.norm[1];
  p.mean[1] = D.norm[2];
  p.inv_std[1] = 1.f / D.norm[3];
  return p;
}
template <typename E>
int patchify(const AmcDesc& D, int Ttok, int K, const float* src, E* A, cudaStream_t st) {
  const size_t total = (size_t)D.B * Ttok * K;
  if (total == 0) return 0;
  const PatchP pp = make_patchp(D, Ttok, K);
  const bool raw = D.input_layout == AMC_INPUT_RAW;
  const int n_per_ch = D.kind == AMC_KIND_RAWIQ ? D.seq_len : D.img_h * D.img_w;
  const int frame_floats = raw ? (D.kind == AMC_KIND_RAWIQ ? 2 * D.seq_len : D.img_h * D.img_w) : D.in_ch * n_per_ch;
  const size_t smem = (size_t)frame_floats * sizeof(float);
  const bool covers = raw || (size_t)Ttok * K == (size_t)frame_floats;      // every input sample is embedded
  if (K % 8 == 0 && frame_floats % 4 == 0 && smem <= 96 * 1024 && covers &&
      (reinterpret_cast<uintptr_t>(src) & 15) == 0 && (reinterpret_cast<uintptr_t>(A) & 15) == 0) {
    if (smem > 48 * 1024)
      AMC_CUDA(cudaFuncSetAttribute(patchify_frames_kernel<E>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
    const int blocks = std::min(D.B, 148 * 8);
    patchify_frames_kernel<E><<<blocks, 256, smem, st>>>(pp, src, A);
    AMC_LAUNCH_CHECK();
    return 0;
  }
  const int blocks = (int)std::min<size_t>((total + 255) / 256, 148 * 16);
  patchify_kernel<E><<<blocks, 256, 0, st>>>(pp, src, A);
  AMC_LAUNCH_CHECK();
  return 0;
}
template int patchify<float>(const AmcDesc&, int, int, const float*, float*, cudaStream_t);
template int patchify<bf16>(const AmcDesc&, int, int, const float*, bf16*, cudaStream_t);

int patch_scatter(const AmcDesc& D, int Ttok, int K, const float* dX, float* dsrc, cudaStream_t st) {
  if (D.B == 0) return 0;
  if ((int64_t)Ttok * K != frame_floats(D))
    AMC_CUDA(cudaMemsetAsync(dsrc, 0, (size_t)D.B * frame_floats(D) * sizeof(float), st));
  const size_t total = (size_t)D.B * Ttok * K;
  const int blocks = (int)std::min<size_t>((total + 255) / 256, 148 * 16);
  patch_scatter_kernel<<<blocks, 256, 0, st>>>(make_patchp(D, Ttok, K), dX, dsrc);
  AMC_LAUNCH_CHECK();
  return 0;
}

template <typename E>
int cls_rows(int B, int T, int d, const float* cls, const float* pos, E* y16, float* y32, const DropoutCfg& drop,
             cudaStream_t st) {
  if (B == 0) return 0;
  cls_rows_kernel<E><<<ceil_div(B * d, 256), 256, 0, st>>>(B, T, d, cls, pos, y16, y32, drop);
  AMC_LAUNCH_CHECK();
  return 0;
}
template int cls_rows<float>(int, int, int, const float*, const float*, float*, float*, const DropoutCfg&,
                             cudaStream_t);
template int cls_rows<bf16>(int, int, int, const float*, const float*, bf16*, float*, const DropoutCfg&,
                            cudaStream_t);

int cls_grad(int B, int T, int d, const float* dx0, float* dcls, const DropoutCfg& drop, cudaStream_t st) {
  if (B == 0) return 0;
  cls_grad_kernel<<<dim3(ceil_div(d, 128), std::max(1, std::min(B / 8, 148 * 4))), 128, 0, st>>>(B, T, d, dx0, dcls, drop);
  AMC_LAUNCH_CHECK();
  return 0;
}

// vector version (d % 4 == 0, 16-byte aligned): one float4 per thread, row arithmetic once per float4
template <typename E>
__global__ void __launch_bounds__(256) gather_tok_rows_vec_kernel(int B, int T, int Ttok, int d4, int has_cls,
                                                                  const float4* __restrict__ dx0, E* __restrict__ out,
                                                                  DropoutCfg drop) {
  const size_t total = (size_t)B * Ttok * d4;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int c4 = (int)(i % d4);
    const size_t row = i / d4;
    const int t = (int)(row % Ttok), b = (int)(row / Ttok);
    const size_t o4 = ((size_t)b * T + has_cls + t) * d4 + c4;
    float4 v = __ldg(dx0 + o4);
    if (drop.p > 0.f) {
      const float4 k = dropout_mult4(drop, site_pe(), (uint64_t)o4);
      v.x *= k.x; v.y *= k.y; v.z *= k.z; v.w *= k.w;
    }
    store4(out + i * 4, v);
  }
}

template <typename E>
int gather_tok_rows(int B, int T, int Ttok, int d, int has_cls, const float* dx0, E* out, const DropoutCfg& drop,
                    cudaStream_t st) {
  const size_t total = (size_t)B * Ttok * d;
  if (total == 0) return 0;
  if (d % 4 == 0 && (reinterpret_cast<uintptr_t>(dx0) & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0) {
    const int blocks = (int)std::min<size_t>((total / 4 + 255) / 256, 148 * 16);
    gather_tok_rows_vec_kernel<E><<<blocks, 256, 0, st>>>(B, T, Ttok, d / 4, has_cls, reinterpret_cast<const float4*>(dx0),
                                                          out, drop);
    AMC_LAUNCH_CHECK();
    return 0;
  }
  const int blocks = (int)std::min<size_t>((total + 255) / 256, 148 * 16);
  gather_tok_rows_kernel<E><<<blocks, 256, 0, st>>>(B, T, Ttok, d, has_cls, dx0, out, drop);
  AMC_LAUNCH_CHECK();
  return 0;
}
template int gather_tok_rows<float>(int, int, int, int, int, const float*, float*, const DropoutCfg&, cudaStream_t);
template int gather_tok_rows<bf16>(int, int, int, int, int, const float*, bf16*, const DropoutCfg&, cudaStream_t);

int head_fwd(int B, int T, int d, int C, int has_cls, int head_ln, float eps, const float* x, const float* lnw,
             const float* lnb, const float* W, const float* bias, float* logits, float* s_hl, float* s_xhat,
             float* s_rstd, cudaStream_t st) {
  AMC_CHECK_ARG(d <= 32 * MAXV, "head: d=%d unsupported", d);
  if (B == 0) return 0;
  head_fwd_kernel<<<ceil_div(B, 4), 128, 0, st>>>(B, T, d, C, has_cls, head_ln, eps, x, lnw, lnb, W, bias, logits,
                                                  s_hl, s_xhat, s_rstd);
  AMC_LAUNCH_CHECK();
  return 0;
}

int head_bwd(int B, int T, int d, int C, int has_cls, int head_ln, const float* dlogits, const float* W,
             const float* lnw, const float* s_hl, const float* s_xhat, const float* s_rstd, float* dhl_scratch,
             float* dxL, float* dW, float* dbias, float* dlnw, float* dlnb, cudaStream_t st) {
  if (B == 0) return 0;
  head_bwd_rows_kernel<<<ceil_div(B, 4), 128, 0, st>>>(B, T, d, C, has_cls, head_ln, dlogits, W, lnw, s_xhat,
                                                       s_rstd, dxL, dW ? dhl_scratch : nullptr);
  AMC_LAUNCH_CHECK();
  if (!dW) return 0;   // input gradient only: no parameter outputs
  const int chunks = ceil_div(B, 32);       // 32 rows per block (the kernel's shared-memory staging size)
  head_bwd_params_kernel<<<dim3(ceil_div(d, 128), chunks), 128, 0, st>>>(B, d, C, head_ln, dlogits, s_hl, dhl_scratch, s_xhat,
                                                              dW, dbias, dlnw, dlnb);
  AMC_LAUNCH_CHECK();
  return 0;
}

int ce_loss(int B, int C, const float* logits, const int64_t* labels, float ls, float grad_scale, float loss_scale,
            float* dlogits, float* stats, cudaStream_t st) {
  if (B == 0) return 0;
  ce_loss_kernel<<<ceil_div(B, 128), 128, 0, st>>>(B, C, logits, labels, ls, grad_scale, loss_scale, dlogits, stats);
  AMC_LAUNCH_CHECK();
  return 0;
}

// first index of the row maximum (torch.max(1) / argmax semantics of R/training/utils.py:311-317; NaN rows give the index
// of the first NaN, as torch does); one thread per frame -- C is 11 or 19
__global__ void argmax_kernel(int B, int C, const float* __restrict__ logits, int64_t* __restrict__ out) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const float* r = logits + (size_t)b * C;
  float best = r[0];
  int bi = 0;
  for (int c = 1; c < C; ++c) {
    const float v = r[c];
    if (best == best && (v > best || v != v)) { best = v; bi = c; }
  }
  out[b] = bi;
}
int argmax_rows(int B, int C, const float* logits, int64_t* out, cudaStream_t st) {
  if (B == 0) return 0;
  argmax_kernel<<<ceil_div(B, 128), 128, 0, st>>>(B, C, logits, out);
  AMC_LAUNCH_CHECK();
  return 0;
}

int cast_blob(int64_t n, const float* src, bf16* dst, cudaStream_t st) {
  AMC_CHECK_ARG(n % 4 == 0, "cast_blob: n must be a multiple of 4");
  if (n == 0) return 0;
  const int blocks = (int)std::min<int64_t>((n / 4 + 255) / 256, 148 * 8);
  cast_blob_kernel<<<blocks, 256, 0, st>>>(n / 4, reinterpret_cast<const float4*>(src),
                                           reinterpret_cast<uint2*>(dst));
  AMC_LAUNCH_CHECK();
  return 0;
}

int transpose_batch(TransposeBatch& tb, cudaStream_t st) {
  int tiles = 0;
  for (int i = 0; i < tb.n; ++i) {
    tb.t[i].tile0 = tiles;
    tiles += ceil_div(tb.t[i].R, 32) * ceil_div(tb.t[i].C, 32);
  }
  if (tiles == 0) return 0;
  transpose_batch_kernel<<<tiles, 256, 0, st>>>(tb);
  AMC_LAUNCH_CHECK();
  return 0;
}

int adamw_clip_dev(int64_t n, float* p, float* g, float* m, float* v, float lr, float b1, float b2, float eps, float wd,
                   float max_norm, float grad_scale, uint32_t* step_counter, float* ws, cudaStream_t st) {
  const int blocks = (int)std::min<int64_t>((n + 255) / 256, 148 * 8);
  if (n > 0) {
    if (max_norm > 0.f) {
      AMC_CUDA(cudaMemsetAsync(ws, 0, 2 * sizeof(float), st));
      sqnorm_kernel<<<blocks, 256, 0, st>>>(n, g, grad_scale, ws);
      AMC_LAUNCH_CHECK();
    }
    adamw_dev_kernel<<<blocks, 256, 0, st>>>(n, p, g, m, v, lr, b1, b2, eps, wd, max_norm, grad_scale, step_counter, ws);
    AMC_LAUNCH_CHECK();
  }
  counter_inc_kernel<<<1, 1, 0, st>>>(step_counter);
  AMC_LAUNCH_CHECK();
  return 0;
}

int adamw_clip(int64_t n, float* p, float* g, float* m, float* v, float lr, float b1, float b2, float eps, float wd,
               float max_norm, float grad_scale, int64_t step, float* ws, cudaStream_t st) {
  AMC_CHECK_ARG(step >= 1, "adamw: step must be >= 1");
  if (n == 0) return 0;
  const int blocks = (int)std::min<int64_t>((n + 255) / 256, 148 * 8);
  if (max_norm > 0.f) {
    AMC_CUDA(cudaMemsetAsync(ws, 0, 2 * sizeof(float), st));
    sqnorm_kernel<<<blocks, 256, 0, st>>>(n, g, grad_scale, ws);
    AMC_LAUNCH_CHECK();
  }
  const float bc1 = 1.f - (float)pow((double)b1, (double)step);
  const float bc2 = (float)sqrt(1.0 - pow((double)b2, (double)step));
  adamw_kernel<<<blocks, 256, 0, st>>>(n, p, g, m, v, lr, b1, b2, eps, wd, max_norm, grad_scale, bc1, bc2, ws);
  AMC_LAUNCH_CHECK();
  return 0;
}

int iq_stats(int64_t n_pairs, const float* x, double* acc, cudaStream_t st) {
  if (n_pairs <= 0) return 0;
  const int blocks = (int)std::min<int64_t>((n_pairs + 255) / 256, 148 * 8);
  iq_stats_kernel<<<blocks, 256, 0, st>>>(n_pairs, reinterpret_cast<const float2*>(x), acc);
  AMC_LAUNCH_CHECK();
  return 0;
}

}  // namespace amc

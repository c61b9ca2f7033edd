// Attention of the TOP encoder layer when only the CLS token feeds the classifier head
// (transformer_rawIQ.py:88-90 `x[:, 0]`, amc_transformer.py:29): of scale_dot_product_attention.py:26-37 only query
// row 0 is live, so per (frame, head)
//   forward : s_j = q_0 . k_j / sqrt(dh),  p = softmax(s),  o_0 = sum_j p_j v_j                     (T dots, not T^2)
//   backward: dp_j = dO_0 . v_j, ds_j = p_j (dp_j - sum p dp) / sqrt(dh),
//             dq_0 = sum_j ds_j k_j,  dk_j = ds_j q_0,  dv_j = p_j dO_0,  dq_{j>0} = 0
// K and V of every token are still needed (and get gradients); Q of the other tokens is dead.  This removes 1/n_layers of
// the attention time of every model with a CLS token.  One group of GS lanes per (frame, head), lanes own keys
// j = lane, lane + GS, ...; rows are read / written as 16-byte chunks straight from / to the [B*T, 3d] q|k|v layout.
// The q / v bias gradients are dq_0 and dO_0 summed over frames (sum_j p_j = 1); the k bias gradient is exactly 0
// (sum_j ds_j = 0: the dead parameter of SURVEY Appendix B).
#include "attention.cuh"
#include "ptx.cuh"

namespace amc {
namespace {

constexpr int KPL_MAX = 9;     // keys per lane: T <= 288 with 32-lane groups

__device__ __forceinline__ float dot8(const uint4& a, const uint4& b) {
  return bf_lo(a.x) * bf_lo(b.x) + bf_hi(a.x) * bf_hi(b.x) + bf_lo(a.y) * bf_lo(b.y) + bf_hi(a.y) * bf_hi(b.y) +
         bf_lo(a.z) * bf_lo(b.z) + bf_hi(a.z) * bf_hi(b.z) + bf_lo(a.w) * bf_lo(b.w) + bf_hi(a.w) * bf_hi(b.w);
}
__device__ __forceinline__ void axpy8(float (&o)[8], float a, const uint4& x) {
  o[0] = fmaf(a, bf_lo(x.x), o[0]); o[1] = fmaf(a, bf_hi(x.x), o[1]); o[2] = fmaf(a, bf_lo(x.y), o[2]); o[3] = fmaf(a, bf_hi(x.y), o[3]);
  o[4] = fmaf(a, bf_lo(x.z), o[4]); o[5] = fmaf(a, bf_hi(x.z), o[5]); o[6] = fmaf(a, bf_lo(x.w), o[6]); o[7] = fmaf(a, bf_hi(x.w), o[7]);
}
__device__ __forceinline__ uint4 scale8(float a, const uint4& x) {
  return make_uint4(pack2(a * bf_lo(x.x), a * bf_hi(x.x)), pack2(a * bf_lo(x.y), a * bf_hi(x.y)), pack2(a * bf_lo(x.z), a * bf_hi(x.z)),
                    pack2(a * bf_lo(x.w), a * bf_hi(x.w)));
}
template <int GS> __device__ __forceinline__ float group_sum(float v) {
#pragma unroll
  for (int o = GS / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
template <int GS> __device__ __forceinline__ float group_max(float v) {
#pragma unroll
  for (int o = GS / 2; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// scores of this lane's keys against q_0 and their softmax; returns the probabilities in p[]
template <int C8, int GS>
__device__ __forceinline__ void cls_probs(const bf16* __restrict__ kbase, int ld, int T, int gl, const uint4 (&q)[C8], float sl2,
                                          float (&p)[KPL_MAX]) {
  float mx = -INFINITY;
#pragma unroll
  for (int i = 0; i < KPL_MAX; ++i) {
    const int j = gl + i * GS;
    p[i] = -INFINITY;
    if (i * GS < T && j < T) {
      const uint4* kr = reinterpret_cast<const uint4*>(kbase + (size_t)j * ld);
      float s = 0.f;
#pragma unroll
      for (int c = 0; c < C8; ++c) s += dot8(q[c], __ldg(kr + c));
      p[i] = s * sl2;                       // log2 domain
      mx = fmaxf(mx, p[i]);
    }
  }
  mx = group_max<GS>(mx);
  float l = 0.f;
#pragma unroll
  for (int i = 0; i < KPL_MAX; ++i) {
    if (i * GS < T) {
      p[i] = exp2f(p[i] - mx);               // exp2(-inf) = 0 for the lanes past T
      l += p[i];
    } else {
      p[i] = 0.f;
    }
  }
  const float inv = 1.f / group_sum<GS>(l);
#pragma unroll
  for (int i = 0; i < KPL_MAX; ++i) p[i] *= inv;
}

template <int C8, int GS>
__global__ void __launch_bounds__(256) attn_cls_fwd_kernel(int B, int T, int h, const bf16* __restrict__ qkv,
                                                           bf16* __restrict__ out, float sl2) {
  constexpr int dh = 8 * C8;
  const int d = h * dh, ld = 3 * d;
  const int lane = threadIdx.x & 31, gl = lane % GS;
  const int groups = (gridDim.x * blockDim.x) / GS, units = B * h;
  // the trip count is warp-uniform (the group reductions are full-warp shuffles): groups past the end redo the last
  // unit and skip the stores
  for (int u0 = ((blockIdx.x * blockDim.x + threadIdx.x) / 32) * (32 / GS); u0 < units; u0 += groups) {
    const int ur = u0 + lane / GS;
    const bool valid = ur < units;
    const int u = valid ? ur : units - 1;
    const int b = u / h, hh = u - b * h;
    const bf16* base = qkv + (size_t)b * T * ld + hh * dh;
    uint4 q[C8];
#pragma unroll
    for (int c = 0; c < C8; ++c) q[c] = __ldg(reinterpret_cast<const uint4*>(base) + c);
    float p[KPL_MAX];
    cls_probs<C8, GS>(base + d, ld, T, gl, q, sl2, p);
    float o[C8][8];
#pragma unroll
    for (int c = 0; c < C8; ++c)
#pragma unroll
      for (int e = 0; e < 8; ++e) o[c][e] = 0.f;
#pragma unroll
    for (int i = 0; i < KPL_MAX; ++i) {
      const int j = gl + i * GS;
      if (i * GS < T && j < T) {
        const uint4* vr = reinterpret_cast<const uint4*>(base + 2 * d + (size_t)j * ld);
#pragma unroll
        for (int c = 0; c < C8; ++c) axpy8(o[c], p[i], __ldg(vr + c));
      }
    }
#pragma unroll
    for (int c = 0; c < C8; ++c)
#pragma unroll
      for (int e = 0; e < 8; ++e) o[c][e] = group_sum<GS>(o[c][e]);
    if (valid && gl < C8) {
      uint4 w = make_uint4(0u, 0u, 0u, 0u);
      // every lane holds every sum; lane gl stores chunk gl (selected without dynamic register indexing)
#pragma unroll
      for (int c = 0; c < C8; ++c)
        if (c == gl) w = make_uint4(pack2(o[c][0], o[c][1]), pack2(o[c][2], o[c][3]), pack2(o[c][4], o[c][5]), pack2(o[c][6], o[c][7]));
      *(reinterpret_cast<uint4*>(out + (size_t)b * T * d + hh * dh) + gl) = w;
    }
  }
}

template <int C8, int GS>
__global__ void __launch_bounds__(256) attn_cls_bwd_kernel(int B, int T, int h, const bf16* __restrict__ qkv,
                                                           const bf16* __restrict__ dO, bf16* __restrict__ dqkv,
                                                           float* __restrict__ dbias, float scale, float sl2) {
  constexpr int dh = 8 * C8;
  extern __shared__ float sbias[];                 // [2][d]: running sums of dq_0 and dO_0 (q and v bias gradients)
  const int d = h * dh, ld = 3 * d;
  const int lane = threadIdx.x & 31, gl = lane % GS;
  if (dbias)
    for (int c = threadIdx.x; c < 2 * d; c += blockDim.x) sbias[c] = 0.f;
  __syncthreads();
  const int groups = (gridDim.x * blockDim.x) / GS, units = B * h;
  const uint4 zero4 = make_uint4(0u, 0u, 0u, 0u);
  // groups % h == 0 (the host rounds the grid): a group always meets the same head, so its bias-gradient partial
  // sums stay in registers until the end of the kernel
  float bq[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, bv[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  int my_head = 0;
  for (int u0 = ((blockIdx.x * blockDim.x + threadIdx.x) / 32) * (32 / GS); u0 < units; u0 += groups) {
    const int ur = u0 + lane / GS;
    const bool valid = ur < units;                 // warp-uniform trip count, see the forward kernel
    const int u = valid ? ur : units - 1;
    const int b = u / h, hh = u - b * h;
    const bf16* base = qkv + (size_t)b * T * ld + hh * dh;
    bf16* gbase = dqkv + (size_t)b * T * ld + hh * dh;
    uint4 q[C8], go[C8];
#pragma unroll
    for (int c = 0; c < C8; ++c) {
      q[c] = __ldg(reinterpret_cast<const uint4*>(base) + c);
      go[c] = __ldg(reinterpret_cast<const uint4*>(dO + (size_t)b * T * d + hh * dh) + c);
    }
    float p[KPL_MAX], ds[KPL_MAX];
    cls_probs<C8, GS>(base + d, ld, T, gl, q, sl2, p);
    float delta = 0.f;
#pragma unroll
    for (int i = 0; i < KPL_MAX; ++i) {
      const int j = gl + i * GS;
      ds[i] = 0.f;
      if (i * GS < T && j < T) {
        const uint4* vr = reinterpret_cast<const uint4*>(base + 2 * d + (size_t)j * ld);
        float dp = 0.f;
#pragma unroll
        for (int c = 0; c < C8; ++c) dp += dot8(go[c], __ldg(vr + c));
        ds[i] = dp;
        delta = fmaf(p[i], dp, delta);
      }
    }
    delta = group_sum<GS>(delta);
    float dq[C8][8];
#pragma unroll
    for (int c = 0; c < C8; ++c)
#pragma unroll
      for (int e = 0; e < 8; ++e) dq[c][e] = 0.f;
#pragma unroll
    for (int i = 0; i < KPL_MAX; ++i) {
      const int j = gl + i * GS;
      if (i * GS < T && j < T) {
        const float dsj = p[i] * (ds[i] - delta) * scale;
        const uint4* kr = reinterpret_cast<const uint4*>(base + d + (size_t)j * ld);
        uint4* gq = reinterpret_cast<uint4*>(gbase + (size_t)j * ld);
        uint4* gk = reinterpret_cast<uint4*>(gbase + d + (size_t)j * ld);
        uint4* gv = reinterpret_cast<uint4*>(gbase + 2 * d + (size_t)j * ld);
#pragma unroll
        for (int c = 0; c < C8; ++c) {
          axpy8(dq[c], dsj, __ldg(kr + c));
          if (valid) {
            gk[c] = scale8(dsj, q[c]);        // dk_j = ds_j q_0
            gv[c] = scale8(p[i], go[c]);      // dv_j = p_j dO_0
            if (j > 0) gq[c] = zero4;         // queries other than the CLS token are dead in this layer
          }
        }
      }
    }
#pragma unroll
    for (int c = 0; c < C8; ++c)
#pragma unroll
      for (int e = 0; e < 8; ++e) dq[c][e] = group_sum<GS>(dq[c][e]);
    if (valid && gl < C8) {
#pragma unroll
      for (int c = 0; c < C8; ++c)
        if (c == gl) {
          *(reinterpret_cast<uint4*>(gbase) + gl) =
              make_uint4(pack2(dq[c][0], dq[c][1]), pack2(dq[c][2], dq[c][3]), pack2(dq[c][4], dq[c][5]), pack2(dq[c][6], dq[c][7]));
          const float g8[8] = {bf_lo(go[c].x), bf_hi(go[c].x), bf_lo(go[c].y), bf_hi(go[c].y),
                               bf_lo(go[c].z), bf_hi(go[c].z), bf_lo(go[c].w), bf_hi(go[c].w)};
#pragma unroll
          for (int e = 0; e < 8; ++e) { bq[e] += dq[c][e]; bv[e] += g8[e]; }
          my_head = hh;
        }
    }
  }
  if (dbias) {
    if (gl < C8) {
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        if (bq[e] != 0.f) atomicAdd(&sbias[my_head * dh + gl * 8 + e], bq[e]);
        if (bv[e] != 0.f) atomicAdd(&sbias[d + my_head * dh + gl * 8 + e], bv[e]);
      }
    }
    __syncthreads();
    for (int c = threadIdx.x; c < d; c += blockDim.x) {
      if (sbias[c] != 0.f) atomicAdd(dbias + c, sbias[c]);                  // q bias
      if (sbias[d + c] != 0.f) atomicAdd(dbias + 2 * d + c, sbias[d + c]);  // v bias (k bias gradient is exactly 0)
    }
  }
}

// ---- T > 288 (embedding_type='conv1d': T = 1025) --------------------------------------------------------------------
// One WARP per (frame, head), lanes own keys j = lane, lane + 32, ...; nothing is kept per key: the forward is a
// single pass with a per-lane online softmax (m, l, o) merged across the warp at the end; the backward recomputes the
// scores in three passes (row statistics; delta = sum_j p_j dp_j; gradients) -- K and V of one head are 32-128 KB and
// stay in L2, the arithmetic is T dot products per pass, so the kernel is bound by the dqkv rows it has to write.
template <int C8>
__device__ __forceinline__ float cls_score(const uint4 (&q)[C8], const uint4* __restrict__ kr, float sl2) {
  float s = 0.f;
#pragma unroll
  for (int c = 0; c < C8; ++c) s += dot8(q[c], __ldg(kr + c));
  return s * sl2;                               // log2 domain
}
__device__ __forceinline__ float warp_sum32(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max32(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

template <int C8>
__global__ void __launch_bounds__(256) attn_cls_long_fwd_kernel(int B, int T, int h, const bf16* __restrict__ qkv,
                                                                bf16* __restrict__ out, float sl2) {
  constexpr int dh = 8 * C8;
  const int d = h * dh, ld = 3 * d;
  const int lane = threadIdx.x & 31;
  const int warps = (gridDim.x * blockDim.x) >> 5, units = B * h;
  for (int u = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; u < units; u += warps) {     // warp-uniform
    const int b = u / h, hh = u - b * h;
    const bf16* base = qkv + (size_t)b * T * ld + hh * dh;
    uint4 q[C8];
#pragma unroll
    for (int c = 0; c < C8; ++c) q[c] = __ldg(reinterpret_cast<const uint4*>(base) + c);
    float m = -INFINITY, l = 0.f, o[C8][8];
#pragma unroll
    for (int c = 0; c < C8; ++c)
#pragma unroll
      for (int e = 0; e < 8; ++e) o[c][e] = 0.f;
    for (int j = lane; j < T; j += 32) {
      const float s = cls_score<C8>(q, reinterpret_cast<const uint4*>(base + d + (size_t)j * ld), sl2);
      const float mn = fmaxf(m, s);
      const float al = exp2f(m - mn), pj = exp2f(s - mn);       // first key of the lane: al = exp2(-inf) = 0
      l = fmaf(l, al, pj);
      const uint4* vr = reinterpret_cast<const uint4*>(base + 2 * d + (size_t)j * ld);
#pragma unroll
      for (int c = 0; c < C8; ++c) {
#pragma unroll
        for (int e = 0; e < 8; ++e) o[c][e] *= al;
        axpy8(o[c], pj, __ldg(vr + c));
      }
      m = mn;
    }
    const float M = warp_max32(m);
    const float w = exp2f(m - M);                                // a lane without keys (T < 32): exp2(-inf) = 0
    const float inv = 1.f / warp_sum32(l * w);
#pragma unroll
    for (int c = 0; c < C8; ++c)
#pragma unroll
      for (int e = 0; e < 8; ++e) o[c][e] = warp_sum32(o[c][e] * w) * inv;
    if (lane < C8) {
      uint4 wv = make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
      for (int c = 0; c < C8; ++c)
        if (c == lane) wv = make_uint4(pack2(o[c][0], o[c][1]), pack2(o[c][2], o[c][3]), pack2(o[c][4], o[c][5]), pack2(o[c][6], o[c][7]));
      *(reinterpret_cast<uint4*>(out + (size_t)b * T * d + hh * dh) + lane) = wv;
    }
  }
}

template <int C8>
__global__ void __launch_bounds__(256) attn_cls_long_bwd_kernel(int B, int T, int h, const bf16* __restrict__ qkv,
                                                                const bf16* __restrict__ dO, bf16* __restrict__ dqkv,
                                                                float* __restrict__ dbias, float scale, float sl2) {
  constexpr int dh = 8 * C8;
  extern __shared__ float sbias[];                 // [2][d]: sums of dq_0 and dO_0 over this CTA's units
  const int d = h * dh, ld = 3 * d;
  const int lane = threadIdx.x & 31;
  if (dbias)
    for (int c = threadIdx.x; c < 2 * d; c += blockDim.x) sbias[c] = 0.f;
  __syncthreads();
  const int warps = (gridDim.x * blockDim.x) >> 5, units = B * h;
  const uint4 zero4 = make_uint4(0u, 0u, 0u, 0u);
  for (int u = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; u < units; u += warps) {
    const int b = u / h, hh = u - b * h;
    const bf16* base = qkv + (size_t)b * T * ld + hh * dh;
    bf16* gbase = dqkv + (size_t)b * T * ld + hh * dh;
    uint4 q[C8], go[C8];
#pragma unroll
    for (int c = 0; c < C8; ++c) {
      q[c] = __ldg(reinterpret_cast<const uint4*>(base) + c);
      go[c] = __ldg(reinterpret_cast<const uint4*>(dO + (size_t)b * T * d + hh * dh) + c);
    }
    // pass 1: softmax row statistics
    float m = -INFINITY, l = 0.f;
    for (int j = lane; j < T; j += 32) {
      const float s = cls_score<C8>(q, reinterpret_cast<const uint4*>(base + d + (size_t)j * ld), sl2);
      const float mn = fmaxf(m, s);
      l = fmaf(l, exp2f(m - mn), exp2f(s - mn));
      m = mn;
    }
    const float M = warp_max32(m);
    const float inv = 1.f / warp_sum32(l * exp2f(m - M));
    // pass 2: delta = sum_j p_j (dO_0 . v_j)
    float delta = 0.f;
    for (int j = lane; j < T; j += 32) {
      const float s = cls_score<C8>(q, reinterpret_cast<const uint4*>(base + d + (size_t)j * ld), sl2);
      const uint4* vr = reinterpret_cast<const uint4*>(base + 2 * d + (size_t)j * ld);
      float dp = 0.f;
#pragma unroll
      for (int c = 0; c < C8; ++c) dp += dot8(go[c], __ldg(vr + c));
      delta = fmaf(exp2f(s - M) * inv, dp, delta);
    }
    delta = warp_sum32(delta);
    // pass 3: gradients
    float dq[C8][8];
#pragma unroll
    for (int c = 0; c < C8; ++c)
#pragma unroll
      for (int e = 0; e < 8; ++e) dq[c][e] = 0.f;
    for (int j = lane; j < T; j += 32) {
      const uint4* kr = reinterpret_cast<const uint4*>(base + d + (size_t)j * ld);
      const uint4* vr = reinterpret_cast<const uint4*>(base + 2 * d + (size_t)j * ld);
      uint4 kv[C8];
      float s = 0.f, dp = 0.f;
#pragma unroll
      for (int c = 0; c < C8; ++c) {
        kv[c] = __ldg(kr + c);
        s += dot8(q[c], kv[c]);
        dp += dot8(go[c], __ldg(vr + c));
      }
      const float p = exp2f(s * sl2 - M) * inv;
      const float dsj = p * (dp - delta) * scale;
      uint4* gq = reinterpret_cast<uint4*>(gbase + (size_t)j * ld);
      uint4* gk = reinterpret_cast<uint4*>(gbase + d + (size_t)j * ld);
      uint4* gv = reinterpret_cast<uint4*>(gbase + 2 * d + (size_t)j * ld);
#pragma unroll
      for (int c = 0; c < C8; ++c) {
        axpy8(dq[c], dsj, kv[c]);
        gk[c] = scale8(dsj, q[c]);          // dk_j = ds_j q_0
        gv[c] = scale8(p, go[c]);           // dv_j = p_j dO_0
        if (j > 0) gq[c] = zero4;           // queries other than the CLS token are dead in this layer
      }
    }
#pragma unroll
    for (int c = 0; c < C8; ++c)
#pragma unroll
      for (int e = 0; e < 8; ++e) dq[c][e] = warp_sum32(dq[c][e]);
    if (lane < C8) {
#pragma unroll
      for (int c = 0; c < C8; ++c)
        if (c == lane) {
          *(reinterpret_cast<uint4*>(gbase) + lane) =
              make_uint4(pack2(dq[c][0], dq[c][1]), pack2(dq[c][2], dq[c][3]), pack2(dq[c][4], dq[c][5]), pack2(dq[c][6], dq[c][7]));
          if (dbias) {
            const float g8[8] = {bf_lo(go[c].x), bf_hi(go[c].x), bf_lo(go[c].y), bf_hi(go[c].y),
                                 bf_lo(go[c].z), bf_hi(go[c].z), bf_lo(go[c].w), bf_hi(go[c].w)};
#pragma unroll
            for (int e = 0; e < 8; ++e) {
              atomicAdd(&sbias[hh * dh + lane * 8 + e], dq[c][e]);
              atomicAdd(&sbias[d + hh * dh + lane * 8 + e], g8[e]);
            }
          }
        }
    }
  }
  if (dbias) {
    __syncthreads();
    for (int c = threadIdx.x; c < d; c += blockDim.x) {
      if (sbias[c] != 0.f) atomicAdd(dbias + c, sbias[c]);                  // q bias
      if (sbias[d + c] != 0.f) atomicAdd(dbias + 2 * d + c, sbias[d + c]);  // v bias (k bias gradient is exactly 0)
    }
  }
}

}  // namespace

bool attn_cls_supported(int T, int h, int dh) {
  return T >= 1 && T <= ATTN_LONG_MAX_T && (dh == 16 || dh == 32 || dh == 64) && h >= 1;
}

#define AMC_CLS_DISPATCH(KERNEL, ...)                                          \
  do {                                                                         \
    if (dh == 16) {                                                            \
      if (gs == 16) KERNEL<2, 16> __VA_ARGS__;                                 \
      else KERNEL<2, 32> __VA_ARGS__;                                          \
    } else if (dh == 32) {                                                     \
      if (gs == 16) KERNEL<4, 16> __VA_ARGS__;                                 \
      else KERNEL<4, 32> __VA_ARGS__;                                          \
    } else {                                                                   \
      if (gs == 16) KERNEL<8, 16> __VA_ARGS__;                                 \
      else KERNEL<8, 32> __VA_ARGS__;                                          \
    }                                                                          \
  } while (0)

// out: only row 0 of every frame is written (row pitch T*d); the other rows are not read by the caller
int attn_cls_fwd(int B, int T, int h, int dh, const bf16* qkv, bf16* out, cudaStream_t st) {
  AMC_CHECK_ARG(attn_cls_supported(T, h, dh), "attn_cls_fwd: unsupported shape T=%d dh=%d", T, dh);
  if (B == 0) return 0;
  const int gs = T <= 16 ? 16 : 32;
  const long long units = (long long)B * h;
  const int blocks = (int)std::min<long long>((units * gs + 255) / 256, 148 * 8);
  const float sl2 = 1.4426950408889634f / sqrtf((float)dh);
  if (T > 32 * KPL_MAX) {
    if (dh == 16) attn_cls_long_fwd_kernel<2><<<blocks, 256, 0, st>>>(B, T, h, qkv, out, sl2);
    else if (dh == 32) attn_cls_long_fwd_kernel<4><<<blocks, 256, 0, st>>>(B, T, h, qkv, out, sl2);
    else attn_cls_long_fwd_kernel<8><<<blocks, 256, 0, st>>>(B, T, h, qkv, out, sl2);
    AMC_LAUNCH_CHECK();
    return 0;
  }
  AMC_CLS_DISPATCH(attn_cls_fwd_kernel, <<<blocks, 256, 0, st>>>(B, T, h, qkv, out, sl2));
  AMC_LAUNCH_CHECK();
  return 0;
}

// dO: row 0 of every frame (row pitch T*d) is read; dqkv [B*T, 3d] is written completely; dbias (nullable, [3d]) +=
int attn_cls_bwd(int B, int T, int h, int dh, const bf16* qkv, const bf16* dO, bf16* dqkv, float* dbias, cudaStream_t st) {
  AMC_CHECK_ARG(attn_cls_supported(T, h, dh), "attn_cls_bwd: unsupported shape T=%d dh=%d", T, dh);
  if (B == 0) return 0;
  const int gs = T <= 16 ? 16 : 32;
  const long long units = (long long)B * h;
  int blocks = (int)std::min<long long>((units * gs + 255) / 256, 148 * 4);
  // groups in the grid (blocks * 256 / gs) must be a multiple of h: a group then always works on the same head
  const int gpb = 256 / gs;
  while ((blocks * gpb) % h != 0) ++blocks;
  const float scale = 1.f / sqrtf((float)dh), sl2 = 1.4426950408889634f * scale;
  const size_t smem = dbias ? (size_t)2 * h * dh * sizeof(float) : 0;
  if (T > 32 * KPL_MAX) {
    const int lb = (int)std::min<long long>((units * 32 + 255) / 256, 148 * 8);
    if (dh == 16) attn_cls_long_bwd_kernel<2><<<lb, 256, smem, st>>>(B, T, h, qkv, dO, dqkv, dbias, scale, sl2);
    else if (dh == 32) attn_cls_long_bwd_kernel<4><<<lb, 256, smem, st>>>(B, T, h, qkv, dO, dqkv, dbias, scale, sl2);
    else attn_cls_long_bwd_kernel<8><<<lb, 256, smem, st>>>(B, T, h, qkv, dO, dqkv, dbias, scale, sl2);
    AMC_LAUNCH_CHECK();
    return 0;
  }
  AMC_CLS_DISPATCH(attn_cls_bwd_kernel, <<<blocks, 256, smem, st>>>(B, T, h, qkv, dO, dqkv, dbias, scale, sl2));
  AMC_LAUNCH_CHECK();
  return 0;
}

}  // namespace amc

// Projected-gradient adversarial attacks (FGSM / PGD, L-inf and L2 balls) on flat input frames: the ascent step with
// its projection, and the random start.  A frame is the n contiguous floats the model reads for one example in the
// caller's input layout; the kernels need neither the model description nor the patch map.
//
// One CTA owns one frame, so the per-frame L2 norms are fp32 tree reductions inside the CTA (warp shuffles, then the 8
// warp partials summed in a fixed order by every thread): deterministic, one launch per step, no atomics.  Up to
// kCacheElems floats per frame (every reference frame: 2048 for raw-IQ 1024 samples and ViT 32x64, 4096 for SPS-2) the
// L2 step keeps x0, x and g in registers between its passes, i.e. 16 B per element of HBM traffic; longer frames
// (conv1d with long seq_len) stream from global memory on every pass.
#include <math.h>

#include "common.cuh"
#include "profile.cuh"

namespace amc {
namespace {

constexpr int kThreads = 256;
constexpr int kCacheElems = 4096;

// V consecutive floats: one 16-byte access for V = 4 (frame start and pointers 16-byte aligned), scalar for V = 1
template <int V> __device__ __forceinline__ void ldv(const float* p, float (&r)[V]) {
  if constexpr (V == 4) {
    const float4 t = __ldg(reinterpret_cast<const float4*>(p));
    r[0] = t.x; r[1] = t.y; r[2] = t.z; r[3] = t.w;
  } else {
    r[0] = __ldg(p);
  }
}
template <int V> __device__ __forceinline__ void stv(float* p, const float (&r)[V]) {
  if constexpr (V == 4) {
    *reinterpret_cast<float4*>(p) = make_float4(r[0], r[1], r[2], r[3]);
  } else {
    p[0] = r[0];
  }
}

// sum of v over the CTA, identical in every thread; `red` is reusable after the call
__device__ __forceinline__ float block_sum(float v, float* red) {
  v = warp_sum(v);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  float t = 0.f;
#pragma unroll
  for (int w = 0; w < kThreads / 32; ++w) t += red[w];
  __syncthreads();
  return t;
}

__device__ __forceinline__ float sgn(float g) { return g > 0.f ? 1.f : (g < 0.f ? -1.f : 0.f); }

// x = min(max(x + a * sign(g), x0 - eps), x0 + eps), a = step_frac * eps
template <int V>
__global__ void __launch_bounds__(kThreads) adv_step_linf_kernel(int64_t n, const float* __restrict__ x0,
                                                                 const float* __restrict__ g,
                                                                 const float* __restrict__ eps, float step_frac,
                                                                 float* __restrict__ x) {
  const int64_t base = (int64_t)blockIdx.x * n;
  const float e = __ldg(eps + blockIdx.x);
  const float a = step_frac * e;
  const int64_t ng = n / V;
  for (int64_t q = threadIdx.x; q < ng; q += kThreads) {
    const int64_t i = base + q * V;
    float xr[V], x0r[V], gr[V];
    ldv<V>(x + i, xr);
    ldv<V>(x0 + i, x0r);
    ldv<V>(g + i, gr);
#pragma unroll
    for (int v = 0; v < V; ++v) {
      const float lo = x0r[v] - e, hi = x0r[v] + e;
      xr[v] = fminf(fmaxf(xr[v] + a * sgn(gr[v]), lo), hi);
    }
    stv<V>(x + i, xr);
  }
}

// v = x + (a / ||g||) g (v = x when ||g|| = 0); d = v - x0; x = ||d|| > eps ? x0 + d (eps / ||d||) : v
// CACHED: n <= kCacheElems, every array is read once into registers.
template <int V, bool CACHED>
__global__ void __launch_bounds__(kThreads) adv_step_l2_kernel(int64_t n, const float* __restrict__ x0,
                                                               const float* __restrict__ g,
                                                               const float* __restrict__ eps, float step_frac,
                                                               float* __restrict__ x) {
  __shared__ float red[kThreads / 32];
  constexpr int J = CACHED ? kCacheElems / (kThreads * V) : 1;
  const int64_t base = (int64_t)blockIdx.x * n;
  const float e = __ldg(eps + blockIdx.x);
  const float a = step_frac * e;
  const int64_t ng = n / V;
  float gc[J][V], xc[J][V], x0c[J][V];

  float s = 0.f;
  if constexpr (CACHED) {
#pragma unroll
    for (int j = 0; j < J; ++j) {
      const int64_t q = threadIdx.x + (int64_t)j * kThreads;
      if (q < ng) {
        ldv<V>(g + base + q * V, gc[j]);
        ldv<V>(x + base + q * V, xc[j]);
        ldv<V>(x0 + base + q * V, x0c[j]);
#pragma unroll
        for (int v = 0; v < V; ++v) s += gc[j][v] * gc[j][v];
      }
    }
  } else {
    for (int64_t q = threadIdx.x; q < ng; q += kThreads) {
      ldv<V>(g + base + q * V, gc[0]);
#pragma unroll
      for (int v = 0; v < V; ++v) s += gc[0][v] * gc[0][v];
    }
  }
  const float gn = sqrtf(block_sum(s, red));
  const float c = gn > 0.f ? a / gn : 0.f;

  // pass 2: ||v - x0||^2 (cached: v replaces x in registers)
  s = 0.f;
  if constexpr (CACHED) {
#pragma unroll
    for (int j = 0; j < J; ++j) {
      const int64_t q = threadIdx.x + (int64_t)j * kThreads;
      if (q < ng) {
#pragma unroll
        for (int v = 0; v < V; ++v) {
          xc[j][v] = xc[j][v] + c * gc[j][v];
          const float d = xc[j][v] - x0c[j][v];
          s += d * d;
        }
      }
    }
  } else {
    for (int64_t q = threadIdx.x; q < ng; q += kThreads) {
      ldv<V>(g + base + q * V, gc[0]);
      ldv<V>(x + base + q * V, xc[0]);
      ldv<V>(x0 + base + q * V, x0c[0]);
#pragma unroll
      for (int v = 0; v < V; ++v) {
        const float d = (xc[0][v] + c * gc[0][v]) - x0c[0][v];
        s += d * d;
      }
    }
  }
  const float dn = sqrtf(block_sum(s, red));
  const bool project = dn > e;
  const float r = project ? e / dn : 1.f;

  // pass 3: write
  if constexpr (CACHED) {
#pragma unroll
    for (int j = 0; j < J; ++j) {
      const int64_t q = threadIdx.x + (int64_t)j * kThreads;
      if (q < ng) {
        if (project) {
#pragma unroll
          for (int v = 0; v < V; ++v) xc[j][v] = x0c[j][v] + (xc[j][v] - x0c[j][v]) * r;
        }
        stv<V>(x + base + q * V, xc[j]);
      }
    }
  } else {
    for (int64_t q = threadIdx.x; q < ng; q += kThreads) {
      ldv<V>(g + base + q * V, gc[0]);
      ldv<V>(x + base + q * V, xc[0]);
      ldv<V>(x0 + base + q * V, x0c[0]);
#pragma unroll
      for (int v = 0; v < V; ++v) {
        const float vv = xc[0][v] + c * gc[0][v];
        xc[0][v] = project ? x0c[0][v] + (vv - x0c[0][v]) * r : vv;
      }
      stv<V>(x + base + q * V, xc[0]);
    }
  }
}

// u in [0, 1) from the top 24 bits of a hash word
__device__ __forceinline__ float unit24(uint32_t w) { return (float)(w >> 8) * 0x1p-24f; }

// standard normal (Box-Muller) of element index q
__device__ __forceinline__ float normal_at(const DropoutCfg& k, uint64_t q) {
  const uint2 hb = counter_hash2(k, site_adv_elem(), q);
  const float u1 = (float)((hb.x >> 8) + 1u) * 0x1p-24f;   // (0, 1]: log finite
  const float u2 = unit24(hb.y);
  return sqrtf(-2.f * logf(u1)) * cospif(2.f * u2);
}

// LINF: x = x0 + eps (2u - 1);  L2: x = x0 + eps r z / ||z||, r = u^(1/n)
template <int NORM>
__global__ void __launch_bounds__(kThreads) adv_init_kernel(int64_t n, const float* __restrict__ x0,
                                                            const float* __restrict__ eps, DropoutCfg key,
                                                            float* __restrict__ x) {
  __shared__ float red[kThreads / 32];
  const int64_t b = blockIdx.x;
  const int64_t base = b * n;
  const float e = __ldg(eps + b);
  if constexpr (NORM == AMC_NORM_LINF) {
    for (int64_t i = threadIdx.x; i < n; i += kThreads) {
      const float u = unit24(counter_hash2(key, site_adv_elem(), (uint64_t)(base + i)).x);
      x[base + i] = __ldg(x0 + base + i) + e * (2.f * u - 1.f);
    }
  } else {
    float s = 0.f;
    for (int64_t i = threadIdx.x; i < n; i += kThreads) {
      const float z = normal_at(key, (uint64_t)(base + i));
      s += z * z;
    }
    const float zn = sqrtf(block_sum(s, red));
    const float u = unit24(counter_hash2(key, site_adv_radius(), (uint64_t)b).x);
    const float rad = e * powf(u, 1.f / (float)n);
    const float c = zn > 0.f ? rad / zn : 0.f;
    for (int64_t i = threadIdx.x; i < n; i += kThreads)
      x[base + i] = __ldg(x0 + base + i) + c * normal_at(key, (uint64_t)(base + i));
  }
}

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

int check_common(int64_t B, int64_t n, int norm) {
  AMC_CHECK_ARG(B >= 0 && B <= 0x7fffffff, "B must be in [0, 2^31), got %lld", (long long)B);
  AMC_CHECK_ARG(n >= 1, "frame size n must be >= 1, got %lld", (long long)n);
  AMC_CHECK_ARG(norm == AMC_NORM_LINF || norm == AMC_NORM_L2, "unknown norm %d (AMC_NORM_LINF or AMC_NORM_L2)", norm);
  return 0;
}

}  // namespace
}  // namespace amc

using namespace amc;

int amc_adv_step(int64_t B, int64_t n, int norm, const float* x0, const float* g, const float* eps, float step_frac,
                 float* x, amc_stream_t stream) {
  DeviceGuard dev_guard(x);
  AMC_TRY(check_common(B, n, norm));
  AMC_CHECK_ARG(isfinite(step_frac) && step_frac >= 0.f, "step_frac must be finite and >= 0, got %g", (double)step_frac);
  if (B == 0) return 0;
  AMC_CHECK_ARG(x0 && g && eps && x, "NULL argument");
  cudaStream_t st = (cudaStream_t)stream;
  const bool vec = n % 4 == 0 && aligned16(x0) && aligned16(g) && aligned16(x);
  ProfScope ps("adv_step", st, 0.0, 16.0 * (double)B * (double)n + 4.0 * (double)B);
  const dim3 grid((unsigned)B);
  if (norm == AMC_NORM_LINF) {
    if (vec) adv_step_linf_kernel<4><<<grid, kThreads, 0, st>>>(n, x0, g, eps, step_frac, x);
    else adv_step_linf_kernel<1><<<grid, kThreads, 0, st>>>(n, x0, g, eps, step_frac, x);
  } else if (n <= kCacheElems) {
    if (vec) adv_step_l2_kernel<4, true><<<grid, kThreads, 0, st>>>(n, x0, g, eps, step_frac, x);
    else adv_step_l2_kernel<1, true><<<grid, kThreads, 0, st>>>(n, x0, g, eps, step_frac, x);
  } else {
    if (vec) adv_step_l2_kernel<4, false><<<grid, kThreads, 0, st>>>(n, x0, g, eps, step_frac, x);
    else adv_step_l2_kernel<1, false><<<grid, kThreads, 0, st>>>(n, x0, g, eps, step_frac, x);
  }
  AMC_LAUNCH_CHECK();
  return 0;
}

int amc_adv_init(int64_t B, int64_t n, int norm, const float* x0, const float* eps, uint64_t seed, uint64_t offset,
                 const uint32_t* step_counter, float* x, amc_stream_t stream) {
  DeviceGuard dev_guard(x);
  AMC_TRY(check_common(B, n, norm));
  if (B == 0) return 0;
  AMC_CHECK_ARG(x0 && eps && x, "NULL argument");
  cudaStream_t st = (cudaStream_t)stream;
  const DropoutCfg key = make_dropout(0.f, seed, offset, false, step_counter);
  ProfScope ps("adv_init", st, 0.0, 8.0 * (double)B * (double)n + 4.0 * (double)B);
  const dim3 grid((unsigned)B);
  if (norm == AMC_NORM_LINF) adv_init_kernel<AMC_NORM_LINF><<<grid, kThreads, 0, st>>>(n, x0, eps, key, x);
  else adv_init_kernel<AMC_NORM_L2><<<grid, kThreads, 0, st>>>(n, x0, eps, key, x);
  AMC_LAUNCH_CHECK();
  return 0;
}

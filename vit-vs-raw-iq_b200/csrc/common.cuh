// Shared helpers for the sm_100a kernels: error plumbing, element types, warp reductions,
// counter-based dropout RNG.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <atomic>
#include <string>

#include "../../include/amc_b200.h"

namespace amc {

typedef __nv_bfloat16 bf16;

// ---- error plumbing ---------------------------------------------------------------------
void set_error(const char* fmt, ...);
#define AMC_CHECK_ARG(cond, ...)                 \
  do {                                           \
    if (!(cond)) {                               \
      ::amc::set_error(__VA_ARGS__);             \
      return -1;                                 \
    }                                            \
  } while (0)
#define AMC_CUDA(expr)                                                                    \
  do {                                                                                    \
    cudaError_t e__ = (expr);                                                             \
    if (e__ != cudaSuccess) {                                                             \
      ::amc::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, \
                       __LINE__);                                                         \
      return (int)e__;                                                                    \
    }                                                                                     \
  } while (0)
extern std::atomic<long long> g_launch_count;   // kernels launched by this library (bench.py's gpu_launches); autograd
                                                 // calls backward from its own thread, hence atomic
#define AMC_LAUNCH_CHECK()          \
  do {                              \
    ::amc::g_launch_count.fetch_add(1, std::memory_order_relaxed); \
    AMC_CUDA(cudaGetLastError());   \
  } while (0)
#define AMC_TRY(expr)          \
  do {                         \
    int r__ = (expr);          \
    if (r__ != 0) return r__;  \
  } while (0)

// ---- element helpers --------------------------------------------------------------------
__device__ __forceinline__ float to_f(float v) { return v; }
__device__ __forceinline__ float to_f(bf16 v) { return __bfloat162float(v); }
template <typename E> __device__ __forceinline__ E from_f(float v);
template <> __device__ __forceinline__ float from_f<float>(float v) { return v; }
template <> __device__ __forceinline__ bf16 from_f<bf16>(float v) { return __float2bfloat16_rn(v); }

// 4 consecutive elements <-> float4 (16-byte fp32 load / 8-byte bf16 load)
__device__ __forceinline__ float4 load4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ float4 load4(const bf16* p) {
  uint2 r = *reinterpret_cast<const uint2*>(p);
  __nv_bfloat162 a = *reinterpret_cast<__nv_bfloat162*>(&r.x);
  __nv_bfloat162 b = *reinterpret_cast<__nv_bfloat162*>(&r.y);
  float2 fa = __bfloat1622float2(a), fb = __bfloat1622float2(b);
  return make_float4(fa.x, fa.y, fb.x, fb.y);
}
__device__ __forceinline__ void store4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
__device__ __forceinline__ void store4(bf16* p, float4 v) {
  __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y), b = __floats2bfloat162_rn(v.z, v.w);
  uint2 r;
  r.x = *reinterpret_cast<uint32_t*>(&a);
  r.y = *reinterpret_cast<uint32_t*>(&b);
  *reinterpret_cast<uint2*>(p) = r;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// ---- dropout RNG ------------------------------------------------------------------------
// Counter-based hash keyed by (seed, offset, site) over the element index.  One call yields the keep
// decisions of 4 consecutive elements.  Stateless: backward regenerates the same masks from
// (seed, offset, site, element index) instead of storing them (SURVEY §7.3 item 7).
struct DropoutCfg {
  float p;          // drop probability; 0 => disabled
  float scale;      // 1/(1-p)
  uint32_t thresh;  // keep iff rnd >= thresh, thresh = p * 2^32
  uint32_t seed_lo, seed_hi;
  uint32_t off_lo, off_hi;
  const uint32_t* ctr;   // device step counter added to the offset (CUDA-graph replays), or nullptr
};
inline DropoutCfg make_dropout(float p, uint64_t seed, uint64_t offset, bool training, const uint32_t* ctr = nullptr) {
  DropoutCfg c;
  c.ctr = ctr;
  // The keep test compares 16-bit fields, so the drop probability is quantised to floor(p * 65536) / 65536 (documented in
  // include/amc_b200.h); the survivors are scaled by the QUANTISED probability, and p < 2^-16 disables dropout altogether
  // (scaling by 1 / (1 - p) with nothing ever dropped would bias the mean).
  double t = (training && p > 0.f) ? (double)p * 4294967296.0 : 0.0;
  c.thresh = t >= 4294967295.0 ? 0xffffffffu : (uint32_t)t;
  const uint32_t t16 = c.thresh >> 16;
  c.p = t16 > 0 ? (float)(t16 / 65536.0) : 0.f;
  c.scale = t16 > 0 && t16 < 65535 ? (float)(1.0 / (1.0 - t16 / 65536.0)) : (t16 > 0 ? 65536.f : 1.f);
  c.seed_lo = (uint32_t)seed;
  c.seed_hi = (uint32_t)(seed >> 32);
  c.off_lo = (uint32_t)offset;
  c.off_hi = (uint32_t)(offset >> 32);
  return c;
}
// One counter hash per group of 4 elements: an affine function of the group index (seed, step offset and site folded
// into the additive key) goes through the murmur3 finaliser (h), and a second word is derived from the first by one
// more multiply + xorshift (b).  The four 16-bit halves of (h, b) are compared with the 16-bit threshold directly on
// the words (high half: h >= t << 16, low half: (h << 16) >= t << 16).  ~6 integer instructions per element including
// the selects -- the dropout mask is ~half of the bias/ReLU/dropout GEMM epilogue's instructions, and those epilogues,
// not the tensor pipe, bound the K = 256 GEMMs.  Statistics (4M groups, p in {0.1, 0.2, 0.5}): drop rate of every
// field within 3e-4 of p; |correlation| between fields, neighbouring groups, rows, seeds, steps and sites < 2e-3.
// Dropout only needs an unbiased, well-mixed keep decision per element; it is not a cryptographic stream.
// the two hash words (h, b) of counter q under key (seed, offset + *ctr, site)
__device__ __forceinline__ uint2 counter_hash2(const DropoutCfg& c, uint32_t site, uint64_t q) {
  const uint32_t off = c.off_lo + (c.ctr != nullptr ? __ldg(c.ctr) : 0u);
  const uint32_t key = c.seed_lo ^ (off * 0x9E3779B9u) ^ (site * 0x85EBCA6Bu) ^ (c.seed_hi * 0x27D4EB2Fu) ^
                       (c.off_hi * 0x165667B1u);                                        // loop-invariant
  uint32_t h = (uint32_t)q * 0x9E3779B1u + ((uint32_t)(q >> 32) * 0x7FEB352Du + key);
  h ^= h >> 16;                                   // murmur3 finaliser: keys that differ in one bit (seed, step, site)
  h *= 0x85EBCA6Bu;                               // must give uncorrelated masks -- a single multiply left 10 %
  h ^= h >> 13;                                   // correlation between neighbouring seeds
  h *= 0xC2B2AE35u;
  h ^= h >> 16;
  uint32_t b = h * 0x27D4EB2Fu;                   // second word derived from the first
  b ^= b >> 15;
  return make_uint2(h, b);
}
// keep-multipliers (0 or scale) for elements [4*q4, 4*q4+4) of dropout site `site`
__device__ __forceinline__ float4 dropout_mult4(const DropoutCfg& c, uint32_t site, uint64_t q4) {
  const uint2 hb = counter_hash2(c, site, q4);
  const uint32_t h = hb.x, b = hb.y;
  const uint32_t t = c.thresh & 0xFFFF0000u;      // keep iff the 16-bit field >= thresh >> 16
  return make_float4((h << 16) >= t ? c.scale : 0.f, h >= t ? c.scale : 0.f, (b << 16) >= t ? c.scale : 0.f,
                     b >= t ? c.scale : 0.f);
}
// dropout sites (layer l): 0 = after positional encoding (encoder.py:111);
// 1+3l = after attention out-proj (encoder_layer.py:24); 2+3l = FFN hidden (position_wise_feed_forward.py:15);
// 3+3l = after FFN (encoder_layer.py:32)
__host__ __device__ __forceinline__ uint32_t site_pe() { return 0; }
__host__ __device__ __forceinline__ uint32_t site_attn(int l) { return 1 + 3 * l; }
__host__ __device__ __forceinline__ uint32_t site_hidden(int l) { return 2 + 3 * l; }
__host__ __device__ __forceinline__ uint32_t site_ffn(int l) { return 3 + 3 * l; }
// random starts of projected-gradient attacks (adversarial.cu): far above every dropout site (n_layers is small)
__host__ __device__ __forceinline__ uint32_t site_adv_elem() { return 0xADF00000u; }
__host__ __device__ __forceinline__ uint32_t site_adv_radius() { return 0xADF00001u; }

// Every entry point runs on the device that owns its buffers, whatever the caller's current device is (a model on
// cuda:1 while cuda:0 is current is plain `.to(device)` usage in the reference): kernels, cudaFuncSetAttribute and tensor-
// map encoding all act on the CURRENT device, so the ABI switches to the buffers' device for the call and back.
struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(const void* device_ptr) {
    cudaPointerAttributes a;
    if (device_ptr != nullptr && cudaPointerGetAttributes(&a, device_ptr) == cudaSuccess &&
        (a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged)) {
      int cur = 0;
      if (cudaGetDevice(&cur) == cudaSuccess && cur != a.device && cudaSetDevice(a.device) == cudaSuccess) prev = cur;
    } else {
      (void)cudaGetLastError();        // a host pointer is an argument error the callee reports; clear the sticky code
    }
  }
  ~DeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
  DeviceGuard(const DeviceGuard&) = delete;
  DeviceGuard& operator=(const DeviceGuard&) = delete;
};
// SM count of the current device (cached per device)
inline int device_sm_count() {
  static std::atomic<int> cache[64];
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64) dev = 0;
  int n = cache[dev].load(std::memory_order_relaxed);
  if (n == 0) {
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
    cache[dev].store(n, std::memory_order_relaxed);
  }
  return n;
}

inline int ceil_div(int a, int b) { return (a + b - 1) / b; }
inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

}  // namespace amc

// Integrated Gradients along the straight path from a baseline x' to the input x (amc_model_integrated_gradients).
// The front end is affine in src, so the embedding of a path point is x0(x') + a (x0(x) - x0(x')): the path points of a
// chunk are blended from the two endpoint embeddings instead of running the front end once per point.  The input
// gradient is linear in the embedding gradient, so the token-row gradients of all points are summed first and the
// dsrc GEMM and scatter run once per call.  Both kernels are HBM-bound element-wise passes; neither uses atomics, so
// repeated calls are bit-identical.
#include "rowops.cuh"

namespace amc {
namespace {

// x32[k, j] = xb[j] + alpha[k] (xx[j] - xb[j]) and x16 = its E copy, j over one endpoint's B*T*d values (frame order
// k*B + b).  xx = x0(x), xb = x0(x') = xx + n_frame.
template <typename E>
__global__ void __launch_bounds__(256) ig_blend_kernel(int n_points, int64_t n_frame, const float* __restrict__ alpha,
                                                       const float* __restrict__ x0e, E* __restrict__ x16,
                                                       float* __restrict__ x32) {
  const int64_t total = (int64_t)n_points * n_frame;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int k = (int)(i / n_frame);
    const int64_t j = i - (int64_t)k * n_frame;
    const float xb = __ldg(x0e + n_frame + j);
    const float v = fmaf(__ldg(alpha + k), __ldg(x0e + j) - xb, xb);
    x32[i] = v;
    if (sizeof(E) == 2) x16[i] = from_f<E>(v);
  }
}

// acc[b, t, c] (+)= sum over k = 0..n-1, in that order, of dx0[(k*B + b), has_cls + t, c]: the gradients of the token
// rows of a chunk's x0 summed over its path points.  `first` starts the sum at 0; with `out` the total also leaves as
// E (the dsrc GEMM's operand; out may alias acc when E is float).
template <typename E>
__global__ void __launch_bounds__(256) ig_reduce_kernel(int B, int T, int Ttok, int d, int has_cls, int n,
                                                        const float* __restrict__ dx0, float* acc, int first, E* out) {
  const int64_t total = (int64_t)B * Ttok * d;
  const int64_t point = (int64_t)B * T * d;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % d);
    const int64_t row = i / d;
    const int t = (int)(row % Ttok), b = (int)(row / Ttok);
    const float* p = dx0 + ((int64_t)b * T + has_cls + t) * d + c;
    float v = first ? 0.f : acc[i];
    for (int k = 0; k < n; ++k) v += __ldg(p + k * point);
    acc[i] = v;
    if (out) out[i] = from_f<E>(v);
  }
}

// the same two passes on float4 (n_frame and d multiples of 4, 16-byte aligned rows): one 16-byte load per operand
template <typename E>
__global__ void __launch_bounds__(256) ig_blend_vec_kernel(int n_points, int64_t n4, const float* __restrict__ alpha,
                                                           const float4* __restrict__ x0e, E* __restrict__ x16,
                                                           float4* __restrict__ x32) {
  const int64_t total = (int64_t)n_points * n4;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int k = (int)(i / n4);
    const int64_t j = i - (int64_t)k * n4;
    const float a = __ldg(alpha + k);
    const float4 xx = __ldg(x0e + j), xb = __ldg(x0e + n4 + j);
    const float4 v = make_float4(fmaf(a, xx.x - xb.x, xb.x), fmaf(a, xx.y - xb.y, xb.y), fmaf(a, xx.z - xb.z, xb.z),
                                 fmaf(a, xx.w - xb.w, xb.w));
    x32[i] = v;
    if (sizeof(E) == 2) store4(x16 + i * 4, v);
  }
}

template <typename E>
__global__ void __launch_bounds__(256) ig_reduce_vec_kernel(int B, int T, int Ttok, int d4, int has_cls, int n,
                                                            const float4* __restrict__ dx0, float4* acc, int first,
                                                            E* out) {
  const int64_t total = (int64_t)B * Ttok * d4;
  const int64_t point = (int64_t)B * T * d4;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % d4);
    const int64_t row = i / d4;
    const int t = (int)(row % Ttok), b = (int)(row / Ttok);
    const float4* p = dx0 + ((int64_t)b * T + has_cls + t) * d4 + c;
    float4 v = first ? make_float4(0.f, 0.f, 0.f, 0.f) : acc[i];
    for (int k = 0; k < n; ++k) {
      const float4 g = __ldg(p + k * point);
      v.x += g.x; v.y += g.y; v.z += g.z; v.w += g.w;
    }
    acc[i] = v;
    if (out) store4(out + i * 4, v);
  }
}

inline int grid_for(int64_t n) { return (int)std::min<int64_t>((n + 255) / 256, 148 * 16); }
inline bool al16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

}  // namespace

template <typename E>
int ig_blend(int n_points, int64_t n_frame, const float* alpha, const float* x0e, E* x16, float* x32, cudaStream_t st) {
  if ((int64_t)n_points * n_frame == 0) return 0;
  if (n_frame % 4 == 0 && al16(x0e) && al16(x16) && al16(x32)) {
    const int64_t n4 = n_frame / 4;
    ig_blend_vec_kernel<E><<<grid_for((int64_t)n_points * n4), 256, 0, st>>>(
        n_points, n4, alpha, reinterpret_cast<const float4*>(x0e), x16, reinterpret_cast<float4*>(x32));
    AMC_LAUNCH_CHECK();
    return 0;
  }
  ig_blend_kernel<E><<<grid_for((int64_t)n_points * n_frame), 256, 0, st>>>(n_points, n_frame, alpha, x0e, x16, x32);
  AMC_LAUNCH_CHECK();
  return 0;
}
template int ig_blend<float>(int, int64_t, const float*, const float*, float*, float*, cudaStream_t);
template int ig_blend<bf16>(int, int64_t, const float*, const float*, bf16*, float*, cudaStream_t);

template <typename E>
int ig_reduce(int B, int T, int Ttok, int d, int has_cls, int n, const float* dx0, float* acc, bool first, E* out,
              cudaStream_t st) {
  const int64_t total = (int64_t)B * Ttok * d;
  if (total == 0) return 0;
  if (d % 4 == 0 && al16(dx0) && al16(acc) && al16(out)) {
    ig_reduce_vec_kernel<E><<<grid_for(total / 4), 256, 0, st>>>(B, T, Ttok, d / 4, has_cls, n,
                                                                reinterpret_cast<const float4*>(dx0),
                                                                reinterpret_cast<float4*>(acc), first ? 1 : 0, out);
    AMC_LAUNCH_CHECK();
    return 0;
  }
  ig_reduce_kernel<E><<<grid_for(total), 256, 0, st>>>(B, T, Ttok, d, has_cls, n, dx0, acc, first ? 1 : 0, out);
  AMC_LAUNCH_CHECK();
  return 0;
}
template int ig_reduce<float>(int, int, int, int, int, int, const float*, float*, bool, float*, cudaStream_t);
template int ig_reduce<bf16>(int, int, int, int, int, int, const float*, float*, bool, bf16*, cudaStream_t);

}  // namespace amc

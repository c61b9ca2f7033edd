// Embedding with a tiny patch width in bf16 mode (K = in_channels * segment_size not a multiple of 8, K <= 16):
// `embedding_type='conv1d'` is Conv1d(2, d, kernel_size=1), i.e. K = 2 (R/models/embedding/patch_embedding.py:26-33).
// A [M, 2] operand has no 16-byte rows for TMA and 2 FLOP per output byte is nothing for a tensor core to do: the
// forward is an HBM-bound elementwise kernel (x0 = a . W[n, :] + bias + PE, dropout -> fp32 + bf16 rows) that shares
// the GEMM epilogue, the backward a column reduction (dW[n, k] += sum_m dY[m, n] A[m, k], db[n] += sum_m dY[m, n]).
// Operands are the same bf16 values the tensor-core path would see, accumulation is fp32.  The input gradient
// (dX[m, k] = sum_n dY[m, n] W[n, k]) is HBM-bound on reading dY and is written straight into the caller's layout.
#include <algorithm>

#include "gemm_common.cuh"
#include "rowops.cuh"

namespace amc {
namespace {

constexpr int SK_MAX = 16;

__global__ void __launch_bounds__(256) embed_smallk_fwd_kernel(int M, int N, int K, const bf16* __restrict__ A,
                                                               const bf16* __restrict__ W, Epi e, int vec_ok) {
  const int n4 = (N + 3) >> 2;
  const long long total = (long long)M * n4;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int m = (int)(idx / n4), n = (int)(idx - (long long)m * n4) * 4;
    float a[SK_MAX];
#pragma unroll
    for (int k = 0; k < SK_MAX; ++k) a[k] = k < K ? to_f(A[(size_t)m * K + k]) : 0.f;
    float v[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (n + j < N) {
        const bf16* wr = W + (size_t)(n + j) * K;
#pragma unroll
        for (int k = 0; k < SK_MAX; ++k)
          if (k < K) v[j] = fmaf(a[k], to_f(wr[k]), v[j]);
      }
    }
    epi_apply4<bf16>(e, m, n, make_float4(v[0], v[1], v[2], v[3]), M, N, vec_ok != 0);
  }
}

// one thread per output column n, a block per slice of rows; per-block partial sums leave through atomics
__global__ void __launch_bounds__(256) embed_smallk_bwd_kernel(int M, int N, int K, const bf16* __restrict__ dY, int ldy,
                                                               const bf16* __restrict__ A, float* __restrict__ dW,
                                                               float* __restrict__ db, int rows_per_block) {
  const int r0 = blockIdx.x * rows_per_block, r1 = min(M, r0 + rows_per_block);
  for (int n = threadIdx.x; n < N; n += blockDim.x) {
    float acc[SK_MAX], sb = 0.f;
#pragma unroll
    for (int k = 0; k < SK_MAX; ++k) acc[k] = 0.f;
    for (int m = r0; m < r1; ++m) {
      const float g = to_f(dY[(size_t)m * ldy + n]);
      sb += g;
#pragma unroll
      for (int k = 0; k < SK_MAX; ++k)
        if (k < K) acc[k] = fmaf(g, to_f(__ldg(A + (size_t)m * K + k)), acc[k]);
    }
#pragma unroll
    for (int k = 0; k < SK_MAX; ++k)
      if (k < K) atomicAdd(dW + (size_t)n * K + k, acc[k]);
    if (db != nullptr) atomicAdd(db + n, sb);
  }
}

// a warp per token row: the row of dY is read once, K <= 16 partial sums per lane are reduced across the warp in a
// fixed order (no atomics: deterministic), lane k writes element k of the patch through the front end's map;
// MUL (Integrated Gradients) also multiplies it by src - base at that offset
template <bool MUL>
__global__ void __launch_bounds__(256) embed_smallk_dgrad_kernel(int M, int N, int K, const bf16* __restrict__ dY,
                                                                 const bf16* __restrict__ W, PatchP p,
                                                                 float* __restrict__ dsrc, const float* __restrict__ src,
                                                                 const float* __restrict__ base) {
  extern __shared__ float sw[];   // W [N, K] in fp32
  for (int i = threadIdx.x; i < N * K; i += blockDim.x) sw[i] = to_f(W[i]);
  __syncthreads();
  const int lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  for (int m = blockIdx.x * nw + (threadIdx.x >> 5); m < M; m += gridDim.x * nw) {
    float acc[SK_MAX];
#pragma unroll
    for (int k = 0; k < SK_MAX; ++k) acc[k] = 0.f;
    for (int n = lane; n < N; n += 32) {
      const float g = to_f(dY[(size_t)m * N + n]);
#pragma unroll
      for (int k = 0; k < SK_MAX; ++k)
        if (k < K) acc[k] = fmaf(g, sw[n * K + k], acc[k]);
    }
    float v = 0.f;
#pragma unroll
    for (int k = 0; k < SK_MAX; ++k) {
      if (k < K) {
        const float s = warp_sum(acc[k]);
        if (lane == k) v = s;
      }
    }
    if (lane < K) {
      const int b = m / p.Ttok, t = m - b * p.Ttok;
      int ch;
      const size_t o = patch_src_offset(p, b, t, lane, &ch);
      const float g = ch < 0 ? v : v * p.inv_std[ch];
      dsrc[o] = MUL ? g * (__ldg(src + o) - __ldg(base + o)) : g;
    }
  }
}

}  // namespace

bool embed_smallk_supported(int K) { return K >= 1 && K <= SK_MAX; }

int embed_smallk_fwd(int M, int N, int K, const bf16* A, const bf16* W, const Epi& epi, cudaStream_t st) {
  AMC_CHECK_ARG(embed_smallk_supported(K), "small-K embedding: K=%d unsupported (1..%d)", K, SK_MAX);
  AMC_CHECK_ARG(epi.drop.p == 0.f || N % 4 == 0, "small-K embedding: dropout needs d_model %% 4 == 0");
  if (M == 0) return 0;
  const long long total = (long long)M * ((N + 3) / 4);
  const int blocks = (int)std::min<long long>((total + 255) / 256, 148 * 16);
  embed_smallk_fwd_kernel<<<blocks, 256, 0, st>>>(M, N, K, A, W, epi, epi_vec_ok<bf16>(epi, N) ? 1 : 0);
  AMC_LAUNCH_CHECK();
  return 0;
}

int embed_smallk_bwd(int M, int N, int K, const bf16* dY, int ldy, const bf16* A, float* dW, float* db, cudaStream_t st) {
  AMC_CHECK_ARG(embed_smallk_supported(K), "small-K embedding: K=%d unsupported (1..%d)", K, SK_MAX);
  if (M == 0) return 0;
  int blocks = std::max(1, std::min(ceil_div(M, 64), 148 * 4));
  const int rpb = ceil_div(M, blocks);
  blocks = ceil_div(M, rpb);
  embed_smallk_bwd_kernel<<<blocks, 256, 0, st>>>(M, N, K, dY, ldy, A, dW, db, rpb);
  AMC_LAUNCH_CHECK();
  return 0;
}

int embed_smallk_dgrad(const AmcDesc& D, int Ttok, int N, int K, const bf16* dY, const bf16* W, float* dsrc,
                       cudaStream_t st, const float* src, const float* base) {
  AMC_CHECK_ARG(embed_smallk_supported(K), "small-K embedding: K=%d unsupported (1..%d)", K, SK_MAX);
  const int M = D.B * Ttok;
  if (M == 0) return 0;
  if ((int64_t)Ttok * K != frame_floats(D))
    AMC_CUDA(cudaMemsetAsync(dsrc, 0, (size_t)D.B * frame_floats(D) * sizeof(float), st));
  const int blocks = std::min(ceil_div(M, 8), 148 * 8);
  const size_t smem = (size_t)N * K * sizeof(float);
  if (src)
    embed_smallk_dgrad_kernel<true><<<blocks, 256, smem, st>>>(M, N, K, dY, W, make_patchp(D, Ttok, K), dsrc, src, base);
  else
    embed_smallk_dgrad_kernel<false><<<blocks, 256, smem, st>>>(M, N, K, dY, W, make_patchp(D, Ttok, K), dsrc, nullptr,
                                                                nullptr);
  AMC_LAUNCH_CHECK();
  return 0;
}

}  // namespace amc

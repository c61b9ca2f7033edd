// Epilogue shared by the fp32 FMA GEMM (gemm_simt.cu) and the bf16 tcgen05 GEMM (gemm_tc.cu).
#pragma once
#include "common.cuh"

namespace amc {

// Everything a GEMM does to an accumulator tile before it leaves the SM.  Order per element:
//   v = acc (+bias[n]) ; relu ; *= (mask_src[m,n] > 0) * mask_scale ; += pos[t,n] ;
//   *= dropout keep/(1-p) ; += res32[m,n] ; -> D16 / D32 (store or atomic add)
struct Epi {
  const float* bias = nullptr;    // [N]
  int relu = 0;
  const void* mask_src = nullptr; // element type E, [M, ldmask]: ReLU backward mask (stored post-ReLU hidden)
  int ldmask = 0;
  float mask_scale = 1.f;
  const float* pos = nullptr;     // [map_T, N] positional encoding (front end)
  int map_Ttok = 0, map_T = 0, map_cls = 0;  // front end: out_row = (m / Ttok) * T + cls + m % Ttok
  DropoutCfg drop = {0.f, 1.f, 0u, 0u, 0u, 0u, 0u, nullptr};
  uint32_t drop_site = 0;
  const float* res32 = nullptr;   // [M, ldres] fp32 residual / skip gradient
  int ldres = 0;
  void* D16 = nullptr;            // element type E
  int ldd16 = 0;
  float* D32 = nullptr;
  int ldd32 = 0;
  int accumulate = 0;             // D32 += (atomic)
  // weight-gradient GEMMs (token-major operands): colsum_out[m] += sum_k A[k, m], i.e. the bias gradient of the
  // same layer, summed from the A tiles while they sit in shared memory (bf16 tcgen05 path only)
  float* colsum_out = nullptr;
  // fused LayerNorm over the row (bf16 tcgen05 path, N <= 256): u = epilogue value, y = gamma*xhat+beta ->
  // D16 (bf16 y), D32 (fp32 y), ln_xhat (bf16, optional, pitch N), ln_rstd (fp32 [M], optional)
  const float* ln_gamma = nullptr;
  const float* ln_beta = nullptr;
  float ln_eps = 0.f;
  void* ln_xhat = nullptr;
  float* ln_rstd = nullptr;
};

// ---- fast path: whole float4 in bounds, every pointer vector-aligned; registers only -------------
template <typename E>
__device__ __forceinline__ void epi_fast4(const Epi& e, int m, int n, float4 v, int N) {
  if (e.bias) {
    const float4 b = __ldg(reinterpret_cast<const float4*>(e.bias + n));
    v.x += b.x; v.y += b.y; v.z += b.z; v.w += b.w;
  }
  if (e.relu) {
    v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f);
  }
  if (e.mask_src) {
    const float4 h = load4(reinterpret_cast<const E*>(e.mask_src) + (size_t)m * e.ldmask + n);
    const float s = e.mask_scale;
    v.x = h.x > 0.f ? v.x * s : 0.f; v.y = h.y > 0.f ? v.y * s : 0.f;
    v.z = h.z > 0.f ? v.z * s : 0.f; v.w = h.w > 0.f ? v.w * s : 0.f;
  }
  int orow = m;
  if (e.map_Ttok > 0) {
    const int b = m / e.map_Ttok, t = m - b * e.map_Ttok + e.map_cls;
    orow = b * e.map_T + t;
    if (e.pos) {
      const float4 q = __ldg(reinterpret_cast<const float4*>(e.pos + (size_t)t * N + n));
      v.x += q.x; v.y += q.y; v.z += q.z; v.w += q.w;
    }
  }
  if (e.drop.p > 0.f) {
    const float4 k = dropout_mult4(e.drop, e.drop_site, ((uint64_t)orow * (uint64_t)N + (uint64_t)n) >> 2);
    v.x *= k.x; v.y *= k.y; v.z *= k.z; v.w *= k.w;
  }
  if (e.res32) {
    const float4 r = *reinterpret_cast<const float4*>(e.res32 + (size_t)orow * e.ldres + n);
    v.x += r.x; v.y += r.y; v.z += r.z; v.w += r.w;
  }
  if (e.D32) {
    float* dp = e.D32 + (size_t)orow * e.ldd32 + n;
    if (e.accumulate) {
      atomicAdd(reinterpret_cast<float4*>(dp), v);     // red.global.add.v4.f32 (sm_90+)
    } else {
      *reinterpret_cast<float4*>(dp) = v;
    }
  }
  if (e.D16) store4(reinterpret_cast<E*>(e.D16) + (size_t)orow * e.ldd16 + n, v);
}

// ---- slow path: ragged right edge or unaligned pointers; element-wise, kept out of line ---------
template <typename E>
__device__ __noinline__ void epi_slow4(const Epi& e, int m, int n, float4 v, int N) {
  const float in[4] = {v.x, v.y, v.z, v.w};
  const int b = e.map_Ttok > 0 ? m / e.map_Ttok : 0;
  const int t = e.map_Ttok > 0 ? m - b * e.map_Ttok + e.map_cls : 0;
  const int orow = e.map_Ttok > 0 ? b * e.map_T + t : m;
  for (int j = 0; j < 4 && n + j < N; ++j) {
    float a = in[j];
    const int c = n + j;
    if (e.bias) a += __ldg(e.bias + c);
    if (e.relu) a = fmaxf(a, 0.f);
    if (e.mask_src)
      a = to_f(reinterpret_cast<const E*>(e.mask_src)[(size_t)m * e.ldmask + c]) > 0.f ? a * e.mask_scale : 0.f;
    if (e.map_Ttok > 0 && e.pos) a += __ldg(e.pos + (size_t)t * N + c);
    if (e.res32) a += e.res32[(size_t)orow * e.ldres + c];
    if (e.D32) {
      float* dp = e.D32 + (size_t)orow * e.ldd32 + c;
      if (e.accumulate) atomicAdd(dp, a);
      else *dp = a;
    }
    if (e.D16) reinterpret_cast<E*>(e.D16)[(size_t)orow * e.ldd16 + c] = from_f<E>(a);
  }
}

template <typename E>
__device__ __forceinline__ void epi_apply4(const Epi& e, int m, int n, float4 v, int M, int N, bool vec_ok) {
  if (m >= M || n >= N) return;
  if (vec_ok && n + 3 < N) epi_fast4<E>(e, m, n, v, N);
  else epi_slow4<E>(e, m, n, v, N);   // (dropout requires N % 4 == 0 and aligned pointers: host-checked)
}

// true when every pointer/ld the epilogue touches allows 16-byte (fp32) / 8-byte (bf16) vectors
template <typename E>
inline bool epi_vec_ok(const Epi& e, int N) {
  auto al = [](const void* p, size_t a) { return p == nullptr || (reinterpret_cast<uintptr_t>(p) % a) == 0; };
  bool ok = (N % 4 == 0);
  ok = ok && al(e.bias, 16) && al(e.pos, 16) && al(e.res32, 16) && al(e.D32, 16);
  ok = ok && al(e.mask_src, sizeof(E) * 4) && al(e.D16, sizeof(E) * 4);
  ok = ok && (e.ldres % 4 == 0) && (e.ldd32 % 4 == 0) && (e.ldmask % 4 == 0) && (e.ldd16 % 4 == 0);
  return ok;
}

struct GemmArgs {
  const char* name = "gemm";  // profiling class
  int M = 0, N = 0, K = 0;
  const void* A = nullptr;  // element type E
  int lda = 0;
  int transA = 0;           // 0: [M,K] row-major; 1: [K,M] row-major
  const void* B = nullptr;
  int ldb = 0;
  int transB = 0;           // 0: [N,K] row-major; 1: [K,N] row-major
  int split_k = 1;          // >1 requires epi.accumulate
  Epi epi;
};

int gemm_f32(const GemmArgs& g, cudaStream_t st);   // gemm_simt.cu
int gemm_bf16(const GemmArgs& g, cudaStream_t st);  // gemm_tc.cu (tcgen05)

// embed_smallk.cu: bf16 embedding whose patch width K is not a multiple of 8 (conv1d embedding: K = 2)
bool embed_smallk_supported(int K);
int embed_smallk_fwd(int M, int N, int K, const bf16* A, const bf16* W, const Epi& epi, cudaStream_t st);
int embed_smallk_bwd(int M, int N, int K, const bf16* dY, int ldy, const bf16* A, float* dW, float* db, cudaStream_t st);
// input gradient dsrc (caller's layout per D.input_layout, overwritten) from dY [B*Ttok, N] and W [N, K]
int embed_smallk_dgrad(const AmcDesc& D, int Ttok, int N, int K, const bf16* dY, const bf16* W, float* dsrc,
                       cudaStream_t st);

// frontend_tc.cu: fused normalise + frame + patchify + embedding GEMM (+bias, +PE, dropout) for the bf16 path.
// *handled = false when the geometry is outside what the fused kernel covers (caller: patchify + gemm);
// probe_only = true answers that question without launching.
int frontend_fused(const AmcDesc& D, int Ttok, int K, const float* src, const bf16* W, const Epi& epi, bf16* Aout,
                   bool probe_only, bool* handled, cudaStream_t st);

}  // namespace amc

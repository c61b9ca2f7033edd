// Host launchers of the fused short-sequence attention kernels (attention.cu).
#pragma once
#include <algorithm>
#include <cmath>
#include <type_traits>

#include "common.cuh"

namespace amc {
// lse (nullable, [B, h, T] fp32): log2-domain softmax row statistics written by the forward tile kernel and read
// by its backward together with `out` (both nullable in backward: the older two-phase kernels are used then).
template <typename E>
int attention_fwd(int B, int T, int h, int dh, const E* qkv, E* out, float* lse, cudaStream_t st);
template <typename E>
int attention_bwd(int B, int T, int h, int dh, const E* qkv, const E* out, const float* lse, const E* dout, E* dqkv,
                  float* dbias, cudaStream_t st);

// attn_tiles.cu: TMA-tiled single-CTA kernels for 16 < T <= 288 (bf16); *handled = false -> caller falls back
bool attn_tiles_supported(int T, int h, int dh);
int attn_tiles_fwd(int B, int T, int h, int dh, const bf16* qkv, bf16* out, float* lse, bool* handled, cudaStream_t st);
int attn_tiles_bwd(int B, int T, int h, int dh, const bf16* qkv, const bf16* out, const float* lse, const bf16* dout,
                   bf16* dqkv, float* dbias, bool* handled, cudaStream_t st);

// attn_tc5.cu: tcgen05 / TMEM kernels for 49 <= T <= 272 (bf16, head dim 16 / 32 / 64); *handled = false -> next kernel
bool attn_tc5_supported(int T, int h, int dh);
int attn_tc5_fwd(int B, int T, int h, int dh, const bf16* qkv, bf16* out, float* lse, bool* handled, cudaStream_t st);
// (needs the forward's out + lse; dbias (nullable, fp32 [3d]) += q | k | v bias gradients)
int attn_tc5_bwd(int B, int T, int h, int dh, const bf16* qkv, const bf16* out, const float* lse, const bf16* dout,
                 bf16* dqkv, float* dbias, bool* handled, cudaStream_t st);

// attn_long.cu: T > 288 (embedding_type='conv1d': one token per IQ sample) -- flash-style tiled kernels; the
// backward needs the forward's `out` and `lse`
constexpr int ATTN_LONG_MAX_T = 16384;
template <typename E>
int attn_long_fwd(int B, int T, int h, int dh, const E* qkv, E* out, float* lse, cudaStream_t st);
template <typename E>
int attn_long_bwd(int B, int T, int h, int dh, const E* qkv, const E* out, const float* lse, const E* dout, E* dqkv,
                  cudaStream_t st);

// attn_cls.cu: attention restricted to query row 0 (the CLS token) for the top layer of a CLS-pooled model (bf16)
bool attn_cls_supported(int T, int h, int dh);
int attn_cls_fwd(int B, int T, int h, int dh, const bf16* qkv, bf16* out, cudaStream_t st);
int attn_cls_bwd(int B, int T, int h, int dh, const bf16* qkv, const bf16* dO, bf16* dqkv, float* dbias, cudaStream_t st);

// attn_maps.cu: attention probabilities fp32 [B, h, T, T] and one rollout step v_out = v_in^T (0.5 mean_h P + 0.5 I),
// v fp32 [B, T], for every (T, dh) attention_fwd takes; neither needs the forward's lse
template <typename E>
int attention_probs(int B, int T, int h, int dh, const E* qkv, float* probs, cudaStream_t st);
template <typename E>
int attention_rollout_step(int B, int T, int h, int dh, const E* qkv, const float* v_in, float* v_out, cudaStream_t st);
// one class-specific relevance step v_out = v_in + (1/h) sum_h v_in^T relu((dO V^T) * P_h); dO [B*T, d] is the gradient of
// the head-concatenated attention output, and its rows whose v_in is 0 are never read
template <typename E>
int attention_relevance_step(int B, int T, int h, int dh, const E* qkv, const E* dout, const float* v_in, float* v_out,
                             cudaStream_t st);
// v = e_0 per frame (CLS pooling) or 1/T (mean pooling)
int rollout_init(int B, int T, int has_cls, float* v, cudaStream_t st);
// dlogits fp32 [B, C] = one_hot(target[b]), or of the first maximum of logits[b] with target NULL; NaN rows for targets
// outside [0, C)
// dlogits[r] = w_k one_hot(t_b) for the n rows r = k * B + b (see relevance_seed_kernel); weight NULL: w_k = 1
int relevance_seed(int n, int B, int C, const float* logits, const int64_t* target, const float* weight, float* dlogits,
                   cudaStream_t st);
}  // namespace amc

// Host launchers of the bandwidth-bound row kernels (rowops.cu).
#pragma once
#include <algorithm>
#include <cmath>

#include "common.cuh"

namespace amc {

struct TransposeTask {
  const float* src;  // [R, C] fp32
  bf16* dst;         // [C, R] bf16
  int R, C, tile0;
};
struct TransposeBatch {
  TransposeTask t[8];
  int n;
};

// Geometry of the front end's patch map (SURVEY §8 a1-a4).
struct PatchP {
  int kind, input_layout, B, Ttok, K, in_ch, seq_len, seg, img_h, img_w, patch;
  float mean[2], inv_std[2];
};
PatchP make_patchp(const AmcDesc& D, int Ttok, int K);

// The one definition of the patch map: element k of token t of frame b in the embedding GEMM's A operand is the sample
// at the returned offset of the caller's input.  *ch is the dataset channel whose z-score the front end applies
// (dataset layout), -1 in model layout.  patchify_kernel reads through it and the input-gradient scatter writes through
// it, so the forward map and its inverse cannot drift apart.  Patches never overlap (stride = kernel size).
__device__ __forceinline__ size_t patch_src_offset(const PatchP& p, int b, int t, int k, int* ch) {
  if (p.kind == AMC_KIND_RAWIQ) {
    const int c = k / p.seg, s = k - c * p.seg;
    const int pos = t * p.seg + s;
    if (p.input_layout == AMC_INPUT_MODEL) {
      *ch = -1;
      return ((size_t)b * p.in_ch + c) * p.seq_len + pos;
    }
    *ch = c;
    return ((size_t)b * p.seq_len + pos) * 2 + c;  // dataset.py:215-222
  }
  const int pp = p.patch * p.patch, wp = p.img_w / p.patch;
  const int c = k / pp, rem = k - c * pp, r = rem / p.patch, cc = rem - r * p.patch;
  const int ph = t / wp, pw = t - ph * wp;
  const int y = ph * p.patch + r, x = pw * p.patch + cc;
  if (p.input_layout == AMC_INPUT_MODEL) {
    *ch = -1;
    return (((size_t)b * p.in_ch + c) * p.img_h + y) * p.img_w + x;
  }
  // V/dataloader/dataset.py:216-224: image = cat(I, Q).view(1, H, W)
  const int L = p.img_h * p.img_w / 2, f = y * p.img_w + x;
  const int chan = f >= L ? 1 : 0, n = f - chan * L;
  *ch = chan;
  return ((size_t)b * L + n) * 2 + chan;
}

// floats of one input frame in either layout; when the patches do not tile it (an image side that is not a multiple of
// the patch size) the uncovered samples get no gradient
inline int64_t frame_floats(const AmcDesc& D) {
  return (int64_t)D.in_ch * (D.kind == AMC_KIND_RAWIQ ? D.seq_len : (int64_t)D.img_h * D.img_w);
}

template <typename E>
int ln_fwd(int M, int d, const float* u, const float* gamma, const float* beta, float eps, E* y16, float* y32,
           E* xhat, float* rstd, cudaStream_t st);
template <typename E>
int ln_bwd(int M, int d, const float* dy, const E* xhat, const float* rstd, const float* gamma, E* du16,
           float* du32, float* dgamma, float* dbeta, float* dbias /* += column sums of du16, nullable */,
           const DropoutCfg& drop, uint32_t site, cudaStream_t st);
template <typename E>
int colsum(int M, int N, const E* X, int ld, float* out, cudaStream_t st);
template <typename E>
int patchify(const AmcDesc& D, int Ttok, int K, const float* src, E* A, cudaStream_t st);
// inverse of patchify for gradients: dsrc[map(row, k)] = dX[row, k] (* 1/std_c in dataset layout); every element of
// dsrc is written (uncovered samples are zeroed)
int patch_scatter(const AmcDesc& D, int Ttok, int K, const float* dX, float* dsrc, cudaStream_t st);
template <typename E>
int cls_rows(int B, int T, int d, const float* cls, const float* pos, E* y16, float* y32, const DropoutCfg& drop,
             cudaStream_t st);
int cls_grad(int B, int T, int d, const float* dx0, float* dcls, const DropoutCfg& drop, cudaStream_t st);
template <typename E>
int gather_tok_rows(int B, int T, int Ttok, int d, int has_cls, const float* dx0, E* out, const DropoutCfg& drop,
                    cudaStream_t st);
int head_fwd(int B, int T, int d, int C, int has_cls, int head_ln, float eps, const float* x, const float* lnw,
             const float* lnb, const float* W, const float* bias, float* logits, float* s_hl, float* s_xhat,
             float* s_rstd, cudaStream_t st);
// dW == NULL: only dxL (the parameter outputs dW, dbias, dlnw, dlnb are all skipped)
int head_bwd(int B, int T, int d, int C, int has_cls, int head_ln, const float* dlogits, const float* W,
             const float* lnw, const float* s_hl, const float* s_xhat, const float* s_rstd, float* dhl_scratch,
             float* dxL, float* dW, float* dbias, float* dlnw, float* dlnb, cudaStream_t st);
int argmax_rows(int B, int C, const float* logits, int64_t* out, cudaStream_t st);
int ce_loss(int B, int C, const float* logits, const int64_t* labels, float ls, float grad_scale, float loss_scale,
            float* dlogits, float* stats, cudaStream_t st);
int cast_blob(int64_t n, const float* src, bf16* dst, cudaStream_t st);
int transpose_batch(TransposeBatch& tb, cudaStream_t st);
int iq_stats(int64_t n_pairs, const float* x, double* acc, cudaStream_t st);
int adamw_clip_dev(int64_t n, float* p, float* g, float* m, float* v, float lr, float b1, float b2, float eps, float wd,
                   float max_norm, float grad_scale, uint32_t* step_counter, float* ws, cudaStream_t st);
int adamw_clip(int64_t n, float* p, float* g, float* m, float* v, float lr, float b1, float b2, float eps, float wd,
               float max_norm, float grad_scale, int64_t step, float* ws, cudaStream_t st);

}  // namespace amc

/*
 * amc_b200.h -- C ABI of the B200-native (sm_100a) transformer-encoder hot path of
 * aliftffd/ViT-vs-Raw-IQ.
 *
 * The reference has no FFI layer: its operator API for this path is the nn.Module surface
 * (SURVEY.md §8b).  This library sits *behind* that surface: the Python host mirror
 * (vit-vs-raw-iq_b200/) keeps the reference's two AMCTransformer classes, forward() and
 * state_dict keys, and reaches the kernels through the entry points below with ctypes.CDLL
 * (no libtorch linkage, plain pointers and sizes only).  Each entry point cites the
 * reference code it replaces; paths are relative to Transformer_Thesis/, R/ =
 * transformer_rawIQ/, V/ = ViT/.
 *
 * Conventions
 *   - every call returns int: 0 = ok, <0 = invalid argument / unsupported shape,
 *     >0 = cudaError_t.  amc_last_error() gives the thread-local message.  There is NO
 *     fallback path: an unsupported configuration is an error.
 *   - all device work is asynchronous on the given cudaStream_t (pass torch's current
 *     stream).  The library never allocates device memory: the caller owns params, grads,
 *     workspace and outputs.  Device pointers must be 16-byte aligned.
 *   - no per-call global state; calls on different streams / threads are independent.
 *   - dtype selects the arithmetic: AMC_F32 = fp32 storage + fp32 FMA GEMMs (the 1e-4
 *     parity mode); AMC_BF16 = bf16 GEMM operands on tcgen05 tensor cores with fp32
 *     accumulation, fp32 residual stream, fp32 LayerNorm/softmax statistics.
 */
#ifndef AMC_B200_H_
#define AMC_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AMC_ABI_VERSION 7

enum { AMC_KIND_RAWIQ = 0, AMC_KIND_VIT = 1 };
enum { AMC_F32 = 0, AMC_BF16 = 1 };
enum { AMC_INPUT_MODEL = 0,   /* [B,C,L] (raw-IQ) or [B,C,H,W] (ViT), already normalised: what
                                 AMCTransformer.forward receives (R/models/transformer_rawIQ.py:72,
                                 V/models/amc_transformer.py:26) */
       AMC_INPUT_RAW = 1 };   /* [B,L,2] interleaved I/Q as stored in the dataset (HDF5 'X'),
                                 normalised + framed inside the front-end kernel
                                 (R/dataloader/dataset.py:215-222, V/dataloader/dataset.py:211-224) */

typedef void* amc_stream_t;   /* cudaStream_t */

/* Static description of one call.  Mirrors the constructor kwargs of the two reference
 * AMCTransformer classes (R/models/transformer_rawIQ.py:14-26, V/models/amc_transformer.py:9). */
typedef struct AmcDesc {
  int32_t kind;          /* AMC_KIND_* */
  int32_t dtype;         /* AMC_F32 | AMC_BF16 */
  int32_t B;             /* frames in this call */
  int32_t d;             /* d_model (multiple of 32, <= 512) */
  int32_t h;             /* n_head (d % h == 0) */
  int32_t F;             /* ffn_hidden */
  int32_t C;             /* num_classes (<= 64) */
  int32_t n_layers;
  int32_t in_ch;         /* 2 raw-IQ / 1 ViT */
  int32_t seq_len;       /* raw-IQ samples per frame; the SPS mode picks 1024 or 2048 */
  int32_t seg;           /* raw-IQ segment size (1 for embedding_type='conv1d') */
  int32_t img_h, img_w, patch;   /* ViT */
  int32_t has_cls;       /* 1 = CLS token prepended; 0 = mean-pool head (raw-IQ use_cls_token=False) */
  int32_t head_ln;       /* 1 = LayerNorm(1e-5)+Linear head (raw-IQ); 0 = Linear head (ViT) */
  int32_t input_layout;  /* AMC_INPUT_* */
  int32_t training;      /* 1 = keep activations for amc_model_bwd */
  float   p_drop;        /* dropout probability applied in this call (encoder_layer.py:12,16; encoder.py:84);
                            pass 0 for module.eval().  The keep test runs on 16-bit hash fields: the effective probability is
                            floor(p * 65536) / 65536, survivors are scaled by 1 / (1 - that), and p < 2^-16 means no dropout */
  float   ln_eps;        /* 1e-12 (layers_norm.py:5) */
  float   head_ln_eps;   /* 1e-5  (nn.LayerNorm default) */
  float   norm[4];       /* i_mean, i_std, q_mean, q_std for AMC_INPUT_RAW */
  uint64_t seed;         /* dropout: counter-based RNG key */
  uint64_t offset;       /* dropout: per-step counter */
  const uint32_t* step_counter;  /* device memory or NULL: its value is added to `offset` on the device, so one captured
                                    CUDA graph of a training step draws fresh masks on every replay (the counter is advanced by
                                    amc_adamw_clip_step_graph) */
} AmcDesc;

/* Offsets (in floats) of every parameter inside the flat fp32 parameter blob.  The same
 * layout is used for the gradient blob and the AdamW moment blobs.  Keys follow the
 * reference state_dict (SURVEY §8b).  w_q/w_k/w_v (and their biases) are adjacent so the
 * fused QKV projection reads one [3d,d] matrix while state_dict keeps three tensors (D2). */
typedef struct AmcParamLayout {
  int64_t total;                 /* floats in the blob (multiple of 64) */
  int64_t emb_w, emb_b;          /* encoder.{sequence,patch}_embedding.projection.{weight,bias} */
  int64_t cls;                   /* encoder.cls_token (-1 when absent) */
  int64_t layer0, layer_stride;  /* first encoder layer, distance between layers */
  /* offsets relative to the start of a layer */
  int64_t wq, wk, wv, bq, bk, bv, wo, bo, g1, be1, w1, b1, w2, b2, g2, be2;
  int64_t head_ln_w, head_ln_b;  /* mlp_head.0.{weight,bias} (-1 for ViT) */
  int64_t head_w, head_b;        /* mlp_head.1.* (raw-IQ) / mlp_head.* (ViT) */
  int32_t T, Ttok, K_embed;      /* derived: tokens incl. CLS, embedded tokens, im2col width */
  int32_t pad_;
} AmcParamLayout;

typedef struct AmcWorkspaceInfo {
  size_t bytes;          /* workspace for one amc_model_fwd (+ matching amc_model_bwd) */
  size_t saved_bytes;    /* part of it that must survive until backward */
} AmcWorkspaceInfo;

int         amc_abi_version(void);
const char* amc_last_error(void);

/* Validates the description (same checks and messages as the reference constructors:
 * R/models/encoder.py:45-48,57; R/training/train.py:132-133) and fills the layout. */
int amc_param_layout(const AmcDesc* desc, AmcParamLayout* out);
int amc_model_workspace(const AmcDesc* desc, AmcWorkspaceInfo* out);

/* ---- whole-path calls -------------------------------------------------------------- */

/* AMCTransformer.forward (R/models/transformer_rawIQ.py:72-98 -> R/models/encoder.py:86-117;
 * V/models/amc_transformer.py:26-31 -> V/models/encoder.py:34-53).
 *   src      device, fp32, layout per desc->input_layout
 *   params   flat fp32 blob (amc_param_layout)
 *   pos      encoder.positional_encoding.encoding buffer [>=T, d] fp32 (read, never regenerated: D10)
 *   logits   [B,C] fp32 out (may be NULL when only enc_out is wanted)
 *   enc_out  [B,T,d] fp32 out or NULL  (Encoder.forward result) */
int amc_model_fwd(const AmcDesc* desc, const float* src, const float* params, const float* pos,
                  void* workspace, float* logits, float* enc_out, amc_stream_t stream);

/* Autograd of the above (SURVEY Appendix B).  Gradients are ACCUMULATED into `grads`
 * (same layout as params; zero it for a fresh step).  Stages let a data-parallel caller
 * overlap the all-reduce of finished gradient slices with the rest of backward:
 *   stage 0 = head, stage 1..n_layers = encoder layers n_layers-1 .. 0, stage n_layers+1 =
 *   embedding front end.  Call with [stage_begin, stage_end) in increasing order.
 *   dlogits  [B,C] fp32 (NULL allowed when denc_out is given)
 *   denc_out [B,T,d] fp32 or NULL (gradient w.r.t. enc_out) */
int amc_model_bwd(const AmcDesc* desc, const float* src, const float* params, void* workspace,
                  const float* dlogits, const float* denc_out, float* grads,
                  int stage_begin, int stage_end, amc_stream_t stream);

/* The same backward with the gradient w.r.t. the input frames (saliency maps, FGSM/PGD adversarial examples and
 * adversarial training on a trained classifier): autograd of R/models/embedding/patch_embedding.py:47-60,
 * V/models/embedding/patch_embedding.py:11-15 and, for AMC_INPUT_RAW, R/dataloader/dataset.py:215-222.
 * amc_model_bwd(...) is amc_model_bwd_ex(..., grads, NULL, ...).
 *   grads  as above, or NULL: no parameter gradients at all (a frozen model).  Only the data-gradient chain runs: no
 *          weight-gradient GEMMs, no bias / LayerNorm / CLS / head parameter sums.  The data gradients are bit-identical
 *          to a run with grads (that chain has no atomics).
 *   dsrc   NULL, or the gradient w.r.t. src, written by stage n_layers+1: fp32, the shape and layout of src as
 *          desc->input_layout defines it ([B,C,L] / [B,C,H,W], or [B,L,2] w.r.t. the UN-normalised dataset frames, i.e.
 *          chained through the fused z-score, 1/std per channel, and the framing).  Overwritten, not accumulated; every
 *          element is written (samples no patch covers get 0).  The CLS token and the positional encoding contribute
 *          nothing to it.
 *   grads and dsrc may not both be NULL. */
int amc_model_bwd_ex(const AmcDesc* desc, const float* src, const float* params, void* workspace,
                     const float* dlogits, const float* denc_out,
                     float* grads, float* dsrc,
                     int stage_begin, int stage_end, amc_stream_t stream);

/* nn.CrossEntropyLoss(label_smoothing) + argmax statistics (R/training/train.py:260,274-277,504).
 *   stats[0] += sum of per-frame losses * loss_scale, stats[1] += #correct (fp32 accumulators)
 *   dlogits = (softmax - smoothed one-hot) * grad_scale   (grad_scale = 1/global_batch)
 *   labels: device int64 [B].  A label outside [0, C) -- where the reference raises -- makes that frame's loss NaN, so
 *   stats[0] is NaN from then on and the host mirror raises when it reads the statistics; that frame is not counted in
 *   stats[1] and its dlogits row uses the all-smoothing target (softmax - ls/C) * grad_scale.
 *   dlogits and stats may each be NULL. */
int amc_ce_loss(int B, int C, const float* logits, const int64_t* labels, float label_smoothing,
                float grad_scale, float loss_scale, float* dlogits, float* stats, amc_stream_t stream);

/* Predicted class per frame: out[b] = index of the first maximum of logits[b, :] (R/training/utils.py:311-317
 * `outputs.max(1)`; V/training/utils.py the same).  logits fp32 [B, C], out device int64 [B]. */
int amc_argmax(int B, int C, const float* logits, int64_t* out, amc_stream_t stream);

/* Zero `bytes` bytes of device memory on `stream` (optimizer.zero_grad() of R/training/train.py:258 for the flat gradient
 * blob; a memset node when captured into a CUDA graph). */
int amc_zero(void* p, size_t bytes, amc_stream_t stream);

/* clip_grad_norm_(max_norm) + AdamW.step fused over the flat blobs (R/training/train.py:266-271,506-511).
 * grads are first multiplied by grad_scale (1/world_size after an all-reduce SUM).  norm_ws: >= 2 floats
 * of device scratch; with clipping (max_norm > 0) the call zeroes it and norm_ws[1] holds the pre-clip global norm of
 * grad_scale * grads afterwards.  max_norm <= 0 disables clipping: no norm is computed and norm_ws is neither read
 * nor written. */
int amc_adamw_clip_step(int64_t n, float* params, float* grads, float* exp_avg, float* exp_avg_sq,
                        float lr, float beta1, float beta2, float eps, float weight_decay,
                        float max_norm, float grad_scale, int64_t step, float* norm_ws,
                        amc_stream_t stream);

/* The same update with the step number kept on the DEVICE: step = *step_counter + 1 is read by the kernels (AdamW bias
 * corrections) and the counter is incremented at the end, so the call -- and the whole training step around it -- can be
 * captured once in a CUDA graph and replayed (R/training/train.py:258-271 at the reference's batch of 256 frames is
 * launch-bound otherwise). */
int amc_adamw_clip_step_graph(int64_t n, float* params, float* grads, float* exp_avg, float* exp_avg_sq,
                              float lr, float beta1, float beta2, float eps, float weight_decay,
                              float max_norm, float grad_scale, uint32_t* step_counter, float* norm_ws,
                              amc_stream_t stream);

/* Dataset-level normalisation statistics on the device (R/dataloader/dataset.py:115-157): for interleaved
 * frames x [n_frames, frame_len, 2] fp32, acc4 (device, fp64, zeroed by the caller) += {sum I, sum I^2, sum Q,
 * sum Q^2}.  mean = s/n, unbiased std = sqrt((ss - s^2/n)/(n-1)), floored at 1e-8 like the reference. */
int amc_iq_stats(int64_t n_frames, int64_t frame_len, const float* x, double* acc4, amc_stream_t stream);

/* ---- operator-level calls (used by the block tests; the whole-path calls are built from
 *      the same kernels) ------------------------------------------------------------- */

/* D[M,N] = op(A) * op(B)^T (+bias[N]) (+res32) (relu) ; dtype AMC_F32: A,B,D16 are fp32;
 * AMC_BF16: A,B,D16 are bf16, accumulation fp32 on tcgen05.
 *   transA=0: A is [M,K] row-major (lda); transA=1: A is [K,M] row-major (weight/activation gradients)
 *   transB=0: B is [N,K] row-major (nn.Linear weight layout); transB=1: B is [K,N] row-major
 *   D16 (dtype, may be NULL), D32 (fp32, may be NULL); accumulate!=0: D32 += (atomic, split-K allowed)
 * Replaces every nn.Linear on the path (multi_head_attention.py:18,28; position_wise_feed_forward.py:13,16). */
int amc_gemm(int dtype, int M, int N, int K, const void* A, int lda, int transA, const void* B, int ldb,
             int transB, const float* bias, const float* res32, int ldres, int relu, void* D16, int ldd16,
             float* D32, int ldd32, int accumulate, amc_stream_t stream);

/* bf16 GEMM with the fused post-LN epilogue used by the encoder block (encoder_layer.py:24-25,32-33):
 *   u = A B^T + bias + res32 ; y = gamma * (u - mean) / sqrt(var + eps) + beta over each row (N <= 256, N % 32 == 0)
 *   y16 (bf16), y32 (fp32), xhat (bf16, nullable), rstd (fp32 [M], nullable). */
int amc_gemm_ln(int M, int N, int K, const void* A, int lda, const void* B, int ldb, const float* bias,
                const float* res32, const float* gamma, const float* beta, float eps, void* y16, float* y32,
                void* xhat, float* rstd, amc_stream_t stream);
/* bf16 GEMM whose epilogue applies the ReLU(+dropout) backward mask taken from the stored hidden activations
 * (position_wise_feed_forward.py:14-15 backward): D16 = (A B^T) * (mask > 0 ? mask_scale : 0). */
int amc_gemm_relu_mask(int M, int N, int K, const void* A, int lda, const void* B, int ldb, const void* mask,
                       float mask_scale, void* D16, amc_stream_t stream);

/* softmax(q k^T / sqrt(dh)) v for every (frame, head); qkv is [B*T, 3d] (q | k | v column blocks,
 * head hh = columns hh*dh..), out is [B*T, d] with heads concatenated
 * (multi_head_attention.py:34-47 + scale_dot_product_attention.py:26-37; mask is always None). */
/*   lse  (nullable, fp32 [B, h, T]): log2-domain softmax row statistics max*c + log2(sum), c = log2(e)/sqrt(dh);
 *        written by the forward when given (training) and read by the backward together with `out`.
 *   out / lse may be NULL in backward for T <= 288 (P is then recomputed with its row statistics by the SIMT kernels --
 *        a convenience form, several times slower than the training path that passes them);
 *   dbias (nullable, fp32 [3d]): += column sums of dqkv = gradients of the q | k | v biases. */
int amc_attention_fwd(int dtype, int B, int T, int h, int dh, const void* qkv, void* out, float* lse,
                      amc_stream_t stream);
int amc_attention_bwd(int dtype, int B, int T, int h, int dh, const void* qkv, const void* out, const float* lse,
                      const void* dout, void* dqkv, float* dbias, amc_stream_t stream);

/* The same attention restricted to query row 0 of every frame, bf16, head dim 16 / 32 / 64: what the TOP encoder layer
 * of a CLS-pooled model needs, since only `x[:, 0]` feeds the classifier head (R/models/transformer_rawIQ.py:88-90,
 * V/models/amc_transformer.py:29).  fwd writes row 0 of every frame of `out` ([B*T, d], other rows untouched);
 * bwd reads row 0 of every frame of `dout` and writes all of dqkv (dq of the other rows is exactly zero);
 * dbias (nullable, fp32 [3d]) += q | k | v bias gradients (the k part is exactly zero). */
int amc_attention_cls_fwd(int B, int T, int h, int dh, const void* qkv, void* out, amc_stream_t stream);
int amc_attention_cls_bwd(int B, int T, int h, int dh, const void* qkv, const void* dout, void* dqkv, float* dbias,
                          amc_stream_t stream);

/* y = gamma * (u - mean) / sqrt(var_biased + eps) + beta over the last dim (layers_norm.py:11-19).
 *   u fp32 [M,d]; y16 (dtype) / y32 (fp32) / xhat (dtype) / rstd (fp32 [M]) may each be NULL. */
int amc_layernorm_fwd(int dtype, int M, int d, const float* u, const float* gamma, const float* beta, float eps,
                      void* y16, float* y32, void* xhat, float* rstd, amc_stream_t stream);
/* du = rstd * (g - mean(g) - xhat * mean(g*xhat)), g = dy*gamma; dgamma += sum dy*xhat; dbeta += sum dy. */
int amc_layernorm_bwd(int dtype, int M, int d, const float* dy, const void* xhat, const float* rstd,
                      const float* gamma, void* du16, float* du32, float* dgamma, float* dbeta,
                      amc_stream_t stream);

/* Embedding front end: normalise (AMC_INPUT_RAW) + frame + patchify + embedding GEMM + bias + CLS row +
 * positional encoding -> x0 [B,T,d] fp32 (R/models/encoder.py:100-111 with
 * R/models/embedding/patch_embedding.py:47-60; V/models/encoder.py:38-47 with V/.../patch_embedding.py:11-15). */
int amc_frontend_fwd(const AmcDesc* desc, const float* src, const float* emb_w, const float* emb_b,
                     const float* cls, const float* pos, void* scratch, size_t scratch_bytes, float* x0,
                     amc_stream_t stream);

/* ---- in-situ kernel timing (measurement only) ------------------------------------------
 * When enabled, every launch site inside the library is bracketed by CUDA events on the launch
 * stream.  amc_profile_dump synchronises the device and writes one line per kernel class:
 *   "<class> <launches> <total_ms> <algorithmic_flops> <algorithmic_bytes>\n", then clears the records. */
long long amc_launch_count(void);   /* kernels launched by the library so far (this process) */
int amc_profile_enable(int on);
int amc_profile_dump(char* buf, size_t cap);

#ifdef __cplusplus
}
#endif
#endif /* AMC_B200_H_ */

// C ABI (include/amc_b200.h): parameter layout, workspace carving and the whole-path
// forward / backward built from the kernels in this directory.
#include <stdarg.h>

#include <vector>

#include "attention.cuh"
#include "gemm_common.cuh"
#include "profile.cuh"
#include "rowops.cuh"

namespace amc {

std::atomic<long long> g_launch_count{0};
static thread_local char g_err[512] = "";
void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

namespace {

#define AMC_PROF(name, flops, bytes, expr)      \
  do {                                        \
    ProfScope ps__(name, st, flops, bytes);   \
    AMC_TRY(expr);                            \
  } while (0)

__global__ void add_inplace_kernel(size_t n, float* __restrict__ a, const float* __restrict__ b) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    a[i] += b[i];
}

// dst[b * ld + c] += src[b * d + c]
__global__ void add_rows_kernel(int B, int d, float* __restrict__ dst, int ld, const float* __restrict__ src) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * d) return;
  const int b = i / d, c = i - b * d;
  dst[(size_t)b * ld + c] += src[i];
}

struct Dims {
  int B, T, Ttok, K, d, h, dh, F, C, L, has_cls;
  int64_t M;  // B*T token rows
};

int validate(const AmcDesc& D, Dims& m) {
  AMC_CHECK_ARG(D.kind == AMC_KIND_RAWIQ || D.kind == AMC_KIND_VIT, "unknown model kind %d", D.kind);
  AMC_CHECK_ARG(D.dtype == AMC_F32 || D.dtype == AMC_BF16, "unknown dtype %d", D.dtype);
  AMC_CHECK_ARG(D.B >= 0, "batch must be >= 0");
  AMC_CHECK_ARG(D.d >= 1 && D.d <= 512, "d_model=%d unsupported (1..512)", D.d);
  AMC_CHECK_ARG(D.h >= 1 && D.d % D.h == 0, "d_model (%d) must be divisible by n_head (%d)", D.d, D.h);
  AMC_CHECK_ARG(D.d / D.h <= 128, "head dim %d unsupported (<= 128)", D.d / D.h);
  AMC_CHECK_ARG(D.F >= 1 && D.C >= 1 && D.C <= 64 && D.n_layers >= 0, "bad ffn_hidden/num_classes/n_layers");
  AMC_CHECK_ARG(D.input_layout == AMC_INPUT_MODEL || D.input_layout == AMC_INPUT_RAW, "bad input_layout");
  AMC_CHECK_ARG(D.p_drop >= 0.f && D.p_drop < 1.f, "drop_prob must be in [0,1)");
  m.B = D.B; m.d = D.d; m.h = D.h; m.dh = D.d / D.h; m.F = D.F; m.C = D.C; m.L = D.n_layers;
  if (D.kind == AMC_KIND_RAWIQ) {
    AMC_CHECK_ARG(D.in_ch >= 1 && D.seq_len >= 1 && D.seg >= 1, "bad raw-IQ geometry");
    // R/models/encoder.py:45-48
    AMC_CHECK_ARG(D.seq_len % D.seg == 0, "seq_length (%d) must be divisible by segment_size (%d)", D.seq_len,
                  D.seg);
    AMC_CHECK_ARG(D.input_layout == AMC_INPUT_MODEL || D.in_ch == 2, "raw interleaved input needs in_channels=2");
    m.Ttok = D.seq_len / D.seg;
    m.K = D.in_ch * D.seg;
    m.has_cls = D.has_cls ? 1 : 0;
  } else {
    AMC_CHECK_ARG(D.in_ch >= 1 && D.patch >= 1 && D.img_h >= D.patch && D.img_w >= D.patch, "bad ViT geometry");
    AMC_CHECK_ARG(D.input_layout == AMC_INPUT_MODEL || (D.in_ch == 1 && (D.img_h * D.img_w) % 2 == 0),
                  "raw interleaved input needs in_channels=1 and an even image");
    m.Ttok = (D.img_h / D.patch) * (D.img_w / D.patch);
    m.K = D.in_ch * D.patch * D.patch;
    m.has_cls = 1;
  }
  m.T = m.Ttok + m.has_cls;
  AMC_CHECK_ARG(m.T <= ATTN_LONG_MAX_T, "T=%d tokens per frame unsupported (<= %d)", m.T, ATTN_LONG_MAX_T);
  if (D.dtype == AMC_BF16) {
    // (a patch width that is not a multiple of 8 -- conv1d embedding, K = 2 -- runs the small-K kernels)
    AMC_CHECK_ARG(D.d % 8 == 0 && D.F % 8 == 0 && (m.K % 8 == 0 || embed_smallk_supported(m.K)),
                  "bf16 path needs d_model and ffn_hidden multiples of 8 and a patch width (%d) that is a multiple "
                  "of 8 or at most 16", m.K);
  }
  if (D.p_drop > 0.f)
    AMC_CHECK_ARG(D.d % 4 == 0 && D.F % 4 == 0, "dropout needs d_model and ffn_hidden multiples of 4");
  m.M = (int64_t)m.B * m.T;
  AMC_CHECK_ARG(m.M * (int64_t)std::max(3 * m.d, m.F) < (int64_t)1 << 40, "problem too large");
  return 0;
}

inline int64_t up64(int64_t v) { return (v + 63) / 64 * 64; }

int make_layout(const AmcDesc& D, const Dims& m, AmcParamLayout& L) {
  int64_t o = 0;
  auto take = [&](int64_t n) { int64_t r = o; o += up64(n); return r; };
  const int64_t d = m.d, F = m.F;
  L.emb_w = take(d * m.K);
  L.emb_b = take(d);
  L.cls = m.has_cls ? take(d) : -1;
  L.layer0 = o;
  int64_t lo = 0;
  auto ltake = [&](int64_t n) { int64_t r = lo; lo += up64(n); return r; };
  // q,k,v adjacent -> one [3d,d] matrix and one [3d] bias (d*d and d are padded only when not %64:
  // adjacency must be exact, so these six are NOT individually padded)
  L.wq = lo; L.wk = lo + d * d; L.wv = lo + 2 * d * d; lo = up64(lo + 3 * d * d);
  L.bq = lo; L.bk = lo + d; L.bv = lo + 2 * d; lo = up64(lo + 3 * d);
  L.wo = ltake(d * d); L.bo = ltake(d);
  L.g1 = ltake(d); L.be1 = ltake(d);
  L.w1 = ltake(F * d); L.b1 = ltake(F);
  L.w2 = ltake(d * F); L.b2 = ltake(d);
  L.g2 = ltake(d); L.be2 = ltake(d);
  L.layer_stride = lo;
  o += lo * m.L;
  if (D.head_ln) { L.head_ln_w = take(d); L.head_ln_b = take(d); } else { L.head_ln_w = L.head_ln_b = -1; }
  L.head_w = take((int64_t)m.C * d);
  L.head_b = take(m.C);
  L.total = o;
  L.T = m.T; L.Ttok = m.Ttok; L.K_embed = m.K; L.pad_ = 0;
  return 0;
}

// ---- workspace ----------------------------------------------------------------------------
struct LayerBuf {
  void *qkv, *o, *xhat1, *x1_16, *hid, *xhat2;
  float *rstd1, *x1_32, *rstd2;
  float* lse;   // [B, h, T] softmax row statistics (training, bf16 tile attention)
};
struct Work {
  bf16* w16 = nullptr;   // bf16 copy of the parameter blob
  bf16* wT = nullptr;    // per layer: wqkvT [d,3d] | woT [d,d] | w1T [d,F] | w2T [F,d]
  int64_t wT_stride = 0;
  void* Apatch = nullptr;
  std::vector<void*> x16;     // L+1 (training) or 2 (inference, ping-pong)
  std::vector<float*> x32;
  std::vector<LayerBuf> lay;  // L (training) or 1
  float *u32, *hl, *hxhat, *hrstd, *dhl;
  // compact [B, .] buffers of the top layer when only its CLS rows are live (see Model::cls_top)
  struct Cls {
    void *x1_16, *hid, *xhat1, *xhat2, *y16, *dw16, *da, *du16;
    float *x1_32, *rstd1, *rstd2, *y32, *u32, *dy32, *dw32, *t32, *du32;
  } c;
  // backward scratch
  float *dy32, *dw32, *t32, *du32;
  void *dw16, *da, *du16, *dO, *dqkv, *demb;
  // input gradient: dX [B*Ttok, K] fp32 and (bf16) W_emb^T [K, d]
  float* dx = nullptr;
  bf16* wembT = nullptr;
  size_t bytes = 0;
};

template <typename E>
void carve(const AmcDesc& D, const Dims& m, const AmcParamLayout& L, char* base, Work& w) {
  size_t off = 0;
  auto take = [&](size_t bytes) -> char* {
    char* p = base ? base + off : nullptr;
    off += align_up(bytes, 256);
    return p;
  };
  const bool bf = D.dtype == AMC_BF16;
  const size_t M = (size_t)m.M, d = m.d, F = m.F, e = sizeof(E);
  if (bf) {
    w.w16 = (bf16*)take((size_t)L.total * 2);
    if (D.training) {
      w.wT_stride = (int64_t)(3 * d * d + d * d + 2 * d * F);
      w.wT = (bf16*)take((size_t)w.wT_stride * m.L * 2);
    }
  }
  w.Apatch = take((size_t)m.B * m.Ttok * m.K * e);
  const int nx = D.training ? m.L + 1 : 2;
  w.x16.resize(nx);
  w.x32.resize(nx);
  for (int i = 0; i < nx; ++i) {
    w.x16[i] = take(M * d * e);
    w.x32[i] = bf ? (float*)take(M * d * 4) : (float*)w.x16[i];
  }
  const int nl = D.training ? m.L : 1;
  w.lay.resize(std::max(nl, 1));
  for (int i = 0; i < (int)w.lay.size(); ++i) {
    LayerBuf& b = w.lay[i];
    b.qkv = take(M * 3 * d * e);
    b.o = take(M * d * e);
    b.x1_16 = take(M * d * e);
    b.x1_32 = bf ? (float*)take(M * d * 4) : (float*)b.x1_16;
    b.hid = take(M * F * e);
    if (D.training) {
      b.xhat1 = take(M * d * e);
      b.xhat2 = take(M * d * e);
      b.rstd1 = (float*)take(M * 4);
      b.rstd2 = (float*)take(M * 4);
      b.lse = (float*)take(M * m.h * 4);
    } else {
      b.xhat1 = b.xhat2 = nullptr;
      b.rstd1 = b.rstd2 = nullptr;
      b.lse = nullptr;
    }
  }
  w.u32 = (float*)take(M * d * 4);
  w.hl = (float*)take((size_t)m.B * d * 4);
  w.hxhat = (float*)take((size_t)m.B * d * 4);
  w.hrstd = (float*)take((size_t)m.B * 4);
  w.dhl = (float*)take((size_t)m.B * d * 4);
  {
    const size_t Bq = (size_t)m.B;
    w.c.x1_16 = take(Bq * d * e);
    w.c.x1_32 = bf ? (float*)take(Bq * d * 4) : (float*)w.c.x1_16;
    w.c.hid = take(Bq * F * e);
    w.c.y16 = take(Bq * d * e);
    w.c.y32 = bf ? (float*)take(Bq * d * 4) : (float*)w.c.y16;
    w.c.u32 = (float*)take(Bq * d * 4);
    w.c.xhat1 = D.training ? take(Bq * d * e) : nullptr;
    w.c.xhat2 = D.training ? take(Bq * d * e) : nullptr;
    w.c.rstd1 = D.training ? (float*)take(Bq * 4) : nullptr;
    w.c.rstd2 = D.training ? (float*)take(Bq * 4) : nullptr;
    if (D.training) {
      w.c.dy32 = (float*)take(Bq * d * 4);
      w.c.dw32 = (float*)take(Bq * d * 4);
      w.c.t32 = (float*)take(Bq * d * 4);
      w.c.du32 = (float*)take(Bq * d * 4);
      w.c.dw16 = take(Bq * d * e);
      w.c.da = take(Bq * F * e);
      w.c.du16 = take(Bq * d * e);
    }
  }
  if (D.training) {
    const size_t dead0 = off;   // dy32 .. dqkv: layer-gradient scratch, dead once stage n_layers+1 has gathered demb
    w.dy32 = (float*)take(M * d * 4);
    w.dw32 = (float*)take(M * d * 4);
    w.t32 = (float*)take(M * d * 4);
    w.du32 = (float*)take(M * d * 4);
    w.dw16 = take(M * d * e);
    w.da = take(M * F * e);
    w.du16 = take(M * d * e);
    w.dO = take(M * d * e);
    w.dqkv = take(M * 3 * d * e);
    // the input gradient's dX and W_emb^T live in that scratch; a buffer of their own only where the patches outgrow it
    // (patch width K well above d * T / Ttok), so the workspace of every geometry that fits is unchanged
    const size_t dx_bytes = align_up((size_t)m.B * m.Ttok * m.K * 4, 256);
    const size_t need = dx_bytes + (bf ? (size_t)m.K * d * 2 : 0);
    char* dx = need <= off - dead0 ? (base ? base + dead0 : nullptr) : take(need);
    w.dx = (float*)dx;
    w.wembT = bf && dx ? (bf16*)(dx + dx_bytes) : nullptr;
    w.demb = take((size_t)m.B * m.Ttok * d * e);
  }
  w.bytes = off;
}

// algorithmic traffic of one GEMM call: operands once, outputs once, residual / mask once
template <typename E> double gemm_bytes(const GemmArgs& g) {
  const double e = sizeof(E), MN = (double)g.M * g.N;
  double b = ((double)g.M * g.K + (double)g.N * g.K) * e;
  if (g.epi.D16) b += MN * e;
  if (g.epi.D32) b += MN * 4 * (g.epi.accumulate ? 2 : 1);
  if (g.epi.res32) b += MN * 4;
  if (g.epi.mask_src) b += MN * e;
  if (g.epi.ln_xhat) b += MN * e;
  return b;
}
template <typename E> int gemm_impl(const GemmArgs& g, cudaStream_t st);
template <> int gemm_impl<float>(const GemmArgs& g, cudaStream_t st) { return gemm_f32(g, st); }
template <> int gemm_impl<bf16>(const GemmArgs& g, cudaStream_t st) { return gemm_bf16(g, st); }
template <typename E> int gemm(const GemmArgs& g, cudaStream_t st) {
  ProfScope ps(g.name, st, 2.0 * g.M * g.N * g.K, gemm_bytes<E>(g));
  return gemm_impl<E>(g, st);
}

inline int pick_split_k(int Mo, int No, int K) {
  const int tiles = ceil_div(Mo, 128) * ceil_div(No, 128);
  int s = std::max(1, (148 * 2) / std::max(tiles, 1));
  // tokens per split: every split pays a full tile of fp32 atomics, so short K ranges (small batches) take fewer splits
  static const int min_k = [] { const char* e = getenv("AMC_WGRAD_MIN_K"); return e ? std::max(64, atoi(e)) : 256; }();
  s = std::min(s, std::max(1, K / min_k));
  return s;
}

template <typename E>
struct Model {
  const AmcDesc& D;
  Dims m;
  AmcParamLayout L;
  Work w;
  const float* params;
  cudaStream_t st;
  DropoutCfg drop;
  float* grads = nullptr;   // backward: parameter-gradient blob, NULL = input gradient only

  Model(const AmcDesc& D_, const float* params_, cudaStream_t st_) : D(D_), params(params_), st(st_) {}

  int init(void* workspace) {
    AMC_TRY(validate(D, m));
    AMC_TRY(make_layout(D, m, L));
    AMC_CHECK_ARG(workspace != nullptr || m.B == 0, "workspace is NULL");
    AMC_CHECK_ARG((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "workspace must be 256-byte aligned");
    carve<E>(D, m, L, (char*)workspace, w);
    drop = make_dropout(D.p_drop, D.seed, D.offset, true, D.step_counter);
    return 0;
  }
  // fp32 parameter inside the blob
  const float* P(int64_t off) const { return params + off; }
  const float* PL(int l, int64_t off) const { return params + L.layer0 + (int64_t)l * L.layer_stride + off; }
  // GEMM-operand view of a weight matrix (element type E)
  const E* WL(int l, int64_t off) const {
    const int64_t o = L.layer0 + (int64_t)l * L.layer_stride + off;
    if (sizeof(E) == 2) return reinterpret_cast<const E*>(w.w16 + o);
    return reinterpret_cast<const E*>(params + o);
  }
  const E* Wemb() const {
    if (sizeof(E) == 2) return reinterpret_cast<const E*>(w.w16 + L.emb_w);
    return reinterpret_cast<const E*>(params + L.emb_w);
  }
  const LayerBuf& LB(int l) const { return w.lay[D.training ? l : 0]; }
  // gradient slots (NULL when no parameter gradients are wanted: every parameter output then takes its null path)
  float* GP(int64_t off) const { return grads ? grads + off : nullptr; }
  float* GL(int l, int64_t off) const { return grads ? grads + L.layer0 + (int64_t)l * L.layer_stride + off : nullptr; }
  // (amc_gemm_ln also takes 256 < N <= 512 -- one single-buffered 512-column accumulator -- but measured inside the d512 L12
  //  step it loses to GEMM + ln_fwd: 4.97 vs 4.54 ms per step for the two LayerNorm sites, the epilogue of a tile no longer
  //  overlapping the next tile's main loop; the model path therefore fuses up to d = 256 only)
  bool fuse_ln() const { return sizeof(E) == 2 && m.d % 32 == 0 && m.d <= 256; }
  int xi(int l) const { return D.training ? l : (l & 1); }

  // bf16 copy of the blob; with `dgrad_operands` also the transposed weights the backward's dgrad GEMMs read
  int pack_weights(bool dgrad_operands) {
    if (sizeof(E) != 2) return 0;
    AMC_PROF("pack_weights", 0.0, (double)L.total * 6, cast_blob(L.total, params, w.w16, st));
    if (!dgrad_operands) return 0;
    const int64_t d = m.d, F = m.F;
    TransposeBatch tb;
    tb.n = 0;
    for (int l = 0; l < m.L; ++l) {
      bf16* t = w.wT + (int64_t)l * w.wT_stride;
      tb.t[tb.n++] = {PL(l, L.wq), t, (int)(3 * d), (int)d, 0};                       // [3d,d] -> [d,3d]
      tb.t[tb.n++] = {PL(l, L.wo), t + 3 * d * d, (int)d, (int)d, 0};                 // [d,d]  -> [d,d]
      tb.t[tb.n++] = {PL(l, L.w1), t + 4 * d * d, (int)F, (int)d, 0};                 // [F,d]  -> [d,F]
      tb.t[tb.n++] = {PL(l, L.w2), t + 4 * d * d + d * F, (int)d, (int)F, 0};         // [d,F]  -> [F,d]
      if (tb.n == 8 || l == m.L - 1) {
        AMC_PROF("pack_weights", 0.0, 0.0, transpose_batch(tb, st));
        tb.n = 0;
      }
    }
    return 0;
  }

  int frontend(const float* src, const float* pos) {
    if (m.B == 0) return 0;
    GemmArgs g;
    g.M = m.B * m.Ttok; g.N = m.d; g.K = m.K;
    g.A = w.Apatch; g.lda = m.K;
    g.B = Wemb(); g.ldb = m.K;
    g.name = "gemm_embed";
    g.epi.bias = P(L.emb_b);
    g.epi.pos = pos;
    g.epi.map_Ttok = m.Ttok; g.epi.map_T = m.T; g.epi.map_cls = m.has_cls;
    g.epi.drop = drop; g.epi.drop_site = site_pe();
    g.epi.D16 = w.x16[0]; g.epi.ldd16 = m.d;
    if (sizeof(E) == 2) { g.epi.D32 = w.x32[0]; g.epi.ldd32 = m.d; }
    bool fused = false;
    if (sizeof(E) == 2) {
      // one kernel: IQ samples -> normalise / frame / patchify in shared memory -> tcgen05 GEMM -> +bias +PE, dropout
      bf16* aout = D.training ? reinterpret_cast<bf16*>(w.Apatch) : nullptr;
      AMC_TRY(frontend_fused(D, m.Ttok, m.K, src, reinterpret_cast<const bf16*>(Wemb()), g.epi, aout, true, &fused, st));
      if (fused) {
        const double by = (double)m.B * m.Ttok * m.K * 4 + (double)g.M * m.d * 6 + (D.training ? (double)g.M * m.K * 2 : 0.0);
        ProfScope ps("frontend_fused", st, 2.0 * g.M * g.N * g.K, by);
        AMC_TRY(frontend_fused(D, m.Ttok, m.K, src, reinterpret_cast<const bf16*>(Wemb()), g.epi, aout, false, &fused, st));
      }
    }
    if (!fused) {
      AMC_PROF("patchify", 0.0, (double)m.B * m.Ttok * m.K * (4 + sizeof(E)), patchify<E>(D, m.Ttok, m.K, src, (E*)w.Apatch, st));
      if (sizeof(E) == 2 && m.K % 8 != 0) {
        AMC_PROF("embed_smallk", 2.0 * g.M * g.N * g.K, (double)g.M * (m.K * 2 + m.d * 6),
                 embed_smallk_fwd(g.M, g.N, g.K, (const bf16*)w.Apatch, (const bf16*)Wemb(), g.epi, st));
      } else {
        AMC_TRY(gemm<E>(g, st));
      }
    }
    if (m.has_cls)
      AMC_PROF("cls_rows", 0.0, 0.0, cls_rows<E>(m.B, m.T, m.d, P(L.cls), pos, (E*)w.x16[0], sizeof(E) == 2 ? w.x32[0] : nullptr, drop, st));
    return 0;
  }

  // The rows a layer's post-attention half (out-proj, norm1, FFN, norm2) works on.  Normally all M = B*T token
  // rows; for the top layer of a CLS-pooled model only the B CLS rows feed the head, so that half runs on a
  // B-row view (attention output and residual read with row pitch T*d, everything else compact).
  struct Rows {
    int n;                                  // rows
    const void* o; int ldo;                 // attention output rows
    const float* xres; int ldxres;          // fp32 residual of the layer input
    const void* xin16; int ldxin;           // layer input rows (weight gradient of nothing here; kept for clarity)
    void *x1_16, *hid, *xhat1, *xhat2, *y16;
    float *x1_32, *rstd1, *rstd2, *y32, *u32;
    // backward
    float *dy32, *dw32, *t32, *du32;
    void *dw16, *da, *du16;
    void* dO; int lddO;                     // where the out-proj input gradient goes (row pitch)
  };
  Rows all_rows(int l) {
    const LayerBuf& b = LB(l);
    Rows r;
    r.n = (int)m.M; r.o = b.o; r.ldo = m.d; r.xres = w.x32[xi(l)]; r.ldxres = m.d;
    r.xin16 = w.x16[xi(l)]; r.ldxin = m.d;
    r.x1_16 = b.x1_16; r.hid = b.hid; r.xhat1 = b.xhat1; r.xhat2 = b.xhat2; r.y16 = w.x16[xi(l + 1)];
    r.x1_32 = b.x1_32; r.rstd1 = b.rstd1; r.rstd2 = b.rstd2; r.y32 = w.x32[xi(l + 1)]; r.u32 = w.u32;
    r.dy32 = w.dy32; r.dw32 = w.dw32; r.t32 = w.t32; r.du32 = w.du32;
    r.dw16 = w.dw16; r.da = w.da; r.du16 = w.du16; r.dO = w.dO; r.lddO = m.d;
    return r;
  }
  Rows cls_rows_view(int l) {
    const LayerBuf& b = LB(l);
    const int Td = m.T * m.d;
    Rows r;
    r.n = m.B; r.o = b.o; r.ldo = Td; r.xres = w.x32[xi(l)]; r.ldxres = Td;
    r.xin16 = w.x16[xi(l)]; r.ldxin = Td;
    r.x1_16 = w.c.x1_16; r.hid = w.c.hid; r.xhat1 = w.c.xhat1; r.xhat2 = w.c.xhat2; r.y16 = w.c.y16;
    r.x1_32 = w.c.x1_32; r.rstd1 = w.c.rstd1; r.rstd2 = w.c.rstd2; r.y32 = w.c.y32; r.u32 = w.c.u32;
    r.dy32 = w.c.dy32; r.dw32 = w.c.dw32; r.t32 = w.c.t32; r.du32 = w.c.du32;
    r.dw16 = w.c.dw16; r.da = w.c.da; r.du16 = w.c.du16; r.dO = w.dO; r.lddO = Td;
    return r;
  }

  // fused QKV projection (one [3d,d] weight: three adjacent state_dict tensors, multi_head_attention.py:18)
  // + attention over all rows
  // the top layer of a CLS-pooled model needs attention for query row 0 only (attn_cls.cu)
  // (T <= 16 stays on the warp-per-(frame, head) tensor-core kernel, which is already at its HBM floor there)
  bool cls_attn() const { return sizeof(E) == 2 && m.T > 16 && attn_cls_supported(m.T, m.h, m.dh) && (m.d % 8) == 0; }

  int qkv_fwd(int l) {
    const int d = m.d;
    GemmArgs g;
    g.M = (int)m.M; g.N = 3 * d; g.K = d; g.A = w.x16[xi(l)]; g.lda = d; g.B = WL(l, L.wq); g.ldb = d;
    g.name = "gemm_qkv";
    g.epi.bias = PL(l, L.bq); g.epi.D16 = LB(l).qkv; g.epi.ldd16 = 3 * d;
    return gemm<E>(g, st);
  }

  int attn_fwd_part(int l, bool cls_only = false) {
    const int M = (int)m.M, d = m.d;
    const LayerBuf& b = LB(l);
    AMC_TRY(qkv_fwd(l));
    if (cls_only && cls_attn()) {
      ProfScope ps("attn_cls_fwd", st, 4.0 * m.M * d, (double)M * 2 * d * sizeof(E));
      AMC_TRY(attn_cls_fwd(m.B, m.T, m.h, m.dh, (const bf16*)b.qkv, (bf16*)b.o, st));
      return 0;
    }
    ProfScope ps("attn_fwd", st, 4.0 * m.M * m.T * d, (double)M * 4 * d * sizeof(E));
    AMC_TRY(attention_fwd<E>(m.B, m.T, m.h, m.dh, (const E*)b.qkv, (E*)b.o, b.lse, st));
    return 0;
  }

  int post_fwd_part(int l, const Rows& r) {
    const int d = m.d, F = m.F, Mr = r.n;
    GemmArgs g;
    // out-proj + dropout1 + residual -> u ; norm1 (encoder_layer.py:24-25)
    g.M = Mr; g.N = d; g.K = d; g.A = r.o; g.lda = r.ldo; g.B = WL(l, L.wo); g.ldb = d;
    g.name = "gemm_outproj";
    g.epi.bias = PL(l, L.bo); g.epi.drop = drop; g.epi.drop_site = site_attn(l);
    g.epi.res32 = r.xres; g.epi.ldres = r.ldxres;
    if (fuse_ln()) {   // bias + dropout + residual + LayerNorm inside the GEMM epilogue (row-owned in TMEM)
      g.name = "gemm_outproj_ln";
      g.epi.ln_gamma = PL(l, L.g1); g.epi.ln_beta = PL(l, L.be1); g.epi.ln_eps = D.ln_eps;
      g.epi.D16 = r.x1_16; g.epi.ldd16 = d; g.epi.D32 = r.x1_32; g.epi.ldd32 = d;
      g.epi.ln_xhat = r.xhat1; g.epi.ln_rstd = r.rstd1;
      AMC_TRY(gemm<E>(g, st));
    } else {
      g.epi.D32 = r.u32; g.epi.ldd32 = d;
      AMC_TRY(gemm<E>(g, st));
      AMC_PROF("ln_fwd", 0.0, (double)Mr * d * (8 + 2 * sizeof(E)),
               ln_fwd<E>(Mr, d, r.u32, PL(l, L.g1), PL(l, L.be1), D.ln_eps, (E*)r.x1_16,
                         sizeof(E) == 2 ? r.x1_32 : nullptr, (E*)r.xhat1, r.rstd1, st));
    }
    // FFN (position_wise_feed_forward.py:12-17): linear1 + ReLU + dropout
    g = GemmArgs();
    g.M = Mr; g.N = F; g.K = d; g.A = r.x1_16; g.lda = d; g.B = WL(l, L.w1); g.ldb = d;
    g.name = "gemm_ffn1";
    g.epi.bias = PL(l, L.b1); g.epi.relu = 1; g.epi.drop = drop; g.epi.drop_site = site_hidden(l);
    g.epi.D16 = r.hid; g.epi.ldd16 = F;
    AMC_TRY(gemm<E>(g, st));
    // linear2 + dropout2 + residual -> u ; norm2 (encoder_layer.py:32-33)
    g = GemmArgs();
    g.M = Mr; g.N = d; g.K = F; g.A = r.hid; g.lda = F; g.B = WL(l, L.w2); g.ldb = F;
    g.name = "gemm_ffn2";
    g.epi.bias = PL(l, L.b2); g.epi.drop = drop; g.epi.drop_site = site_ffn(l);
    g.epi.res32 = r.x1_32; g.epi.ldres = d;
    if (fuse_ln()) {
      g.name = "gemm_ffn2_ln";
      g.epi.ln_gamma = PL(l, L.g2); g.epi.ln_beta = PL(l, L.be2); g.epi.ln_eps = D.ln_eps;
      g.epi.D16 = r.y16; g.epi.ldd16 = d; g.epi.D32 = r.y32; g.epi.ldd32 = d;
      g.epi.ln_xhat = r.xhat2; g.epi.ln_rstd = r.rstd2;
      AMC_TRY(gemm<E>(g, st));
    } else {
      g.epi.D32 = r.u32; g.epi.ldd32 = d;
      AMC_TRY(gemm<E>(g, st));
      AMC_PROF("ln_fwd", 0.0, (double)Mr * d * (8 + 2 * sizeof(E)),
               ln_fwd<E>(Mr, d, r.u32, PL(l, L.g2), PL(l, L.be2), D.ln_eps, (E*)r.y16,
                         sizeof(E) == 2 ? r.y32 : nullptr, (E*)r.xhat2, r.rstd2, st));
    }
    return 0;
  }

  int layer_fwd(int l, bool cls_only) {
    AMC_TRY(attn_fwd_part(l, cls_only));
    return post_fwd_part(l, cls_only ? cls_rows_view(l) : all_rows(l));
  }

  int forward(const float* src, const float* pos, float* logits, float* enc_out) {
    if (m.B == 0) return 0;
    AMC_TRY(pack_weights(D.training));
    AMC_TRY(frontend(src, pos));
    return forward_layers(logits, enc_out);
  }
  // the encoder layers and the head, from the x0 rows in w.x16[0] / w.x32[0] (the weights packed)
  int forward_layers(float* logits, float* enc_out) {
    // Only the CLS rows of the top layer reach the head (transformer_rawIQ.py:88-90, amc_transformer.py:29): when
    // just the logits are wanted, the top layer's out-proj / FFN / LayerNorms run on those B rows alone.
    const bool cls_top = m.has_cls && logits && !enc_out && m.L >= 1;
    for (int l = 0; l < m.L; ++l) AMC_TRY(layer_fwd(l, cls_top && l == m.L - 1));
    const float* xL = cls_top ? w.c.y32 : w.x32[xi(m.L)];
    const int headT = cls_top ? 1 : m.T;
    if (enc_out)
      AMC_CUDA(cudaMemcpyAsync(enc_out, xL, (size_t)m.M * m.d * 4, cudaMemcpyDeviceToDevice, st));
    if (logits)
      AMC_PROF("head", 0.0, 0.0, head_fwd(m.B, headT, m.d, m.C, m.has_cls, D.head_ln, D.head_ln_eps, xL,
                       D.head_ln ? P(L.head_ln_w) : nullptr, D.head_ln ? P(L.head_ln_b) : nullptr, P(L.head_w),
                       P(L.head_b), logits, w.hl, w.hxhat, w.hrstd, st));
    return 0;
  }

  // Attention maps (amc_model_attention): every layer below the top on all rows, and of the top layer only its QKV
  // projection on all rows (no CLS-row top layer: its maps need every row; nothing reads its attention output, FFN or
  // norms), then the probabilities of the masked layers and the rollout from layer L-1 down to 0.  No backward follows,
  // so the transposed dgrad weights are not packed.  The training-mode carve keeps every
  // layer's qkv; the rollout ping-pongs between `rollout` and w.u32 ([M, d] fp32, dead once the forward is done), started
  // so that the last step lands in `rollout`.
  int attention(const float* src, const float* pos, uint32_t mask, float* probs, float* rollout) {
    AMC_CHECK_ARG(D.training == 1 && D.p_drop == 0.f, "amc_model_attention needs desc.training=1 and desc.p_drop=0");
    AMC_CHECK_ARG(mask != 0 || rollout, "amc_model_attention: empty layer_mask and no rollout");
    AMC_CHECK_ARG(m.L >= 32 || (mask >> m.L) == 0, "amc_model_attention: layer_mask 0x%x names a layer >= n_layers (%d)",
                  mask, m.L);
    AMC_CHECK_ARG(mask == 0 || probs, "amc_model_attention: probs is NULL");
    if (m.B == 0) return 0;
    AMC_TRY(pack_weights(false));
    AMC_TRY(frontend(src, pos));
    for (int l = 0; l + 1 < m.L; ++l) AMC_TRY(layer_fwd(l, false));
    if (m.L >= 1) AMC_TRY(qkv_fwd(m.L - 1));
    const size_t per = (size_t)m.B * m.h * m.T * m.T;
    const double s_flops = 2.0 * m.M * m.T * m.d, qk_bytes = (double)m.M * 2 * m.d * sizeof(E);
    float* out = probs;
    for (int l = 0; l < m.L && l < 32; ++l) {
      if (!((mask >> l) & 1u)) continue;
      AMC_PROF("attn_probs", s_flops, qk_bytes + 4.0 * per,
               attention_probs<E>(m.B, m.T, m.h, m.dh, (const E*)LB(l).qkv, out, st));
      out += per;
    }
    if (rollout) {
      float* v[2] = {rollout, w.u32};
      int cur = m.L & 1;
      AMC_PROF("attn_rollout", 0.0, (double)m.M * 4, rollout_init(m.B, m.T, m.has_cls, v[cur], st));
      for (int l = m.L - 1; l >= 0; --l, cur ^= 1)
        AMC_PROF("attn_rollout", 2.0 * s_flops, qk_bytes + (double)m.M * 8,
                 attention_rollout_step<E>(m.B, m.T, m.h, m.dh, (const E*)LB(l).qkv, v[cur], v[cur ^ 1], st));
    }
    return 0;
  }

  // Class-specific relevance (amc_model_relevance): the forward of forward() with logits, the one-hot dlogits of the
  // target (or argmax) class, then the frozen backward (grads = NULL) from the head down, with one relevance step on each
  // layer's attention-output gradient dO_l as layer_bwd_out leaves it.  Layer 0's attention backward, dgrad QKV and the
  // front end would only feed layers below it, so they do not run.  The vector ping-pongs between `relevance` and w.u32,
  // and the one-hot dlogits sit in w.u32 behind it: w.u32 ([M, d] fp32) is forward scratch that no backward kernel
  // writes (post_bwd_part, layer_bwd_attn and the head backward use dy32 / dw32 / t32 / du32 and their CLS-view copies).
  int relevance(const float* src, const float* pos, const int64_t* target, float* logits, float* relevance) {
    AMC_CHECK_ARG(D.training == 1 && D.p_drop == 0.f, "amc_model_relevance needs desc.training=1 and desc.p_drop=0");
    AMC_CHECK_ARG(logits && relevance, "amc_model_relevance: logits or relevance is NULL");
    AMC_CHECK_ARG(m.L >= 1, "amc_model_relevance: the model has no encoder layer");
    if (m.B == 0) return 0;
    const size_t vn = align_up((size_t)m.M, 64);
    AMC_CHECK_ARG(vn + (size_t)m.B * m.C <= m.M * (size_t)m.d, "amc_model_relevance: scratch too small");
    AMC_TRY(forward(src, pos, logits, nullptr));
    float* dlogits = w.u32 + vn;
    AMC_PROF("relevance", 0.0, 0.0, relevance_seed(m.B, m.B, m.C, logits, target, nullptr, dlogits, st));
    AMC_TRY(backward(dlogits, nullptr, nullptr, nullptr, 0, 1));   // head
    const bool cls_top = m.has_cls;                                 // forward() ran with logits: mirrors its choice
    float* v[2] = {relevance, w.u32};
    int cur = m.L & 1;
    AMC_PROF("relevance", 0.0, (double)m.M * 4, rollout_init(m.B, m.T, m.has_cls, v[cur], st));
    const double s_flops = 2.0 * m.M * m.T * m.d, qkv_bytes = (double)m.M * 3 * m.d * sizeof(E);
    for (int l = m.L - 1; l >= 0; --l, cur ^= 1) {
      const bool cls_only = cls_top && l == m.L - 1;
      AMC_TRY(layer_bwd_out(l, cls_only));
      AMC_PROF("relevance", 3.0 * s_flops, qkv_bytes + (double)m.M * m.d * sizeof(E) + (double)m.M * 8,
               attention_relevance_step<E>(m.B, m.T, m.h, m.dh, (const E*)LB(l).qkv, (const E*)w.dO, v[cur],
                                           v[cur ^ 1], st));
      if (l > 0) AMC_TRY(layer_bwd_attn(l, cls_only));
    }
    return 0;
  }

  // ---- backward ---------------------------------------------------------------------------
  // weight-gradient GEMM: dW[No, Ki] += dY[M, No]^T X[M, Ki]
  // ... and db[No] += column sums of dY: inside the same kernel on the bf16 path, a colsum launch in fp32
  int wgrad(int No, int Ki, const void* dY, int ldy, const void* X, int ldx, float* dW, float* db) {
    if (!dW) return 0;
    if (db && sizeof(E) != 2) AMC_PROF("colsum", 0.0, 0.0, colsum<E>((int)m.M, No, (const E*)dY, ldy, db, st));
    GemmArgs g;
    if (sizeof(E) == 2) g.epi.colsum_out = db;
    g.M = No; g.N = Ki; g.K = (int)m.M;
    g.A = dY; g.lda = ldy; g.transA = 1;
    g.B = X; g.ldb = ldx; g.transB = 1;
    g.split_k = pick_split_k(No, Ki, g.K);
    g.name = "gemm_wgrad";
    g.epi.D32 = dW; g.epi.ldd32 = Ki; g.epi.accumulate = 1;
    return gemm<E>(g, st);
  }
  // activation-gradient GEMM: dX[M, Ki] = dY[M, No] W[No, Ki]; the bf16 path reads the pre-transposed copy
  void dgrad_operand(GemmArgs& g, int l, int64_t woff, int64_t wT_off, int No, int Ki) {
    if (sizeof(E) == 2) {
      g.B = w.wT + (int64_t)l * w.wT_stride + wT_off;  // [Ki, No]
      g.ldb = No; g.transB = 0;
    } else {
      g.B = PL(l, woff);                                // [No, Ki] read as [K=No, N=Ki]
      g.ldb = Ki; g.transB = 1;
    }
  }

  // wgrad with an explicit token count (the CLS view has B token rows)
  int wgrad_n(int Ktok, int No, int Ki, const void* dY, int ldy, const void* X, int ldx, float* dW, float* db) {
    if (!dW) return 0;
    if (db && sizeof(E) != 2) AMC_PROF("colsum", 0.0, 0.0, colsum<E>(Ktok, No, (const E*)dY, ldy, db, st));
    GemmArgs g;
    if (sizeof(E) == 2) g.epi.colsum_out = db;
    g.M = No; g.N = Ki; g.K = Ktok;
    g.A = dY; g.lda = ldy; g.transA = 1;
    g.B = X; g.ldb = ldx; g.transB = 1;
    g.split_k = pick_split_k(No, Ki, g.K);
    g.name = "gemm_wgrad";
    g.epi.D32 = dW; g.epi.ldd32 = Ki; g.epi.accumulate = 1;
    return gemm<E>(g, st);
  }

  // With fuse_ln(), LayerNorm backward runs in the epilogue of the dgrad GEMM that produces the gradient of the norm's
  // output: dgrad FFN1 for norm1, and for norm2 of layer l the dgrad QKV of layer l + 1.  The top layer's norm2 takes its
  // output gradient from the head (or denc_out) and keeps the separate ln_bwd.
  bool ln2_bwd_fused(int l) const { return fuse_ln() && l < m.L - 1; }
  // ... the epilogue: norm (gamma at goff, beta at boff) of layer l with its saved xhat / rstd, dropout `site` on du16,
  // and dbias (offset dboff) += column sums of du16: the bias gradient of the sub-layer whose output the norm took
  void ln_bwd_epilogue(GemmArgs& g, int l, const void* xhat, const float* rstd, int64_t goff, int64_t boff, int64_t dboff,
                       uint32_t site, void* du16, float* du32) {
    g.epi.ln_bwd = 1;
    g.epi.ln_xhat = const_cast<void*>(xhat); g.epi.ln_rstd = const_cast<float*>(rstd); g.epi.ln_gamma = PL(l, goff);
    g.epi.ln_dgamma = GL(l, goff); g.epi.ln_dbeta = GL(l, boff); g.epi.colsum_out = GL(l, dboff);
    g.epi.drop = drop; g.epi.drop_site = site;
    g.epi.D16 = du16; g.epi.ldd16 = m.d; g.epi.D32 = du32; g.epi.ldd32 = m.d;
  }

  // backward of post_fwd_part on the same row view: consumes r.dy32 (or, when the dgrad QKV of layer l + 1 has done
  // norm2's backward, r.dw16 / r.dw32; only on all rows, the CLS view being the top layer's), leaves the out-proj input gradient in r.dO (row pitch r.lddO) and the skip
  // gradient of the layer input in r.du32
  int post_bwd_part(int l, const Rows& r) {
    const int d = m.d, F = m.F, Mr = r.n;
    const int64_t dd = (int64_t)d * d;
    GemmArgs g;
    // norm2 backward; dw16 carries dropout2's mask (operand of the FFN2 gradients), dw32 is the skip path
    if (!ln2_bwd_fused(l))
      AMC_PROF("ln_bwd", 0.0, (double)Mr * d * (8 + 2 * sizeof(E)),
               ln_bwd<E>(Mr, d, r.dy32, (const E*)r.xhat2, r.rstd2, PL(l, L.g2), (E*)r.dw16, r.dw32, GL(l, L.g2),
                         GL(l, L.be2), GL(l, L.b2), drop, site_ffn(l), st));
    AMC_TRY(wgrad_n(Mr, d, F, r.dw16, d, r.hid, F, GL(l, L.w2), nullptr));
    // dgrad FFN2 with the ReLU/dropout mask taken from the stored hidden
    g.M = Mr; g.N = F; g.K = d; g.A = r.dw16; g.lda = d;
    dgrad_operand(g, l, L.w2, 4 * dd + (int64_t)d * F, d, F);
    g.name = "gemm_dgrad_ffn2";
    g.epi.mask_src = r.hid; g.epi.ldmask = F; g.epi.mask_scale = drop.scale;
    g.epi.D16 = r.da; g.epi.ldd16 = F;
    const bool fuse_db1 = sizeof(E) == 2 && F % 32 == 0 && F <= 2048;   // bias gradient summed in the mask epilogue
    if (fuse_db1) g.epi.colsum_out = GL(l, L.b1);
    AMC_TRY(gemm<E>(g, st));
    AMC_TRY(wgrad_n(Mr, F, d, r.da, F, r.x1_16, d, GL(l, L.w1), fuse_db1 ? nullptr : GL(l, L.b1)));
    // dgrad FFN1 + skip -> gradient w.r.t. x1
    g = GemmArgs();
    g.M = Mr; g.N = d; g.K = F; g.A = r.da; g.lda = F;
    dgrad_operand(g, l, L.w1, 4 * dd, F, d);
    g.name = "gemm_dgrad_ffn1";
    g.epi.res32 = r.dw32; g.epi.ldres = d;
    if (fuse_ln()) {   // + norm1 backward
      g.name = "gemm_dgrad_ffn1_lnb";
      ln_bwd_epilogue(g, l, r.xhat1, r.rstd1, L.g1, L.be1, L.bo, site_attn(l), r.du16, r.du32);
      AMC_TRY(gemm<E>(g, st));
    } else {
      g.epi.D32 = r.t32; g.epi.ldd32 = d;
      AMC_TRY(gemm<E>(g, st));
      // norm1 backward
      AMC_PROF("ln_bwd", 0.0, (double)Mr * d * (8 + 2 * sizeof(E)),
               ln_bwd<E>(Mr, d, r.t32, (const E*)r.xhat1, r.rstd1, PL(l, L.g1), (E*)r.du16, r.du32, GL(l, L.g1),
                         GL(l, L.be1), GL(l, L.bo), drop, site_attn(l), st));
    }
    AMC_TRY(wgrad_n(Mr, d, d, r.du16, d, r.o, r.ldo, GL(l, L.wo), nullptr));
    g = GemmArgs();
    g.M = Mr; g.N = d; g.K = d; g.A = r.du16; g.lda = d;
    dgrad_operand(g, l, L.wo, 3 * dd, d, d);
    g.name = "gemm_dgrad_outproj";
    g.epi.D16 = r.dO; g.epi.ldd16 = r.lddO;
    AMC_TRY(gemm<E>(g, st));
    return 0;
  }

  int layer_bwd(int l, bool cls_only) {
    AMC_TRY(layer_bwd_out(l, cls_only));
    return layer_bwd_attn(l, cls_only);
  }
  // the first half of layer_bwd: leaves the attention-output gradient in w.dO
  int layer_bwd_out(int l, bool cls_only) {
    if (cls_only) {
      // every non-CLS row of the attention-output gradient is exactly zero (the CLS-row kernel never reads them)
      if (!cls_attn()) AMC_CUDA(cudaMemsetAsync(w.dO, 0, (size_t)m.M * m.d * sizeof(E), st));
      return post_bwd_part(l, cls_rows_view(l));
    }
    return post_bwd_part(l, all_rows(l));
  }
  // the second half: attention backward, dgrad QKV and the skip path into the gradient of the layer input
  int layer_bwd_attn(int l, bool cls_only) {
    const int M = (int)m.M, d = m.d;
    const LayerBuf& b = LB(l);
    const bool cls_kernel = cls_only && cls_attn();
    if (cls_kernel) {
      ProfScope ps("attn_cls_bwd", st, 10.0 * m.M * d, (double)M * 5 * d * sizeof(E));
      AMC_TRY(attn_cls_bwd(m.B, m.T, m.h, m.dh, (const bf16*)b.qkv, (const bf16*)w.dO, (bf16*)w.dqkv, GL(l, L.bq), st));
    } else {
      ProfScope ps("attn_bwd", st, 10.0 * m.M * m.T * d, (double)M * 7 * d * sizeof(E));
      AMC_TRY(attention_bwd<E>(m.B, m.T, m.h, m.dh, (const E*)b.qkv, (const E*)b.o, b.lse, (const E*)w.dO, (E*)w.dqkv, GL(l, L.bq), st));
    }
    AMC_TRY(wgrad(3 * d, d, w.dqkv, 3 * d, w.x16[l], d, GL(l, L.wq), nullptr));
    // dgrad QKV + skip -> gradient w.r.t. the layer input
    GemmArgs g;
    g.M = M; g.N = d; g.K = 3 * d; g.A = w.dqkv; g.lda = 3 * d;
    dgrad_operand(g, l, L.wq, 0, 3 * d, d);
    g.name = "gemm_dgrad_qkv";
    if (l > 0 && ln2_bwd_fused(l - 1)) {
      // + norm2 backward of layer l - 1: its dw16 / dw32 are written here
      if (cls_only) {   // the skip gradient exists on the CLS rows only: spread it over a zeroed full-size residual
        AMC_CUDA(cudaMemsetAsync(w.du32, 0, (size_t)M * d * 4, st));
        add_rows_kernel<<<ceil_div(m.B * d, 256), 256, 0, st>>>(m.B, d, w.du32, m.T * d, w.c.du32);
        AMC_LAUNCH_CHECK();
      }
      const LayerBuf& bp = LB(l - 1);
      g.name = "gemm_dgrad_qkv_lnb";
      g.epi.res32 = w.du32; g.epi.ldres = d;
      ln_bwd_epilogue(g, l - 1, bp.xhat2, bp.rstd2, L.g2, L.be2, L.b2, site_ffn(l - 1), w.dw16, w.dw32);
      return gemm<E>(g, st);
    }
    g.epi.D32 = w.dy32; g.epi.ldd32 = d;
    if (!cls_only) { g.epi.res32 = w.du32; g.epi.ldres = d; }
    AMC_TRY(gemm<E>(g, st));
    if (cls_only) {   // the skip gradient exists on the CLS rows only
      add_rows_kernel<<<ceil_div(m.B * d, 256), 256, 0, st>>>(m.B, d, w.dy32, m.T * d, w.c.du32);
      AMC_LAUNCH_CHECK();
    }
    return 0;
  }

  // Input gradient (stage n_layers+1), autograd of the patch embedding and of the dataset z-score + framing:
  // dX = demb W_emb, then the transpose of the patch map into dsrc (caller's layout, * 1/std_c for dataset input).
  // With src and base (Integrated Gradients) every element is also multiplied by src - base.
  int input_grad(const E* demb, float* dsrc, const float* src = nullptr, const float* base = nullptr) {
    const int Mt = m.B * m.Ttok;
    const double mul_bytes = src ? 8.0 * Mt * m.K : 0.0;
    if (sizeof(E) == 2 && m.K % 8 != 0) {
      AMC_PROF("frontend_bwd_dsrc", 2.0 * Mt * m.d * m.K, (double)Mt * (m.d * 2 + m.K * 4) + mul_bytes,
               embed_smallk_dgrad(D, m.Ttok, m.d, m.K, (const bf16*)demb, (const bf16*)Wemb(), dsrc, st, src, base));
      return 0;
    }
    GemmArgs g;
    g.M = Mt; g.N = m.K; g.K = m.d;
    g.A = demb; g.lda = m.d;
    if (sizeof(E) == 2) {   // tcgen05 needs both operands K-major: W_emb [d, K] -> [K, d]
      TransposeBatch tb;
      tb.n = 1;
      tb.t[0] = {P(L.emb_w), w.wembT, m.d, m.K, 0};
      AMC_PROF("frontend_bwd_dsrc", 0.0, (double)m.d * m.K * 6, transpose_batch(tb, st));
      g.B = w.wembT; g.ldb = m.d;
    } else {
      g.B = P(L.emb_w); g.ldb = m.K; g.transB = 1;   // [d, K] read as [K=d, N=K]
    }
    g.name = "frontend_bwd_dsrc";
    g.epi.D32 = w.dx; g.epi.ldd32 = m.K;
    AMC_TRY(gemm<E>(g, st));
    AMC_PROF("frontend_bwd_dsrc", 0.0, (double)Mt * m.K * 8 + mul_bytes,
             patch_scatter(D, m.Ttok, m.K, w.dx, dsrc, st, src, base));
    return 0;
  }

  int backward(const float* dlogits, const float* denc_out, float* grads_, float* dsrc, int s0, int s1) {
    AMC_CHECK_ARG(D.training, "amc_model_bwd needs a forward run with desc.training=1");
    AMC_CHECK_ARG(0 <= s0 && s0 <= s1 && s1 <= m.L + 2, "bad stage range [%d,%d)", s0, s1);
    if (m.B == 0) return 0;
    grads = grads_;
    const size_t nx = (size_t)m.M * m.d;
    const bool cls_top = m.has_cls && dlogits && !denc_out && m.L >= 1;   // must mirror forward()
    for (int s = s0; s < s1; ++s) {
      if (s == 0) {
        AMC_CHECK_ARG(dlogits || denc_out, "amc_model_bwd: dlogits and denc_out are both NULL");
        if (dlogits) {
          AMC_PROF("head", 0.0, 0.0, head_bwd(m.B, cls_top ? 1 : m.T, m.d, m.C, m.has_cls, D.head_ln, dlogits, P(L.head_w),
                           D.head_ln ? P(L.head_ln_w) : nullptr, w.hl, w.hxhat, w.hrstd, w.dhl,
                           cls_top ? w.c.dy32 : w.dy32,
                           GP(L.head_w), GP(L.head_b), D.head_ln ? GP(L.head_ln_w) : nullptr,
                           D.head_ln ? GP(L.head_ln_b) : nullptr, st));
          if (denc_out) {
            add_inplace_kernel<<<148 * 4, 256, 0, st>>>(nx, w.dy32, denc_out);
            AMC_LAUNCH_CHECK();
          }
        } else {
          AMC_CUDA(cudaMemcpyAsync(w.dy32, denc_out, nx * 4, cudaMemcpyDeviceToDevice, st));
        }
      } else if (s <= m.L) {
        AMC_TRY(layer_bwd(m.L - s, cls_top && s == 1));
      } else {
        // embedding front end: dcls, dW_emb, db_emb (when parameter gradients are wanted) and the input gradient
        if (m.has_cls && grads) AMC_PROF("frontend_bwd_misc", 0.0, 0.0, cls_grad(m.B, m.T, m.d, w.dy32, GP(L.cls), drop, st));
        AMC_PROF("frontend_bwd_misc", 0.0, 0.0, gather_tok_rows<E>(m.B, m.T, m.Ttok, m.d, m.has_cls, w.dy32, (E*)w.demb, drop, st));
        const int Mt = m.B * m.Ttok;
        if (grads && sizeof(E) == 2 && m.K % 8 != 0) {
          AMC_PROF("embed_smallk", 2.0 * Mt * m.d * m.K, (double)Mt * (m.K + m.d) * 2,
                   embed_smallk_bwd(Mt, m.d, m.K, (const bf16*)w.demb, m.d, (const bf16*)w.Apatch, GP(L.emb_w),
                                    GP(L.emb_b), st));
        } else if (grads) {
          if (sizeof(E) != 2) AMC_PROF("colsum", 0.0, 0.0, colsum<E>(Mt, m.d, (const E*)w.demb, m.d, GP(L.emb_b), st));
          GemmArgs g;
          if (sizeof(E) == 2) g.epi.colsum_out = GP(L.emb_b);
          g.M = m.d; g.N = m.K; g.K = Mt;
          g.A = w.demb; g.lda = m.d; g.transA = 1;
          g.B = w.Apatch; g.ldb = m.K; g.transB = 1;
          g.split_k = pick_split_k(m.d, m.K, Mt);
          g.name = "gemm_wgrad";
          g.epi.D32 = GP(L.emb_w); g.epi.ldd32 = m.K; g.epi.accumulate = 1;
          AMC_TRY(gemm<E>(g, st));
        }
        if (dsrc) AMC_TRY(input_grad((const E*)w.demb, dsrc));
      }
    }
    return 0;
  }
};

template <typename E>
size_t model_ws_bytes(const AmcDesc& D, const Dims& m, const AmcParamLayout& L) {
  Work w;
  carve<E>(D, m, L, nullptr, w);
  return std::max<size_t>(w.bytes, 256);
}
size_t model_ws_bytes(const AmcDesc& D, const Dims& m, const AmcParamLayout& L) {
  return D.dtype == AMC_BF16 ? model_ws_bytes<bf16>(D, m, L) : model_ws_bytes<float>(D, m, L);
}

// ---- Integrated Gradients -----------------------------------------------------------------
// Workspace of amc_model_integrated_gradients for chunks of `chunk` path points, in order: [src; baseline] as one
// 2B-frame batch, the endpoint embeddings x0e = [x0(x); x0(x')] fp32, the fp32 sum of the token-row gradients over the
// points, its E copy (the dsrc GEMM's operand), the chunk's seed and logits, then the training-mode workspace of the
// larger of the 2B-frame endpoint forward and the chunk's chunk * B frames, which each pass carves afresh.
struct IgPlan {
  size_t src2, x0e, acc, demb, dlogits, clogits, model, bytes;
};
int ig_plan(const AmcDesc& D, int chunk, IgPlan& p) {
  Dims m;
  AmcParamLayout L;
  AMC_TRY(validate(D, m));
  AMC_TRY(make_layout(D, m, L));
  AMC_CHECK_ARG(chunk >= 1, "integrated_gradients: chunk must be >= 1");
  AMC_CHECK_ARG(std::max<int64_t>((int64_t)chunk * D.B, 2 * (int64_t)D.B) <= INT32_MAX,
                "integrated_gradients: too many frames per pass");
  AmcDesc D2 = D, Dc = D;
  D2.B = 2 * D.B;
  Dc.B = chunk * D.B;
  Dims m2, mc;
  AMC_TRY(validate(D2, m2));
  AMC_TRY(validate(Dc, mc));
  const size_t e = D.dtype == AMC_BF16 ? 2 : 4, B = D.B, tok = B * m.Ttok * m.d;
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t r = off; off += align_up(bytes, 256); return r; };
  p.src2 = take(2 * B * frame_floats(D) * 4);
  p.x0e = take(2 * B * m.T * m.d * 4);
  p.acc = take(tok * 4);
  p.demb = e == 4 ? p.acc : take(tok * e);
  p.dlogits = take((size_t)chunk * B * m.C * 4);
  p.clogits = take((size_t)chunk * B * m.C * 4);
  p.model = take(std::max(model_ws_bytes(D2, m2, L), model_ws_bytes(Dc, mc, L)));
  p.bytes = off;
  return 0;
}

// IG_t(x) = (x - x') * sum_k w_k dy_t/dx (x' + a_k (x - x')) over `steps` path points (a_k, w_k device fp32).
//  1. one forward of [x; x'] (2B frames) gives both endpoints' logits and x0 rows;
//  2. per chunk of n points: x0 rows blended in frame order k*B + b, the layers and head forward, the seed w_k e_t,
//     the frozen backward (grads = NULL) down to dx0, and the token rows of dx0 summed over the chunk's points into acc
//     (fixed order, no atomics);
//  3. once: the dsrc GEMM on that sum and the scatter multiplied by src - base.
// Each model pass carves the same region afresh; what lives across passes is in the plan's first buffers.
template <typename E>
int integrated_gradients(const AmcDesc& D, const float* src, const float* base, const float* params, const float* pos,
                         char* ws, const int64_t* target, int steps, const float* alpha, const float* weight, int chunk,
                         float* logits, float* attr, cudaStream_t st) {
  AMC_CHECK_ARG(D.training == 1 && D.p_drop == 0.f,
                "amc_model_integrated_gradients needs desc.training=1 and desc.p_drop=0");
  AMC_CHECK_ARG(steps >= 1, "amc_model_integrated_gradients: steps must be >= 1");
  IgPlan p;
  AMC_TRY(ig_plan(D, chunk, p));
  if (D.B == 0) return 0;
  AMC_CHECK_ARG(ws != nullptr && (reinterpret_cast<uintptr_t>(ws) & 255) == 0,
                "workspace is NULL or not 256-byte aligned");
  const int B = D.B;
  float* src2 = (float*)(ws + p.src2);
  float* x0e = (float*)(ws + p.x0e);
  float* acc = (float*)(ws + p.acc);
  E* demb = (E*)(ws + p.demb);
  float* dlogits = (float*)(ws + p.dlogits);
  float* clogits = (float*)(ws + p.clogits);
  const size_t nsrc = (size_t)B * frame_floats(D);
  AMC_CUDA(cudaMemcpyAsync(src2, src, nsrc * 4, cudaMemcpyDeviceToDevice, st));
  AMC_CUDA(cudaMemcpyAsync(src2 + nsrc, base, nsrc * 4, cudaMemcpyDeviceToDevice, st));
  AmcDesc D2 = D;
  D2.B = 2 * B;
  Dims m;
  {
    Model<E> me(D2, params, st);
    AMC_TRY(me.init(ws + p.model));
    AMC_TRY(me.forward(src2, pos, logits, nullptr));
    AMC_CUDA(cudaMemcpyAsync(x0e, me.w.x32[0], (size_t)me.m.M * me.m.d * 4, cudaMemcpyDeviceToDevice, st));
    m = me.m;
  }
  const int64_t n_frame = (int64_t)B * m.T * m.d;
  for (int k0 = 0; k0 < steps; k0 += chunk) {
    const int n = std::min(chunk, steps - k0);
    AmcDesc Dc = D;
    Dc.B = n * B;
    Model<E> mc(Dc, params, st);
    AMC_TRY(mc.init(ws + p.model));
    AMC_TRY(mc.pack_weights(true));
    AMC_PROF("ig_blend", 0.0, (double)n * n_frame * (4 + sizeof(E)) + 2.0 * n_frame * 4,
             ig_blend<E>(n, n_frame, alpha + k0, x0e, (E*)mc.w.x16[0], mc.w.x32[0], st));
    AMC_TRY(mc.forward_layers(clogits, nullptr));
    AMC_PROF("ig_seed", 0.0, 0.0, relevance_seed(n * B, B, m.C, logits, target, weight + k0, dlogits, st));
    AMC_TRY(mc.backward(dlogits, nullptr, nullptr, nullptr, 0, m.L + 1));
    const bool last = k0 + n >= steps;
    const double tok = (double)B * m.Ttok * m.d;
    AMC_PROF("ig_reduce", 0.0, tok * (4.0 * n + (k0 ? 8 : 4) + (last ? sizeof(E) : 0)),
             ig_reduce<E>(B, m.T, m.Ttok, m.d, m.has_cls, n, mc.w.dy32, acc, k0 == 0, last ? demb : nullptr, st));
  }
  Model<E> mb(D, params, st);
  AMC_TRY(mb.init(ws + p.model));
  AMC_TRY(mb.pack_weights(false));
  return mb.input_grad(demb, attr, src, base);
}

}  // namespace
}  // namespace amc

using namespace amc;

extern "C" {

int amc_abi_version(void) { return AMC_ABI_VERSION; }
long long amc_launch_count(void) { return g_launch_count.load(std::memory_order_relaxed); }
const char* amc_last_error(void) { return g_err; }

int amc_param_layout(const AmcDesc* desc, AmcParamLayout* out) {
  AMC_CHECK_ARG(desc && out, "NULL argument");
  Dims m;
  AMC_TRY(validate(*desc, m));
  return make_layout(*desc, m, *out);
}

int amc_model_workspace(const AmcDesc* desc, AmcWorkspaceInfo* out) {
  AMC_CHECK_ARG(desc && out, "NULL argument");
  Dims m;
  AmcParamLayout L;
  AMC_TRY(validate(*desc, m));
  AMC_TRY(make_layout(*desc, m, L));
  out->bytes = model_ws_bytes(*desc, m, L);
  out->saved_bytes = out->bytes;
  return 0;
}

int amc_model_ig_workspace(const AmcDesc* desc, int chunk, AmcWorkspaceInfo* out) {
  AMC_CHECK_ARG(desc && out, "NULL argument");
  IgPlan p;
  AMC_TRY(ig_plan(*desc, chunk, p));
  out->bytes = p.bytes;
  out->saved_bytes = p.bytes;
  return 0;
}

int amc_model_integrated_gradients(const AmcDesc* desc, const float* src, const float* baseline, const float* params,
                                   const float* pos, void* workspace, const int64_t* target, int steps,
                                   const float* alpha, const float* weight, int chunk, float* logits, float* attr,
                                   amc_stream_t stream) {
  DeviceGuard dev_guard(params);
  AMC_CHECK_ARG(desc && params && pos, "NULL argument");
  AMC_CHECK_ARG(desc->B == 0 || (src && baseline && alpha && weight && logits && attr), "NULL argument");
  cudaStream_t st = (cudaStream_t)stream;
  if (desc->dtype == AMC_BF16)
    return integrated_gradients<bf16>(*desc, src, baseline, params, pos, (char*)workspace, target, steps, alpha, weight,
                                      chunk, logits, attr, st);
  return integrated_gradients<float>(*desc, src, baseline, params, pos, (char*)workspace, target, steps, alpha, weight,
                                     chunk, logits, attr, st);
}

int amc_model_fwd(const AmcDesc* desc, const float* src, const float* params, const float* pos, void* workspace,
                  float* logits, float* enc_out, amc_stream_t stream) {
  DeviceGuard dev_guard(params);
  AMC_CHECK_ARG(desc && params && pos, "NULL argument");
  AMC_CHECK_ARG(src || desc->B == 0, "src is NULL");
  cudaStream_t st = (cudaStream_t)stream;
  if (desc->dtype == AMC_BF16) {
    Model<bf16> mdl(*desc, params, st);
    AMC_TRY(mdl.init(workspace));
    return mdl.forward(src, pos, logits, enc_out);
  }
  Model<float> mdl(*desc, params, st);
  AMC_TRY(mdl.init(workspace));
  return mdl.forward(src, pos, logits, enc_out);
}

int amc_model_bwd_ex(const AmcDesc* desc, const float* src, const float* params, void* workspace, const float* dlogits,
                     const float* denc_out, float* grads, float* dsrc, int stage_begin, int stage_end,
                     amc_stream_t stream) {
  DeviceGuard dev_guard(params);
  (void)src;   // the input gradient's shape follows from desc; the kernels never read src in backward
  AMC_CHECK_ARG(desc && params && (grads || dsrc), "NULL argument");
  cudaStream_t st = (cudaStream_t)stream;
  if (desc->dtype == AMC_BF16) {
    Model<bf16> mdl(*desc, params, st);
    AMC_TRY(mdl.init(workspace));
    return mdl.backward(dlogits, denc_out, grads, dsrc, stage_begin, stage_end);
  }
  Model<float> mdl(*desc, params, st);
  AMC_TRY(mdl.init(workspace));
  return mdl.backward(dlogits, denc_out, grads, dsrc, stage_begin, stage_end);
}

int amc_model_attention(const AmcDesc* desc, const float* src, const float* params, const float* pos, void* workspace,
                        uint32_t layer_mask, float* probs, float* rollout, amc_stream_t stream) {
  DeviceGuard dev_guard(params);
  AMC_CHECK_ARG(desc && params && pos, "NULL argument");
  AMC_CHECK_ARG(src || desc->B == 0, "src is NULL");
  cudaStream_t st = (cudaStream_t)stream;
  if (desc->dtype == AMC_BF16) {
    Model<bf16> mdl(*desc, params, st);
    AMC_TRY(mdl.init(workspace));
    return mdl.attention(src, pos, layer_mask, probs, rollout);
  }
  Model<float> mdl(*desc, params, st);
  AMC_TRY(mdl.init(workspace));
  return mdl.attention(src, pos, layer_mask, probs, rollout);
}

int amc_model_relevance(const AmcDesc* desc, const float* src, const float* params, const float* pos, void* workspace,
                        const int64_t* target, float* logits, float* relevance, amc_stream_t stream) {
  DeviceGuard dev_guard(params);
  AMC_CHECK_ARG(desc && params && pos, "NULL argument");
  AMC_CHECK_ARG(src || desc->B == 0, "src is NULL");
  cudaStream_t st = (cudaStream_t)stream;
  if (desc->dtype == AMC_BF16) {
    Model<bf16> mdl(*desc, params, st);
    AMC_TRY(mdl.init(workspace));
    return mdl.relevance(src, pos, target, logits, relevance);
  }
  Model<float> mdl(*desc, params, st);
  AMC_TRY(mdl.init(workspace));
  return mdl.relevance(src, pos, target, logits, relevance);
}

int amc_model_bwd(const AmcDesc* desc, const float* src, const float* params, void* workspace, const float* dlogits,
                  const float* denc_out, float* grads, int stage_begin, int stage_end, amc_stream_t stream) {
  AMC_CHECK_ARG(grads, "NULL argument");
  return amc_model_bwd_ex(desc, src, params, workspace, dlogits, denc_out, grads, nullptr, stage_begin, stage_end,
                          stream);
}

int amc_ce_loss(int B, int C, const float* logits, const int64_t* labels, float label_smoothing, float grad_scale,
                float loss_scale, float* dlogits, float* stats, amc_stream_t stream) {
  DeviceGuard dev_guard(logits);
  AMC_CHECK_ARG(B >= 0 && C >= 1 && logits && labels, "bad argument");
  ProfScope ps("ce_loss", (cudaStream_t)stream);
  return ce_loss(B, C, logits, labels, label_smoothing, grad_scale, loss_scale, dlogits, stats, (cudaStream_t)stream);
}

int amc_argmax(int B, int C, const float* logits, int64_t* out, amc_stream_t stream) {
  DeviceGuard dev_guard(logits);
  AMC_CHECK_ARG(B >= 0 && C >= 1 && logits && out, "bad argument");
  ProfScope ps("argmax", (cudaStream_t)stream);
  return argmax_rows(B, C, logits, out, (cudaStream_t)stream);
}

int amc_zero(void* p, size_t bytes, amc_stream_t stream) {
  DeviceGuard dev_guard(p);
  AMC_CHECK_ARG(p != nullptr || bytes == 0, "bad argument");
  if (bytes) AMC_CUDA(cudaMemsetAsync(p, 0, bytes, (cudaStream_t)stream));
  return 0;
}

int amc_adamw_clip_step(int64_t n, float* params, float* grads, float* exp_avg, float* exp_avg_sq, float lr,
                        float beta1, float beta2, float eps, float weight_decay, float max_norm, float grad_scale,
                        int64_t step, float* norm_ws, amc_stream_t stream) {
  DeviceGuard dev_guard(params);
  AMC_CHECK_ARG(n >= 0 && params && grads && exp_avg && exp_avg_sq && norm_ws, "bad argument");
  ProfScope ps("adamw_clip", (cudaStream_t)stream, 0.0, (double)n * 32);
  return adamw_clip(n, params, grads, exp_avg, exp_avg_sq, lr, beta1, beta2, eps, weight_decay, max_norm, grad_scale,
                    step, norm_ws, (cudaStream_t)stream);
}

int amc_adamw_clip_step_graph(int64_t n, float* params, float* grads, float* exp_avg, float* exp_avg_sq, float lr,
                              float beta1, float beta2, float eps, float weight_decay, float max_norm, float grad_scale,
                              uint32_t* step_counter, float* norm_ws, amc_stream_t stream) {
  DeviceGuard dev_guard(params);
  AMC_CHECK_ARG(n >= 0 && params && grads && exp_avg && exp_avg_sq && norm_ws && step_counter, "bad argument");
  ProfScope ps("adamw_clip", (cudaStream_t)stream, 0.0, (double)n * 32);
  return adamw_clip_dev(n, params, grads, exp_avg, exp_avg_sq, lr, beta1, beta2, eps, weight_decay, max_norm, grad_scale,
                        step_counter, norm_ws, (cudaStream_t)stream);
}

int amc_iq_stats(int64_t n_frames, int64_t frame_len, const float* x, double* acc4, amc_stream_t stream) {
  DeviceGuard dev_guard(x);
  AMC_CHECK_ARG(n_frames >= 0 && frame_len >= 1 && x && acc4, "bad argument");
  AMC_CHECK_ARG((reinterpret_cast<uintptr_t>(x) & 7) == 0, "frames must be 8-byte aligned");
  return iq_stats(n_frames * frame_len, x, acc4, (cudaStream_t)stream);
}

int amc_gemm(int dtype, int M, int N, int K, const void* A, int lda, int transA, const void* B, int ldb, int transB,
             const float* bias, const float* res32, int ldres, int relu, void* D16, int ldd16, float* D32, int ldd32,
             int accumulate, amc_stream_t stream) {
  DeviceGuard dev_guard(A);
  AMC_CHECK_ARG(A && B && (D16 || D32), "NULL argument");
  GemmArgs g;
  g.M = M; g.N = N; g.K = K; g.A = A; g.lda = lda; g.transA = transA; g.B = B; g.ldb = ldb; g.transB = transB;
  g.epi.bias = bias; g.epi.res32 = res32; g.epi.ldres = ldres; g.epi.relu = relu;
  g.epi.D16 = D16; g.epi.ldd16 = ldd16; g.epi.D32 = D32; g.epi.ldd32 = ldd32; g.epi.accumulate = accumulate;
  if (accumulate && !bias && !res32 && !D16) g.split_k = pick_split_k(M, N, K);
  if (dtype == AMC_BF16) return gemm_bf16(g, (cudaStream_t)stream);
  AMC_CHECK_ARG(dtype == AMC_F32, "unknown dtype %d", dtype);
  return gemm_f32(g, (cudaStream_t)stream);
}

int amc_gemm_ln(int M, int N, int K, const void* A, int lda, const void* B, int ldb, const float* bias,
                const float* res32, const float* gamma, const float* beta, float eps, void* y16, float* y32,
                void* xhat, float* rstd, amc_stream_t stream) {
  DeviceGuard dev_guard(A);
  AMC_CHECK_ARG(A && B && res32 && gamma && beta && y16 && y32, "NULL argument");
  GemmArgs g;
  g.M = M; g.N = N; g.K = K; g.A = A; g.lda = lda; g.B = B; g.ldb = ldb;
  g.epi.bias = bias; g.epi.res32 = res32; g.epi.ldres = N; g.epi.ln_gamma = gamma; g.epi.ln_beta = beta;
  g.epi.ln_eps = eps; g.epi.D16 = y16; g.epi.ldd16 = N; g.epi.D32 = y32; g.epi.ldd32 = N; g.epi.ln_xhat = xhat;
  g.epi.ln_rstd = rstd;
  return gemm_bf16(g, (cudaStream_t)stream);
}

int amc_gemm_ln_bwd(int M, int N, int K, const void* A, int lda, const void* B, int ldb, const float* res32,
                    const void* xhat, const float* rstd, const float* gamma, void* du16, float* du32, float* dgamma,
                    float* dbeta, float* dbias, amc_stream_t stream) {
  DeviceGuard dev_guard(A);
  AMC_CHECK_ARG(A && B && res32 && xhat && rstd && gamma && du16 && du32, "NULL argument");
  GemmArgs g;
  g.M = M; g.N = N; g.K = K; g.A = A; g.lda = lda; g.B = B; g.ldb = ldb;
  g.epi.ln_bwd = 1; g.epi.res32 = res32; g.epi.ldres = N; g.epi.ln_xhat = const_cast<void*>(xhat);
  g.epi.ln_rstd = const_cast<float*>(rstd); g.epi.ln_gamma = gamma; g.epi.D16 = du16; g.epi.ldd16 = N; g.epi.D32 = du32;
  g.epi.ldd32 = N; g.epi.ln_dgamma = dgamma; g.epi.ln_dbeta = dbeta; g.epi.colsum_out = dbias;
  return gemm_bf16(g, (cudaStream_t)stream);
}

int amc_gemm_relu_mask(int M, int N, int K, const void* A, int lda, const void* B, int ldb, const void* mask,
                       float mask_scale, void* D16, amc_stream_t stream) {
  DeviceGuard dev_guard(A);
  AMC_CHECK_ARG(A && B && mask && D16, "NULL argument");
  GemmArgs g;
  g.M = M; g.N = N; g.K = K; g.A = A; g.lda = lda; g.B = B; g.ldb = ldb;
  g.epi.mask_src = mask; g.epi.ldmask = N; g.epi.mask_scale = mask_scale; g.epi.D16 = D16; g.epi.ldd16 = N;
  return gemm_bf16(g, (cudaStream_t)stream);
}

int amc_attention_fwd(int dtype, int B, int T, int h, int dh, const void* qkv, void* out, float* lse,
                      amc_stream_t stream) {
  DeviceGuard dev_guard(qkv);
  AMC_CHECK_ARG(qkv && out, "NULL argument");
  if (dtype == AMC_BF16)
    return attention_fwd<bf16>(B, T, h, dh, (const bf16*)qkv, (bf16*)out, lse, (cudaStream_t)stream);
  return attention_fwd<float>(B, T, h, dh, (const float*)qkv, (float*)out, lse, (cudaStream_t)stream);
}
int amc_attention_probs(int dtype, int B, int T, int h, int dh, const void* qkv, float* probs, amc_stream_t stream) {
  DeviceGuard dev_guard(qkv);
  AMC_CHECK_ARG(qkv && probs, "NULL argument");
  if (dtype == AMC_BF16) return attention_probs<bf16>(B, T, h, dh, (const bf16*)qkv, probs, (cudaStream_t)stream);
  AMC_CHECK_ARG(dtype == AMC_F32, "unknown dtype %d", dtype);
  return attention_probs<float>(B, T, h, dh, (const float*)qkv, probs, (cudaStream_t)stream);
}
int amc_attention_rollout_step(int dtype, int B, int T, int h, int dh, const void* qkv, const float* v_in, float* v_out,
                               amc_stream_t stream) {
  DeviceGuard dev_guard(qkv);
  AMC_CHECK_ARG(qkv && v_in && v_out, "NULL argument");
  AMC_CHECK_ARG(v_in != v_out, "attention_rollout_step: v_in and v_out must be distinct buffers");
  if (dtype == AMC_BF16)
    return attention_rollout_step<bf16>(B, T, h, dh, (const bf16*)qkv, v_in, v_out, (cudaStream_t)stream);
  AMC_CHECK_ARG(dtype == AMC_F32, "unknown dtype %d", dtype);
  return attention_rollout_step<float>(B, T, h, dh, (const float*)qkv, v_in, v_out, (cudaStream_t)stream);
}
int amc_attention_relevance_step(int dtype, int B, int T, int h, int dh, const void* qkv, const void* dout,
                                 const float* v_in, float* v_out, amc_stream_t stream) {
  DeviceGuard dev_guard(qkv);
  AMC_CHECK_ARG(qkv && dout && v_in && v_out, "NULL argument");
  AMC_CHECK_ARG(v_in != v_out, "attention_relevance_step: v_in and v_out must be distinct buffers");
  if (dtype == AMC_BF16)
    return attention_relevance_step<bf16>(B, T, h, dh, (const bf16*)qkv, (const bf16*)dout, v_in, v_out,
                                          (cudaStream_t)stream);
  AMC_CHECK_ARG(dtype == AMC_F32, "unknown dtype %d", dtype);
  return attention_relevance_step<float>(B, T, h, dh, (const float*)qkv, (const float*)dout, v_in, v_out,
                                         (cudaStream_t)stream);
}
int amc_attention_cls_fwd(int B, int T, int h, int dh, const void* qkv, void* out, amc_stream_t stream) {
  DeviceGuard dev_guard(qkv);
  AMC_CHECK_ARG(qkv && out, "NULL argument");
  AMC_CHECK_ARG((h * dh) % 8 == 0 && ((reinterpret_cast<uintptr_t>(qkv) | reinterpret_cast<uintptr_t>(out)) & 15) == 0,
                "attention_cls: rows must be 16-byte aligned");
  return attn_cls_fwd(B, T, h, dh, (const bf16*)qkv, (bf16*)out, (cudaStream_t)stream);
}
int amc_attention_cls_bwd(int B, int T, int h, int dh, const void* qkv, const void* dout, void* dqkv, float* dbias,
                          amc_stream_t stream) {
  DeviceGuard dev_guard(qkv);
  AMC_CHECK_ARG(qkv && dout && dqkv, "NULL argument");
  AMC_CHECK_ARG((h * dh) % 8 == 0 && ((reinterpret_cast<uintptr_t>(qkv) | reinterpret_cast<uintptr_t>(dout) |
                                       reinterpret_cast<uintptr_t>(dqkv)) & 15) == 0,
                "attention_cls: rows must be 16-byte aligned");
  return attn_cls_bwd(B, T, h, dh, (const bf16*)qkv, (const bf16*)dout, (bf16*)dqkv, dbias, (cudaStream_t)stream);
}
int amc_attention_bwd(int dtype, int B, int T, int h, int dh, const void* qkv, const void* out, const float* lse,
                      const void* dout, void* dqkv, float* dbias, amc_stream_t stream) {
  DeviceGuard dev_guard(qkv);
  AMC_CHECK_ARG(qkv && dout && dqkv, "NULL argument");
  if (dtype == AMC_BF16)
    return attention_bwd<bf16>(B, T, h, dh, (const bf16*)qkv, (const bf16*)out, lse, (const bf16*)dout, (bf16*)dqkv, dbias,
                               (cudaStream_t)stream);
  return attention_bwd<float>(B, T, h, dh, (const float*)qkv, (const float*)out, lse, (const float*)dout, (float*)dqkv,
                              dbias, (cudaStream_t)stream);
}

int amc_layernorm_fwd(int dtype, int M, int d, const float* u, const float* gamma, const float* beta, float eps,
                      void* y16, float* y32, void* xhat, float* rstd, amc_stream_t stream) {
  DeviceGuard dev_guard(u);
  AMC_CHECK_ARG(u && gamma && beta, "NULL argument");
  if (dtype == AMC_BF16)
    return ln_fwd<bf16>(M, d, u, gamma, beta, eps, (bf16*)y16, y32, (bf16*)xhat, rstd, (cudaStream_t)stream);
  return ln_fwd<float>(M, d, u, gamma, beta, eps, (float*)y16, y32, (float*)xhat, rstd, (cudaStream_t)stream);
}
int amc_layernorm_bwd(int dtype, int M, int d, const float* dy, const void* xhat, const float* rstd,
                      const float* gamma, void* du16, float* du32, float* dgamma, float* dbeta, amc_stream_t stream) {
  DeviceGuard dev_guard(dy);
  AMC_CHECK_ARG(dy && xhat && rstd && gamma, "NULL argument");
  DropoutCfg nodrop = make_dropout(0.f, 0, 0, false);
  if (dtype == AMC_BF16)
    return ln_bwd<bf16>(M, d, dy, (const bf16*)xhat, rstd, gamma, (bf16*)du16, du32, dgamma, dbeta, nullptr, nodrop, 0,
                        (cudaStream_t)stream);
  return ln_bwd<float>(M, d, dy, (const float*)xhat, rstd, gamma, (float*)du16, du32, dgamma, dbeta, nullptr, nodrop, 0,
                       (cudaStream_t)stream);
}

int amc_frontend_fwd(const AmcDesc* desc, const float* src, const float* emb_w, const float* emb_b, const float* cls,
                     const float* pos, void* scratch, size_t scratch_bytes, float* x0, amc_stream_t stream) {
  DeviceGuard dev_guard(src);
  AMC_CHECK_ARG(desc && src && emb_w && emb_b && pos && x0, "NULL argument");
  AMC_CHECK_ARG(desc->dtype == AMC_F32, "amc_frontend_fwd operator call is fp32-only; use amc_model_fwd for bf16");
  Dims m;
  AMC_TRY(validate(*desc, m));
  AMC_CHECK_ARG(!m.has_cls || cls, "cls is NULL");
  const size_t need = (size_t)m.B * m.Ttok * m.K * sizeof(float);
  AMC_CHECK_ARG(scratch && scratch_bytes >= need, "scratch too small: need %zu bytes", need);
  cudaStream_t st = (cudaStream_t)stream;
  AMC_TRY(patchify<float>(*desc, m.Ttok, m.K, src, (float*)scratch, st));
  GemmArgs g;
  g.M = m.B * m.Ttok; g.N = m.d; g.K = m.K; g.A = scratch; g.lda = m.K; g.B = emb_w; g.ldb = m.K;
  g.epi.bias = emb_b; g.epi.pos = pos; g.epi.map_Ttok = m.Ttok; g.epi.map_T = m.T; g.epi.map_cls = m.has_cls;
  g.epi.D32 = x0; g.epi.ldd32 = m.d;
  AMC_TRY(gemm_f32(g, st));
  if (m.has_cls) {
    DropoutCfg nodrop = make_dropout(0.f, 0, 0, false);
    AMC_TRY(cls_rows<float>(m.B, m.T, m.d, cls, pos, x0, nullptr, nodrop, st));
  }
  return 0;
}

}  // extern "C"

// Fused embedding front end (bf16 path): dataset z-score + framing + patchify + embedding GEMM + bias +
// positional encoding + dropout in ONE kernel -- SURVEY §8 rows a1-a5:
//   R/dataloader/dataset.py:215-222, V/dataloader/dataset.py:211-224 (normalise, transpose / cat(I,Q).view(1,32,64))
//   R/models/embedding/patch_embedding.py:38-60, V/models/embedding/patch_embedding.py:9-15 (Conv1d / Conv2d as a GEMM)
//   R/models/encoder.py:104-111 (CLS row shift, + encoding[:T], dropout)
//
// The IQ samples are read from HBM exactly once, as coalesced 128-bit loads (every warp-wide load is 512 contiguous
// bytes of a frame), normalised, converted to bf16 and written by the converter warps straight into the
// 128B-swizzled K-major shared-memory tile that tcgen05.mma consumes as its A operand: the patchified operand never
// exists in HBM in inference (training also streams it out once, for the embedding weight gradient).  The embedding
// weight W[d, K] is TMA-loaded once per CTA and stays resident; accumulators are double-buffered in TMEM so the
// epilogue (bias + positional encoding + dropout, CLS-shifted fp32 and bf16 rows) of tile i overlaps tile i+1.
//
// Warp roles (448 threads): warp 0 = W loader (TMA), warp 1 = MMA issuer (one thread), warps 2-9 = converters,
// warps 10-13 = epilogue (one per TMEM lane quadrant).  Bound: HBM (8 B per IQ sample in, 6 B per embedding
// element out); the GEMM (K <= 256) is a small fraction of the tensor pipe.
#include <algorithm>

#include "gemm_common.cuh"
#include "rowops.cuh"
#include "ptx.cuh"

namespace amc {
namespace {

constexpr int FBM = 128, FBK = 64;
constexpr int F_NCONV = 8, F_NEPI = 4;
constexpr int F_THREADS = 64 + 32 * (F_NCONV + F_NEPI);
constexpr int F_CONV_WARP0 = 2, F_EPI_WARP0 = 2 + F_NCONV;
constexpr int F_STG_LD = 32;

struct FrontParams {
  int kind, raw;          // AMC_KIND_*, input layout (1 = dataset [B,L,2] interleaved, 0 = model layout)
  int B, M;               // frames, token rows B * Ttok
  int Ttok, K, d;
  int kb_total;           // ceil(K / 64)
  int S, L, lg_ttok;      // raw-IQ: segment size, samples per frame, log2(tokens per frame)
  int p;                  // ViT: patch size (image is 32 x 64)
  float mean[2], inv_std[2];
  int tiles_m, tiles_n, vec_ok;
  bf16* Aout;             // nullable: the patchified operand [M, K] (training: embedding weight gradient)
};

template <int BN> struct FrontCfg {
  static constexpr int A_BYTES = FBM * FBK * 2;                    // 16 KB per k-block
  static constexpr int W_BLOCK = BN * FBK * 2;                     // one k-block of W
  static constexpr int STG_BYTES = F_NEPI * 32 * F_STG_LD * 4;     // 32 KB
  static constexpr int AUX_BYTES = 1024;
  static constexpr int TMEM_COLS = 2 * BN;
  static size_t smem(int kb_total, int nstage) {
    return 1024 + (size_t)kb_total * W_BLOCK + (size_t)nstage * A_BYTES + STG_BYTES + AUX_BYTES;
  }
};

// byte offset of element (row, kcol) inside a 128-row x 64-column K-major SWIZZLE_128B tile
__device__ __forceinline__ uint32_t a_off(int row, int kcol) {
  return (uint32_t)(row * 128 + ((((kcol >> 3) ^ (row & 7)) << 4) | ((kcol & 7) << 1)));
}

// One converter warp's share of k-block `kb` of the A tile starting at token row m0.  The work is a list of
// warp-wide 512-byte loads (lane = one float4); they are issued FB at a time before any of their values is
// consumed, so a warp keeps FB * 512 bytes in flight (the scatter's st.shared would otherwise serialise them).
constexpr int FB = 8;

struct Slot {              // where one float4 of the input lands
  const float4* src;       // nullptr: out of range (zero fill)
  int row0, row1, k0, k1;  // raw layouts: (I pair -> row0,k0), (Q pair -> row1,k1); model layouts: 4 values at (row0,k0)
};


__device__ __forceinline__ Slot slot_of(const FrontParams& p, const float* __restrict__ src, int m0, int kb, int wl,
                                        int lane) {
  Slot s;
  s.src = nullptr; s.row0 = s.row1 = 0; s.k0 = s.k1 = 0;
  if (p.kind == AMC_KIND_RAWIQ) {
    const int S = p.S;
    if (p.raw) {
      // tile = 128 * S consecutive (I, Q) pairs of the frame stream; float4 = samples n, n + 1
      const int n = wl * 64 + 2 * lane, row = n / S, sidx = n - row * S;
      s.row0 = s.row1 = row; s.k0 = sidx; s.k1 = S + sidx;
      if (m0 + row < p.M) s.src = reinterpret_cast<const float4*>(src + (size_t)m0 * S * 2) + wl * 32 + lane;
    } else {
      // model layout [B, 2, L] (already normalised): S warp-loads (128 samples each) per channel
      const int c = wl / S, n = (wl - c * S) * 128 + lane * 4, row = n / S, sidx = n - row * S, gr = m0 + row;
      s.row0 = row; s.k0 = c * S + sidx;
      if (gr < p.M) {
        const int b = gr / p.Ttok, t = gr - b * p.Ttok;
        s.src = reinterpret_cast<const float4*>(src + ((size_t)b * 2 + c) * p.L + (size_t)t * S + sidx);
      }
    }
  } else {
    // ViT, image 32 x 64, patch p in {4, 8, 16}: token = ph * (64/p) + pw, k = r * p + cc  (patch_embedding.py:12-14)
    const int pp = p.p, wp = 64 / pp, rpk = min(pp, 64 / pp), f0 = m0 / p.Ttok;
    if (p.raw) {
      // dataset layout: image = cat(I, Q).view(32, 64) -> image rows 0-15 = I samples, 16-31 = Q samples
      // (V/dataloader/dataset.py:216-224); one warp-load = one image row of I and the matching row of Q
      const int nph = 16 / pp;
      const int rr = wl % rpk, t2 = wl / rpk, ph = t2 % nph, f = t2 / nph;
      const int r = kb * rpk + rr, x = 2 * lane, pw = x / pp, cc = x - pw * pp;
      s.row0 = f * p.Ttok + ph * wp + pw; s.row1 = s.row0 + nph * wp; s.k0 = s.k1 = rr * pp + cc;
      if (f0 + f < p.B) s.src = reinterpret_cast<const float4*>(src + ((size_t)(f0 + f) * 1024 + (ph * pp + r) * 64 + x) * 2);
    } else {
      // model layout [B, 1, 32, 64]: a half-warp reads one image row (64 px), a warp two consecutive selected rows
      const int nphh = 32 / pp, ir = 2 * wl + (lane >> 4);
      const int rr = ir % rpk, t2 = ir / rpk, phh = t2 % nphh, f = t2 / nphh;
      const int r = kb * rpk + rr, x = (lane & 15) * 4, pw = x / pp, cc = x - pw * pp;
      s.row0 = f * p.Ttok + phh * wp + pw; s.k0 = rr * pp + cc;
      if (f0 + f < p.B) s.src = reinterpret_cast<const float4*>(src + ((size_t)(f0 + f) * 32 + phh * pp + r) * 64 + x);
    }
  }
  return s;
}

// number of warp-loads that make up k-block kb of one tile
__device__ __forceinline__ int warp_loads(const FrontParams& p) {
  if (p.kind == AMC_KIND_RAWIQ) return 2 * p.S;
  const int rpk = min(p.p, 64 / p.p), fpt = FBM / p.Ttok;
  return p.raw ? fpt * (16 / p.p) * rpk : fpt * (32 / p.p) * rpk / 2;
}

// Per-thread, tile-invariant description of the FB float4s a converter lane handles in every k-block: computed once
// per kernel (the index arithmetic has runtime divisors), so the per-tile work is one add + bounds test per load.
struct LaneSlots {
  int off[FB];          // float offset from the tile's base pointer (k-block 0); < 0: slot unused
  uint32_t meta[FB];    // row0 | row1 << 8 | k0 << 16 | k1 << 24
  uint32_t soff[FB];    // byte offsets inside the swizzled A stage: (row0,k0) | (row1,k1) << 16
  int kb_stride;        // floats added per k-block
};

__device__ __forceinline__ void make_lane_slots(const FrontParams& p, int cw, int lane, LaneSlots& ls) {
  const int nwl = warp_loads(p);
  ls.kb_stride = 0;
  if (p.kind == AMC_KIND_VIT) {
    const int rpk = min(p.p, 64 / p.p);
    ls.kb_stride = p.raw ? rpk * 64 * 2 : rpk * 64;
  }
  const int per = (nwl + F_NCONV - 1) / F_NCONV;      // consecutive warp-loads per warp: contiguous DRAM runs
#pragma unroll
  for (int j = 0; j < FB; ++j) {
    const int wl = j < per ? cw * per + j : nwl;
    ls.off[j] = -1;
    ls.meta[j] = 0u;
    ls.soff[j] = 0u;
    if (wl < nwl) {
      // base pointer = nullptr + offsets of tile 0 / k-block 0; only the offset part is kept
      const Slot t = slot_of(p, reinterpret_cast<const float*>(0), 0, 0, wl, lane);
      ls.meta[j] = (uint32_t)t.row0 | ((uint32_t)t.row1 << 8) | ((uint32_t)t.k0 << 16) | ((uint32_t)t.k1 << 24);
      ls.off[j] = (int)(reinterpret_cast<uintptr_t>(t.src) >> 2);
      ls.soff[j] = a_off(t.row0, t.k0) | (a_off(t.row1, t.k1) << 16);
    }
  }
}

// issue the FB loads of (tile m0, k-block kb); `okmask` bit j = slot j holds real data
__device__ __forceinline__ void load_block(const FrontParams& p, const LaneSlots& ls, const float* __restrict__ src, int m0,
                                           int kb, float4 (&v)[FB], uint32_t& okmask) {
  const float* tbase;
  int limit;                            // rows available from the tile start (raw-IQ: token rows; ViT: rows of whole frames)
  const bool by_row = p.kind == AMC_KIND_RAWIQ;
  if (by_row) {
    tbase = p.raw ? src + (size_t)m0 * p.S * 2 : src;
    limit = p.M - m0;
  } else {
    const int f0 = m0 / p.Ttok;
    tbase = src + (size_t)f0 * 2048 + (size_t)kb * ls.kb_stride;
    limit = (p.B - f0) * p.Ttok;
  }
  okmask = 0u;
#pragma unroll
  for (int j = 0; j < FB; ++j) {
    const int row0 = ls.meta[j] & 0xFF;
    const bool ok = ls.off[j] >= 0 && row0 < limit;
    v[j] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (ok) {
      okmask |= 1u << j;
      const float* a;
      if (by_row && !p.raw) {           // model layout [B, 2, L]: frame / token of the row (Ttok is a power of two)
        const int gr = m0 + row0, b = gr >> p.lg_ttok, t = gr & (p.Ttok - 1);
        const int k0 = (ls.meta[j] >> 16) & 0xFF, c = k0 >= p.S ? 1 : 0;
        a = src + ((size_t)b * 2 + c) * p.L + (size_t)t * p.S + (k0 - c * p.S);
      } else {
        a = tbase + ls.off[j];
      }
      v[j] = __ldg(reinterpret_cast<const float4*>(a));
    }
  }
}

// normalise, convert and scatter the loaded values into the swizzled A stage (and stream them to Aout in training)
__device__ __forceinline__ void store_block(const FrontParams& p, const LaneSlots& ls, uint32_t sa, int m0, int kb,
                                            const float4 (&v)[FB], uint32_t okmask) {
  const int kbase = kb * FBK;          // column of this k-block inside the [M, K] operand (Aout)
#pragma unroll
  for (int j = 0; j < FB; ++j) {
    if (ls.off[j] < 0) continue;
    const bool ok = (okmask >> j) & 1u;
    const int row0 = ls.meta[j] & 0xFF, row1 = (ls.meta[j] >> 8) & 0xFF, k0 = (ls.meta[j] >> 16) & 0xFF, k1 = ls.meta[j] >> 24;
    if (p.raw) {
      uint32_t wi = 0u, wq = 0u;
      if (ok) {
        wi = pack2((v[j].x - p.mean[0]) * p.inv_std[0], (v[j].z - p.mean[0]) * p.inv_std[0]);
        wq = pack2((v[j].y - p.mean[1]) * p.inv_std[1], (v[j].w - p.mean[1]) * p.inv_std[1]);
        if (p.Aout) {
          *reinterpret_cast<uint32_t*>(p.Aout + (size_t)(m0 + row0) * p.K + kbase + k0) = wi;
          *reinterpret_cast<uint32_t*>(p.Aout + (size_t)(m0 + row1) * p.K + kbase + k1) = wq;
        }
      }
      sts32(sa + (ls.soff[j] & 0xFFFFu), wi);
      sts32(sa + (ls.soff[j] >> 16), wq);
    } else {
      const uint32_t w0_ = pack2(v[j].x, v[j].y), w1_ = pack2(v[j].z, v[j].w);
      if (ok && p.Aout)
        *reinterpret_cast<uint2*>(p.Aout + (size_t)(m0 + row0) * p.K + kbase + k0) = make_uint2(w0_, w1_);
      sts64(sa + (ls.soff[j] & 0xFFFFu), w0_, w1_);
    }
  }
}

template <int BN>
__global__ void __launch_bounds__(F_THREADS, 1)
frontend_tc_kernel(const __grid_constant__ CUtensorMap mapW, const FrontParams p, const Epi epi,
                   const float* __restrict__ src, int nstage) {
  using C = FrontCfg<BN>;
  extern __shared__ unsigned char smem_dyn[];
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023) & ~(uintptr_t)1023);
  unsigned char* sW = smem;                                            // [kb_total][BN x 64] bf16, SWIZZLE_128B
  unsigned char* sA = sW + (size_t)p.kb_total * C::W_BLOCK;           // ring of nstage A k-blocks
  float* stage_base = reinterpret_cast<float*>(sA + (size_t)nstage * C::A_BYTES);
  uint64_t* bars = reinterpret_cast<uint64_t*>(reinterpret_cast<unsigned char*>(stage_base) + C::STG_BYTES);
  uint64_t* wfull = bars;
  uint64_t* full_bar = bars + 1;            // [nstage <= 8]
  uint64_t* empty_bar = full_bar + 8;
  uint64_t* tfull_bar = empty_bar + 8;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tn = blockIdx.x % p.tiles_n, cta_m = blockIdx.x / p.tiles_n, m_stride = gridDim.x / p.tiles_n;
  const int n0 = tn * BN;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&mapW);
    mbar_init(wfull, 1);
    for (int s = 0; s < nstage; ++s) {
      mbar_init(full_bar + s, F_NCONV);
      mbar_init(empty_bar + s, 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(tfull_bar + s, 1);
      mbar_init(tempty_bar + s, F_NEPI);
    }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, C::TMEM_COLS);
  // columns of the A tiles beyond K (K % 64 != 0) are never written by the converters: they must read as zero
  for (int i = threadIdx.x; i < nstage * C::A_BYTES / 16; i += blockDim.x)
    reinterpret_cast<uint4*>(sA)[i] = make_uint4(0u, 0u, 0u, 0u);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      mbar_expect_tx(wfull, (uint32_t)(p.kb_total * C::W_BLOCK));
      for (int kb = 0; kb < p.kb_total; ++kb)
        tma_load_2d(&mapW, wfull, smem_u32(sW + (size_t)kb * C::W_BLOCK), kb * FBK, n0);
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc(FBM, BN, 0, 0);
      mbar_wait(wfull, 0);
      int stage = 0, as = 0;
      uint32_t phase = 0, aphase = 0;
      for (int tm = cta_m; tm < p.tiles_m; tm += m_stride) {
        mbar_wait(tempty_bar + as, aphase ^ 1);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + (uint32_t)(as * BN);
        for (int kb = 0; kb < p.kb_total; ++kb) {
          mbar_wait(full_bar + stage, phase);
          tc_fence_after();
          const uint32_t sa = smem_u32(sA + (size_t)stage * C::A_BYTES);
          const uint32_t sb = smem_u32(sW + (size_t)kb * C::W_BLOCK);
          const int ksteps = min(FBK, p.K - kb * FBK + 15) / 16;
          for (int k = 0; k < ksteps; ++k)
            umma_bf16(tmem_d, make_smem_desc(sa + k * 32, 16, 1024, 2), make_smem_desc(sb + k * 32, 16, 1024, 2), idesc,
                      (kb > 0 || k > 0) ? 1u : 0u);
          umma_commit(empty_bar + stage);
          if (++stage == nstage) { stage = 0; phase ^= 1; }
        }
        umma_commit(tfull_bar + as);
        if (++as == 2) { as = 0; aphase ^= 1; }
      }
    }
  } else if (warp < F_EPI_WARP0) {
    // ===================== converter warps =====================
    const int cw = warp - F_CONV_WARP0;
    LaneSlots ls;
    make_lane_slots(p, cw, lane, ls);
    int stage = 0;
    uint32_t phase = 0;
    // the FB loads of a k-block are issued before waiting for its shared-memory stage, so DRAM latency overlaps the
    // wait for the tensor core to release the stage
    for (int tm = cta_m; tm < p.tiles_m; tm += m_stride) {
      for (int kb = 0; kb < p.kb_total; ++kb) {
        float4 cur[FB];
        uint32_t ok_cur = 0u;
        load_block(p, ls, src, tm * FBM, kb, cur, ok_cur);
        mbar_wait(empty_bar + stage, phase ^ 1);
        store_block(p, ls, smem_u32(sA + (size_t)stage * C::A_BYTES), tm * FBM, kb, cur, ok_cur);
        fence_proxy_async();   // generic-proxy writes -> visible to the tensor core's async-proxy reads
        __syncwarp();
        if (lane == 0) mbar_arrive(full_bar + stage);
        if (++stage == nstage) { stage = 0; phase ^= 1; }
      }
    }
  } else {
    // ===================== epilogue warps =====================
    const int ew = warp - F_EPI_WARP0;
    const int quad = warp & 3;                         // TMEM lane quadrant this warp may access
    int as = 0;
    uint32_t aphase = 0;
    const uint32_t stg = smem_u32(stage_base + ew * (32 * F_STG_LD));
    const int sub_r = lane >> 3, sub_c = (lane & 7) * 4;
    float* const D32 = epi.D32;
    bf16* const D16 = reinterpret_cast<bf16*>(epi.D16);
    for (int tm = cta_m; tm < p.tiles_m; tm += m_stride) {
      const int m_base = tm * FBM + quad * 32;
      // output row (CLS-shifted, encoder.py:104-105) and token index of the 8 rows this lane touches in every chunk
      int orow[8], tok[8];
#pragma unroll
      for (int it = 0; it < 8; ++it) {
        const int m = m_base + it * 4 + sub_r;
        const int b = m / epi.map_Ttok, t = m - b * epi.map_Ttok + epi.map_cls;
        tok[it] = t;
        orow[it] = m < p.M ? b * epi.map_T + t : -1;
      }
      mbar_wait(tfull_bar + as, aphase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(as * BN);
      const int c_begin = 0;
      const int c_end = min(BN, p.d - n0);
      uint32_t r[32];
      if (c_begin < c_end) tmem_ld32(taddr + c_begin, r);
#pragma unroll 1
      for (int c = c_begin; c < c_end; c += 32) {
        tmem_ld_wait(r);
#pragma unroll
        for (int j = 0; j < 32; j += 4)
          sts128(stg + (uint32_t)(lane * F_STG_LD + (((j >> 2) ^ (lane & 7)) << 2)) * 4, r[j], r[j + 1], r[j + 2], r[j + 3]);
        if (c + 32 < c_end) tmem_ld32(taddr + c + 32, r);
        __syncwarp();
        const int n = n0 + c + sub_c;
        if (n < p.d) {                    // d % 8 == 0: a float4 is never ragged
          const float4 bias = __ldg(reinterpret_cast<const float4*>(epi.bias + n));
          float4 pe[8];
#pragma unroll
          for (int it = 0; it < 8; ++it) pe[it] = __ldg(reinterpret_cast<const float4*>(epi.pos + (size_t)tok[it] * p.d + n));
#pragma unroll
          for (int it = 0; it < 8; ++it) {
            const int rr = it * 4 + sub_r;
            float4 v = lds128f(stg + (uint32_t)(rr * F_STG_LD + ((((lane & 7)) ^ (rr & 7)) << 2)) * 4);
            if (orow[it] < 0) continue;
            v.x += bias.x + pe[it].x; v.y += bias.y + pe[it].y; v.z += bias.z + pe[it].z; v.w += bias.w + pe[it].w;
            const size_t o = (size_t)orow[it] * p.d + n;
            if (epi.drop.p > 0.f) {
              const float4 k = dropout_mult4(epi.drop, epi.drop_site, (uint64_t)o >> 2);
              v.x *= k.x; v.y *= k.y; v.z *= k.z; v.w *= k.w;
            }
            if (D32) *reinterpret_cast<float4*>(D32 + o) = v;
            if (D16) store4(D16 + o, v);
          }
        }
        __syncwarp();
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar + as);
      if (++as == 2) { as = 0; aphase ^= 1; }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, C::TMEM_COLS);
  }
}

inline bool pow2(int v) { return v > 0 && (v & (v - 1)) == 0; }

template <int BN>
int launch_front(const AmcDesc& D, FrontParams p, const Epi& epi, const float* src, const bf16* W, cudaStream_t st) {
  using C = FrontCfg<BN>;
  CUtensorMap mapW;
  const cuuint64_t dims[2] = {(cuuint64_t)p.K, (cuuint64_t)p.d};
  const cuuint64_t strides[1] = {(cuuint64_t)p.K * 2};
  const cuuint32_t box[2] = {(cuuint32_t)FBK, (cuuint32_t)BN};
  AMC_TRY(encode_tiled_map(&mapW, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, W, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B,
                           CU_TENSOR_MAP_L2_PROMOTION_L2_256B));
  p.tiles_n = ceil_div(p.d, BN);
  p.tiles_m = ceil_div(p.M, FBM);
  int nstage = std::min(8, std::max(2, 2 * p.kb_total));
  while (nstage > 2 && C::smem(p.kb_total, nstage) > 227 * 1024) --nstage;
  const size_t smem = C::smem(p.kb_total, nstage);
  AMC_CHECK_ARG(smem <= 227 * 1024, "front end: K=%d d=%d needs %zu bytes of shared memory", p.K, p.d, smem);
  const int per_n = std::max(1, std::min(p.tiles_m, device_sm_count() / p.tiles_n));
  auto kern = frontend_tc_kernel<BN>;
  AMC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
  kern<<<per_n * p.tiles_n, F_THREADS, smem, st>>>(mapW, p, epi, src, nstage);
  AMC_LAUNCH_CHECK();
  (void)D;
  return 0;
}

}  // namespace

// Returns 0 and sets *handled when the geometry is one the fused kernel covers; otherwise the caller runs the
// patchify kernel + generic GEMM.
int frontend_fused(const AmcDesc& D, int Ttok, int K, const float* src, const bf16* W, const Epi& epi, bf16* Aout,
                   bool probe_only, bool* handled, cudaStream_t st) {
  *handled = false;
  const int d = D.d;
  if (D.B <= 0 || d % 8 != 0 || K % 8 != 0 || K > 256 || d > 512) return 0;
  if ((reinterpret_cast<uintptr_t>(src) & 15) != 0) return 0;
  FrontParams p = {};
  p.kind = D.kind; p.raw = D.input_layout == AMC_INPUT_RAW;
  p.B = D.B; p.Ttok = Ttok; p.M = D.B * Ttok; p.K = K; p.d = d;
  p.kb_total = ceil_div(K, FBK);
  if (D.kind == AMC_KIND_RAWIQ) {
    const int S = D.seg;
    // one k-block (2S <= 64); 128-token tiles made of whole 64-sample warp-loads; float4 never straddles a token
    if (D.in_ch != 2 || !pow2(S) || S < 4 || 2 * S > 64 || K != 2 * S) return 0;
    if (!p.raw && (Ttok % 1 != 0 || D.seq_len % 4 != 0)) return 0;
    if (!pow2(Ttok)) return 0;
    p.S = S; p.L = D.seq_len;
    p.lg_ttok = 0;
    while ((1 << p.lg_ttok) < Ttok) ++p.lg_ttok;
  } else {
    if (D.in_ch != 1 || D.img_h != 32 || D.img_w != 64 || (D.patch != 4 && D.patch != 8 && D.patch != 16)) return 0;
    if (FBM % Ttok != 0 && Ttok % FBM != 0) return 0;
    p.p = D.patch;
  }
  p.vec_ok = epi_vec_ok<bf16>(epi, d) ? 1 : 0;
  if (!p.vec_ok || epi.bias == nullptr || epi.pos == nullptr || epi.D16 == nullptr || epi.ldd16 != d ||
      (epi.D32 && epi.ldd32 != d))
    return 0;
  if (probe_only) {
    *handled = true;
    return 0;
  }
  p.mean[0] = D.norm[0]; p.inv_std[0] = 1.f / D.norm[1];
  p.mean[1] = D.norm[2]; p.inv_std[1] = 1.f / D.norm[3];
  p.Aout = Aout;
  if (d <= 128) AMC_TRY(launch_front<128>(D, p, epi, src, W, st));
  else AMC_TRY(launch_front<256>(D, p, epi, src, W, st));
  *handled = true;
  return 0;
}

}  // namespace amc

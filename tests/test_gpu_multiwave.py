"""The persistent GEMM, attention and LayerNorm-backward kernels past each CTA's first work item.

Every kernel here launches grid = min(items, SMs x CTAs per SM) and loops over items with a stride of gridDim.x,
carrying state from one item to the next: TMEM accumulator buffers and phases, input-ring parities, slabs and O / lse
prefetched for the next item, column-sum partials.  The operator tests elsewhere stay within one item per CTA.  Here
every case is sized so that each CTA takes at least three items (printed at run time from the SM count and the bound
on CTAs per SM named in the table), with a ragged last item, and three checks run:

  1. single-wave replay: the problem again in chunks of at most 148 items, so every item is the first of its CTA
     (the regime the single-wave float64 tests validate); outputs pre-filled with NaN must equal the whole-problem
     outputs bit for bit, for every output written without atomics (GEMMs: over several whole runs, since a race
     between items need not show on every run);
  2. float64 element by element, with the per-element bounds of tests/multiwave_ref.py;
  3. (GEMMs) integer operands in -3..3: exact in bf16, products exact, every partial sum below 9 K < 2^24, so any fp32
     accumulation order -- tensor-core adder, TMEM double buffer, split-K atomics -- gives the exact result: D32 must
     equal float64, D16 its RNE bf16.  The LayerNorm epilogues are compared with float64 LayerNorm (backward) of the
     exact u / t under a bound of the LayerNorm arithmetic alone.
Outputs carry padding rows past M (and padding columns where ld > N) that must never be written."""
import pytest
import torch

pytestmark = pytest.mark.gpu

import isolated_ref as R  # noqa: E402
import multiwave_ref as MW  # noqa: E402

from vit_vs_raw_iq_b200 import _lib  # noqa: E402

DEV = "cuda:0"
M_ROWS = 444 * 128 + 73          # 56,905 token rows: 445 row tiles, the last one ragged (73 rows)
PAD_ROWS = 128                   # rows past M in every output buffer: must stay NaN
TOKENS = 294912                  # bench.py's default token count (32,768 frames x 9 tokens)
EPS = 1e-5
WHOLE_RUNS = 4                   # whole-problem runs compared with the single-wave replay


def stream():
    return torch.cuda.current_stream().cuda_stream


def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def report_items(what, items, ctas_per_sm, need=3):
    n = MW.min_items_per_cta(items, sms(), ctas_per_sm)
    print(f"  {what}: {items} items, <= {ctas_per_sm} CTAs/SM on {sms()} SMs -> every CTA takes >= {n} items")
    assert n >= need, (what, items, n)
    return n


def nan_rows(t, M):
    assert torch.isnan(t[M:].float()).all(), "rows past M were written"


# ---------------------------------------------------------------------------------------------------------------------
# GEMMs with a row epilogue (gemm_tc_row_kernel) and the generic-epilogue kernel (gemm_tc_kernel), M = 56,905
# ---------------------------------------------------------------------------------------------------------------------
# Dispatch: gemm_bf16 in csrc/gemm_tc.cu.  One CTA per SM for every GEMM: launch / launch_row use grid = min(tiles,
# SMs) with __launch_bounds__(..., 1) and more than half of the shared memory.  BN is the N tile the dispatch picks.
GEMM_CASES = [
    dict(id="bf16-w8-qkv", entry="gemm", N=768, K=256, bn=256, bias=1,
         kernel="gemm_tc_row_kernel<256, RE_BF16, 8>: D16 only, no ReLU / dropout"),
    dict(id="bf16-w16-ffn1-relu", entry="gemm", N=1024, K=256, bn=256, bias=1, relu=1,
         kernel="gemm_tc_row_kernel<256, RE_BF16, 16>: e.relu"),
    dict(id="bf16-w8-ragged-n288", entry="gemm", N=288, K=256, bn=64, bias=1,
         kernel="gemm_tc_row_kernel<64, RE_BF16, 8>: N = 288 pads least at BN = 64, last N tile half full"),
    dict(id="res32-ffn2", entry="gemm", N=256, K=1024, bn=256, bias=1, res=1,
         kernel="gemm_tc_row_kernel<256, RE_RES32, 4>: res32, D32 only"),
    dict(id="mask-dgrad-ffn2", entry="mask", N=1024, K=256, bn=256,
         kernel="gemm_tc_row_kernel<256, RE_MASK, 16>: amc_gemm_relu_mask"),
    dict(id="ln-w8-k256", entry="ln", N=256, K=256, bn=256,
         kernel="gemm_tc_row_kernel<256, RE_LN, 8>: K <= 256, two warps per quadrant"),
    dict(id="ln-w4-k1024", entry="ln", N=256, K=1024, bn=256,
         kernel="gemm_tc_row_kernel<256, RE_LN, 4>: K > 256, one warp per quadrant"),
    dict(id="ln-n384", entry="ln", N=384, K=384, bn=512,
         kernel="gemm_tc_row_kernel<512, RE_LN, 4>: N > 256, single-buffered 512-column accumulator"),
    dict(id="ln-n512", entry="ln", N=512, K=512, bn=512,
         kernel="gemm_tc_row_kernel<512, RE_LN, 4>: N > 256, single-buffered 512-column accumulator"),
    dict(id="lnb-n64-k768", entry="lnb", N=64, K=768, bn=64, kernel="gemm_tc_row_kernel<64, RE_LNB, 8>"),
    dict(id="lnb-n128-k1024", entry="lnb", N=128, K=1024, bn=128, kernel="gemm_tc_row_kernel<128, RE_LNB, 8>"),
    dict(id="lnb-n256-k768", entry="lnb", N=256, K=768, bn=256, kernel="gemm_tc_row_kernel<256, RE_LNB, 8>"),
    dict(id="lnb-n256-k1024", entry="lnb", N=256, K=1024, bn=256, kernel="gemm_tc_row_kernel<256, RE_LNB, 8>"),
    dict(id="generic-d16-d32-padded", entry="gemm", N=192, K=128, bn=64, bias=1, out16=1, out32=1, lda=136,
         ldd16=200, ldd32=196,
         kernel="gemm_tc_kernel<64, 0>: D16 and D32 together take no row epilogue (unfused embedding)"),
]


def gemm_outputs(c):
    """name -> (buffer with PAD_ROWS extra rows, NaN-filled; replayed bit for bit?)"""
    M, N = M_ROWS, c["N"]
    e = c["entry"]
    nan = lambda cols, dt: torch.full((M + PAD_ROWS, cols), float("nan"), device=DEV, dtype=dt)  # noqa
    if e == "gemm":
        out = {}
        if c.get("out16", not c.get("res")):
            out["D16"] = nan(c.get("ldd16", N), torch.bfloat16)
        if c.get("out32", c.get("res")):
            out["D32"] = nan(c.get("ldd32", N), torch.float32)
        return out
    if e == "mask":
        return {"D16": nan(N, torch.bfloat16)}
    if e == "ln":
        return {"y16": nan(N, torch.bfloat16), "y32": nan(N, torch.float32), "xhat": nan(N, torch.bfloat16),
                "rstd": torch.full((M + PAD_ROWS,), float("nan"), device=DEV)}
    return {"du16": nan(N, torch.bfloat16), "du32": nan(N, torch.float32)}


def gemm_inputs(c, integer, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    M, N, K = M_ROWS, c["N"], c["K"]

    def draw(shape, scale=1.0, ints=integer):
        if ints:
            return torch.randint(-3, 4, shape, generator=g, device=DEV).float()
        return torch.randn(shape, generator=g, device=DEV) * scale

    X = dict(A=draw((M, c.get("lda", K))).bfloat16(), B=draw((N, K), K ** -0.5).bfloat16())
    e = c["entry"]
    if c.get("bias") or e == "ln":
        X["bias"] = draw((N,))
    if c.get("res") or e in ("ln", "lnb"):
        X["res"] = draw((M, N))
    if e == "mask":
        X["mask"] = (torch.randint(-1, 2, (M, N), generator=g, device=DEV).float() if integer
                     else torch.randn(M, N, generator=g, device=DEV).clamp_min(0)).bfloat16()
        X["scale"] = 2.0 if integer else 1.25           # 2: acc * scale stays exact in fp32
    if e in ("ln", "lnb"):
        X["gamma"] = draw((N,), ints=False)
        X["beta"] = draw((N,), ints=False)
    if e == "lnb":
        X["xhat"] = draw((M, N)).bfloat16()
        X["rstd"] = 0.5 + torch.rand(M, generator=g, device=DEV)
        X["dgamma"], X["dbeta"], X["dbias"] = (torch.zeros(N, device=DEV) for _ in range(3))
    return X


def gemm_call(c, X, O, r0, r1, colsums=None):
    """Rows [r0, r1) of the problem: every pointer offset by r0 rows (16-byte aligned: r0 is a multiple of 128)."""
    N, K, m = c["N"], c["K"], r1 - r0
    A = X["A"][r0:r1]
    lda = X["A"].stride(0)
    ptr, lib = _lib.ptr, _lib.lib
    rows = lambda name: O[name][r0:r1] if name in O else None  # noqa
    e = c["entry"]
    if e == "gemm":
        res = X["res"][r0:r1] if "res" in X else None
        d16, d32 = rows("D16"), rows("D32")
        rc = lib.amc_gemm(_lib.BF16, m, N, K, A.data_ptr(), lda, 0, X["B"].data_ptr(), K, 0, ptr(X.get("bias")),
                          ptr(res), N, c.get("relu", 0), ptr(d16), O["D16"].stride(0) if d16 is not None else 0,
                          ptr(d32), O["D32"].stride(0) if d32 is not None else 0, 0, stream())
    elif e == "mask":
        rc = lib.amc_gemm_relu_mask(m, N, K, A.data_ptr(), lda, X["B"].data_ptr(), K, X["mask"][r0:r1].data_ptr(),
                                    X["scale"], rows("D16").data_ptr(), stream())
    elif e == "ln":
        rc = lib.amc_gemm_ln(m, N, K, A.data_ptr(), lda, X["B"].data_ptr(), K, X["bias"].data_ptr(),
                             X["res"][r0:r1].data_ptr(), X["gamma"].data_ptr(), X["beta"].data_ptr(), EPS,
                             rows("y16").data_ptr(), rows("y32").data_ptr(), rows("xhat").data_ptr(),
                             O["rstd"][r0:r1].data_ptr(), stream())
    else:
        cs = colsums or (X["dgamma"], X["dbeta"], X["dbias"])
        rc = lib.amc_gemm_ln_bwd(m, N, K, A.data_ptr(), lda, X["B"].data_ptr(), K, X["res"][r0:r1].data_ptr(),
                                 X["xhat"][r0:r1].data_ptr(), X["rstd"][r0:r1].data_ptr(), X["gamma"].data_ptr(),
                                 rows("du16").data_ptr(), rows("du32").data_ptr(), *(t.data_ptr() for t in cs),
                                 stream())
    _lib.check(rc, c["id"])


def gemm_reference(c, X, exact):
    """name -> (ref, bound) in float64 on the device.  ``exact``: integer operands, the GEMM part has no error."""
    N, K = c["N"], c["K"]
    A = X["A"][:, :K].double()
    B = X["B"].double()
    acc = A @ B.T
    mag = A.abs() @ B.abs().T
    del A, B
    zero = torch.zeros((), device=DEV, dtype=torch.float64)
    e = c["entry"]
    if e == "gemm":
        bias = X["bias"].double() if "bias" in X else zero
        u = acc + bias
        mag += bias.abs()
        extra = 1
        if c.get("relu"):
            u = u.clamp_min(0)
        if "res" in X:
            res = X["res"].double()
            u, mag, extra = u + res, mag + res.abs(), 2
        err = zero if exact else MW.gemm_bound(mag, K, extra)
        return {"D16": (u, MW.bf16_bound(u, err)), "D32": (u, err)}
    if e == "mask":
        keep = (X["mask"].double() > 0) * X["scale"]
        u = acc * keep
        err = zero if exact else MW.gemm_bound(mag, K) * keep
        return {"D16": (u, MW.bf16_bound(u, err))}
    if e == "ln":
        res = X["res"].double()
        u = acc + X["bias"].double() + res
        e_u = torch.zeros_like(u) if exact else MW.gemm_bound(mag + X["bias"].double().abs() + res.abs(), K, 2)
        L = MW.ln_fwd_ref(u, e_u, X["gamma"].double(), X["beta"].double(), EPS)
        return {"y32": (L["y"], L["e_y"]), "y16": (L["y"], MW.bf16_bound(L["y"], L["e_y"])),
                "xhat": (L["xhat"], MW.bf16_bound(L["xhat"], L["e_xhat"])), "rstd": (L["rstd"], L["e_rstd"])}
    res = X["res"].double()
    t = acc + res
    e_t = torch.zeros_like(t) if exact else MW.gemm_bound(mag + res.abs(), K)
    xh = X["xhat"].double()
    du, e_du = MW.ln_bwd_ref(t, e_t, xh, X["rstd"].double(), X["gamma"].double())
    e_du16 = MW.bf16_bound(du, e_du)
    return {"du32": (du, e_du), "du16": (du, e_du16),
            "dgamma": ((t * xh).sum(0), MW.colsum_bound(t * xh, e_t * xh.abs())),
            "dbeta": (t.sum(0), MW.colsum_bound(t, e_t)),
            "dbias": (du.sum(0), MW.colsum_bound(du, e_du16))}


def check_outputs(c, X, O, refs, exact):
    M, N = M_ROWS, c["N"]
    for name, buf in O.items():
        ref, bound = refs[name]
        got = buf[:M, :N] if buf.dim() == 2 else buf[:M]
        nan_rows(buf, M)
        if buf.dim() == 2 and buf.shape[1] > N:
            assert torch.isnan(buf[:, N:].float()).all(), f"{name}: padding columns were written"
        if exact and name in ("D16", "D32"):
            want = ref.float() if name == "D32" else ref.float().bfloat16()
            assert torch.equal(got, want), f"{name}: integer-operand result differs from the exact one"
            print(f"  {name}: exact")
        else:
            R.check(name, got, ref, bound)
    if c["entry"] == "gemm" and "D16" in O and "D32" in O:
        assert torch.equal(O["D16"][:M, :N], O["D32"][:M, :N].bfloat16())      # D16 = RNE of the same fp32 value
    if c["entry"] == "lnb":
        for name in ("dgamma", "dbeta", "dbias"):
            R.check(name, X[name], *refs[name])


@pytest.mark.parametrize("c", GEMM_CASES, ids=[c["id"] for c in GEMM_CASES])
def test_gemm_multiwave(c):
    M, N = M_ROWS, c["N"]
    tiles_n = -(-N // c["bn"])
    print(f"\n{c['id']}: {c['kernel']}; M={M} N={N} K={c['K']}")
    report_items("tiles", -(-M // MW.BM) * tiles_n, 1)

    # 1. chunks of at most 148 tiles, then the whole problem WHOLE_RUNS times (a race between items need not show on
    #    every run): every whole run equal to the single-wave replay, bit for bit
    X = gemm_inputs(c, False, M + N + c["K"])
    scratch = [torch.zeros(N, device=DEV) for _ in range(3)]
    O1 = gemm_outputs(c)
    rows = MW.gemm_chunk_rows(tiles_n)
    for r0, r1 in MW.spans(M, rows):
        gemm_call(c, X, O1, r0, r1, colsums=scratch)
    for run in range(WHOLE_RUNS):
        O = gemm_outputs(c)
        gemm_call(c, X, O, 0, M, colsums=None if run == 0 else scratch)
        torch.cuda.synchronize()
        for name in O:
            whole, chunked = (O[name][:M], O1[name][:M]) if O[name].dim() == 1 else (O[name][:M, :N], O1[name][:M, :N])
            diff = (whole.double() - chunked.double()).abs().nan_to_num(float("inf"))
            bad = (diff > 0).nonzero()[:, 0].unique()[:8].tolist()
            assert torch.equal(whole, chunked), (f"{name}, whole run {run}: differs from the replay in chunks of {rows} "
                                                 f"rows in {int((diff > 0).sum())} elements, rows {bad}..., max |diff| "
                                                 f"{float(diff.max())}")
    print(f"  {WHOLE_RUNS} whole runs and the replay in chunks of {rows} rows: {', '.join(O)} equal bit for bit")
    del O1

    # 2. float64 element by element
    check_outputs(c, X, O, gemm_reference(c, X, False), False)
    del X, O

    # 3. integer operands: the main loop is exact
    X = gemm_inputs(c, True, 7 * M + N)
    O = gemm_outputs(c)
    gemm_call(c, X, O, 0, M)
    torch.cuda.synchronize()
    check_outputs(c, X, O, gemm_reference(c, X, True), True)


# ---------------------------------------------------------------------------------------------------------------------
# split-K weight gradients: amc_gemm, transA = transB = 1, accumulate (gemm_tc_kernel<BN, 1>, one CTA per SM)
# ---------------------------------------------------------------------------------------------------------------------
# At the bench's token count, pick_split_k (api.cu) sizes the splits to about two waves of 128 x 128 tiles, and these
# N take BN = 256: 144 (tile, split) items on 148 SMs, one per CTA.  The main loop of each item is long (192 to 256
# k-blocks), and the integer check is the one that can see a missing or duplicated split at that K.  N = 320 pads least
# at BN = 64 (five N tiles against three of 128), which gives 480 items: the same kernel past the first item.
WGRAD_CASES = [
    # id, M (dW rows), N (dW cols), K (tokens), multi-wave
    ("qkv-d256", 768, 256, TOKENS, False),
    ("ffn1-d256", 1024, 256, TOKENS, False),
    ("ffn2-d256", 256, 1024, TOKENS, False),
    ("qkv-d320", 960, 320, TOKENS, True),
    ("qkv-d320-ragged-k", 960, 320, 73719, True),
]


@pytest.mark.parametrize("case", WGRAD_CASES, ids=[c[0] for c in WGRAD_CASES])
def test_wgrad_split_k(case):
    name, M, N, K, multi = case
    items, splits = MW.split_k_items(M, N, K)
    print(f"\n{name}: gemm_tc_kernel<{MW.pick_bn(N)}, 1>, dW[{M}, {N}] += A[{K}, {M}]^T B[{K}, {N}], {splits} splits")
    if multi:
        report_items("(tile, split) items", items, 1)
    else:
        assert items <= MW.LAUNCH_SMS
        print(f"  {items} (tile, split) items: one per CTA")
    for integer in (False, True):
        g = torch.Generator(device=DEV).manual_seed(M + N + K + integer)
        draw = ((lambda s: torch.randint(-3, 4, s, generator=g, device=DEV).float()) if integer
                else (lambda s: torch.randn(s, generator=g, device=DEV)))
        A, B = draw((K, M)).bfloat16(), draw((K, N)).bfloat16()
        D0 = torch.full((M, N), 5.0, device=DEV) if integer else torch.randn(M, N, generator=g, device=DEV)
        D = torch.full((M + PAD_ROWS, N), float("nan"), device=DEV)
        D[:M] = D0
        _lib.check(_lib.lib.amc_gemm(_lib.BF16, M, N, K, A.data_ptr(), M, 1, B.data_ptr(), N, 1, None, None, 0, 0,
                                     None, 0, D.data_ptr(), N, 1, stream()), name)
        acc = D0.double()
        mag = D0.double().abs()
        for k0, k1 in MW.spans(K, 32768):
            a, b = A[k0:k1].double(), B[k0:k1].double()
            acc += a.T @ b
            mag += a.abs().T @ b.abs()
        nan_rows(D, M)
        if integer:
            assert torch.equal(D[:M].double(), acc), "integer-operand dW differs from the exact sum"
            print("  integer operands: dW exact")
        else:
            R.check("dW", D[:M], acc, MW.gemm_bound(mag, K, splits + 1))


# ---------------------------------------------------------------------------------------------------------------------
# attention, training form: forward keeps lse, backward reads out + lse and writes dbias
# ---------------------------------------------------------------------------------------------------------------------
# Dispatch: the comment at the top of csrc/attention.cu.  Each direction names its kernel, the bound on CTAs per SM and
# (frames, heads) per item at most, so that items >= ceil(B / frames) * (h / heads).
TC5_F = ("attn_tc5_fwd_kernel (tc5_preferred: T > 80 or dh = 64)", 4, 1, 1)     # 512 / tmem_cols, tmem_cols >= 128
TC5_B = ("attn_tc5_bwd_kernel (tc5_preferred: dh = 32 at T > 80, dh = 64)", 1, 1, 1)   # occ = 1 in attn_tc5_bwd
TILE = ("attn_tile_*_kernel (attn_tiles.cu; a unit is G | h heads of a frame)", 32, 1, None)  # occupancy API: hw ceiling
MMA = ("attn_mma_*_kernel (T <= 16; F <= 8 frames per item)", 8, 8, None)      # mma_ctas_per_sm <= 8
FRAMES = ("attn_frames_*_kernel<float, 16> (fp32, T <= 32, dh <= 32; F <= 256 / (h T) frames per item)", 2, None, None)

ATTN_CASES = [
    # id, dtype, B, T, h, dh, forward, backward, lse kept
    ("tc5-T129-dh32", _lib.BF16, 229, 129, 8, 32, TC5_F, TC5_B, True),
    ("tc5-T257-dh32-two-threads-per-row", _lib.BF16, 229, 257, 8, 32, TC5_F, TC5_B, True),
    ("tc5-T65-dh64-64-row-tiles", _lib.BF16, 449, 65, 4, 64, TC5_F, TC5_B, True),
    ("tc5-fwd-tile-bwd-T129-dh16", _lib.BF16, 14209, 129, 8, 16, TC5_F, TILE, True),
    ("tiles-T33-dh32", _lib.BF16, 14209, 33, 8, 32, TILE, TILE, True),
    ("tiles-T65-dh16", _lib.BF16, 14209, 65, 4, 16, TILE, TILE, True),
    ("tiles-T288-dh16", _lib.BF16, 14209, 288, 2, 16, TILE, TILE, True),
    ("mma-T9-dh32-bench", _lib.BF16, 32768, 9, 8, 32, MMA, MMA, False),
    ("mma-T16-dh16", _lib.BF16, 28501, 16, 8, 16, MMA, MMA, False),
    ("frames-fp32-T9-dh32", _lib.F32, 2711, 9, 8, 32, FRAMES, FRAMES, False),
]


def attn_items(spec, B, T, h):
    _, ctas, frames, heads = spec
    frames = frames or max(1, 256 // (h * T))
    return -(-B // frames) * (h // (heads or h)), ctas


def attn_buffers(dt, B, T, h, dh):
    d = h * dh
    et = torch.float32 if dt == _lib.F32 else torch.bfloat16
    nan = float("nan")
    return dict(out=torch.full((B * T, d), nan, device=DEV, dtype=et), lse=torch.full((B, h, T), nan, device=DEV),
                dqkv=torch.full((B * T, 3 * d), nan, device=DEV, dtype=et), dbias=torch.zeros(3 * d, device=DEV))


def attn_call(dt, T, h, dh, qkv, dout, Z, f0, f1, keep_lse):
    b = f1 - f0
    rows = slice(f0 * T, f1 * T)
    lse = Z["lse"][f0:f1].data_ptr() if keep_lse else None
    _lib.check(_lib.lib.amc_attention_fwd(dt, b, T, h, dh, qkv[rows].data_ptr(), Z["out"][rows].data_ptr(), lse,
                                          stream()), "amc_attention_fwd")
    _lib.check(_lib.lib.amc_attention_bwd(dt, b, T, h, dh, qkv[rows].data_ptr(), Z["out"][rows].data_ptr(), lse,
                                          dout[rows].data_ptr(), Z["dqkv"][rows].data_ptr(), Z["dbias"].data_ptr(),
                                          stream()), "amc_attention_bwd")


def attn_inputs(dt, B, T, h, dh, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    et = torch.float32 if dt == _lib.F32 else torch.bfloat16
    d = h * dh
    return (torch.randn(B * T, 3 * d, device=DEV, generator=g).to(et),
            torch.randn(B * T, d, device=DEV, generator=g).to(et))


def check_attention(dt, B, T, h, dh, qkv, dout, Z, keep_lse):
    """Check 2: out, lse, dqkv element by element (reference in frame chunks), dbias against the column sums."""
    ref_frames = max(1, (1 << 25) // (h * T * T))        # [frames, h, T, T] float64 temporaries of <= 256 MB
    names = ["out", "dqkv"] + (["lse"] if keep_lse else [])
    worst = {n: 0.0 for n in names}
    db_ref = torch.zeros(3 * h * dh, device=DEV, dtype=torch.float64)
    db_mag = torch.zeros_like(db_ref)
    db_err = torch.zeros_like(db_ref)
    for f0, f1 in MW.spans(B, ref_frames):
        rows = slice(f0 * T, f1 * T)
        r = MW.attention_ref(qkv[rows].double(), dout[rows].double(), Z["out"][rows].double(), T, h, dh,
                             dt == _lib.BF16)
        for n in names:
            got = Z[n][f0:f1] if n == "lse" else Z[n][rows]
            worst[n] = max(worst[n], R.check(f"{n}[{f0}:{f1}]", got, r[n], r["e_" + n], quiet=True))
        db_ref += r["dqkv"].sum(0)
        db_mag += r["dqkv"].abs().sum(0)
        db_err += r["e_dqkv"].sum(0)
    for n in names:
        print(f"  {n}: worst err/bound {worst[n]:.3g}")
    R.check("dbias", Z["dbias"], db_ref, db_err + R.C_ACC * (B * T + 1) * R.U * db_mag)


@pytest.mark.parametrize("case", ATTN_CASES, ids=[c[0] for c in ATTN_CASES])
def test_attention_multiwave(case):
    name, dt, B, T, h, dh, fwd, bwd, keep_lse = case
    print(f"\n{name}: B={B} T={T} h={h} dh={dh}\n  forward: {fwd[0]}\n  backward: {bwd[0]}")
    report_items("forward", *attn_items(fwd, B, T, h))
    report_items("backward", *attn_items(bwd, B, T, h))
    qkv, dout = attn_inputs(dt, B, T, h, dh, B + T * 31 + dh)
    Z = attn_buffers(dt, B, T, h, dh)
    attn_call(dt, T, h, dh, qkv, dout, Z, 0, B, keep_lse)
    torch.cuda.synchronize()

    # 1. chunks of at most 148 (frame, head) units: every output without atomics equal bit for bit
    Z1 = attn_buffers(dt, B, T, h, dh)
    fc = MW.attn_chunk_frames(T, h)
    for f0, f1 in MW.spans(B, fc):
        attn_call(dt, T, h, dh, qkv, dout, Z1, f0, f1, keep_lse)
    torch.cuda.synchronize()
    for n in ("out", "dqkv") + (("lse",) if keep_lse else ()):
        assert not torch.isnan(Z[n].float()).any(), f"{n}: not written completely"
        assert torch.equal(Z[n], Z1[n]), f"{n}: chunked replay ({fc} frames) differs"
    print(f"  replay in chunks of {fc} frames: out, dqkv{', lse' if keep_lse else ''} equal bit for bit")
    del Z1

    # 2. float64
    check_attention(dt, B, T, h, dh, qkv, dout, Z, keep_lse)


# The bound of multiwave_ref.attention_ref at single-wave shapes test_gpu_ops.py passes (one per kernel), before it is
# relied on at the multi-wave sizes above.
@pytest.mark.parametrize("dt,B,T,h,dh,keep_lse", [(_lib.BF16, 2, 129, 8, 32, True), (_lib.BF16, 1, 257, 8, 32, True),
                                                  (_lib.BF16, 3, 65, 8, 16, True), (_lib.BF16, 4, 33, 8, 32, True),
                                                  (_lib.BF16, 1, 288, 2, 16, True), (_lib.BF16, 2, 129, 8, 16, True),
                                                  (_lib.BF16, 50, 9, 8, 32, False), (_lib.BF16, 4, 16, 4, 16, False),
                                                  (_lib.F32, 37, 9, 8, 32, False)])
def test_attention_bound_single_wave(dt, B, T, h, dh, keep_lse):
    qkv, dout = attn_inputs(dt, B, T, h, dh, T * 31 + dh)
    Z = attn_buffers(dt, B, T, h, dh)
    attn_call(dt, T, h, dh, qkv, dout, Z, 0, B, keep_lse)
    torch.cuda.synchronize()
    check_attention(dt, B, T, h, dh, qkv, dout, Z, keep_lse)


# ---------------------------------------------------------------------------------------------------------------------
# amc_layernorm_bwd: ln_bwd_vec_kernel (rowops.cu ln_bwd, d % 128 == 0), grid = min(items, 148 x 2)
# ---------------------------------------------------------------------------------------------------------------------
LN_M = 30011        # >= 3 x 296 x 32 rows; an item is 8 warps x R rows (R = 4 for d <= 256, 2 above)


@pytest.mark.parametrize("d", [256, 512])
@pytest.mark.parametrize("dt", [_lib.F32, _lib.BF16], ids=["fp32", "bf16"])
def test_layernorm_bwd_multiwave(dt, d):
    M = LN_M
    per_item = 8 * (4 if d <= 256 else 2)
    print(f"\nln_bwd_vec_kernel<{'float' if dt == _lib.F32 else 'bf16'}, {d // 128}>: M={M} d={d}")
    report_items(f"{per_item}-row items", -(-M // per_item), 2)
    et = torch.float32 if dt == _lib.F32 else torch.bfloat16
    g = torch.Generator(device=DEV).manual_seed(M + d + dt)
    dy = torch.randn(M, d, device=DEV, generator=g)
    xh = torch.randn(M, d, device=DEV, generator=g).to(et)
    rstd = 0.5 + torch.rand(M, device=DEV, generator=g)
    gamma = torch.randn(d, device=DEV, generator=g)

    def outputs():
        return (torch.full((M + PAD_ROWS, d), float("nan"), device=DEV, dtype=et),
                torch.full((M + PAD_ROWS, d), float("nan"), device=DEV), torch.zeros(d, device=DEV),
                torch.zeros(d, device=DEV))

    def call(out, r0, r1):
        du16, du32, dgamma, dbeta = out
        _lib.check(_lib.lib.amc_layernorm_bwd(dt, r1 - r0, d, dy[r0:r1].data_ptr(), xh[r0:r1].data_ptr(),
                                              rstd[r0:r1].data_ptr(), gamma.data_ptr(), du16[r0:r1].data_ptr(),
                                              du32[r0:r1].data_ptr(), dgamma.data_ptr(), dbeta.data_ptr(), stream()),
                   "amc_layernorm_bwd")

    O = outputs()
    call(O, 0, M)
    O1 = outputs()
    rows = MW.LAUNCH_SMS * per_item
    for r0, r1 in MW.spans(M, rows):
        call(O1, r0, r1)
    torch.cuda.synchronize()
    assert torch.equal(O[0][:M], O1[0][:M]) and torch.equal(O[1][:M], O1[1][:M]), "chunked replay differs"
    print(f"  replay in chunks of {rows} rows: du16, du32 equal bit for bit")
    nan_rows(O[0], M)
    nan_rows(O[1], M)
    x = xh.double()
    du, e_du = MW.ln_bwd_ref(dy.double(), torch.zeros(M, d, device=DEV, dtype=torch.float64), x, rstd.double(),
                             gamma.double())
    R.check("du32", O[1][:M], du, e_du)
    R.check("du16", O[0][:M], du, MW.bf16_bound(du, e_du) if dt == _lib.BF16 else e_du)
    zero = torch.zeros(M, d, device=DEV, dtype=torch.float64)
    R.check("dgamma", O[2], (dy.double() * x).sum(0), MW.colsum_bound(dy.double() * x, zero))
    R.check("dbeta", O[3], dy.double().sum(0), MW.colsum_bound(dy.double(), zero))

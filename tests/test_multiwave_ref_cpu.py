"""CPU checks of tests/multiwave_ref.py: the items-per-CTA arithmetic, the chunking that makes every launch single-wave,
and the bound functions, which must hold for emulated fp32 / bf16 kernels and reject each planted defect of the kind a
persistent kernel's carried state can produce.  For each defect the test also records whether the max-normalised
``relerr < 2e-2`` check of test_gpu_ops.py would have caught it: it catches every defect planted at full size, and
lets the two small ones through."""
import math

import numpy as np
import pytest
import torch

import isolated_ref as R
import multiwave_ref as MW

F64 = torch.float64


def t64(a):
    return torch.from_numpy(np.asarray(a, dtype=np.float64))


def relerr_catches(got, ref):
    got, ref = np.asarray(got, dtype=np.float64), np.asarray(ref, dtype=np.float64)
    return float(np.abs(got - ref).max() / max(np.abs(ref).max(), 1e-30)) >= 2e-2


# ---------------------------------------------------------------------------------------------------------------------
# items per CTA and chunking
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("items,sms,ctas", [(445, 148, 1), (1335, 148, 1), (4096, 148, 8), (1832, 148, 4), (100, 148, 1),
                                            (14209, 148, 32), (938, 132, 2), (5000, 160, 1)])
def test_min_items_per_cta_matches_the_persistent_loop(items, sms, ctas):
    grid = min(items, MW.grid_cap(sms, ctas))
    counts = [len(range(b, items, grid)) for b in range(grid)]
    assert min(counts) >= MW.min_items_per_cta(items, sms, ctas)
    if grid == MW.grid_cap(sms, ctas):          # the full grid: the bound is attained
        assert min(counts) == MW.min_items_per_cta(items, sms, ctas)


def test_multiwave_case_sizes_give_three_items():
    assert MW.min_items_per_cta(445 * 1, 148, 1) == 3             # M = 56,905, one N tile
    assert MW.min_items_per_cta(14209, 148, 32) == 3              # tile attention, hardware ceiling
    assert MW.min_items_per_cta(-(-32768 // 8), 148, 8) == 3      # attn_mma at the bench's B
    assert MW.min_items_per_cta(-(-30011 // 32), 148, 2) == 3     # ln_bwd_vec at d = 256


def test_spans_cover_in_order():
    for n, size in [(56905, 4736), (10, 3), (7, 7), (1, 5)]:
        s = MW.spans(n, size)
        assert s[0][0] == 0 and s[-1][1] == n
        assert all(a[1] == b[0] for a, b in zip(s, s[1:]))
        assert all(0 < i1 - i0 <= size for i0, i1 in s)


@pytest.mark.parametrize("tiles_n", [1, 2, 3, 4, 5, 8, 148])
def test_gemm_chunks_are_single_wave(tiles_n):
    rows = MW.gemm_chunk_rows(tiles_n)
    assert rows % MW.BM == 0                                       # offsets stay 16-byte aligned
    assert (rows // MW.BM) * tiles_n <= MW.LAUNCH_SMS
    assert (rows // MW.BM + 1) * tiles_n > MW.LAUNCH_SMS           # and as large as that allows


@pytest.mark.parametrize("T,h", [(129, 8), (257, 8), (65, 4), (33, 8), (288, 2), (9, 8), (16, 8), (129, 3), (9, 5)])
def test_attention_chunks_are_single_wave_and_aligned(T, h):
    f = MW.attn_chunk_frames(T, h)
    assert f * h <= MW.LAUNCH_SMS
    assert (f * h * T * 4) % 16 == 0                               # lse offsets
    for dh in (16, 32, 64):
        assert (f * T * 3 * h * dh * 2) % 16 == 0 and (f * T * h * dh * 2) % 16 == 0


def test_gemm_tiles_and_split_k_plan():
    assert [MW.pick_bn(n) for n in (64, 128, 192, 256, 288, 320, 768, 1024)] == [64, 128, 64, 256, 64, 64, 256, 256]
    # the bench's weight gradients: about two waves of 128 x 128 tiles, BN = 256 -> 144 items on 148 SMs
    assert MW.split_k_items(768, 256, 294912) == (144, 24)
    assert MW.split_k_items(1024, 256, 294912) == (144, 18)
    assert MW.split_k_items(256, 1024, 294912) == (144, 18)
    assert MW.split_k_items(960, 320, 294912) == (480, 12)
    assert MW.split_k_items(960, 320, 73719) == (480, 12)
    assert MW.split_k_items(64, 32, 1000) == (3, 3)                # short K: K / 256 splits


# ---------------------------------------------------------------------------------------------------------------------
# GEMM: an emulated kernel passes, planted defects fail
# ---------------------------------------------------------------------------------------------------------------------
M, N, K, BN = 512, 256, 256, 64          # 4 row tiles, 4 N tiles, 4 k-blocks


def gemm_case(seed=0, small_kblock=False):
    g = np.random.default_rng(seed)
    A = R.bf16_rne(g.standard_normal((M, K)).astype(np.float32))
    if small_kblock:                                                # k-block 1 of A 64 times smaller (still exact bf16)
        A[:, 64:128] *= np.float32(2.0 ** -6)
    B = R.bf16_rne((g.standard_normal((N, K)) / np.sqrt(K)).astype(np.float32))
    bias = g.standard_normal(N).astype(np.float32)
    res = g.standard_normal((M + 32, N)).astype(np.float32)
    acc = A @ B.T                                                   # fp32 accumulation
    ref = A.astype(np.float64) @ B.T.astype(np.float64)
    mag = np.abs(A).astype(np.float64) @ np.abs(B.T).astype(np.float64)
    return A, B, bias, res, acc, ref, mag


def gemm_defects():
    A, B, bias, res, acc, ref, mag = gemm_case()
    good = acc + bias + res[:M]
    r64 = ref + bias + res[:M].astype(np.float64)
    bound = MW.gemm_bound(t64(mag + np.abs(bias) + np.abs(res[:M])), K, 2)
    out = {}
    d = good.copy()                                                 # tile 1 misses its second k-block
    d[128:256] -= A[128:256, 64:128] @ B[:, 64:128].T
    out["missing k-block"] = d
    d = good.copy()                                                 # tile 2 accumulates onto tile 1's accumulator
    d[256:384] += acc[128:256]
    out["previous tile's accumulator"] = d
    d = good.copy()                                                 # N tile 1 adds the bias of N tile 2
    d[:, BN:2 * BN] += bias[2 * BN:3 * BN] - bias[BN:2 * BN]
    out["neighbouring N tile's bias"] = d
    d = good.copy()                                                 # tile 1's residual slab one quadrant late
    d[128:256] = acc[128:256] + bias + res[160:288]
    out["residual shifted by one quadrant"] = d
    A, B, bias, res, acc, ref, mag = gemm_case(small_kblock=True)  # the same k-block missing, small operands
    d = acc + bias + res[:M]
    d[128:256] -= A[128:256, 64:128] @ B[:, 64:128].T
    out["missing k-block, small operands"] = (d, ref + bias + res[:M].astype(np.float64),
                                              MW.gemm_bound(t64(mag + np.abs(bias) + np.abs(res[:M])), K, 2))
    return good, r64, bound, out


# which planted defects the max-normalised relerr < 2e-2 would let through (False = let through).  At full size every
# defect of the list is caught by it too; the small ones (a k-block of operands 64 times smaller, an lse 1.5 % off in
# its exponential, as a neighbour of nearly equal row statistics would give) are rejected only by the per-element bound.
RELERR_CATCHES = {"missing k-block": True, "previous tile's accumulator": True, "neighbouring N tile's bias": True,
                  "residual shifted by one quadrant": True, "missing k-block, small operands": False,
                  "neighbour's lse": True, "leftover row, neighbour's V": True, "neighbour's lse, 1.5 % off": False}


def test_gemm_bound_holds_for_fp32_accumulation():
    good, r64, bound, _ = gemm_defects()
    R.check("emulated D32", t64(good), t64(r64), bound)
    bf = R.bf16_rne(good)
    R.check("emulated D16", t64(bf), t64(r64), MW.bf16_bound(t64(r64), bound))


@pytest.mark.parametrize("name", ["missing k-block", "previous tile's accumulator", "neighbouring N tile's bias",
                                  "residual shifted by one quadrant", "missing k-block, small operands"])
def test_gemm_defect_is_rejected(name):
    _, r64, bound, defects = gemm_defects()
    bad = defects[name]
    if isinstance(bad, tuple):                                      # a defect planted in its own case
        bad, r64, bound = bad
    with pytest.raises(AssertionError, match="out of bound"):
        R.check(name, t64(bad), t64(r64), bound)
    with pytest.raises(AssertionError, match="out of bound"):       # also after the bf16 output rounding
        R.check(name, t64(R.bf16_rne(bad)), t64(r64), MW.bf16_bound(t64(r64), bound))
    print(f"  {name}: relerr < 2e-2 {'catches' if relerr_catches(bad, r64) else 'lets it through'}")
    assert relerr_catches(bad, r64) == RELERR_CATCHES[name]


def test_integer_operands_are_exact_in_any_order():
    """The premise of check 3: integer bf16 operands in -3..3 give the exact sum in fp32 whatever the order."""
    g = np.random.default_rng(3)
    K_ = 294912
    a = g.integers(-3, 4, K_).astype(np.float32)
    b = g.integers(-3, 4, K_).astype(np.float32)
    p = a * b
    exact = float(np.dot(a.astype(np.float64), b.astype(np.float64)))
    assert 9 * K_ < 2 ** 24
    for order in (np.arange(K_), g.permutation(K_)):
        s = np.float32(0)
        for chunk in np.array_split(p[order], 24):                   # split-K: partial sums, then added
            s = np.float32(s + np.cumsum(chunk, dtype=np.float32)[-1])
        assert float(s) == exact


# ---------------------------------------------------------------------------------------------------------------------
# attention: an emulated bf16 kernel passes, planted defects fail
# ---------------------------------------------------------------------------------------------------------------------
NB, T, H, DH = 2, 129, 2, 32            # 4 (frame, head) units, T = 129: a 128-row tile and a leftover row


def attention_case(seed=1):
    g = np.random.default_rng(seed)
    d = H * DH
    qkv = R.bf16_rne(g.standard_normal((NB * T, 3 * d)).astype(np.float32))
    q, k, v = (qkv.reshape(NB, T, 3, H, DH)[:, :, i].transpose(0, 2, 1, 3).astype(np.float32) for i in range(3))
    s = (q @ k.transpose(0, 1, 3, 2)) * np.float32(1 / math.sqrt(DH))
    mx = s.max(-1, keepdims=True)
    e = np.exp(s - mx)
    lse = mx + np.log(e.sum(-1, keepdims=True))                     # fp32 row statistics
    return qkv, q, k, v, s, lse


def emulate_out(q, k, v, s, lse, lse_used=None, v_row128=None):
    """The tensor-core forward in fp32 with bf16 P and a bf16 output; optional defects."""
    P = np.exp(s - (lse if lse_used is None else lse_used)).astype(np.float32)
    o = R.bf16_rne(P) @ v
    if v_row128 is not None:
        o[:, :, 128] = (R.bf16_rne(P[:, :, 128])[:, :, None, :] @ v_row128)[:, :, 0]
    return R.bf16_rne(o.transpose(0, 2, 1, 3).reshape(NB * T, H * DH))


def attention_defects():
    qkv, q, k, v, s, lse = attention_case()
    ref = MW.attention_ref(t64(qkv), torch.zeros(NB * T, H * DH, dtype=F64), torch.zeros(NB * T, H * DH, dtype=F64),
                           T, H, DH)
    good = emulate_out(q, k, v, s, lse)
    u = lambda x: x.reshape(NB * H, *x.shape[2:])                    # noqa: E731  (units: frame-major, head-minor)
    uu = lambda x: x.reshape(NB, H, *x.shape[1:])                    # noqa: E731
    lse_bad = u(lse).copy()
    lse_bad[1] = u(lse)[2]                                           # unit 1 normalised with unit 2's lse
    v_bad = u(v).copy()
    v_bad[1] = u(v)[2]
    lse_near = u(lse).copy()
    lse_near[1] += np.float32(0.015)                                # unit 1: P scaled by exp(-0.015)
    out = {"neighbour's lse": emulate_out(q, k, v, s, lse, lse_used=uu(lse_bad)),
           "neighbour's lse, 1.5 % off": emulate_out(q, k, v, s, lse, lse_used=uu(lse_near)),
           "leftover row, neighbour's V": emulate_out(q, k, v, s, lse, v_row128=uu(v_bad))}
    return good, ref, out


def test_attention_bound_holds_for_the_emulated_kernel():
    good, ref, _ = attention_defects()
    R.check("emulated out", t64(good), ref["out"], ref["e_out"])


@pytest.mark.parametrize("name", ["neighbour's lse", "leftover row, neighbour's V", "neighbour's lse, 1.5 % off"])
def test_attention_defect_is_rejected(name):
    _, ref, defects = attention_defects()
    bad = defects[name]
    with pytest.raises(AssertionError, match="out of bound"):
        R.check(name, t64(bad), ref["out"], ref["e_out"])
    print(f"  {name}: relerr < 2e-2 {'catches' if relerr_catches(bad, ref['out']) else 'lets it through'}")
    assert relerr_catches(bad, ref["out"].numpy()) == RELERR_CATCHES[name]


def test_attention_gradient_bound_holds_for_float32_math():
    """dqkv of fp32 math on the same operands (no bf16 rounding of P or dS) is inside the bf16 bound, and the fp32 bound
    (c = 0 rounding term) holds for it as well."""
    qkv, *_ = attention_case()
    g = np.random.default_rng(2)
    dout = R.bf16_rne(g.standard_normal((NB * T, H * DH)).astype(np.float32))
    x = torch.from_numpy(qkv).requires_grad_(True)
    q, k, v = [y.view(NB, T, H, DH).transpose(1, 2) for y in x.view(NB, T, 3 * H * DH).split(H * DH, -1)]
    o = (torch.softmax(q @ k.transpose(2, 3) / math.sqrt(DH), -1) @ v).transpose(1, 2).reshape(NB * T, -1)
    o.backward(torch.from_numpy(dout))
    for bf16 in (True, False):
        ref = MW.attention_ref(t64(qkv), t64(dout), o.detach().double(), T, H, DH, bf16)
        R.check(f"fp32 out (bf16 bound {bf16})", o.detach().double(), ref["out"], ref["e_out"])
        R.check(f"fp32 dqkv (bf16 bound {bf16})", x.grad.double(), ref["dqkv"], ref["e_dqkv"])


# ---------------------------------------------------------------------------------------------------------------------
# LayerNorm bounds against fp32 arithmetic, and a neighbouring N tile's gamma rejected
# ---------------------------------------------------------------------------------------------------------------------
def test_layernorm_bounds_hold_for_fp32_and_reject_a_neighbours_gamma():
    g = np.random.default_rng(4)
    Mr, Nc = 300, 256
    u = (g.standard_normal((Mr, Nc)) * 2 + 0.3).astype(np.float32)
    gamma = g.standard_normal(Nc).astype(np.float32)
    beta = g.standard_normal(Nc).astype(np.float32)
    mean = u.mean(-1, keepdims=True, dtype=np.float32)
    var = ((u - mean) ** 2).mean(-1, keepdims=True, dtype=np.float32)
    rstd = (np.float32(1) / np.sqrt(var + np.float32(1e-5))).astype(np.float32)
    xhat = (u - mean) * rstd
    y = gamma * xhat + beta
    L = MW.ln_fwd_ref(t64(u), torch.zeros(Mr, Nc, dtype=F64), t64(gamma), t64(beta), 1e-5)
    R.check("y32", t64(y), L["y"], L["e_y"])
    R.check("xhat16", t64(R.bf16_rne(xhat)), L["xhat"], MW.bf16_bound(L["xhat"], L["e_xhat"]))
    R.check("rstd", t64(rstd[:, 0]), L["rstd"], L["e_rstd"])
    y_bad = y.copy()
    y_bad[:, 64:128] = gamma[128:192] * xhat[:, 64:128] + beta[64:128]
    with pytest.raises(AssertionError, match="out of bound"):
        R.check("y32, neighbouring gamma", t64(y_bad), L["y"], L["e_y"])

    dy = g.standard_normal((Mr, Nc)).astype(np.float32)
    xh = R.bf16_rne(xhat)
    gg = dy * gamma
    s1 = gg.mean(-1, keepdims=True, dtype=np.float32)
    s2 = (gg * xh).mean(-1, keepdims=True, dtype=np.float32)
    du = rstd * (gg - s1 - xh * s2)
    ref, e = MW.ln_bwd_ref(t64(dy), torch.zeros(Mr, Nc, dtype=F64), t64(xh), t64(rstd[:, 0]), t64(gamma))
    R.check("du32", t64(du), ref, e)
    du_bad = rstd * (dy * np.roll(gamma, -64) - s1 - xh * s2)
    with pytest.raises(AssertionError, match="out of bound"):
        R.check("du32, neighbouring gamma", t64(du_bad), ref, e)

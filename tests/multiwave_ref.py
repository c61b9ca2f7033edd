"""Helpers of tests/test_gpu_multiwave.py: how many work items the persistent kernels give each CTA, the chunking that
replays a problem with one item per CTA, and float64 references with per-element error bounds (torch, any device).

Persistent launches (csrc/gemm_tc.cu launch / launch_row, attn_tc5.cu, attn_tiles.cu, attention.cu, rowops.cu ln_bwd)
size the grid as min(items, SMs x CTAs per SM) and loop ``for (item = blockIdx.x; item < n; item += gridDim.x)``.  The
launch code multiplies by ``device_sm_count()`` or by the literal 148 of the B200; ``max(sms, 148)`` covers both.

Bounds follow tests/isolated_ref.py: fp32 sums of n terms are within C_ACC * n * u * sum|terms|, and a bf16 result is
within 2^-9 of its fp32 value, relative (written 2^-8 * (|ref| + e), which also covers the fp32 error e it rounds)."""
import math

import torch

from isolated_ref import C_ACC, U

LAUNCH_SMS = 148        # the B200's SM count, written into some of the launch code
BM = 128                # rows of a GEMM tile (csrc/gemm_tc.cu)
BK = 64                 # k-block of the GEMM main loop
BF16_REL = 2.0 ** -8    # two bf16 roundings (2 x 2^-9), or one of a value carrying an fp32 error


def grid_cap(sms, ctas_per_sm):
    """Largest grid a persistent launch can have on ``sms`` SMs with at most ``ctas_per_sm`` resident CTAs."""
    return max(sms, LAUNCH_SMS) * ctas_per_sm


def min_items_per_cta(items, sms, ctas_per_sm):
    """Least number of items any CTA of the launch processes: grid <= grid_cap, CTA b takes items b, b + grid, ..."""
    return items // grid_cap(sms, ctas_per_sm)


def spans(n, size):
    """[(i0, i1)] covering range(n) in pieces of ``size`` (the last one ragged)."""
    assert size > 0
    return [(i, min(n, i + size)) for i in range(0, n, size)]


def gemm_chunk_rows(tiles_n, cap=LAUNCH_SMS):
    """Rows of a GEMM chunk whose launch has at most ``cap`` tiles: floor(cap / tiles_n) row tiles of 128."""
    assert 1 <= tiles_n <= cap
    return (cap // tiles_n) * BM


def attn_chunk_frames(T, h, units_per_frame=None, cap=LAUNCH_SMS):
    """Frames of an attention chunk with at most ``cap`` units (a unit is a (frame, head) or (frame, head group)), cut
    so that every chunk offset of the fp32 lse [B, h, T] stays 16-byte aligned (the bf16 rows are: d % 16 == 0)."""
    f = cap // (units_per_frame or h)
    while f > 1 and (f * h * T) % 4:
        f -= 1
    assert f >= 1 and (f * h * T) % 4 == 0, (T, h)
    return f


def pick_bn(N):
    """N tile of gemm_bf16 for the plain row epilogues and the generic kernel: least padding, ties to the larger."""
    best, pad = 256, -(-N // 256) * 256
    for bn in (128, 64):
        p = -(-N // bn) * bn
        if p < pad:
            best, pad = bn, p
    return best


def split_k_items(M, N, K):
    """(tile, split) items of amc_gemm's split-K weight gradient: pick_split_k in api.cu, then launch<BN, 1>."""
    tiles128 = -(-M // 128) * (-(-N // 128))
    s = max(1, 296 // max(tiles128, 1))
    s = min(s, max(1, K // 256))
    kb_total = -(-K // BK)
    s = max(1, min(s, kb_total))
    per = -(-kb_total // s)
    splits = -(-kb_total // per)
    return -(-M // BM) * (-(-N // pick_bn(N))) * splits, splits


# ---------------------------------------------------------------------------------------------------------------------
# float64 references and bounds
# ---------------------------------------------------------------------------------------------------------------------
def bf16_bound(ref, e):
    """Bound of a bf16 output whose fp32 value is within e of ref."""
    return e + BF16_REL * (ref.abs() + e)


def gemm_bound(mag, K, extra_terms=1):
    """fp32 accumulation of K exact products plus ``extra_terms`` fp32 additions; ``mag`` is the sum of the absolute
    values of every term (|A| |B| + |bias| + |res| ...)."""
    return C_ACC * (K + extra_terms) * U * mag


def ln_fwd_ref(u, e_u, gamma, beta, eps):
    """LayerNorm of rows u [M, N] (float64) whose values are within e_u of the kernel's fp32 u: y, xhat, rstd and their
    bounds.  Mean and variance are N-term fp32 sums (a one-pass E[u^2] - mean^2 form is covered: its error scales with
    mean(u^2)); rsqrtf is within 2 ulp."""
    N = u.shape[-1]
    mean = u.mean(-1, keepdim=True)
    c = u - mean
    var = (c * c).mean(-1, keepdim=True)
    rstd = 1.0 / torch.sqrt(var + eps)
    xhat = c * rstd
    y = gamma * xhat + beta
    a = C_ACC * (N + 4) * U
    e_mean = a * u.abs().mean(-1, keepdim=True) + e_u.mean(-1, keepdim=True)
    e_var = a * (u * u).mean(-1, keepdim=True) + 2 * (c.abs() * (e_u + e_mean)).mean(-1, keepdim=True)
    e_rstd = rstd * (e_var / (2 * (var + eps)) + 4 * U)
    e_xhat = c.abs() * e_rstd + rstd * (e_u + e_mean) + 2 * U * xhat.abs()
    e_y = gamma.abs() * e_xhat + 2 * U * ((gamma * xhat).abs() + beta.abs())
    return dict(y=y, e_y=e_y, xhat=xhat, e_xhat=e_xhat, rstd=rstd.squeeze(-1), e_rstd=e_rstd.squeeze(-1))


def ln_bwd_ref(t, e_t, xh, rstd, gamma):
    """du = rstd (g - mean(g) - xh mean(g xh)), g = t gamma, for the forward's xhat / rstd as stored, and its bound (the
    form of isolated_ref.head_bwd_ref); t is within e_t of the kernel's fp32 t."""
    N = t.shape[-1]
    rs = rstd.unsqueeze(-1)
    g = t * gamma
    du = rs * (g - g.mean(-1, keepdim=True) - xh * (g * xh).mean(-1, keepdim=True))
    ag, axh = g.abs(), xh.abs()
    e_g = gamma.abs() * e_t + U * ag
    e_du = rs * (C_ACC * (N + 4) * U * (ag + ag.mean(-1, keepdim=True) + axh * (ag * axh).mean(-1, keepdim=True))
                 + e_g + e_g.mean(-1, keepdim=True) + axh * (e_g * axh).mean(-1, keepdim=True)) + 2 * U * du.abs()
    return du, e_du


def colsum_bound(x, e_x):
    """Bound of fp32 column sums of M rows accumulated through per-CTA partials and atomics."""
    return C_ACC * (x.shape[0] + 1) * U * x.abs().sum(0) + e_x.sum(0)


def attention_ref(qkv, dout, out_k, T, h, dh, bf16=True, c=2.0):
    """Training-form attention of frames qkv [b T, 3 d] (float64 holding the kernels' input values) in float64: out,
    the log2-domain lse, and for dL/dout = dout the gradient dqkv, each with a per-element bound.  out_k is the forward
    output the backward reads (its D = rowsum(dO o O) uses those values, as the kernels do).

    Bound (bf16 kernels): the tensor-core kernels round P to bf16 before P V and before P^T dO, round dS = P (dP - D) to
    bf16 before dS K and dS^T Q, and store bf16 outputs: two roundings of 2^-9 on each path, c 2^-8 with c = 2 for
    slack, times the absolute-value product of the path: |P| |V| for out, |dS| |K| for dq, |dS|^T |Q| for dk, |P|^T |dO|
    for dv.  What the fp32 arithmetic adds is within C_ACC (T + dh + 4) u of the same products, plus the error of P
    itself (fp32 scores, the fp32 exponent argument s log2e - lse, ex2.approx): relative C_ACC (T + dh + 4) u
    (|Q| |K|^T scale + |lse| + 1), carried through P V, P (dP - D) and P^T dO; D carries C_ACC (T + dh + 4) u, and
    2^-8 where a kernel forms it from its own fp32 O, of sum |dO o O|.  fp32 kernels: no rounding term."""
    b = qkv.shape[0] // T
    d = h * dh
    split = lambda x, n: [y.reshape(b, T, h, dh).transpose(1, 2) for y in x.reshape(b, T, n * d).split(d, -1)]  # noqa
    q, k, v = split(qkv, 3)
    do, = split(dout, 1)
    o, = split(out_k, 1)
    sc = 1.0 / math.sqrt(dh)
    kt = k.transpose(-1, -2)
    s = (q @ kt) * sc
    lse = torch.logsumexp(s, -1, keepdim=True)
    P = torch.exp(s - lse)
    rnd = c * BF16_REL if bf16 else 0.0
    acc = C_ACC * (T + dh + 4) * U
    eP = P * acc * ((q.abs() @ kt.abs()) * sc + lse.abs() + 1.0)
    out = P @ v
    e_out = (rnd + acc) * (P @ v.abs()) + eP @ v.abs()
    dP = do @ v.transpose(-1, -2)
    D = (do * o).sum(-1, keepdim=True)
    dS = P * (dP - D)
    # (kernels that recompute O instead of reading out_k form D from their fp32 O: within 2^-9 of the bf16 out_k)
    e_D = (acc + (BF16_REL if bf16 else 0.0)) * (do * o).abs().sum(-1, keepdim=True)
    e_dS = P * (acc * (do.abs() @ v.abs().transpose(-1, -2)) + e_D) + eP * (dP - D).abs()
    aS = dS.abs()
    dq = (dS @ k) * sc
    dk = (dS.transpose(-1, -2) @ q) * sc
    dv = P.transpose(-1, -2) @ do
    e_dq = ((rnd + acc) * (aS @ k.abs()) + e_dS @ k.abs()) * sc
    e_dk = ((rnd + acc) * (aS.transpose(-1, -2) @ q.abs()) + e_dS.transpose(-1, -2) @ q.abs()) * sc
    e_dv = (rnd + acc) * (P.transpose(-1, -2) @ do.abs()) + eP.transpose(-1, -2) @ do.abs()
    rows = lambda x: x.transpose(1, 2).reshape(b * T, -1)  # noqa
    lse2 = lse.squeeze(-1) / math.log(2.0)
    e_lse2 = acc * (lse.abs().squeeze(-1) + s.abs().amax(-1) + 1.0) / math.log(2.0)
    return dict(out=rows(out), e_out=rows(e_out), lse=lse2, e_lse=e_lse2,
                dqkv=torch.cat([rows(dq), rows(dk), rows(dv)], -1),
                e_dqkv=torch.cat([rows(e_dq), rows(e_dk), rows(e_dv)], -1))

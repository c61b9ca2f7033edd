"""float64 references for the kernels around the encoder: the embedding front end (forward and backward, both input
layouts), the classifier head, cross-entropy with label smoothing, argmax, clip + AdamW and the IQ statistics sums.

Each reference starts from the operands the kernel actually multiplies: where the bf16 path rounds (the front end's
patch operand, W_emb, the token-row gradient demb, the transposed W_emb of the input gradient) the reference applies
the same round-to-nearest-even with ``bf16_rne`` and then computes in float64.  What is left between kernel and
reference is fp32 accumulation, which the ``*_bound`` values returned next to the results bound element by element.

Rounding points (vit-vs-raw-iq_b200/csrc/api.cu, Model::frontend / Model::backward / Model::input_grad):
  - patch operand: dataset layout z = fp32(fp32(x - mean) * fp32(1 / std)) (frontend_tc.cu store_block, rowops.cu
    patchify kernels; a subtract then a multiply, nothing to contract into an FMA), then bf16 in bf16 mode;
  - W_emb: bf16 copy of the fp32 blob (cast_blob) for the forward and the small-K kernels, bf16 transpose
    (transpose_batch) for the input-gradient GEMM: the same RNE values;
  - demb = bf16(fp32(dx0 * dropout scale)) (gather_tok_rows); the emb_w / emb_b gradients and the input gradient all
    read it; dcls sums fp32 dx0 (cls_grad);
  - dsrc = fp32(dX * fp32(1 / std)) in dataset layout (patch_scatter, embed_smallk_dgrad).
"""
from typing import Dict, Optional

import numpy as np

from oracle import amc_oracle as O

U = 2.0 ** -24          # unit roundoff of fp32
C_ACC = 4.0             # slack on the classical gamma_n = n*u bound (tensor-core adders, atomics, fused adds)


def check(what, got, ref, bound, quiet=False):
    """|got - ref| <= bound element by element (a zero bound demands exact equality).  numpy arrays or torch tensors;
    tensors are compared in float64 on the device of ``ref``.  Prints (unless ``quiet``) and returns the worst
    err/bound over the elements with a positive bound."""
    import torch

    def f64(x, device=None):        # numpy arrays and Python scalars go through float64 without an fp32 rounding
        if isinstance(x, torch.Tensor):
            return x.to(device or x.device, torch.float64)
        return torch.from_numpy(np.array(x, dtype=np.float64)).to(device or "cpu")

    ref = f64(ref)
    got = f64(got, ref.device)
    bound = f64(bound, ref.device).expand(ref.shape)
    assert got.shape == ref.shape, (what, tuple(got.shape), tuple(ref.shape))
    err = (got - ref).abs()
    bad = ~(err <= bound)
    pos = bound > 0
    worst = float((err[pos] / bound[pos]).max()) if bool(pos.any()) else 0.0
    if not quiet:
        print(f"  {what}: worst err/bound {worst:.3g}")
    if bool(bad.any()):
        i = np.unravel_index(int(bad.flatten().nonzero()[0, 0]), tuple(ref.shape))
        raise AssertionError(f"{what}: {int(bad.sum())} of {ref.numel()} elements out of bound; first at {i}: "
                             f"got {float(got[i])!r} ref {float(ref[i])!r} bound {float(bound[i])!r}")
    return worst


def bf16_rne(x):
    """float32 -> nearest bfloat16 (ties to even), computed on the float32 bit pattern; returned as float32."""
    a = np.ascontiguousarray(x, dtype=np.float32)
    u = a.view(np.uint32).astype(np.uint64)
    r = ((u + 0x7FFF + ((u >> 16) & 1)) >> 16) << 16
    r = np.where(np.isnan(a), (u | 0x400000) & 0xFFFF0000, r)     # NaN stays a (quiet) NaN
    return r.astype(np.uint32).view(np.float32).reshape(a.shape)


def p_effective(p: float) -> float:
    """The dropout probability the kernels apply: floor(p * 65536) / 65536 (include/amc_b200.h, AmcDesc.p_drop)."""
    return np.floor(float(np.float32(p)) * 65536.0) / 65536.0


def keep_scale(p: float) -> np.float32:
    return np.float32(1.0 / (1.0 - p_effective(p))) if p_effective(p) > 0 else np.float32(1.0)


def emb_key(cfg):
    return "encoder.sequence_embedding.projection" if cfg.kind == "rawiq" else "encoder.patch_embedding.projection"


def head_keys(cfg, head_ln):
    if head_ln:
        return "mlp_head.1.weight", "mlp_head.1.bias", "mlp_head.0.weight", "mlp_head.0.bias"
    return "mlp_head.weight", "mlp_head.bias", None, None


# ---------------------------------------------------------------------------------------------------------------------
# front end
# ---------------------------------------------------------------------------------------------------------------------
def zscore_f32(x, stats):
    """The kernel's fp32 z-score of interleaved dataset frames [B, L, 2]: (x - mean) * (1 / std), every step in fp32."""
    x = np.asarray(x, dtype=np.float32)
    mean = np.array([stats["i_mean"], stats["q_mean"]], dtype=np.float32)
    inv = np.float32(1.0) / np.array([stats["i_std"], stats["q_std"]], dtype=np.float32)
    return (x - mean) * inv


def model_layout(x, cfg, layout, stats=None, exact=False):
    """The model-layout frames the patch map reads: ``x`` itself, or the framed z-score of dataset frames (in fp32 as
    the kernel computes it, or with ``exact`` in float64 by division as the dataset code writes it)."""
    if layout == "model":
        return np.asarray(x, dtype=np.float64)
    if exact:
        z = np.asarray(x, dtype=np.float64).copy()
        z[..., 0] = (z[..., 0] - stats["i_mean"]) / stats["i_std"]
        z[..., 1] = (z[..., 1] - stats["q_mean"]) / stats["q_std"]
    else:
        z = zscore_f32(x, stats).astype(np.float64)
    if cfg.kind == "rawiq":
        return O.frame_rawiq(z)
    return O.frame_vit(z, cfg.img_size_h, cfg.img_size_w)


def patch_operand(x, cfg, layout, stats=None, bf16=False, exact=False):
    """A [B, Ttok, K]: the embedding GEMM's left operand as the kernel forms it (float64 holding fp32 / bf16 values)."""
    src = model_layout(x, cfg, layout, stats, exact)
    if cfg.kind == "rawiq":
        A = O.patchify_rawiq(src, cfg)
    else:                       # the strided Conv2d drops the rows / columns past the last whole patch
        p = cfg.patch_size
        A = O.patchify_vit(src[:, :, :src.shape[2] // p * p, :src.shape[3] // p * p], cfg)
    return bf16_rne(A).astype(np.float64) if bf16 else A


def emb_weight(params, cfg, bf16):
    W = np.asarray(params[emb_key(cfg) + ".weight"], dtype=np.float32)
    W = W.reshape(W.shape[0], -1)
    return (bf16_rne(W) if bf16 else W).astype(np.float64)


def frontend_ref(x, params, pos, cfg, layout="model", stats=None, bf16=False, exact=False):
    """x0 [B, T, d] of the front end (dropout off), the operand A [B, Ttok, K] it multiplied, and the per-element
    error bound of an fp32 computation of it.

    Bound: x0 = sum_k a_k w_k (K products, exact in fp32 for bf16 operands, one FMA rounding each in fp32 mode)
    + bias + pe: K + 2 fp32 additions, |err| <= C_ACC * (K + 2) * u * (|A| |W|^T + |bias| + |pe|)."""
    A = patch_operand(x, cfg, layout, stats, bf16, exact)
    W = emb_weight(params, cfg, bf16)
    b = np.asarray(params[emb_key(cfg) + ".bias"], dtype=np.float64)
    pos = np.asarray(pos, dtype=np.float64)
    B, Ttok, K = A.shape
    c = 1 if cfg.has_cls else 0
    pe = pos[c:c + Ttok]
    x0 = A @ W.T + b + pe
    mag = np.abs(A) @ np.abs(W).T + np.abs(b) + np.abs(pe)
    if cfg.has_cls:
        cls = np.asarray(params["encoder.cls_token"], dtype=np.float64).reshape(1, 1, -1)
        x0 = np.concatenate([np.broadcast_to(cls + pos[0], (B, 1, x0.shape[2])), x0], 1)
        mag = np.concatenate([np.broadcast_to(np.abs(cls) + np.abs(pos[0]), (B, 1, x0.shape[2])), mag], 1)
    return x0, A, C_ACC * (K + 2) * U * mag


def frontend_bwd_ref(dx0, A, params, cfg, layout="model", stats=None, bf16=False, mult=None):
    """Gradients of the front end for dL/dx0 = dx0 [B, T, d]: emb_w, emb_b, cls (None without a CLS token) and dsrc in
    the caller's layout, each with its error bound.  ``mult`` [B, T, d] is the dropout multiplier (0 or 1 / (1 - p))
    the forward applied; the backward applies the same one.

    Bounds (fp32 sums of n terms: C_ACC * n * u * sum |terms|):
      emb_w, emb_b: n = B * Ttok rows of demb^T A;  cls: n = B;  dsrc: n = d (+1 for the 1/std product)."""
    dx0 = np.asarray(dx0, dtype=np.float64)
    if mult is not None:        # the fp32 product the kernels form
        dx0 = (dx0.astype(np.float32) * np.asarray(mult, dtype=np.float32)).astype(np.float64)
    c = 1 if cfg.has_cls else 0
    B, T, d = dx0.shape
    demb = dx0[:, c:]
    demb = (bf16_rne(demb).astype(np.float64) if bf16 else demb).reshape(-1, d)
    Am = A.reshape(-1, A.shape[-1])
    W = emb_weight(params, cfg, bf16)
    n = demb.shape[0]
    out = {}
    out["emb_w"] = demb.T @ Am
    out["emb_w_bound"] = C_ACC * n * U * (np.abs(demb).T @ np.abs(Am))
    out["emb_b"] = demb.sum(0)
    out["emb_b_bound"] = C_ACC * n * U * np.abs(demb).sum(0)
    if cfg.has_cls:
        g = dx0[:, 0].astype(np.float64)
        out["cls"] = g.sum(0)
        out["cls_bound"] = C_ACC * B * U * np.abs(g).sum(0)
    else:
        out["cls"] = out["cls_bound"] = None
    dA = (demb @ W).reshape(A.shape)
    dA_mag = (np.abs(demb) @ np.abs(W)).reshape(A.shape)
    unpatch = unpatchify_rawiq if cfg.kind == "rawiq" else unpatchify_vit
    dsrc, mag = unpatch(dA, cfg), unpatch(dA_mag, cfg)
    if layout == "dataset":
        inv = np.float32(1.0) / np.array([stats["i_std"], stats["q_std"]], dtype=np.float32)
        dsrc, mag = to_dataset(dsrc, cfg, inv.astype(np.float64)), to_dataset(mag, cfg, inv.astype(np.float64))
    out["dsrc"] = dsrc
    out["dsrc_bound"] = C_ACC * (d + 1) * U * mag
    return out


def unpatchify_rawiq(dA, cfg):
    """Transpose of O.patchify_rawiq: [B, Tt, C*S] -> [B, C, Tt*S]."""
    B, Tt, K = dA.shape
    S = 1 if cfg.embedding_type == "conv1d" else cfg.segment_size
    return np.ascontiguousarray(dA.reshape(B, Tt, K // S, S).transpose(0, 2, 1, 3).reshape(B, K // S, Tt * S))


def unpatchify_vit(dA, cfg):
    """Transpose of O.patchify_vit: [B, N, C*p*p] -> [B, C, H, W]; pixels no patch covers are 0."""
    B = dA.shape[0]
    p, C, H, W = cfg.patch_size, cfg.in_channels, cfg.img_size_h, cfg.img_size_w
    hp, wp = H // p, W // p
    out = np.zeros((B, C, H, W))
    out[:, :, :hp * p, :wp * p] = dA.reshape(B, hp, wp, C, p, p).transpose(0, 3, 1, 4, 2, 5).reshape(B, C, hp * p, wp * p)
    return out


def to_dataset(dsrc, cfg, inv):
    """Model-layout gradient -> gradient w.r.t. the interleaved dataset frames [B, L, 2] (framing transposed, * 1/std)."""
    B = dsrc.shape[0]
    if cfg.kind == "rawiq":
        g = dsrc.transpose(0, 2, 1)
    else:
        flat = dsrc.reshape(B, -1)
        L = flat.shape[1] // 2
        g = np.stack([flat[:, :L], flat[:, L:]], -1)
    return np.ascontiguousarray(g * inv)


# ---------------------------------------------------------------------------------------------------------------------
# classifier head
# ---------------------------------------------------------------------------------------------------------------------
def head_ref(x0, params, cfg, head_ln, eps=1e-5):
    """logits of the head on the encoder output x0 [B, T, d] (CLS row or mean over T, optional LayerNorm), its cache
    and the per-element bound of an fp32 computation.

    Bounds: pooling adds T terms (mean: and a division): e_pool = C_ACC (T + 1) u mean_t|x|.  LayerNorm: mean and
    variance are d-term sums, rsqrtf is within 2 ulp: e_xhat = C_ACC (d + 4) u (|xhat| + rstd (|v| + mean|v|))
    + rstd e_pool.  logits: d-term dot product plus bias, plus what the xhat error carries through gamma and W."""
    x0 = np.asarray(x0, dtype=np.float64)
    B, T, d = x0.shape
    kw, kb, kg, kbeta = head_keys(cfg, head_ln)
    if cfg.has_cls:
        v, e_pool = x0[:, 0], np.zeros((B, d))
    else:
        v = x0.mean(1)
        e_pool = C_ACC * (T + 1) * U * np.abs(x0).mean(1)
    cache = dict(v=v, T=T, head_ln=head_ln, has_cls=cfg.has_cls)
    if head_ln:
        g, be = (np.asarray(params[k], dtype=np.float64) for k in (kg, kbeta))
        mean = v.mean(1, keepdims=True)
        rstd = 1.0 / np.sqrt(((v - mean) ** 2).mean(1, keepdims=True) + eps)
        xhat = (v - mean) * rstd
        hl = g * xhat + be
        e_xhat = C_ACC * (d + 4) * U * (np.abs(xhat) + rstd * (np.abs(v) + np.abs(v).mean(1, keepdims=True))) \
            + rstd * (e_pool + e_pool.mean(1, keepdims=True))
        e_hl = np.abs(g) * e_xhat + C_ACC * U * (np.abs(g * xhat) + np.abs(be))
        cache.update(xhat=xhat, rstd=rstd, gamma=g, e_xhat=e_xhat)
    else:
        hl, e_hl = v, e_pool
    W = np.asarray(params[kw], dtype=np.float64)
    b = np.asarray(params[kb], dtype=np.float64)
    logits = hl @ W.T + b
    bound = C_ACC * (d + 2) * U * (np.abs(hl) @ np.abs(W).T + np.abs(b)) + e_hl @ np.abs(W).T
    cache.update(hl=hl, e_hl=e_hl, W=W)
    return logits, cache, bound


def head_bwd_ref(dlogits, cache):
    """Gradients of the head for dL/dlogits: head_w, head_b, (head_ln) ln_w, ln_b, and dx0 [B, T, d] (the CLS row or
    dpool / T on every row), each with its bound (first-order propagation of the forward's hl / xhat bounds plus fp32
    sums: C dlogits terms per dhl element, d terms per LayerNorm-backward mean, B rows per parameter gradient)."""
    dl = np.asarray(dlogits, dtype=np.float64)
    B, Cn = dl.shape
    W, hl, e_hl, T = cache["W"], cache["hl"], cache["e_hl"], cache["T"]
    d = W.shape[1]
    out = {}
    out["head_w"] = dl.T @ hl
    out["head_w_bound"] = C_ACC * (B + 1) * U * (np.abs(dl).T @ np.abs(hl)) + np.abs(dl).T @ e_hl
    out["head_b"] = dl.sum(0)
    out["head_b_bound"] = C_ACC * (B + 1) * U * np.abs(dl).sum(0)
    dhl = dl @ W
    e_dhl = C_ACC * (Cn + 1) * U * (np.abs(dl) @ np.abs(W))
    if cache["head_ln"]:
        xh, rs, gm, e_xh = cache["xhat"], cache["rstd"], cache["gamma"], cache["e_xhat"]
        out["ln_w"] = (dhl * xh).sum(0)
        out["ln_w_bound"] = C_ACC * (B + 1) * U * np.abs(dhl * xh).sum(0) + (e_dhl * np.abs(xh) + np.abs(dhl) * e_xh).sum(0)
        out["ln_b"] = dhl.sum(0)
        out["ln_b_bound"] = C_ACC * (B + 1) * U * np.abs(dhl).sum(0) + e_dhl.sum(0)
        g = dhl * gm
        s1 = g.mean(1, keepdims=True)
        s2 = (g * xh).mean(1, keepdims=True)
        dpool = rs * (g - s1 - xh * s2)
        ag, e_g = np.abs(g), np.abs(gm) * e_dhl
        m_g, m_gx = ag.mean(1, keepdims=True), (ag * np.abs(xh)).mean(1, keepdims=True)
        e_dpool = rs * (C_ACC * (d + 4) * U * (ag + m_g + np.abs(xh) * m_gx)
                        + e_g + e_g.mean(1, keepdims=True) + np.abs(xh) * (e_g * np.abs(xh)).mean(1, keepdims=True)
                        + e_xh * m_gx + np.abs(xh) * (ag * e_xh).mean(1, keepdims=True))
    else:
        out["ln_w"] = out["ln_b"] = out["ln_w_bound"] = out["ln_b_bound"] = None
        dpool, e_dpool = dhl, e_dhl
    dx0 = np.zeros((B, T, d))
    ex0 = np.zeros((B, T, d))
    if cache["has_cls"]:
        dx0[:, 0], ex0[:, 0] = dpool, e_dpool
    else:                                   # g * fp32(1 / T): two more roundings
        dx0[:] = (dpool / T)[:, None]
        ex0[:] = ((e_dpool + 2 * U * np.abs(dpool)) / T)[:, None]
    out["dx0"], out["dx0_bound"] = dx0, ex0
    return out


# ---------------------------------------------------------------------------------------------------------------------
# loss, argmax, optimizer, statistics
# ---------------------------------------------------------------------------------------------------------------------
def ce_ref(logits, labels, ls):
    """Per-frame nn.CrossEntropyLoss(label_smoothing=ls) losses [B] and d loss_b / d logits [B, C] (unscaled) in
    float64.  Labels outside [0, C) get a NaN loss and the gradient of an all-smoothing target."""
    z = np.asarray(logits, dtype=np.float64)
    labels = np.asarray(labels, dtype=np.int64)
    B, C = z.shape
    zs = z - z.max(1, keepdims=True)
    logp = zs - np.log(np.exp(zs).sum(1, keepdims=True))
    ok = (labels >= 0) & (labels < C)
    tgt = np.full((B, C), ls / C)
    tgt[np.arange(B)[ok], labels[ok]] += 1.0 - ls
    loss = -(tgt * logp).sum(1)
    loss[~ok] = np.nan
    return loss, np.exp(logp) - tgt


def argmax_ref(logits):
    """torch.max(1) indices: the first maximum; a row with a NaN gives its first NaN."""
    z = np.asarray(logits)
    out = np.argmax(z, 1)
    nan = np.isnan(z)
    rows = nan.any(1)
    out[rows] = np.argmax(nan[rows], 1)
    return out


def adamw_ref(p, g, m, v, step, lr, beta1, beta2, eps, wd, max_norm, grad_scale):
    """clip_grad_norm_(max_norm) (disabled for max_norm <= 0) + torch.optim.AdamW step, float64.  Returns
    (p, m, v, pre-clip norm of grad_scale * g)."""
    g = np.asarray(g, dtype=np.float64) * grad_scale
    norm = float(np.sqrt((g * g).sum()))
    if max_norm > 0:
        g = g * min(1.0, max_norm / (norm + 1e-6))
    p = np.asarray(p, dtype=np.float64) * (1.0 - lr * wd)
    m = beta1 * np.asarray(m, dtype=np.float64) + (1.0 - beta1) * g
    v = beta2 * np.asarray(v, dtype=np.float64) + (1.0 - beta2) * g * g
    denom = np.sqrt(v) / np.sqrt(1.0 - beta2 ** step) + eps
    p = p - lr / (1.0 - beta1 ** step) * m / denom
    return p, m, v, norm


def adamw_bound(p, g, m, v, step, lr, beta1, beta2, eps, wd, max_norm, grad_scale, n_chain):
    """Per-element bounds (p, m, v) of one fp32 clip + AdamW step from the fp32 state (p, g, m, v), and the relative
    bound of the pre-clip norm.  The squared norm is a sum of positive fp32 terms along a chain of at most ``n_chain``
    additions (grid-stride loop, warp and block trees, one atomic per block): relative error C_ACC n_chain u; the clip
    coefficient max_norm / (norm + 1e-6) adds a sqrtf, an add and a division.  The update itself is a fixed sequence of
    fp32 operations whose roundings are propagated to first order."""
    g = np.asarray(g, dtype=np.float64) * grad_scale
    norm = float(np.sqrt((g * g).sum()))
    e_norm = C_ACC * n_chain * U / 2 + 2 * U
    coef, e_coef = 1.0, 0.0
    if max_norm > 0 and max_norm / (norm + 1e-6) < 1.0:
        coef = max_norm / (norm + 1e-6)
        e_coef = coef * (e_norm + 4 * U)
    gi = g * coef
    e_g = C_ACC * U * np.abs(gi) + np.abs(g) * e_coef
    m = np.asarray(m, dtype=np.float64)
    v = np.asarray(v, dtype=np.float64)
    m1 = beta1 * m + (1 - beta1) * gi
    v1 = beta2 * v + (1 - beta2) * gi * gi
    e_m = C_ACC * U * (np.abs(beta1 * m) + np.abs((1 - beta1) * gi)) + (1 - beta1) * e_g
    e_v = C_ACC * U * (beta2 * v + (1 - beta2) * gi * gi) + (1 - beta2) * 2 * np.abs(gi) * e_g
    bc2 = np.sqrt(1.0 - beta2 ** step)
    sv = np.sqrt(v1)
    denom = sv / bc2 + eps
    e_den = C_ACC * U * denom + np.where(sv > 0, e_v / (2 * np.maximum(sv, 1e-300) * bc2), np.sqrt(e_v) / bc2)
    step_size = lr / (1.0 - beta1 ** step)
    upd = step_size * m1 / denom
    e_upd = 2 * C_ACC * U * np.abs(upd) + step_size * (e_m / denom + np.abs(m1) * e_den / denom ** 2)
    p = np.asarray(p, dtype=np.float64)
    e_p = C_ACC * U * (np.abs(p) + np.abs(upd)) + e_upd
    return e_p, e_m, e_v, e_norm


def iq_stats_ref(x):
    """{sum I, sum I^2, sum Q, sum Q^2} of interleaved frames [..., 2] in float64 (fp32 inputs are exact in float64 and
    so are their squares), and a bound for a float64 accumulation of them: (n + 64) * 2^-53 * sum of |terms|."""
    x = np.asarray(x, dtype=np.float64).reshape(-1, 2)
    i, q = x[:, 0], x[:, 1]
    s = np.array([i.sum(), (i * i).sum(), q.sum(), (q * q).sum()])
    mag = np.array([np.abs(i).sum(), (i * i).sum(), np.abs(q).sum(), (q * q).sum()])
    return s, (x.shape[0] + 64) * 2.0 ** -53 * mag

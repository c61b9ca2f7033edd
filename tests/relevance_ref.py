"""float64 reference for the class-specific attention relevance (tests only).

Chefer, Gur & Wolf, "Generic Attention-model Explainability" (ICCV 2021): A_l = mean_h relu(dy_t/dP_l * P_l) and
r = u^T (I + A_{L-1}) ... (I + A_0), u = e_0 (CLS pooling) or 1/T (mean pooling).  y_t is the logit of class t_b.  The
gradient comes from the oracle's forward cache and its per-layer backward (oracle/amc_oracle.py, SURVEY Appendix B):
per layer the attention-output gradient `do` is formed as encoder_layer_bwd forms it, and dy_t/dP = doh @ vh^T.
"""
from __future__ import annotations

import numpy as np

from oracle import amc_oracle as O


def _lp(params, i, name):
    return params[f"encoder.layers.{i}.{name}"]


def _head_bwd(dlogits, cache, params, cfg):
    """Gradient of the logits' weighted sum w.r.t. the top layer's output [B, T, d]."""
    B = dlogits.shape[0]
    if cfg.kind == "rawiq":
        _, hxhat, hrstd = cache["head"]
        dhl = dlogits @ params["mlp_head.1.weight"]
        dpool, _, _ = O.layer_norm_bwd(dhl, hxhat, hrstd, params["mlp_head.0.weight"])
    else:
        dpool = dlogits @ params["mlp_head.weight"]
    dx = np.zeros((B, cfg.T, cfg.d_model), dtype=dlogits.dtype)
    if cfg.has_cls:
        dx[:, 0] = dpool
    else:
        dx[:] = dpool[:, None, :] / cfg.T
    return dx


def _attn_out_grad(dx2, c, params, i):
    """encoder_layer_bwd (oracle/amc_oracle.py:241-263) up to `do`, the gradient of the head-concatenated attention
    output."""
    dw, _, _ = O.layer_norm_bwd(dx2, c["xhat2"], c["rstd2"], _lp(params, i, "norm2.gamma"))
    da = (dw @ _lp(params, i, "ffn.linear2.weight")) * (c["hid"] > 0)
    dx1 = da @ _lp(params, i, "ffn.linear1.weight") + dw
    du, _, _ = O.layer_norm_bwd(dx1, c["xhat1"], c["rstd1"], _lp(params, i, "norm1.gamma"))
    return du @ _lp(params, i, "attention.w_concat.weight")


def probs_and_grads(src, params, cfg, target=None):
    """(logits, t, [(P_l, dy_t/dP_l) for l = 0 .. L-1]), each P / dP float64 [B, h, T, T].  target None -> argmax."""
    p64 = {k: np.asarray(v, np.float64) for k, v in params.items()}
    logits, cache = O.model_forward(np.asarray(src, np.float64), p64, cfg, want_cache=True)
    B, C = logits.shape
    t = np.argmax(logits, 1) if target is None else np.asarray(target, np.int64)
    dlogits = np.zeros((B, C))
    dlogits[np.arange(B), t] = 1.0
    dx = _head_bwd(dlogits, cache, p64, cfg)
    out = [None] * cfg.n_layers
    for i in reversed(range(cfg.n_layers)):
        c = cache["caches"][i]
        doh = O.split_heads(_attn_out_grad(dx, c, p64, i), cfg.n_head)
        out[i] = (c["p"], doh @ c["vh"].transpose(0, 1, 3, 2))
        dx = O.encoder_layer_bwd(dx, c, p64, i, cfg, {})
    return logits, t, out


def layer_weight(p, dp):
    """A_l = mean_h relu(dP * P): [B, T, T]."""
    return np.maximum(dp * p, 0.0).mean(1)


def readout(B, T, has_cls):
    u = np.zeros((B, T)) if has_cls else np.full((B, T), 1.0 / T)
    if has_cls:
        u[:, 0] = 1.0
    return u


def relevance_step(v, p, dp):
    """v [B, T] -> v + v^T A_l."""
    return v + np.einsum("bi,bij->bj", v, layer_weight(p, dp))


def relevance(src, params, cfg, target=None):
    """(logits, r [B, T]) in float64."""
    logits, _, pg = probs_and_grads(src, params, cfg, target)
    B, _, T, _ = pg[0][0].shape
    v = readout(B, T, cfg.has_cls)
    for p, dp in reversed(pg):
        v = relevance_step(v, p, dp)
    return logits, v

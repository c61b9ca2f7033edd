"""float64 reference for Integrated Gradients (tests only).

Sundararajan, Taly & Yan, "Axiomatic Attribution for Deep Networks" (ICML 2017):
IG_t(x) = (x - x') * integral_0^1 dy_t/dx (x' + a (x - x')) da, here with the Gauss-Legendre rule on [0, 1], as
model.integrated_gradients computes it.  The gradient at each node is tests/input_grad_ref.py::input_grad with
dlogits = e_t (the oracle's forward cache and per-layer backward), in either input layout: for dataset-layout frames
[B, L, 2] the path runs between the un-normalised frames and the attribution is w.r.t. them.
"""
from __future__ import annotations

import numpy as np

import input_grad_ref as IR
from oracle import amc_oracle as O


def nodes(steps):
    """Gauss-Legendre nodes and weights on [0, 1]."""
    x, w = np.polynomial.legendre.leggauss(steps)
    return (x + 1.0) / 2.0, w / 2.0


def model_layout(x, cfg, norm_stats=None):
    """The model-layout frames the front end sees: x itself, or for dataset frames [B, L, 2] the z-score + framing
    (R/dataloader/dataset.py:215-222, V/dataloader/dataset.py:211-224)."""
    if norm_stats is None:
        return x
    i = (x[:, :, 0] - norm_stats["i_mean"]) / norm_stats["i_std"]
    q = (x[:, :, 1] - norm_stats["q_mean"]) / norm_stats["q_std"]
    if cfg.kind == "rawiq":
        return np.stack([i, q], 1)
    return np.concatenate([i, q], 1).reshape(x.shape[0], 1, cfg.img_size_h, cfg.img_size_w)


def integrated_gradients(src, baseline, params, cfg, target=None, steps=32, norm_stats=None):
    """(attr, logits of src, logits of baseline, t): attr float64 in the layout of src; target None -> argmax at src."""
    p64 = {k: np.asarray(v, np.float64) for k, v in params.items()}
    src = np.asarray(src, np.float64)
    baseline = np.asarray(baseline, np.float64)
    lx = O.model_forward(model_layout(src, cfg, norm_stats), p64, cfg)
    lb = O.model_forward(model_layout(baseline, cfg, norm_stats), p64, cfg)
    B, C = lx.shape
    t = np.argmax(lx, 1) if target is None else np.asarray(target, np.int64)
    alpha, w = nodes(steps)
    total = np.zeros_like(src)
    for a, wk in zip(alpha, w):
        x = baseline + a * (src - baseline)
        _, cache = O.model_forward(model_layout(x, cfg, norm_stats), p64, cfg, want_cache=True)
        dlogits = np.zeros((B, C))
        dlogits[np.arange(B), t] = 1.0
        total += wk * IR.input_grad(dlogits, cache, p64, cfg, norm_stats)
    return (src - baseline) * total, lx, lb, t


def delta(attr, lx, lb, t):
    """attr[b].sum() - (y_t(x_b) - y_t(x'_b)): the completeness gap."""
    B = attr.shape[0]
    r = np.arange(B)
    return attr.reshape(B, -1).sum(1) - (lx[r, t] - lb[r, t])

"""float64 references for the attention maps and the attention rollout (tests only).

Maps come from the oracle's forward cache (``caches[i]["p"]``: R/models/layers/scale_dot_product_attention.py:26-39).
Rollout is u^T A_{L-1} ... A_0 with A_l = 0.5 * mean_h(P_l) + 0.5 * I and u = e_0 (CLS pooling) or 1/T (mean pooling).
"""
from __future__ import annotations

import numpy as np

from oracle import amc_oracle as O


def maps(src, params, cfg):
    """[P_0, ..., P_{L-1}], each float64 [B, h, T, T]."""
    p64 = {k: np.asarray(v, np.float64) for k, v in params.items()}
    _, cache = O.model_forward(np.asarray(src, np.float64), p64, cfg, want_cache=True)
    return [c["p"] for c in cache["caches"]]


def rollout_step(v, p):
    """v [B, T], p [B, h, T, T] -> 0.5 v + (0.5 / h) sum_hh v^T P_hh."""
    return 0.5 * v + 0.5 * np.einsum("bi,bhij->bj", v, p) / p.shape[1]


def rollout(ps, has_cls):
    B, _, T, _ = ps[0].shape if ps else (0, 0, 0, 0)
    v = np.zeros((B, T)) if has_cls else np.full((B, T), 1.0 / T)
    if has_cls:
        v[:, 0] = 1.0
    for p in reversed(ps):
        v = rollout_step(v, p)
    return v


def probs_from_qkv(qkv, B, T, h, dh):
    """softmax(q k^T / sqrt(dh)) from a [B*T, 3d] qkv buffer (q | k | v column blocks, head hh = columns hh*dh ..)."""
    x = np.asarray(qkv, np.float64).reshape(B, T, 3, h, dh)
    q, k = x[:, :, 0].transpose(0, 2, 1, 3), x[:, :, 1].transpose(0, 2, 1, 3)
    s = q @ k.transpose(0, 1, 3, 2) / np.sqrt(dh)
    e = np.exp(s - s.max(-1, keepdims=True))
    return e / e.sum(-1, keepdims=True)

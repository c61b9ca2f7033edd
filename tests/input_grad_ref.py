"""Reference input gradient (d loss / d src) in numpy, built on the oracle's forward cache and its per-layer backward
(oracle/amc_oracle.py, SURVEY Appendix B): head backward, encoder layers in reverse, then the embedding's dgrad
dA = demb . W_emb, un-patchified into the input layout (segments / patches never overlap), and for dataset-layout input
chained through the framing and the z-score (R/dataloader/dataset.py:215-222, V/dataloader/dataset.py:211-224).
The CLS token and the positional encoding do not reach src.  Pinned to autograd of oracle/amc_torch_port.py by
tests/test_oracle_input_grad.py."""
from typing import Dict, Optional

import numpy as np

from oracle import amc_oracle as O


def unpatchify_rawiq(dA, cfg):
    """Transpose of O.patchify_rawiq: [B,Tt,C*S] -> [B,C,Tt*S]."""
    B, Tt, K = dA.shape
    S = 1 if cfg.embedding_type == "conv1d" else cfg.segment_size
    C = K // S
    return np.ascontiguousarray(dA.reshape(B, Tt, C, S).transpose(0, 2, 1, 3).reshape(B, C, Tt * S))


def unpatchify_vit(dA, cfg):
    """Transpose of O.patchify_vit: [B,N,C*p*p] -> [B,C,H,W]; pixels no patch covers (H or W not a multiple of p,
    dropped by the strided Conv2d) get 0."""
    B = dA.shape[0]
    p, C, H, W = cfg.patch_size, cfg.in_channels, cfg.img_size_h, cfg.img_size_w
    hp, wp = H // p, W // p
    x = dA.reshape(B, hp, wp, C, p, p).transpose(0, 3, 1, 4, 2, 5).reshape(B, C, hp * p, wp * p)
    out = np.zeros((B, C, H, W), dtype=dA.dtype)
    out[:, :, :hp * p, :wp * p] = x
    return out


def dataset_input_grad(dsrc, cfg, stats: Dict[str, float]):
    """Model-layout input gradient -> gradient w.r.t. the un-normalised interleaved frames [B,L,2]."""
    B = dsrc.shape[0]
    if cfg.kind == "rawiq":
        d = dsrc.transpose(0, 2, 1)                                   # [B,2,L] -> [B,L,2]
    else:
        flat = dsrc.reshape(B, -1)                                    # cat(I, Q).view(1, H, W)
        L = flat.shape[1] // 2
        d = np.stack([flat[:, :L], flat[:, L:]], axis=-1)
    inv = np.array([1.0 / stats["i_std"], 1.0 / stats["q_std"]], dtype=dsrc.dtype)
    return np.ascontiguousarray(d * inv)


def input_grad(dlogits, cache, params, cfg, norm_stats: Optional[Dict[str, float]] = None):
    """d loss / d src for a forward cache of O.model_forward(..., want_cache=True); with the dataset z-score
    ``norm_stats`` the gradient w.r.t. the un-normalised dataset frames [B,L,2]."""
    B = dlogits.shape[0]
    T, d = cfg.T, cfg.d_model
    if cfg.kind == "rawiq":
        _, hxhat, hrstd = cache["head"]
        dhl = dlogits @ params["mlp_head.1.weight"]
        dpool, _, _ = O.layer_norm_bwd(dhl, hxhat, hrstd, params["mlp_head.0.weight"])
    else:
        dpool = dlogits @ params["mlp_head.weight"]
    dx = np.zeros((B, T, d), dtype=dlogits.dtype)
    if cfg.has_cls:
        dx[:, 0] = dpool
    else:
        dx[:] = dpool[:, None, :] / T
    scratch = {}
    for i in reversed(range(cfg.n_layers)):
        dx = O.encoder_layer_bwd(dx, cache["caches"][i], params, i, cfg, scratch)
    demb = dx[:, 1:] if cfg.has_cls else dx
    key = "encoder.sequence_embedding.projection" if cfg.kind == "rawiq" else "encoder.patch_embedding.projection"
    W = params[key + ".weight"]
    dA = demb @ W.reshape(W.shape[0], -1).astype(demb.dtype)
    dsrc = unpatchify_rawiq(dA, cfg) if cfg.kind == "rawiq" else unpatchify_vit(dA, cfg)
    return dsrc if norm_stats is None else dataset_input_grad(dsrc, cfg, norm_stats)

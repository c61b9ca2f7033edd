"""CPU pins of the float64 attention-map and rollout references in attention_ref.py."""
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import attention_ref as R
from oracle import amc_oracle as O

CFGS = [
    O.Config(kind="vit", in_channels=1, num_classes=5, d_model=32, n_head=4, n_layers=2, ffn_hidden=64, patch_size=16),
    O.Config(kind="rawiq", num_classes=5, d_model=32, n_head=2, n_layers=3, ffn_hidden=64, seq_length=128,
             embedding_type="segment", segment_size=8),
    O.Config(kind="rawiq", num_classes=5, d_model=16, n_head=2, n_layers=2, ffn_hidden=32, seq_length=24,
             embedding_type="conv1d", use_cls_token=False),
]


def _src(cfg, B, seed):
    rng = np.random.default_rng(seed)
    shape = (B, 1, cfg.img_size_h, cfg.img_size_w) if cfg.kind == "vit" else (B, cfg.in_channels, cfg.seq_length)
    return rng.standard_normal(shape)


def _setup(cfg, seed, B=3):
    params = {k: v.astype(np.float64) for k, v in O.init_params(cfg, seed).items()}
    return params, _src(cfg, B, seed + 100)


@pytest.mark.parametrize("cfg", CFGS, ids=["vit_p16", "rawiq_seg8", "rawiq_conv1d_meanpool"])
def test_maps_match_an_independent_softmax(cfg):
    """q, k from the layer inputs with the torch port's operator sequence (oracle/amc_torch_port.py:60-67), softmax in
    float64: the oracle's cached P is the same."""
    params, src = _setup(cfg, 1)
    ps = R.maps(src, params, cfg)
    _, cache = O.model_forward(src, params, cfg, want_cache=True)
    h = cfg.n_head
    for i, (p, c) in enumerate(zip(ps, cache["caches"])):
        x = torch.from_numpy(c["x"])
        B, T, d = x.shape
        dh = d // h
        pre = f"encoder.layers.{i}.attention."
        w = {k: torch.from_numpy(params[pre + k]) for k in ("w_q.weight", "w_q.bias", "w_k.weight", "w_k.bias")}
        q = F.linear(x, w["w_q.weight"], w["w_q.bias"]).view(B, T, h, dh).transpose(1, 2)
        k = F.linear(x, w["w_k.weight"], w["w_k.bias"]).view(B, T, h, dh).transpose(1, 2)
        ref = torch.softmax((q @ k.transpose(2, 3)) / math.sqrt(dh), dim=-1).numpy()
        assert p.shape == (B, h, T, T)
        np.testing.assert_allclose(p, ref, rtol=0, atol=1e-13)


def test_probs_from_qkv_matches_the_oracle_layout():
    """The [B*T, 3d] q | k | v buffer layout of the kernels gives the oracle's P."""
    cfg = CFGS[1]
    params, src = _setup(cfg, 2)
    _, cache = O.model_forward(src, params, cfg, want_cache=True)
    c = cache["caches"][0]
    B, T, d = c["x"].shape
    pre = "encoder.layers.0.attention."
    qkv = np.concatenate([c["x"] @ params[pre + f"w_{n}.weight"].T + params[pre + f"w_{n}.bias"] for n in "qkv"], -1)
    p = R.probs_from_qkv(qkv.reshape(B * T, 3 * d), B, T, cfg.n_head, d // cfg.n_head)
    np.testing.assert_allclose(p, c["p"], rtol=0, atol=1e-13)


@pytest.mark.parametrize("seed", [0, 1, 2])
@pytest.mark.parametrize("cfg", CFGS, ids=["vit_p16", "rawiq_seg8", "rawiq_conv1d_meanpool"])
def test_invariants_on_random_models(cfg, seed):
    params, src = _setup(cfg, seed)
    ps = R.maps(src, params, cfg)
    for p in ps:
        assert (p >= 0).all()
        np.testing.assert_allclose(p.sum(-1), 1.0, rtol=0, atol=1e-12)
    r = R.rollout(ps, cfg.has_cls)
    assert r.shape == (src.shape[0], cfg.T)
    assert (r >= 0).all()
    np.testing.assert_allclose(r.sum(-1), 1.0, rtol=0, atol=1e-12)


def test_one_layer_rollout_is_half_e0_plus_half_the_mean_cls_row():
    cfg = O.Config(kind="vit", in_channels=1, num_classes=5, d_model=32, n_head=4, n_layers=1, ffn_hidden=64,
                   patch_size=16)
    params, src = _setup(cfg, 3)
    (p,) = R.maps(src, params, cfg)
    e0 = np.zeros(cfg.T)
    e0[0] = 1.0
    expect = 0.5 * e0[None] + 0.5 * p[:, :, 0, :].mean(1)
    np.testing.assert_allclose(R.rollout([p], True), expect, rtol=0, atol=1e-15)


def test_mean_pool_rollout_of_uniform_attention_is_uniform():
    B, h, T = 2, 3, 7
    p = np.full((B, h, T, T), 1.0 / T)
    np.testing.assert_allclose(R.rollout([p, p], False), np.full((B, T), 1.0 / T), rtol=0, atol=1e-15)

"""The numpy input-gradient reference (tests/input_grad_ref.py, built on the oracle) against autograd of the PyTorch-eager port, which
test_torch_port_golden.py pins to the unmodified reference.  float64 on both sides, every golden configuration, both
input layouts: model layout ([B,C,L] / [B,C,H,W]) and dataset frames [B,L,2] through the z-score and the framing."""
import numpy as np
import pytest
import torch

import input_grad_ref as R
from conftest import GOLDEN_CASES, GOLDEN_HP, load_golden
from oracle import amc_oracle as O
from oracle import amc_torch_port as TP


def _frame(raw, cfg, stats, lib):
    """dataset.py:215-224 in float64: z-score, then [B,2,L] (raw-IQ) or cat(I, Q).view(1, H, W) (ViT)."""
    i = (raw[:, :, 0] - stats["i_mean"]) / stats["i_std"]
    q = (raw[:, :, 1] - stats["q_mean"]) / stats["q_std"]
    if cfg.kind == "rawiq":
        return lib.stack([i, q], 1)
    cat = lib.cat([i, q], 1) if lib is torch else np.concatenate([i, q], 1)
    return cat.reshape(raw.shape[0], 1, cfg.img_size_h, cfg.img_size_w)


@pytest.mark.parametrize("layout", ["model", "dataset"])
@pytest.mark.parametrize("name", list(GOLDEN_CASES))
def test_oracle_input_grad_matches_torch_port_autograd(name, layout):
    z, params, _, _ = load_golden(name)
    kind, kw = GOLDEN_CASES[name]
    cfg = O.Config(kind=kind, **kw)
    p64 = {k: v.astype(np.float64) for k, v in params.items()}
    labels = z["labels"].astype(np.int64)
    B = labels.shape[0]
    stats = None
    if layout == "model":
        x = z["src"].astype(np.float64)
        src = x
    else:
        L = cfg.seq_length if kind == "rawiq" else cfg.img_size_h * cfg.img_size_w // 2
        x = np.random.default_rng(7).standard_normal((B, L, 2)) * 0.7 + 0.05
        stats = {"i_mean": 0.03, "i_std": 0.8, "q_mean": -0.02, "q_std": 1.3}
        src = _frame(x, cfg, stats, np)
    logits, cache = O.model_forward(src, p64, cfg, want_cache=True)
    _, dlogits = O.cross_entropy_ls(logits, labels, GOLDEN_HP["label_smoothing"])
    dsrc = R.input_grad(dlogits, cache, p64, cfg, norm_stats=stats)

    tp = TP.params_from_numpy(p64, requires_grad=False)
    xt = torch.from_numpy(x).requires_grad_(True)
    st = xt if layout == "model" else _frame(xt, cfg, stats, torch)
    out = TP.model_forward(st, tp, cfg)
    torch.nn.functional.cross_entropy(out, torch.from_numpy(labels),
                                      label_smoothing=GOLDEN_HP["label_smoothing"]).backward()
    ref = xt.grad.numpy()
    assert dsrc.shape == x.shape
    assert np.abs(dsrc - ref).max() <= 1e-10 * np.abs(ref).max()


def test_unpatchify_is_the_transpose_of_patchify():
    """<patchify(x), a> == <x, unpatchify(a)>, including a ViT image whose sides are not multiples of the patch."""
    rng = np.random.default_rng(0)
    for cfg, shape in ((O.Config(kind="rawiq", seq_length=64, segment_size=8), (3, 2, 64)),
                       (O.Config(kind="rawiq", seq_length=16, embedding_type="conv1d"), (3, 2, 16)),
                       (O.Config(kind="vit", in_channels=1, img_size_h=10, img_size_w=13, patch_size=4), (2, 1, 10, 13))):
        x = rng.standard_normal(shape)
        if cfg.kind == "rawiq":
            A = O.patchify_rawiq(x, cfg)
            back = R.unpatchify_rawiq
        else:
            A = O.patchify_vit(x[:, :, :8, :12], cfg)
            back = R.unpatchify_vit
        a = rng.standard_normal(A.shape)
        y = back(a, cfg)
        assert y.shape == x.shape
        assert abs(float((A * a).sum()) - float((x * y).sum())) < 1e-9

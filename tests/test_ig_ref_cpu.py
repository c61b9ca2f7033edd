"""CPU pins of the float64 Integrated Gradients reference in ig_ref.py, on every golden configuration and in both input
layouts: (a) it equals IG formed by float64 autograd through the PyTorch-eager port (oracle/amc_torch_port.py, pinned
to the unmodified reference by test_torch_port_golden.py) at the same Gauss-Legendre nodes; (b) a baseline equal to
the input gives exactly zero; (c) the completeness gap shrinks from 4 to 64 nodes."""
import numpy as np
import pytest
import torch

import ig_ref as R
from conftest import GOLDEN_CASES, load_golden
from oracle import amc_oracle as O
from oracle import amc_torch_port as TP

STATS = {"i_mean": 0.03, "i_std": 0.8, "q_mean": -0.02, "q_std": 1.3}


def _case(name, layout):
    z, params, _, _ = load_golden(name)
    kind, kw = GOLDEN_CASES[name]
    cfg = O.Config(kind=kind, **kw)
    p64 = {k: v.astype(np.float64) for k, v in params.items()}
    src = z["src"].astype(np.float64)
    if layout == "model":
        return cfg, p64, src, None
    # the dataset frames whose z-score + framing is src
    B = src.shape[0]
    if cfg.kind == "rawiq":
        i, q = src[:, 0], src[:, 1]
    else:
        flat = src.reshape(B, -1)
        i, q = flat[:, :flat.shape[1] // 2], flat[:, flat.shape[1] // 2:]
    x = np.stack([i * STATS["i_std"] + STATS["i_mean"], q * STATS["q_std"] + STATS["q_mean"]], -1)
    return cfg, p64, x, STATS


def _torch_model_layout(x, cfg, stats):
    if stats is None:
        return x
    i = (x[:, :, 0] - stats["i_mean"]) / stats["i_std"]
    q = (x[:, :, 1] - stats["q_mean"]) / stats["q_std"]
    if cfg.kind == "rawiq":
        return torch.stack([i, q], 1)
    return torch.cat([i, q], 1).reshape(x.shape[0], 1, cfg.img_size_h, cfg.img_size_w)


def _baseline(src):
    return 0.3 * np.random.default_rng(1).standard_normal(src.shape)


@pytest.mark.parametrize("layout", ["model", "dataset"])
@pytest.mark.parametrize("name", list(GOLDEN_CASES))
def test_reference_matches_torch_port_autograd(name, layout):
    cfg, p64, src, stats = _case(name, layout)
    base = _baseline(src)
    B = src.shape[0]
    target = (np.arange(B) * 5 + 2) % cfg.num_classes
    steps = 4
    attr, _, _, t = R.integrated_gradients(src, base, p64, cfg, target, steps, stats)
    tp = TP.params_from_numpy(p64, requires_grad=False)
    alpha, w = R.nodes(steps)
    total = torch.zeros(src.shape, dtype=torch.float64)
    for a, wk in zip(alpha, w):
        x = torch.from_numpy(base + a * (src - base)).requires_grad_(True)
        out = TP.model_forward(_torch_model_layout(x, cfg, stats), tp, cfg)
        (g,) = torch.autograd.grad(out[torch.arange(B), torch.from_numpy(t)].sum(), x)
        total += wk * g
    ref = ((torch.from_numpy(src) - torch.from_numpy(base)) * total).numpy()
    assert attr.shape == src.shape
    assert np.abs(attr - ref).max() <= 1e-10 * np.abs(ref).max()


@pytest.mark.parametrize("name", list(GOLDEN_CASES))
def test_baseline_equal_to_input_gives_zero(name):
    cfg, p64, src, _ = _case(name, "model")
    attr, lx, lb, t = R.integrated_gradients(src, src.copy(), p64, cfg, steps=3)
    assert (attr == 0).all()
    assert (R.delta(attr, lx, lb, t) == 0).all()


@pytest.mark.parametrize("name", list(GOLDEN_CASES))
def test_completeness_gap_shrinks_with_more_nodes(name):
    cfg, p64, src, _ = _case(name, "model")
    base = np.zeros_like(src)
    gaps = {}
    for steps in (4, 64):
        attr, lx, lb, t = R.integrated_gradients(src, base, p64, cfg, steps=steps)
        gaps[steps] = np.abs(R.delta(attr, lx, lb, t)).mean()
    print(f"{name}: mean |delta| at 4 nodes {gaps[4]:.3e}, at 64 nodes {gaps[64]:.3e}")
    assert gaps[64] < gaps[4]

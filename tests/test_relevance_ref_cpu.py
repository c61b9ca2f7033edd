"""CPU pins of the float64 class-specific relevance reference in relevance_ref.py, on every golden configuration:
(a) its dy_t/dP_l equals autograd through the PyTorch-eager port (oracle/amc_torch_port.py, pinned to the unmodified
reference by test_torch_port_golden.py) with the softmax outputs' gradients retained; (b) its vector chain equals the
read-out row of Chefer's full-matrix recursion R <- R + A R."""
import numpy as np
import pytest
import torch

import relevance_ref as R
from conftest import GOLDEN_CASES, load_golden
from oracle import amc_oracle as O
from oracle import amc_torch_port as TP


def _case(name):
    z, params, _, _ = load_golden(name)
    kind, kw = GOLDEN_CASES[name]
    cfg = O.Config(kind=kind, **kw)
    p64 = {k: v.astype(np.float64) for k, v in params.items()}
    return cfg, p64, z["src"].astype(np.float64)


@pytest.mark.parametrize("given", [False, True], ids=["argmax", "target"])
@pytest.mark.parametrize("name", list(GOLDEN_CASES))
def test_grad_wrt_p_matches_torch_port_autograd(name, given, monkeypatch):
    cfg, p64, src = _case(name)
    B = src.shape[0]
    target = (np.arange(B) * 7 + 3) % cfg.num_classes if given else None
    logits, t, pg = R.probs_and_grads(src, p64, cfg, target)

    kept = []
    softmax = torch.softmax

    def keep(x, dim=None, **kw):
        y = softmax(x, dim=dim, **kw)
        y.retain_grad()
        kept.append(y)
        return y

    monkeypatch.setattr(torch, "softmax", keep)
    xs = torch.from_numpy(src).requires_grad_(True)     # frozen parameters: the graph hangs off the input
    out = TP.model_forward(xs, TP.params_from_numpy(p64, requires_grad=False), cfg)
    np.testing.assert_allclose(out.detach().numpy(), logits, rtol=0, atol=1e-10)
    out[torch.arange(B), torch.from_numpy(t)].sum().backward()
    assert len(kept) == cfg.n_layers
    for (p, dp), y in zip(pg, kept):
        np.testing.assert_allclose(y.detach().numpy(), p, rtol=0, atol=1e-12)
        g = y.grad.numpy()
        assert np.abs(dp - g).max() <= 1e-10 * max(np.abs(g).max(), 1e-30)


@pytest.mark.parametrize("name", list(GOLDEN_CASES))
def test_vector_chain_is_the_readout_row_of_the_full_matrix_recursion(name):
    cfg, p64, src = _case(name)
    _, _, pg = R.probs_and_grads(src, p64, cfg)
    B, _, T, _ = pg[0][0].shape
    Rm = np.broadcast_to(np.eye(T), (B, T, T)).copy()
    for p, dp in pg:                                    # Chefer: layers in forward order, R <- R + A R
        Rm = Rm + R.layer_weight(p, dp) @ Rm
    row = Rm[:, 0] if cfg.has_cls else Rm.mean(1)
    _, r = R.relevance(src, p64, cfg)
    np.testing.assert_allclose(r, row, rtol=1e-12, atol=1e-14)
    u = R.readout(B, T, cfg.has_cls)
    assert (r >= u).all()
    if cfg.has_cls:
        assert (r[:, 0] >= 1.0).all()

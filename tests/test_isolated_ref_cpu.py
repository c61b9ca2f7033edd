"""Pins the float64 references of tests/isolated_ref.py (used by test_gpu_isolated.py) to the oracle and to PyTorch:
with rounding off, the front end and head references equal the oracle's forward and backward on every golden
configuration cut to 0 encoder layers; the AdamW reference equals torch.optim.AdamW + clip_grad_norm_; the CE and
argmax references equal torch; bf16_rne equals torch's float32 -> bfloat16 conversion."""
import numpy as np
import pytest
import torch

import input_grad_ref
import isolated_ref as R
from conftest import GOLDEN_CASES, GOLDEN_HP, load_golden
from oracle import amc_oracle as O

STATS = {"i_mean": 0.03, "i_std": 0.8, "q_mean": -0.02, "q_std": 1.3}


def close(a, b, tol=1e-12):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    assert a.shape == b.shape, (a.shape, b.shape)
    assert np.abs(a - b).max() <= tol * max(np.abs(b).max(), 1e-300)


def test_bf16_rne_matches_torch_on_edge_cases():
    f = np.float32
    bits = np.array([0x3F808000, 0x3F818000, 0x3F80C000, 0x3F807FFF, 0x3F80FFFF,   # ties to even (down, up), above, below
                     0x00000001, 0x00008000, 0x00018000, 0x007FFFFF, 0x80008000,   # subnormals, ties among them
                     0x7F7FFFFF, 0x7F7F7FFF, 0x7F7F8000, 0xFF7FFFFF,               # largest finite values
                     0x7F800000, 0xFF800000, 0x00000000, 0x80000000], dtype=np.uint32)
    rng = np.random.default_rng(0)
    x = np.concatenate([bits.view(np.float32), rng.standard_normal(100000).astype(f) * f(1e3),
                        rng.integers(0, 2 ** 32, 100000, dtype=np.uint64).astype(np.uint32).view(np.float32)])
    x = x[~np.isnan(x)]
    ref = torch.from_numpy(x).bfloat16().float().numpy()
    got = R.bf16_rne(x)
    assert np.array_equal(got.view(np.uint32), ref.view(np.uint32))
    assert np.isnan(R.bf16_rne(np.array([np.nan], dtype=f)))[0]


def _zero_layer(name):
    z, params, _, _ = load_golden(name)
    kind, kw = GOLDEN_CASES[name]
    cfg = O.Config(kind=kind, **dict(kw, n_layers=0))
    p64 = {k: v.astype(np.float64) for k, v in params.items()}
    return z, cfg, p64


@pytest.mark.parametrize("name", list(GOLDEN_CASES))
def test_frontend_and_head_refs_equal_the_oracle_without_rounding(name):
    z, cfg, p = _zero_layer(name)
    src = z["src"].astype(np.float64)
    labels = z["labels"].astype(np.int64)
    pos = p["encoder.positional_encoding.encoding"]
    logits, cache = O.model_forward(src, p, cfg, want_cache=True)
    x0, A, _ = R.frontend_ref(src, p, pos, cfg)
    close(A, cache["A"])
    close(x0, cache["xL"])
    head_ln = cfg.kind == "rawiq"
    hlog, hcache, _ = R.head_ref(x0, p, cfg, head_ln)
    close(hlog, logits)

    _, dlogits = O.cross_entropy_ls(logits, labels, GOLDEN_HP["label_smoothing"])
    grads = O.model_backward(dlogits, cache, p, cfg)
    hb = R.head_bwd_ref(dlogits, hcache)
    kw, kb, kg, kbeta = R.head_keys(cfg, head_ln)
    close(hb["head_w"], grads[kw])
    close(hb["head_b"], grads[kb])
    if head_ln:
        close(hb["ln_w"], grads[kg])
        close(hb["ln_b"], grads[kbeta])
    fb = R.frontend_bwd_ref(hb["dx0"], A, p, cfg)
    key = R.emb_key(cfg)
    close(fb["emb_w"], grads[key + ".weight"].reshape(fb["emb_w"].shape))
    close(fb["emb_b"], grads[key + ".bias"])
    if cfg.has_cls:
        close(fb["cls"], grads["encoder.cls_token"].ravel())
    close(fb["dsrc"], input_grad_ref.input_grad(dlogits, cache, p, cfg))


@pytest.mark.parametrize("name", ["rawiq_seg16", "rawiq_conv1d", "vit_p8"])
def test_dataset_layout_operand_and_input_gradient(name):
    """Dataset frames: the oracle's fp32 z-score (a subtraction and a division) and the kernel's (a subtraction, then a
    multiplication by fp32(1 / std)) lie within a few roundings of the exact one; the dataset-layout input gradient
    equals input_grad_ref's up to the rounding of fp32(1 / std)."""
    z, cfg, p = _zero_layer(name)
    B = z["src"].shape[0]
    L = cfg.seq_length if cfg.kind == "rawiq" else cfg.img_size_h * cfg.img_size_w // 2
    x = (np.random.default_rng(1).standard_normal((B, L, 2)) * 0.7 + 0.05).astype(np.float32)
    exact = R.patch_operand(x, cfg, "dataset", STATS, exact=True)
    framed = O.frame_rawiq(O.normalize_iq(x, STATS)) if cfg.kind == "rawiq" else O.frame_vit(O.normalize_iq(x, STATS))
    oracle_A = O.patchify_rawiq(framed, cfg) if cfg.kind == "rawiq" else O.patchify_vit(framed, cfg)
    # both round mean and std to fp32 first: u |mean| / std absolute, u |z| relative
    mu = R.U * max(abs(STATS["i_mean"]) / STATS["i_std"], abs(STATS["q_mean"]) / STATS["q_std"])
    assert np.all(np.abs(exact - oracle_A) <= 3.001 * R.U * np.abs(exact) + mu)
    fp32 = R.patch_operand(x, cfg, "dataset", STATS)
    assert np.all(np.abs(fp32 - exact) <= 4.001 * R.U * np.abs(exact) + mu)

    src = R.model_layout(x, cfg, "dataset", STATS, exact=True)
    logits, cache = O.model_forward(src, p, cfg, want_cache=True)
    _, dlogits = O.cross_entropy_ls(logits, z["labels"].astype(np.int64), 0.1)
    hb = R.head_bwd_ref(dlogits, R.head_ref(cache["xL"], p, cfg, cfg.kind == "rawiq")[1])
    fb = R.frontend_bwd_ref(hb["dx0"], cache["A"], p, cfg, layout="dataset", stats=STATS)
    close(fb["dsrc"], input_grad_ref.input_grad(dlogits, cache, p, cfg, norm_stats=STATS), tol=2 * R.U)


@pytest.mark.parametrize("max_norm", [0.0, 1.0, 1e-3])
def test_adamw_ref_equals_torch_adamw(max_norm):
    rng = np.random.default_rng(2)
    shapes = [(7, 5), (13,), (3, 4, 2)]
    p0 = [rng.standard_normal(s) for s in shapes]
    tp = [torch.tensor(a, requires_grad=True) for a in p0]
    lr, betas, eps, wd, gs = 1e-3, (0.9, 0.99), 1e-8, 0.01, 0.5
    opt = torch.optim.AdamW(tp, lr=lr, betas=betas, eps=eps, weight_decay=wd, foreach=False)
    flat = np.concatenate([a.ravel() for a in p0])
    m = np.zeros_like(flat)
    v = np.zeros_like(flat)
    for step in range(1, 6):
        g = [rng.standard_normal(s) * 0.3 for s in shapes]
        for t, gi in zip(tp, g):
            t.grad = torch.tensor(gi * gs)
        tnorm = float(torch.nn.utils.clip_grad_norm_(tp, max_norm)) if max_norm > 0 else None
        opt.step()
        flat, m, v, norm = R.adamw_ref(flat, np.concatenate([a.ravel() for a in g]), m, v, step, lr, betas[0],
                                       betas[1], eps, wd, max_norm, gs)
        if tnorm is not None:
            assert abs(norm - tnorm) <= 1e-12 * tnorm
        close(flat, np.concatenate([t.detach().numpy().ravel() for t in tp]))
        st = [opt.state[t] for t in tp]
        close(m, np.concatenate([s["exp_avg"].numpy().ravel() for s in st]))
        close(v, np.concatenate([s["exp_avg_sq"].numpy().ravel() for s in st]))


@pytest.mark.parametrize("ls", [0.0, 0.1, 0.3])
def test_ce_and_argmax_refs_equal_torch(ls):
    rng = np.random.default_rng(3)
    z = rng.standard_normal((40, 11)) * 5
    z[3] = 80.0
    z[4, :3] = -80.0
    y = rng.integers(0, 11, 40)
    loss, dl = R.ce_ref(z, y, ls)
    zt = torch.tensor(z, requires_grad=True)
    lt = torch.nn.functional.cross_entropy(zt, torch.tensor(y), label_smoothing=ls, reduction="none")
    lt.sum().backward()
    close(loss, lt.detach().numpy())
    close(dl, zt.grad.numpy())
    z[5, 2] = np.nan
    z[6, 4] = z[6, 7] = np.nan
    z[7] = z[7, 1]                       # ties
    z[8] = -np.inf
    assert np.array_equal(R.argmax_ref(z), torch.tensor(z).max(1).indices.numpy())
    assert np.isnan(R.ce_ref(z[:2], np.array([11, -1]), ls)[0]).all()


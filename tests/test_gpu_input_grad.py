"""Gradients w.r.t. the input IQ frames through the nn.Module surface (``x.requires_grad_(True); loss.backward();
x.grad``): parity with the numpy oracle in both input layouts and both compute dtypes, finite differences, the
frozen-model backward (no parameter gradients, no weight-gradient GEMMs, bit-identical input gradient), the encoder
entry points, and the unchanged path when the input needs no gradient.

Tolerances as for the parameter gradients (test_gpu_model.py): L2-relative 1e-3 in fp32, 6e-2 in bf16."""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import input_grad_ref as R  # noqa: E402
from conftest import GOLDEN_CASES, l2_rel, load_golden  # noqa: E402
from oracle import amc_oracle as O  # noqa: E402
from oracle import amc_torch_port as TP  # noqa: E402

import vit_vs_raw_iq_b200 as amc  # noqa: E402
from vit_vs_raw_iq_b200 import _lib  # noqa: E402

DEV = "cuda:0"
TOL = {"fp32": 1e-3, "bf16": 6e-2}
STATS = {"i_mean": 0.03, "i_std": 0.8, "q_mean": -0.02, "q_std": 1.3}

# test_gpu_model.py::test_oracle_parity_at_reference_shapes
REF_SHAPES = [
    ("rawiq", dict(in_channels=2, seq_length=1024, num_classes=11, d_model=128, n_head=8, n_layers=3,
                   ffn_hidden=512, use_cls_token=True, embedding_type="segment", segment_size=16), 16),
    ("vit", dict(in_channels=1, img_size_h=32, img_size_w=64, patch_size=16, num_classes=19, d_model=256, n_head=8,
                 n_layers=2, ffn_hidden=1024), 33),
    ("vit", dict(in_channels=1, img_size_h=32, img_size_w=64, patch_size=4, num_classes=19, d_model=128, n_head=8,
                 n_layers=2, ffn_hidden=512), 7),
    ("rawiq", dict(in_channels=2, seq_length=2048, num_classes=11, d_model=256, n_head=8, n_layers=1,
                   ffn_hidden=1024, use_cls_token=True, embedding_type="segment", segment_size=8), 3),
    ("rawiq", dict(in_channels=2, seq_length=1024, num_classes=11, d_model=128, n_head=8, n_layers=2,
                   ffn_hidden=256, use_cls_token=True, embedding_type="conv1d", segment_size=64), 2),
    ("rawiq", dict(in_channels=2, seq_length=512, num_classes=11, d_model=64, n_head=2, n_layers=1,
                   ffn_hidden=128, use_cls_token=False, embedding_type="conv1d", segment_size=64), 3),
]


def make(kind, kw, dtype, drop=0.0):
    cls = amc.RawIQAMCTransformer if kind == "rawiq" else amc.ViTAMCTransformer
    return cls(**kw, drop_prob=drop, device=DEV, compute_dtype=dtype)


def bf16_supported(kind, kw):
    K = kw["in_channels"] * (kw["patch_size"] ** 2 if kind == "vit" else
                             (1 if kw["embedding_type"] == "conv1d" else kw["segment_size"]))
    return (K % 8 == 0 or (K <= 16 and kw["d_model"] >= 32)) and kw["d_model"] % 8 == 0


def input_batch(kind, kw, B, layout, seed):
    """(tensor fed to the model, model-layout float64 src for the oracle)"""
    rng = np.random.default_rng(seed)
    if layout == "model":
        shape = (B, kw["in_channels"], kw["seq_length"]) if kind == "rawiq" else (B, 1, kw["img_size_h"], kw["img_size_w"])
        x = rng.standard_normal(shape).astype(np.float32)
        return x, x.astype(np.float64)
    L = kw["seq_length"] if kind == "rawiq" else kw["img_size_h"] * kw["img_size_w"] // 2
    x = (rng.standard_normal((B, L, 2)) * 0.7 + 0.05).astype(np.float32)
    x64 = x.astype(np.float64)
    i = (x64[:, :, 0] - STATS["i_mean"]) / STATS["i_std"]
    q = (x64[:, :, 1] - STATS["q_mean"]) / STATS["q_std"]
    src = np.stack([i, q], 1) if kind == "rawiq" else np.concatenate([i, q], 1).reshape(B, 1, kw["img_size_h"],
                                                                                         kw["img_size_w"])
    return x, src


def oracle_dsrc(model, kind, kw, src64, labels, layout):
    cfg = O.Config(kind=kind, **kw)
    p64 = {k: v.detach().cpu().numpy().astype(np.float64) for k, v in model.state_dict().items()}
    logits, cache = O.model_forward(src64, p64, cfg, want_cache=True)
    _, dlogits = O.cross_entropy_ls(logits, labels, 0.1)
    return R.input_grad(dlogits, cache, p64, cfg, norm_stats=STATS if layout == "dataset" else None)


def check_against_oracle(model, kind, kw, B, layout, dtype, seed):
    if layout == "dataset":
        model.set_raw_input(STATS)
    x, src64 = input_batch(kind, kw, B, layout, seed)
    labels = np.random.default_rng(seed + 1).integers(0, kw["num_classes"], B)
    xt = torch.from_numpy(x).to(DEV).requires_grad_(True)
    out = model(xt)
    torch.nn.functional.cross_entropy(out, torch.from_numpy(labels).to(DEV), label_smoothing=0.1).backward()
    ref = oracle_dsrc(model, kind, kw, src64, labels, layout)
    got = xt.grad.cpu().numpy()
    assert got.shape == x.shape
    e = l2_rel(got, ref)
    assert e < TOL[dtype], e


@pytest.mark.parametrize("layout", ["model", "dataset"])
@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
@pytest.mark.parametrize("name", list(GOLDEN_CASES))
def test_input_grad_matches_oracle_on_golden_configs(name, dtype, layout):
    kind, kw = GOLDEN_CASES[name]
    if dtype == "bf16" and not bf16_supported(kind, kw):
        pytest.skip("tiny fixture outside the bf16 path's shapes")
    _, params, _, _ = load_golden(name)
    model = make(kind, kw, dtype)
    model.load_state_dict({k: torch.from_numpy(v) for k, v in params.items()}, strict=True)
    model.eval()
    check_against_oracle(model, kind, kw, 4, layout, dtype, seed=11)


@pytest.mark.parametrize("layout", ["model", "dataset"])
@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
@pytest.mark.parametrize("kind,kw,B", REF_SHAPES)
def test_input_grad_matches_oracle_at_reference_shapes(kind, kw, B, dtype, layout):
    torch.manual_seed(3)
    model = make(kind, kw, dtype)
    with torch.no_grad():
        for n, p in model.named_parameters():
            if n.endswith(("gamma", "beta", "mlp_head.0.weight", "mlp_head.0.bias")):
                p.add_(0.1 * torch.randn_like(p))
    model.train()          # drop_prob = 0: the training-mode path, masks off
    check_against_oracle(model, kind, kw, B, layout, dtype, seed=5)


def test_input_grad_central_finite_differences():
    """fp32, drop_prob = 0: d loss / d x at single input elements (both layouts) against central differences."""
    torch.manual_seed(0)
    cases = [("rawiq", dict(in_channels=2, seq_length=128, num_classes=11, d_model=32, n_head=4, n_layers=2,
                            ffn_hidden=64, use_cls_token=True, embedding_type="segment", segment_size=16), "model"),
             ("vit", dict(in_channels=1, img_size_h=32, img_size_w=64, patch_size=8, num_classes=19, d_model=32,
                          n_head=4, n_layers=2, ffn_hidden=64), "dataset")]
    for kind, kw, layout in cases:
        model = make(kind, kw, "fp32")
        model.eval()
        if layout == "dataset":
            model.set_raw_input(STATS)
        x, _ = input_batch(kind, kw, 3, layout, seed=2)
        x = torch.from_numpy(x).to(DEV)
        wgt = torch.randn(3, kw["num_classes"], device=DEV)
        xg = x.clone().requires_grad_(True)
        (model(xg) * wgt).sum().backward()
        g = xg.grad.reshape(-1)
        # input-gradient elements are ~1e-2 here (the dataset z-score divides by std): the step has to lift the loss change
        # (2 * eps * g) well above the fp32 rounding of the loss (~1e-6)
        eps = 3e-2
        for idx in torch.topk(g.abs(), 4).indices.tolist() + [int(g.numel() // 2)]:
            with torch.no_grad():
                xp, xm = x.clone().reshape(-1), x.clone().reshape(-1)
                xp[idx] += eps
                xm[idx] -= eps
                fp = float((model(xp.view_as(x)) * wgt).double().sum())
                fm = float((model(xm.view_as(x)) * wgt).double().sum())
            numeric = (fp - fm) / (2 * eps)
            analytic = float(g[idx])
            assert abs(analytic - numeric) < 2e-2 * max(abs(analytic), abs(numeric), 5e-2 * float(g.abs().max())), \
                (kind, idx, analytic, numeric)


FROZEN_CASES = [
    ("vit", dict(in_channels=1, img_size_h=32, img_size_w=64, patch_size=16, num_classes=19, d_model=256, n_head=8,
                 n_layers=2, ffn_hidden=1024), 64),
    ("rawiq", dict(in_channels=2, seq_length=1024, num_classes=11, d_model=128, n_head=4, n_layers=2, ffn_hidden=256,
                   use_cls_token=True, embedding_type="segment", segment_size=8), 16),
    ("rawiq", dict(in_channels=2, seq_length=1024, num_classes=11, d_model=128, n_head=8, n_layers=1, ffn_hidden=256,
                   use_cls_token=True, embedding_type="conv1d", segment_size=64), 2),
    ("rawiq", dict(in_channels=2, seq_length=128, num_classes=24, d_model=32, n_head=2, n_layers=1, ffn_hidden=96,
                   use_cls_token=False, embedding_type="segment", segment_size=8), 8),
]


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
@pytest.mark.parametrize("kind,kw,B", FROZEN_CASES)
def test_frozen_model_fgsm_backward(kind, kw, B, dtype):
    """The FGSM case: a frozen .eval() model, torch.autograd.grad(loss, src).  No parameter gradient is created, no
    weight-gradient GEMM runs, and the input gradient is bit-identical to the one computed alongside the parameter
    gradients (the data-gradient chain has no atomics) and from run to run."""
    torch.manual_seed(4)
    model = make(kind, kw, dtype)
    model.eval()
    x, _ = input_batch(kind, kw, B, "model", seed=9)
    x = torch.from_numpy(x).to(DEV)
    labels = torch.randint(0, kw["num_classes"], (B,), device=DEV)

    def input_grad():
        xg = x.clone().requires_grad_(True)
        loss = torch.nn.functional.cross_entropy(model(xg), labels)
        return torch.autograd.grad(loss, xg)[0]

    model.requires_grad_(False)
    _lib.profile(True)
    try:
        g_frozen = input_grad()
        prof = _lib.profile_dump()
    finally:
        _lib.profile(False)
    assert all(p.grad is None for p in model.parameters())
    assert "gemm_wgrad" not in prof and "colsum" not in prof
    assert prof["frontend_bwd_dsrc"]["n"] >= 1
    assert torch.equal(g_frozen, input_grad())

    model.requires_grad_(True)
    xg = x.clone().requires_grad_(True)
    torch.nn.functional.cross_entropy(model(xg), labels).backward()
    assert all(p.grad is not None for p in model.parameters())
    assert torch.equal(xg.grad, g_frozen)
    assert float(g_frozen.abs().max()) > 0


@pytest.mark.parametrize("which", ["encoder", "cls", "sequence"])
@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_encoder_entry_points_give_the_input_gradient(which, dtype):
    """model.encoder(src), get_cls_token_output and get_sequence_output with src.requires_grad: the gradient of the
    output's sum, against autograd of the PyTorch-eager port in float64."""
    kind, kw = "rawiq", dict(in_channels=2, seq_length=256, num_classes=11, d_model=64, n_head=4, n_layers=2,
                             ffn_hidden=128, use_cls_token=True, embedding_type="segment", segment_size=16)
    torch.manual_seed(6)
    model = make(kind, kw, dtype)
    model.eval()
    x, _ = input_batch(kind, kw, 5, "model", seed=3)
    xg = torch.from_numpy(x).to(DEV).requires_grad_(True)
    enc = model.encoder
    out = {"encoder": enc, "cls": enc.get_cls_token_output, "sequence": enc.get_sequence_output}[which](xg)
    wgt = torch.randn(out.shape, generator=torch.Generator().manual_seed(1)).to(DEV)
    (out * wgt).sum().backward()

    cfg = O.Config(kind=kind, **kw)
    p64 = TP.params_from_numpy({k: v.detach().cpu().numpy().astype(np.float64) for k, v in model.state_dict().items()},
                               requires_grad=False)
    x64 = torch.from_numpy(x.astype(np.float64)).requires_grad_(True)
    ref = TP.encoder_forward(x64, p64, cfg)
    ref = {"encoder": ref, "cls": ref[:, 0], "sequence": ref[:, 1:]}[which]
    (ref * wgt.cpu().double()).sum().backward()
    assert l2_rel(xg.grad.cpu().numpy(), x64.grad.numpy()) < TOL[dtype]


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_bwd_without_input_gradient_is_the_old_path(dtype):
    """amc_model_bwd_ex(..., dsrc=NULL) and amc_model_bwd launch the same kernels, and the module surface still calls
    no input-gradient kernel when src does not require a gradient."""
    kind, kw = "vit", dict(in_channels=1, img_size_h=32, img_size_w=64, patch_size=8, num_classes=19, d_model=128,
                           n_head=4, n_layers=2, ffn_hidden=256)
    torch.manual_seed(2)
    model = make(kind, kw, dtype)
    core = model._core
    src = torch.randn(8, 1, 32, 64, device=DEV)
    dlogits = torch.randn(8, 19, device=DEV) * 1e-2
    stream = torch.cuda.current_stream().cuda_stream

    def run(ex):
        desc = core.make_desc(src, training=True, module_training=False)
        ws = torch.empty(_lib.workspace_bytes(desc), dtype=torch.uint8, device=DEV)
        logits = torch.empty(8, 19, device=DEV)
        _lib.check(_lib.lib.amc_model_fwd(C.byref(desc), src.data_ptr(), core.flat.data_ptr(),
                                          core.pos_buffer().data_ptr(), ws.data_ptr(), logits.data_ptr(), 0, stream),
                   "fwd")
        grads = torch.zeros(core.layout.total, device=DEV)
        torch.cuda.synchronize()
        _lib.profile(True)
        try:
            n0 = _lib.lib.amc_launch_count()
            if ex:
                rc = _lib.lib.amc_model_bwd_ex(C.byref(desc), src.data_ptr(), core.flat.data_ptr(), ws.data_ptr(),
                                               dlogits.data_ptr(), 0, grads.data_ptr(), 0, 0, core.n_layers + 2, stream)
            else:
                rc = _lib.lib.amc_model_bwd(C.byref(desc), src.data_ptr(), core.flat.data_ptr(), ws.data_ptr(),
                                            dlogits.data_ptr(), 0, grads.data_ptr(), 0, core.n_layers + 2, stream)
            _lib.check(rc, "bwd")
            n = _lib.lib.amc_launch_count() - n0
            prof = _lib.profile_dump()
        finally:
            _lib.profile(False)
        return n, {k: v["n"] for k, v in prof.items()}, grads

    n_old, prof_old, g_old = run(False)
    n_ex, prof_ex, g_ex = run(True)
    assert n_old == n_ex and prof_old == prof_ex
    assert "frontend_bwd_dsrc" not in prof_ex
    assert l2_rel(g_ex.cpu().numpy(), g_old.cpu().numpy()) < 1e-5

    _lib.profile(True)
    try:
        torch.nn.functional.cross_entropy(model(src), torch.zeros(8, dtype=torch.long, device=DEV)).backward()
        prof = _lib.profile_dump()
    finally:
        _lib.profile(False)
    assert "frontend_bwd_dsrc" not in prof and "gemm_wgrad" in prof
    # both NULL: nothing to compute is an argument error
    with pytest.raises(RuntimeError):
        desc = core.make_desc(src, training=True, module_training=False)
        _lib.check(_lib.lib.amc_model_bwd_ex(C.byref(desc), src.data_ptr(), core.flat.data_ptr(), None,
                                             dlogits.data_ptr(), 0, 0, 0, 0, core.n_layers + 2, stream), "bwd_ex")


def test_train_mode_dropout_input_grad_by_finite_differences():
    """.train() with dropout: the backward regenerates the forward's masks, so with the dropout counter frozen the
    input gradient's directional derivative matches a central difference taken with the same masks."""
    torch.manual_seed(0)
    kind, kw = "rawiq", dict(in_channels=2, seq_length=128, num_classes=11, d_model=32, n_head=4, n_layers=2,
                             ffn_hidden=64, use_cls_token=True, embedding_type="segment", segment_size=16)
    model = make(kind, kw, "fp32", drop=0.3)
    model.train()
    model.set_raw_input(STATS)
    core = model._core
    x, _ = input_batch(kind, kw, 6, "dataset", seed=8)
    x = torch.from_numpy(x).to(DEV)
    wgt = torch.randn(6, 11, device=DEV)

    def f(inp):
        core.calls = 7          # freeze the dropout counter -> identical masks on every call
        return (model(inp) * wgt).sum()

    xg = x.clone().requires_grad_(True)
    f(xg).backward()
    v = torch.randn_like(x)
    v /= v.norm()
    analytic = float((xg.grad * v).sum())
    eps = 3e-3
    with torch.no_grad():
        numeric = (float(f(x + eps * v)) - float(f(x - eps * v))) / (2 * eps)
    assert abs(analytic - numeric) < 3e-2 * max(abs(analytic), abs(numeric), 1e-3), (analytic, numeric)
    # and the masks are really on: a different counter gives a different input gradient
    core.calls = 8
    xh = x.clone().requires_grad_(True)
    (model(xh) * wgt).sum().backward()
    assert not torch.equal(xh.grad, xg.grad)

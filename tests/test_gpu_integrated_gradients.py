"""Integrated Gradients on the device (model.integrated_gradients, amc_model_integrated_gradients).

Whole path against ig_ref.py (float64 on the oracle) at the reference shapes of test_gpu_attention_maps.py, in both
dtypes (L2-rel 1e-4 fp32; bf16 at the input-gradient tolerance of test_gpu_input_grad.py, 6e-2), and in the dataset
layout.  The blend, the weighted seed and the multiply-scatter are checked through the entry point: one path point
against the frozen input gradient of the module surface at the blended input times (x - x'), a baseline equal to the
input giving exactly zero, and an out-of-range target giving a NaN row.  Against the module surface: the host loop of
torch.autograd.grad at the same nodes (1e-5 in fp32).  Surface: argmax default, internal_batch_size, bit-identical
repeats, batch independence, return_delta, no side effects, validation."""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import ig_ref as R  # noqa: E402
from conftest import l2_rel  # noqa: E402
from oracle import amc_oracle as O  # noqa: E402
from test_gpu_attention_maps import REF_IDS, REF_SHAPES, make, model_src  # noqa: E402

from vit_vs_raw_iq_b200 import _lib  # noqa: E402

DEV = "cuda:0"
TOL = {"fp32": 1e-4, "bf16": 6e-2}
STATS = {"i_mean": 0.03, "i_std": 0.8, "q_mean": -0.02, "q_std": 1.3}
SURF = REF_SHAPES[0]
STEPS = 8


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _baseline(src, seed=9):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return 0.3 * torch.randn(src.shape, device=DEV, generator=g)


def _params64(model):
    return {k: v.detach().cpu().numpy().astype(np.float64) for k, v in model.state_dict().items()}


def _autograd_loop(model, src, base, t, steps):
    """IG by the host loop a user would write: a frozen forward + torch.autograd.grad per Gauss-Legendre node."""
    B = src.shape[0]
    alpha, w = R.nodes(steps)
    for p in model.parameters():
        p.requires_grad_(False)
    try:
        total = torch.zeros_like(src, dtype=torch.float64)
        for a, wk in zip(alpha, w):
            x = (base + float(a) * (src - base)).requires_grad_(True)
            (g,) = torch.autograd.grad(model(x)[torch.arange(B, device=DEV), t].sum(), x)
            total += float(wk) * g.double()
    finally:
        for p in model.parameters():
            p.requires_grad_(True)
    return ((src - base).double() * total).float()


# ---- whole path against the float64 reference ----------------------------------------------------------------------
@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
@pytest.mark.parametrize("shape", REF_SHAPES, ids=REF_IDS)
def test_whole_path_against_reference(shape, dtype):
    kind, kw, B = shape
    torch.manual_seed(11)
    model = make(kind, kw, dtype).eval()
    src = model_src(kind, kw, B, 5)
    base = _baseline(src)
    t = (torch.arange(B, device=DEV) * 5 + 1) % kw["num_classes"]
    attr = model.integrated_gradients(src, t, base, steps=STEPS)
    assert attr.shape == src.shape and attr.dtype == torch.float32
    cfg = O.Config(kind=kind, **kw)
    ref, _, _, _ = R.integrated_gradients(src.cpu().numpy(), base.cpu().numpy(), _params64(model), cfg,
                                          t.cpu().numpy(), STEPS)
    e = l2_rel(attr.cpu().numpy(), ref)
    assert e <= TOL[dtype], e


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
@pytest.mark.parametrize("kind", ["rawiq", "vit"])
def test_dataset_layout_against_reference(kind, dtype):
    kw = SURF[1] if kind == "rawiq" else REF_SHAPES[2][1]
    torch.manual_seed(2)
    model = make(kind, kw, dtype).eval().set_raw_input(STATS)
    B = 3
    L = kw["seq_length"] if kind == "rawiq" else kw["img_size_h"] * kw["img_size_w"] // 2
    g = torch.Generator(device=DEV).manual_seed(4)
    x = torch.randn(B, L, 2, device=DEV, generator=g) * 0.7 + 0.05
    t = torch.arange(B, device=DEV) % kw["num_classes"]
    attr = model.integrated_gradients(x, t, steps=STEPS)      # baseline: zero dataset frames
    assert attr.shape == x.shape
    cfg = O.Config(kind=kind, **kw)
    ref, _, _, _ = R.integrated_gradients(x.cpu().numpy(), np.zeros(x.shape), _params64(model), cfg, t.cpu().numpy(),
                                          STEPS, STATS)
    e = l2_rel(attr.cpu().numpy(), ref)
    assert e <= TOL[dtype], e


@pytest.mark.parametrize("shape", [REF_SHAPES[0], REF_SHAPES[1], REF_SHAPES[5]], ids=["seg16", "vit_p16", "conv1d_meanpool"])
def test_against_the_autograd_host_loop(shape):
    kind, kw, B = shape
    torch.manual_seed(12)
    model = make(kind, kw, "fp32").eval()
    src = model_src(kind, kw, B, 6)
    base = _baseline(src, 3)
    t = (torch.arange(B, device=DEV) * 3 + 2) % kw["num_classes"]
    attr = model.integrated_gradients(src, t, base, steps=STEPS)
    loop = _autograd_loop(model, src, base, t, STEPS)
    e = l2_rel(attr.cpu().numpy(), loop.cpu().numpy())
    assert e <= 1e-5, e


# ---- the blend, the weighted seed and the multiply-scatter through the entry point ------------------------------------
@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
@pytest.mark.parametrize("shape", [REF_SHAPES[0], REF_SHAPES[4]], ids=["seg16", "conv1d_cls"])
def test_one_point_is_the_input_gradient_at_the_midpoint_times_the_difference(shape, dtype):
    """steps = 1: the node a = 1/2 with weight 1, so attr = (x - x') * dy_t/dx at the midpoint.  The blended embedding
    differs from the front end run on the midpoint only by rounding (fp32) or by where the bf16 rounding of the patch
    operand happens (bf16)."""
    kind, kw, B = shape
    torch.manual_seed(13)
    model = make(kind, kw, dtype).eval()
    src = model_src(kind, kw, B, 7)
    base = _baseline(src, 5)
    t = (torch.arange(B, device=DEV) + 3) % kw["num_classes"]
    attr = model.integrated_gradients(src, t, base, steps=1)
    ref = _autograd_loop(model, src, base, t, 1)
    e = l2_rel(attr.cpu().numpy(), ref.cpu().numpy())
    assert e <= (1e-5 if dtype == "fp32" else TOL["bf16"]), e


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_baseline_equal_to_input_gives_exactly_zero(dtype):
    kind, kw, B = SURF
    torch.manual_seed(14)
    model = make(kind, kw, dtype).eval()
    src = model_src(kind, kw, B, 8)
    attr, delta = model.integrated_gradients(src, baseline=src.clone(), steps=4, return_delta=True)
    assert torch.equal(attr, torch.zeros_like(attr))
    assert torch.equal(delta, torch.zeros_like(delta))


def _call_entry(model, src, base, t, steps, chunk):
    core = model._core
    B = src.shape[0]
    desc = core.make_desc(src, training=True, module_training=False)
    alpha, w = R.nodes(steps)
    alpha = torch.tensor(alpha, dtype=torch.float32, device=DEV)
    w = torch.tensor(w, dtype=torch.float32, device=DEV)
    ws = torch.empty(_lib.ig_workspace_bytes(desc, chunk), dtype=torch.uint8, device=DEV)
    logits = torch.empty(2, B, core.C, device=DEV)
    attr = torch.empty_like(src)
    rc = _lib.lib.amc_model_integrated_gradients(C.byref(desc), src.data_ptr(), base.data_ptr(), core.flat.data_ptr(),
                                                 core.pos_buffer().data_ptr(), ws.data_ptr(), _lib.ptr(t), steps,
                                                 alpha.data_ptr(), w.data_ptr(), chunk, logits.data_ptr(),
                                                 attr.data_ptr(), _stream())
    return rc, logits, attr


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
@pytest.mark.parametrize("shape", [REF_SHAPES[0], REF_SHAPES[5]], ids=["seg16", "conv1d_meanpool"])
def test_out_of_range_target_gives_a_nan_row(shape, dtype):
    kind, kw, B = shape
    torch.manual_seed(6)
    model = make(kind, kw, dtype).eval()
    src = model_src(kind, kw, B, 6)
    base = _baseline(src)
    C_ = kw["num_classes"]
    good = torch.arange(B, device=DEV) % C_
    bad = good.clone()
    bad[1], bad[B - 1] = C_, -1
    rc0, lg0, a0 = _call_entry(model, src, base, good, 4, 2)
    rc1, lg1, a1 = _call_entry(model, src, base, bad, 4, 2)
    assert rc0 == 0 and rc1 == 0
    assert bool(torch.isnan(a1[1]).all()) and bool(torch.isnan(a1[B - 1]).all())
    keep = [b for b in range(B) if b not in (1, B - 1)]
    assert bool(torch.isfinite(a0).all()) and bool(torch.isfinite(a1[keep]).all())
    assert torch.allclose(a1[keep], a0[keep], rtol=1e-6, atol=0)
    assert torch.equal(lg1, lg0)
    # the logits of both endpoints, as a forward of each gives them
    with torch.no_grad():
        assert torch.allclose(lg0[0], model(src), rtol=1e-5, atol=1e-5)
        assert torch.allclose(lg0[1], model(base), rtol=1e-5, atol=1e-5)


def test_entry_point_validates_its_arguments():
    kind, kw, B = SURF
    model = make(kind, kw, "bf16")
    src = model_src(kind, kw, B, 0)
    base = torch.zeros_like(src)
    assert _call_entry(model, src, base, None, 4, 2)[0] == 0
    core = model._core
    for desc in (core.make_desc(src, training=False, module_training=False),
                 core._desc(B=B, dtype=_lib.BF16, training=True, p_drop=0.1)):
        out = _lib.AmcWorkspaceInfo()
        assert _lib.lib.amc_model_ig_workspace(C.byref(desc), 2, C.byref(out)) == 0
        ws = torch.empty(out.bytes, dtype=torch.uint8, device=DEV)
        a = torch.empty_like(src)
        lg = torch.empty(2, B, core.C, device=DEV)
        nodes = torch.full((4,), 0.25, device=DEV)
        assert _lib.lib.amc_model_integrated_gradients(C.byref(desc), src.data_ptr(), base.data_ptr(),
                                                       core.flat.data_ptr(), core.pos_buffer().data_ptr(), ws.data_ptr(),
                                                       None, 4, nodes.data_ptr(), nodes.data_ptr(), 2, lg.data_ptr(),
                                                       a.data_ptr(), _stream()) != 0
    ok = core.make_desc(src, training=True, module_training=False)
    out = _lib.AmcWorkspaceInfo()
    assert _lib.lib.amc_model_ig_workspace(C.byref(ok), 0, C.byref(out)) != 0
    torch.cuda.synchronize()


# ---- surface properties ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_argmax_default_and_bit_identical_repeats(dtype):
    kind, kw, B = SURF
    torch.manual_seed(0)
    model = make(kind, kw, dtype).eval()
    src = model_src(kind, kw, B, 1)
    a0 = model.integrated_gradients(src)
    with torch.no_grad():
        t = model(src).argmax(1).contiguous()
    assert torch.equal(model.integrated_gradients(src, t), a0)
    assert torch.equal(model.integrated_gradients(src), a0)
    other = ((t + 1) % kw["num_classes"]).contiguous()
    assert not torch.equal(model.integrated_gradients(src, other), a0)


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_internal_batch_size_changes_only_the_summation_order(dtype):
    kind, kw, B = SURF
    torch.manual_seed(1)
    model = make(kind, kw, dtype).eval()
    src = model_src(kind, kw, B, 2)
    t = torch.arange(B, device=DEV) % kw["num_classes"]
    ref = model.integrated_gradients(src, t, steps=7)
    scale = ref.abs().max().item()
    for ibs in (1, 3 * B, 10 ** 6):          # one point a pass, 3 + 3 + 1, all seven at once
        a = model.integrated_gradients(src, t, steps=7, internal_batch_size=ibs)
        err = (a - ref).abs().max().item()
        assert err <= 1e-5 * scale, (ibs, err)


def test_a_frame_does_not_depend_on_its_batch_neighbours():
    kind, kw, B = SURF
    torch.manual_seed(4)
    model = make(kind, kw, "fp32").eval()
    src = model_src(kind, kw, B, 3)
    base = _baseline(src)
    t = (torch.arange(B, device=DEV) * 3) % kw["num_classes"]
    full = model.integrated_gradients(src, t, base, steps=4)
    for b in (0, B - 1):
        one = model.integrated_gradients(src[b:b + 1].contiguous(), t[b:b + 1].contiguous(),
                                         base[b:b + 1].contiguous(), steps=4)
        err = (one[0] - full[b]).abs().max().item()
        assert err <= 1e-5 * max(1.0, full[b].abs().max().item()), err


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_return_delta_is_the_completeness_gap(dtype):
    kind, kw, B = SURF
    torch.manual_seed(5)
    model = make(kind, kw, dtype).eval()
    src = model_src(kind, kw, B, 4)
    base = _baseline(src)
    attr, delta = model.integrated_gradients(src, baseline=base, steps=32, return_delta=True)
    assert torch.equal(attr, model.integrated_gradients(src, baseline=base, steps=32))
    with torch.no_grad():
        lx, lb = model(src).double(), model(base).double()
    t = lx.argmax(1)
    r = torch.arange(B, device=DEV)
    gap = lx[r, t] - lb[r, t]
    assert delta.shape == (B,) and delta.dtype == torch.float32
    want = attr.double().reshape(B, -1).sum(1) - gap
    assert torch.allclose(delta.double(), want, rtol=1e-4, atol=1e-4 * gap.abs().max().item())
    if dtype == "fp32":
        # completeness: the gap is small against the logit difference it accounts for (in bf16 the rounding of the
        # path's gradients, about 1e-2 relative, is of the size of these untrained logits' differences)
        assert (delta.double().abs() <= 0.05 * gap.abs().max()).all(), (delta, gap)


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_no_side_effects_dropout_off(dtype):
    kind, kw, B = SURF
    torch.manual_seed(3)
    model = make(kind, kw, dtype, drop=0.3).eval()
    src = model_src(kind, kw, B, 2)
    with torch.no_grad():
        logits0 = model(src).clone()
    flat0 = model.flat_parameters().clone()
    params = list(model.parameters())
    params[0].grad = torch.full_like(params[0], 0.25)
    a0 = model.integrated_gradients(src, steps=4)
    model.train()                                   # dropout stays off whatever model.training is
    a1 = model.integrated_gradients(src, steps=4)
    assert model.training
    model.eval()
    assert torch.equal(a0, a1) and not a0.requires_grad
    assert torch.equal(params[0].grad, torch.full_like(params[0], 0.25))
    assert all(p.grad is None for p in params[1:])
    assert all(p.requires_grad for p in params)
    with torch.no_grad():
        assert torch.equal(model(src), logits0)
    assert torch.equal(model.flat_parameters(), flat0)


def test_bad_arguments_raise():
    kind, kw, B = SURF
    model = make(kind, kw, "bf16")
    src = model_src(kind, kw, B, 0)
    C_ = kw["num_classes"]
    ok = torch.zeros(B, dtype=torch.int64, device=DEV)
    bad_targets = [ok.to(torch.int32), ok.float(), ok[:-1].contiguous(), ok.view(B, 1), ok.cpu(),
                   torch.zeros(2 * B, dtype=torch.int64, device=DEV)[::2], ok - 1, ok + C_, [0] * B]
    for t in bad_targets:
        with pytest.raises(ValueError):
            model.integrated_gradients(src, t)
    bad_baselines = [src[:-1], src.double(), src.cpu(), src.reshape(B, -1), src[0].tolist()]
    for b in bad_baselines:
        with pytest.raises(ValueError):
            model.integrated_gradients(src, baseline=b)
    for kwargs in (dict(steps=0), dict(steps=-3), dict(steps=2.5), dict(steps=True), dict(internal_batch_size=0),
                   dict(internal_batch_size=-1), dict(internal_batch_size=1.5)):
        with pytest.raises(ValueError):
            model.integrated_gradients(src, **kwargs)
    assert model.integrated_gradients(src, ok + (C_ - 1), steps=np.int64(2)).shape == src.shape

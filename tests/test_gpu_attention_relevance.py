"""Class-specific attention relevance on the device.

Op level: amc_attention_relevance_step against float64 computed from the same qkv / dO / v values (max abs error 1e-5),
at the shapes of test_gpu_attention_maps.py, with the dO rows of queries whose v_in is 0 filled with NaN.  Whole path:
model.attention_relevance against relevance_ref.py (float64 on the oracle), compared on r - u so that the identity term
cannot hide an error (L2-rel 1e-3 fp32, 6e-2 bf16: the gradient tolerances of DESIGN §3).  Surface: argmax default,
determinism, dataset-layout input, batch independence, no side effects, validation, and the NaN row an out-of-range
target gives through the C entry point."""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import relevance_ref as RR  # noqa: E402
from conftest import l2_rel  # noqa: E402
from oracle import amc_oracle as O  # noqa: E402
from test_gpu_attention_maps import OP_CASES, OP_IDS, REF_IDS, REF_SHAPES, make, model_src  # noqa: E402

from vit_vs_raw_iq_b200 import _lib  # noqa: E402

DEV = "cuda:0"
DT = {"fp32": (_lib.F32, torch.float32), "bf16": (_lib.BF16, torch.bfloat16)}
TOL = {"fp32": 1e-3, "bf16": 6e-2}
STATS = {"i_mean": 0.03, "i_std": 0.8, "q_mean": -0.02, "q_std": 1.3}


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _rand(shape, dtype, seed, scale):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return (torch.randn(*shape, device=DEV, generator=g) * scale).to(DT[dtype][1]).contiguous()


def _ref_step(qkv, dout, v, B, T, h, dh):
    x = qkv.double().view(B, T, 3, h, dh)
    q, k, vv = (x[:, :, i].transpose(1, 2) for i in range(3))
    p = torch.softmax(q @ k.transpose(2, 3) / dh ** 0.5, dim=-1)
    do = dout.double().view(B, T, h, dh).transpose(1, 2)
    do = torch.where((v > 0)[:, None, :, None], do, torch.zeros_like(do))   # rows with v_in = 0 carry no weight
    a = torch.relu((do @ vv.transpose(2, 3)) * p).mean(1)
    return v.double() + torch.einsum("bi,bij->bj", v.double(), a)


@pytest.mark.parametrize("case", OP_CASES, ids=OP_IDS)
def test_relevance_step_op_against_float64(case):
    dtype, B, T, h, dh = case
    qkv = _rand((B * T, 3 * h * dh), dtype, 5, 1.5)
    dout = _rand((B * T, h * dh), dtype, 6, 0.1)
    g = torch.Generator(device=DEV).manual_seed(7)
    v = torch.rand(B, T, device=DEV, generator=g)
    v[:, 1::3] = 0.0                      # rows with v_in = 0 are skipped ...
    v[0] = 0.0
    v[0, 0] = 1.0                         # e_0: the top layer of a CLS model
    v = v / v.sum(1, keepdim=True)
    dout.view(B, T, -1)[v == 0] = float("nan")   # ... and their dO is never read
    out = torch.full((B, T), float("nan"), device=DEV)
    _lib.check(_lib.lib.amc_attention_relevance_step(DT[dtype][0], B, T, h, dh, qkv.data_ptr(), dout.data_ptr(),
                                                     v.data_ptr(), out.data_ptr(), _stream()))
    ref = _ref_step(qkv, dout, v, B, T, h, dh)
    err = (out.double() - ref).abs().max().item()
    assert err <= 1e-5, err
    # bit-reproducible
    out2 = torch.empty_like(out)
    _lib.check(_lib.lib.amc_attention_relevance_step(DT[dtype][0], B, T, h, dh, qkv.data_ptr(), dout.data_ptr(),
                                                     v.data_ptr(), out2.data_ptr(), _stream()))
    assert torch.equal(out, out2)


def test_relevance_step_rejects_bad_arguments():
    qkv = _rand((9, 48), "bf16", 0, 1.0)
    dout = _rand((9, 16), "bf16", 1, 1.0)
    v = torch.ones(9, device=DEV)
    out = torch.empty(9, device=DEV)
    step = _lib.lib.amc_attention_relevance_step
    assert step(_lib.BF16, 1, 9, 1, 16, qkv.data_ptr(), dout.data_ptr(), v.data_ptr(), v.data_ptr(), _stream()) != 0
    assert step(_lib.BF16, 1, 9, 1, 16, qkv.data_ptr(), None, v.data_ptr(), out.data_ptr(), _stream()) != 0
    assert step(_lib.BF16, 1, 9, 1, 129, qkv.data_ptr(), dout.data_ptr(), v.data_ptr(), out.data_ptr(), _stream()) != 0
    assert step(7, 1, 9, 1, 16, qkv.data_ptr(), dout.data_ptr(), v.data_ptr(), out.data_ptr(), _stream()) != 0
    assert step(_lib.BF16, 1, 9, 1, 16, qkv.data_ptr(), dout.data_ptr(), v.data_ptr(), out.data_ptr(), _stream()) == 0
    torch.cuda.synchronize()


# ---- whole path against the float64 reference ----------------------------------------------------------------------
def _ref(model, kind, kw, src, target):
    cfg = O.Config(kind=kind, **kw)
    params = {k: v.detach().cpu().numpy() for k, v in model.state_dict().items()}
    return cfg, RR.relevance(src.cpu().numpy(), params, cfg, target)


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
@pytest.mark.parametrize("shape", REF_SHAPES, ids=REF_IDS)
def test_whole_path_against_reference(shape, dtype):
    kind, kw, B = shape
    torch.manual_seed(11)
    model = make(kind, kw, dtype).eval()
    src = model_src(kind, kw, B, 5)
    # the target is given, so that a near-tie between two bf16 logits cannot pick another class than float64 does
    t = (torch.arange(B, device=DEV) * 5 + 1) % kw["num_classes"]
    cfg, (_, ref) = _ref(model, kind, kw, src, t.cpu().numpy())
    r = model.attention_relevance(src, t)
    assert r.shape == (B, cfg.T) and r.dtype == torch.float32
    u = RR.readout(B, cfg.T, cfg.has_cls)
    e = l2_rel(r.cpu().numpy().astype(np.float64) - u, ref - u)
    assert e <= TOL[dtype], e
    assert bool((r.cpu().numpy() >= u.astype(np.float32)).all())
    if cfg.has_cls:
        assert bool((r[:, 0] >= 1.0).all())


# ---- surface properties ---------------------------------------------------------------------------------------------
SURF = REF_SHAPES[0]


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_argmax_default_and_bit_identical_repeats(dtype):
    kind, kw, B = SURF
    torch.manual_seed(0)
    model = make(kind, kw, dtype).eval()
    src = model_src(kind, kw, B, 1)
    r0 = model.attention_relevance(src)
    with torch.no_grad():
        t = model(src).argmax(1).contiguous()
    assert torch.equal(model.attention_relevance(src, t), r0)
    assert torch.equal(model.attention_relevance(src), r0)
    other = ((t + 1) % kw["num_classes"]).contiguous()
    assert not torch.equal(model.attention_relevance(src, other), r0)   # the map depends on the class asked about


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
@pytest.mark.parametrize("kind", ["rawiq", "vit"])
def test_dataset_layout_frames_give_the_model_layout_result(kind, dtype):
    kw = SURF[1] if kind == "rawiq" else REF_SHAPES[2][1]
    torch.manual_seed(2)
    model = make(kind, kw, dtype).eval()
    B = 3
    L = kw["seq_length"] if kind == "rawiq" else kw["img_size_h"] * kw["img_size_w"] // 2
    g = torch.Generator(device=DEV).manual_seed(4)
    x = torch.randn(B, L, 2, device=DEV, generator=g) * 0.7 + 0.05
    i = (x[:, :, 0] - STATS["i_mean"]) / STATS["i_std"]
    q = (x[:, :, 1] - STATS["q_mean"]) / STATS["q_std"]
    src = (torch.stack([i, q], 1) if kind == "rawiq"
           else torch.cat([i, q], 1).view(B, 1, kw["img_size_h"], kw["img_size_w"])).contiguous()
    t = torch.arange(B, device=DEV) % kw["num_classes"]
    ref = model.attention_relevance(src, t)
    model.set_raw_input(STATS)
    r = model.attention_relevance(x, t)
    model.set_raw_input(None)
    u = RR.readout(B, ref.shape[1], True)
    e = l2_rel(r.cpu().numpy() - u, ref.cpu().numpy() - u)
    assert e <= (1e-4 if dtype == "fp32" else TOL["bf16"]), e


def test_a_frame_does_not_depend_on_its_batch_neighbours():
    kind, kw, B = SURF
    torch.manual_seed(4)
    model = make(kind, kw, "fp32").eval()
    src = model_src(kind, kw, B, 3)
    t = (torch.arange(B, device=DEV) * 3) % kw["num_classes"]
    full = model.attention_relevance(src, t)
    for b in (0, B - 1):
        one = model.attention_relevance(src[b:b + 1].contiguous(), t[b:b + 1].contiguous())
        err = (one[0] - full[b]).abs().max().item()
        assert err <= 1e-5 * max(1.0, full[b].abs().max().item()), err


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
    r0 = model.attention_relevance(src)
    model.train()                                   # dropout stays off whatever model.training is
    r1 = model.attention_relevance(src)
    assert model.training
    model.eval()
    assert torch.equal(r0, r1) and not r0.requires_grad
    assert torch.equal(params[0].grad, torch.full_like(params[0], 0.25))
    assert all(p.grad is None for p in params[1:])
    assert all(p.requires_grad for p in params)
    with torch.no_grad():
        assert torch.equal(model(src), logits0)
    assert torch.equal(model.flat_parameters(), flat0)


def test_bad_target_raises():
    kind, kw, B = SURF
    model = make(kind, kw, "bf16")
    src = model_src(kind, kw, B, 0)
    C_ = kw["num_classes"]
    ok = torch.zeros(B, dtype=torch.int64, device=DEV)
    bad = [ok.to(torch.int32), ok.float(), ok[:-1].contiguous(), torch.zeros(B + 1, dtype=torch.int64, device=DEV),
           ok.view(B, 1), ok.cpu(), torch.zeros(2 * B, dtype=torch.int64, device=DEV)[::2], ok - 1, ok + C_, [0] * B]
    for t in bad:
        with pytest.raises(ValueError):
            model.attention_relevance(src, t)
    assert model.attention_relevance(src, ok + (C_ - 1)).shape == (B, model._core.layout.T)


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
@pytest.mark.parametrize("shape", [REF_SHAPES[0], REF_SHAPES[5]], ids=["seg16", "conv1d_meanpool"])
def test_out_of_range_target_gives_a_nan_row(shape, dtype):
    """The C entry point takes any int64 target: a value outside [0, C) makes that frame's row NaN (the amc_ce_loss
    convention), and the other frames keep what a valid call gives them."""
    kind, kw, B = shape
    torch.manual_seed(6)
    model = make(kind, kw, dtype).eval()
    src = model_src(kind, kw, B, 6)
    core = model._core
    C_, T = kw["num_classes"], core.layout.T

    def call(t):
        desc = core.make_desc(src, training=True, module_training=False)
        ws = torch.empty(_lib.workspace_bytes(desc), dtype=torch.uint8, device=DEV)
        lg = torch.empty(B, C_, device=DEV)
        r = torch.empty(B, T, device=DEV)
        _lib.check(_lib.lib.amc_model_relevance(C.byref(desc), src.data_ptr(), core.flat.data_ptr(),
                                                core.pos_buffer().data_ptr(), ws.data_ptr(), t.data_ptr(),
                                                lg.data_ptr(), r.data_ptr(), _stream()), "amc_model_relevance")
        return lg, r

    good = torch.arange(B, device=DEV) % C_
    bad = good.clone()
    bad[1], bad[B - 1] = C_, -1
    lg0, r0 = call(good)
    lg1, r1 = call(bad)
    assert bool(torch.isnan(r1[1]).all()) and bool(torch.isnan(r1[B - 1]).all())
    keep = [b for b in range(B) if b not in (1, B - 1)]
    assert bool(torch.isfinite(r0).all()) and bool(torch.isfinite(r1[keep]).all())
    assert torch.allclose(r1[keep], r0[keep], rtol=1e-6, atol=0)
    assert torch.equal(lg1, lg0)


def test_model_relevance_validates_the_description():
    kind, kw, B = SURF
    model = make(kind, kw, "bf16")
    src = model_src(kind, kw, B, 0)
    core = model._core
    T = core.layout.T
    logits = torch.empty(B, kw["num_classes"], device=DEV)
    rel = torch.empty(B, T, device=DEV)

    def call(desc, lg=logits, r=rel):
        ws = torch.empty(_lib.workspace_bytes(desc), dtype=torch.uint8, device=DEV)
        return _lib.lib.amc_model_relevance(C.byref(desc), src.data_ptr(), core.flat.data_ptr(),
                                            core.pos_buffer().data_ptr(), ws.data_ptr(), None, _lib.ptr(lg),
                                            _lib.ptr(r), _stream())

    ok = core.make_desc(src, training=True, module_training=False)
    assert call(ok) == 0
    assert call(ok, lg=None) != 0
    assert call(ok, r=None) != 0
    assert call(core.make_desc(src, training=False, module_training=False)) != 0
    assert call(core._desc(B=B, dtype=_lib.BF16, training=True, p_drop=0.1)) != 0
    torch.cuda.synchronize()

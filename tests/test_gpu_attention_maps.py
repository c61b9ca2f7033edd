"""Attention maps and attention rollout on the device.

Op level: amc_attention_probs / amc_attention_rollout_step against float64 computed from the same bf16 / fp32 qkv values
(max abs error 1e-5), at shapes that mirror each forward attention regime.  Whole path: model.attention_maps /
model.attention_rollout against the numpy oracle (fp32: P 1e-4 max abs, rollout 1e-4 L2-rel; bf16: 2e-2 for both, the
bf16 logit bound of DESIGN §3).  Surface: layer subsets, dataset-layout input, no side effects, determinism, validation."""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import attention_ref as R  # noqa: E402
from conftest import l2_rel  # noqa: E402
from oracle import amc_oracle as O  # noqa: E402

import vit_vs_raw_iq_b200 as amc  # noqa: E402
from vit_vs_raw_iq_b200 import _lib  # noqa: E402

DEV = "cuda:0"
DT = {"fp32": (_lib.F32, torch.float32), "bf16": (_lib.BF16, torch.bfloat16)}

# (dtype, B, T, h, dh): the forward attention regime each shape mirrors
OP_CASES = [
    ("bf16", 5, 9, 4, 16),      # T <= 16 attn_mma (ViT p16)
    ("bf16", 3, 17, 2, 32),     # attn_tiles
    ("bf16", 2, 33, 4, 64),     # attn_tiles
    ("bf16", 3, 65, 2, 16),     # tcgen05 / attn_tiles boundary
    ("bf16", 1, 129, 8, 16),    # tcgen05 (ViT p4, raw-IQ seg8 SPS-1)
    ("bf16", 2, 129, 2, 32),    # tcgen05
    ("bf16", 3, 257, 2, 64),    # tcgen05 (SPS-2 seg8), probs rows staged whole
    ("bf16", 2, 1025, 2, 32),   # attn_long (conv1d): probs in two passes, rollout streamed
    ("bf16", 1, 1025, 1, 16),
    ("bf16", 2, 40, 2, 24),     # head dim that is not a multiple of 16 (zero-padded k)
    ("bf16", 3, 33, 2, 20),     # head dim not a multiple of 8: element-wise q / k loads
    ("bf16", 1, 300, 1, 20),    # the same, rows of more than 288 tokens
    ("fp32", 5, 9, 2, 16),      # attn_frames (fp32 parity path)
    ("fp32", 3, 33, 2, 32),
    ("fp32", 1, 65, 2, 64),
    ("fp32", 3, 129, 2, 48),    # SIMT head dims 48 / 96 / 128
    ("fp32", 2, 257, 1, 96),
    ("fp32", 2, 129, 1, 128),
    ("fp32", 1, 1025, 2, 32),   # attn_long fp32
    ("fp32", 2, 65, 3, 18),     # head dim not a multiple of 4: element-wise loads
]
OP_IDS = [f"{c[0]}-B{c[1]}-T{c[2]}-h{c[3]}-dh{c[4]}" for c in OP_CASES]


def _qkv(dtype, B, T, h, dh, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    x = torch.randn(B * T, 3 * h * dh, device=DEV, generator=g) * 1.5
    return x.to(DT[dtype][1]).contiguous()


def _ref_probs(qkv, B, T, h, dh):
    x = qkv.double().view(B, T, 3, h, dh)
    q, k = x[:, :, 0].transpose(1, 2), x[:, :, 1].transpose(1, 2)
    return torch.softmax(q @ k.transpose(2, 3) / dh ** 0.5, dim=-1)


def _stream():
    return torch.cuda.current_stream().cuda_stream


@pytest.mark.parametrize("case", OP_CASES, ids=OP_IDS)
def test_probs_op_against_float64(case):
    dtype, B, T, h, dh = case
    qkv = _qkv(dtype, B, T, h, dh, 1)
    out = torch.full((B, h, T, T), float("nan"), device=DEV)
    _lib.check(_lib.lib.amc_attention_probs(DT[dtype][0], B, T, h, dh, qkv.data_ptr(), out.data_ptr(), _stream()))
    err = (out.double() - _ref_probs(qkv, B, T, h, dh)).abs().max().item()
    assert err <= 1e-5, err


@pytest.mark.parametrize("case", OP_CASES, ids=OP_IDS)
def test_rollout_step_op_against_float64(case):
    dtype, B, T, h, dh = case
    qkv = _qkv(dtype, B, T, h, dh, 2)
    g = torch.Generator(device=DEV).manual_seed(3)
    v = torch.rand(B, T, device=DEV, generator=g)
    v[:, 1::3] = 0.0                      # rows with v_in = 0 are skipped
    v[0] = 0.0
    v[0, 0] = 1.0                         # e_0: the top layer of a CLS model
    v = v / v.sum(1, keepdim=True)
    out = torch.full((B, T), float("nan"), device=DEV)
    _lib.check(_lib.lib.amc_attention_rollout_step(DT[dtype][0], B, T, h, dh, qkv.data_ptr(), v.data_ptr(),
                                                   out.data_ptr(), _stream()))
    p = _ref_probs(qkv, B, T, h, dh)
    ref = 0.5 * v.double() + 0.5 * torch.einsum("bi,bhij->bj", v.double(), p) / h
    err = (out.double() - ref).abs().max().item()
    assert err <= 1e-5, err


def test_ops_reject_bad_arguments():
    qkv = _qkv("bf16", 1, 9, 1, 16, 0)
    out = torch.empty(81, device=DEV)
    assert _lib.lib.amc_attention_probs(_lib.BF16, 1, 9, 1, 129, qkv.data_ptr(), out.data_ptr(), _stream()) != 0
    assert _lib.lib.amc_attention_probs(7, 1, 9, 1, 16, qkv.data_ptr(), out.data_ptr(), _stream()) != 0
    assert _lib.lib.amc_attention_rollout_step(_lib.BF16, 1, 9, 1, 16, qkv.data_ptr(), out.data_ptr(), out.data_ptr(),
                                               _stream()) != 0


# ---- whole path against the oracle --------------------------------------------------------------------------------
# the shapes of test_gpu_input_grad.py::REF_SHAPES: ViT p4 / p16, raw-IQ seg16, SPS-2 seg8, conv1d with and without CLS
REF_SHAPES = [
    ("rawiq", dict(in_channels=2, seq_length=1024, num_classes=11, d_model=128, n_head=8, n_layers=3,
                   ffn_hidden=512, use_cls_token=True, embedding_type="segment", segment_size=16), 5),
    ("vit", dict(in_channels=1, img_size_h=32, img_size_w=64, patch_size=16, num_classes=19, d_model=256, n_head=8,
                 n_layers=2, ffn_hidden=1024), 9),
    ("vit", dict(in_channels=1, img_size_h=32, img_size_w=64, patch_size=4, num_classes=19, d_model=128, n_head=8,
                 n_layers=2, ffn_hidden=512), 3),
    ("rawiq", dict(in_channels=2, seq_length=2048, num_classes=11, d_model=256, n_head=8, n_layers=2,
                   ffn_hidden=1024, use_cls_token=True, embedding_type="segment", segment_size=8), 2),
    ("rawiq", dict(in_channels=2, seq_length=1024, num_classes=11, d_model=128, n_head=8, n_layers=2,
                   ffn_hidden=256, use_cls_token=True, embedding_type="conv1d", segment_size=64), 2),
    ("rawiq", dict(in_channels=2, seq_length=512, num_classes=11, d_model=64, n_head=2, n_layers=2,
                   ffn_hidden=128, use_cls_token=False, embedding_type="conv1d", segment_size=64), 3),
]
REF_IDS = ["seg16", "vit_p16", "vit_p4", "sps2_seg8", "conv1d_cls", "conv1d_meanpool"]
TOL = {"fp32": (1e-4, 1e-4), "bf16": (2e-2, 2e-2)}


def make(kind, kw, dtype, drop=0.0):
    cls = amc.RawIQAMCTransformer if kind == "rawiq" else amc.ViTAMCTransformer
    return cls(**kw, drop_prob=drop, device=DEV, compute_dtype=dtype)


def model_src(kind, kw, B, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    shape = (B, kw["in_channels"], kw["seq_length"]) if kind == "rawiq" else (B, 1, kw["img_size_h"], kw["img_size_w"])
    return torch.randn(*shape, device=DEV, generator=g)


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
@pytest.mark.parametrize("shape", REF_SHAPES, ids=REF_IDS)
def test_whole_path_against_oracle(shape, dtype):
    kind, kw, B = shape
    torch.manual_seed(11)
    model = make(kind, kw, dtype).eval()
    src = model_src(kind, kw, B, 5)
    maps = model.attention_maps(src)
    roll = model.attention_rollout(src)
    cfg = O.Config(kind=kind, **kw)
    params = {k: v.detach().cpu().numpy() for k, v in model.state_dict().items()}
    ref = R.maps(src.cpu().numpy(), params, cfg)
    ptol, rtol = TOL[dtype]
    assert len(maps) == kw["n_layers"]
    for m, r in zip(maps, ref):
        assert m.shape == r.shape and m.dtype == torch.float32
        err = np.abs(m.cpu().numpy() - r).max()
        assert err <= ptol, err
    rref = R.rollout(ref, cfg.has_cls)
    assert roll.shape == (B, cfg.T)
    e = l2_rel(roll.cpu().numpy().astype(np.float64), rref)
    assert e <= rtol, e
    np.testing.assert_allclose(roll.sum(1).cpu().numpy(), 1.0, atol=1e-5)


# ---- surface properties ---------------------------------------------------------------------------------------------
SURF = REF_SHAPES[0]
STATS = {"i_mean": 0.03, "i_std": 0.8, "q_mean": -0.02, "q_std": 1.3}


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_layer_subset_comes_back_in_the_order_asked(dtype):
    kind, kw, B = SURF
    torch.manual_seed(0)
    model = make(kind, kw, dtype).eval()
    src = model_src(kind, kw, B, 1)
    full = model.attention_maps(src)
    sub = model.attention_maps(src, layers=[2, 0])
    assert len(sub) == 2
    assert torch.equal(sub[0], full[2]) and torch.equal(sub[1], full[0])
    one = model.attention_maps(src, layers=(1,))
    assert len(one) == 1 and torch.equal(one[0], full[1])
    # any integer type; a repeated layer is its own copy
    arr = model.attention_maps(src, layers=np.array([1, 1]))
    assert torch.equal(arr[0], full[1]) and torch.equal(arr[1], full[1])
    assert arr[0].untyped_storage().data_ptr() != arr[1].untyped_storage().data_ptr()
    assert torch.equal(model.attention_maps(src, layers=[np.int64(2)])[0], full[2])


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
@pytest.mark.parametrize("kind", ["rawiq", "vit"])
def test_dataset_layout_frames_give_the_same_maps(kind, dtype):
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
    ref_maps, ref_roll = model.attention_maps(src), model.attention_rollout(src)
    model.set_raw_input(STATS)
    maps, roll = model.attention_maps(x), model.attention_rollout(x)
    model.set_raw_input(None)
    tol = 1e-5 if dtype == "fp32" else 2e-2
    for a, b in zip(maps, ref_maps):
        assert (a - b).abs().max().item() <= tol
    assert (roll - ref_roll).abs().max().item() <= tol


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_no_side_effects_dropout_off_and_bit_identical_repeats(dtype):
    kind, kw, B = SURF
    torch.manual_seed(3)
    model = make(kind, kw, dtype, drop=0.3).eval()
    src = model_src(kind, kw, B, 2)
    with torch.no_grad():
        logits0 = model(src).clone()
    flat0 = model.flat_parameters().clone()
    maps0, roll0 = model.attention_maps(src), model.attention_rollout(src)
    model.train()                                   # dropout stays off in the maps whatever model.training is
    maps1, roll1 = model.attention_maps(src), model.attention_rollout(src)
    model.eval()
    for a, b in zip(maps0, maps1):
        assert torch.equal(a, b)
    assert torch.equal(roll0, roll1)
    assert not roll0.requires_grad and not maps0[0].requires_grad
    with torch.no_grad():
        assert torch.equal(model(src), logits0)
    assert torch.equal(model.flat_parameters(), flat0)


@pytest.mark.parametrize("layers", [[3], [-1], [], ["0"], [True], [0, 5], [1.0], [np.bool_(True)]])
def test_invalid_layers_raise(layers):
    kind, kw, B = SURF
    model = make(kind, kw, "bf16")
    with pytest.raises(ValueError):
        model.attention_maps(model_src(kind, kw, B, 0), layers=layers)


def test_model_attention_validates_the_description():
    kind, kw, B = SURF
    model = make(kind, kw, "bf16")
    src = model_src(kind, kw, B, 0)
    core = model._core
    T, h = core.layout.T, kw["n_head"]
    out = torch.empty(B * h * T * T, device=DEV)
    roll = torch.empty(B * T, device=DEV)

    def call(desc, mask, probs, rollout):
        ws = torch.empty(_lib.workspace_bytes(desc), dtype=torch.uint8, device=DEV)
        return _lib.lib.amc_model_attention(C.byref(desc), src.data_ptr(), core.flat.data_ptr(),
                                            core.pos_buffer().data_ptr(), ws.data_ptr(), mask, _lib.ptr(probs),
                                            _lib.ptr(rollout), _stream())

    ok = core.make_desc(src, training=True, module_training=False)
    assert call(ok, 1, out, roll) == 0
    assert call(ok, 0, None, None) != 0                       # nothing asked for
    assert call(ok, 1 << kw["n_layers"], out, None) != 0      # a layer that does not exist
    assert call(ok, 1, None, None) != 0                       # maps asked for, nowhere to write them
    assert call(core.make_desc(src, training=False, module_training=False), 1, out, None) != 0
    drop = core._desc(B=B, dtype=_lib.BF16, training=True, p_drop=0.1)
    assert call(drop, 1, out, None) != 0
    torch.cuda.synchronize()

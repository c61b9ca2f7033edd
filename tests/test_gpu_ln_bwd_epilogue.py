"""The LayerNorm-backward GEMM epilogue (RE_LNB in csrc/gemm_tc.cu): in isolation through amc_gemm_ln_bwd against
float64, and on the model path, where the dgrad FFN1 / dgrad QKV GEMMs carry the backward of norm1 / the previous
layer's norm2: dropout masks equal to the forward's, and a staged backward equal to a single call."""
import ctypes as C

import pytest
import torch

pytestmark = pytest.mark.gpu

import vit_vs_raw_iq_b200 as amc  # noqa: E402
from vit_vs_raw_iq_b200 import _lib  # noqa: E402

DEV = "cuda:0"


def stream():
    return torch.cuda.current_stream().cuda_stream


def relerr(a, b):
    a, b = a.double(), b.double()
    return ((a - b).abs().max() / b.abs().max().clamp_min(1e-30)).item()


def l2_rel(a, b):
    a, b = a.double(), b.double()
    return ((a - b).norm() / b.norm().clamp_min(1e-30)).item()


def gemm_ln_bwd(A, B, res, xhat, rstd, gamma, dgamma=None, dbeta=None, dbias=None):
    M, K = A.shape
    N = B.shape[0]
    du16 = torch.empty(M, N, device=DEV, dtype=torch.bfloat16)
    du32 = torch.empty(M, N, device=DEV)
    _lib.check(_lib.lib.amc_gemm_ln_bwd(M, N, K, A.data_ptr(), K, B.data_ptr(), K, res.data_ptr(), xhat.data_ptr(),
                                        rstd.data_ptr(), gamma.data_ptr(), du16.data_ptr(), du32.data_ptr(),
                                        _lib.ptr(dgamma), _lib.ptr(dbeta), _lib.ptr(dbias), stream()),
               "amc_gemm_ln_bwd")
    torch.cuda.synchronize()
    return du16, du32


# N = d of the encoder (64 / 128 / 256) at K = 3d (dgrad QKV) and F (dgrad FFN1); M not a multiple of the 128-row tile
@pytest.mark.parametrize("M,N,K", [(1000, 256, 1024), (4096, 256, 768), (513, 128, 1024), (77, 64, 64)])
def test_gemm_ln_bwd_epilogue_against_float64(M, N, K):
    g = torch.Generator(device=DEV).manual_seed(M + N + K)
    A = torch.randn(M, K, device=DEV, generator=g).bfloat16()
    B = (torch.randn(N, K, device=DEV, generator=g) / K ** 0.5).bfloat16()
    res = torch.randn(M, N, device=DEV, generator=g)
    xhat = torch.randn(M, N, device=DEV, generator=g).bfloat16()
    rstd = 0.5 + torch.rand(M, device=DEV, generator=g)
    gamma = torch.randn(N, device=DEV, generator=g)
    dg0, db0, dbias0 = (torch.randn(N, device=DEV, generator=g) for _ in range(3))
    dgamma, dbeta, dbias = dg0.clone(), db0.clone(), dbias0.clone()
    du16, du32 = gemm_ln_bwd(A, B, res, xhat, rstd, gamma, dgamma, dbeta, dbias)

    t = A.double() @ B.double().t() + res.double()
    xh = xhat.double()
    gg = t * gamma.double()
    du = rstd.double()[:, None] * (gg - gg.mean(-1, keepdim=True) - xh * (gg * xh).mean(-1, keepdim=True))
    assert relerr(du32, du) < 1e-4
    assert relerr(du16.float(), du) < 1e-2
    # the column sums accumulate into what the outputs held
    assert relerr(dgamma - dg0, (t * xh).sum(0)) < 1e-4
    assert relerr(dbeta - db0, t.sum(0)) < 1e-4
    assert relerr(dbias - dbias0, du.sum(0)) < 1e-4
    assert relerr(dgamma, dg0.double() + (t * xh).sum(0)) < 1e-4

    # without parameter gradients the row outputs are unchanged, bit for bit
    n16, n32 = gemm_ln_bwd(A, B, res, xhat, rstd, gamma)
    assert torch.equal(n16, du16) and torch.equal(n32, du32)
    # any one of the sums alone
    only = torch.zeros(N, device=DEV)
    gemm_ln_bwd(A, B, res, xhat, rstd, gamma, dbeta=only)
    assert relerr(only, t.sum(0)) < 1e-4


def test_gemm_ln_bwd_rejects_unsupported_shapes():
    A = torch.zeros(64, 64, device=DEV, dtype=torch.bfloat16)
    for N in (512, 96 + 8):   # N > 256, N % 32 != 0
        B = torch.zeros(N, 64, device=DEV, dtype=torch.bfloat16)
        res, xhat = torch.zeros(64, N, device=DEV), torch.zeros(64, N, device=DEV, dtype=torch.bfloat16)
        with pytest.raises(RuntimeError, match="LayerNorm-backward"):
            gemm_ln_bwd(A, B, res, xhat, torch.ones(64, device=DEV), torch.ones(N, device=DEV))


def _rawiq(d, dtype, n_layers=3, drop=0.3):
    torch.manual_seed(11)
    return amc.RawIQAMCTransformer(in_channels=2, seq_length=256, num_classes=11, d_model=d, n_head=4,
                                   n_layers=n_layers, ffn_hidden=2 * d, drop_prob=drop, device=DEV,
                                   use_cls_token=True, embedding_type="segment", segment_size=16,
                                   compute_dtype=dtype)


@pytest.mark.parametrize("d", [64, 256])
def test_bf16_backward_masks_match_fp32(d):
    """The dropout masks depend on (seed, offset, site, element index) only, so a bf16 model and an fp32 model with the
    same weights and a frozen call counter draw the same ones; the bf16 backward, whose norm backward runs in the dgrad
    GEMM epilogues (d <= 256), must regenerate the masks the forward used.  A wrong site or element index moves whole
    masked entries and fails this by far more than the bf16 rounding allowed for."""
    src = torch.randn(24, 2, 256, device=DEV)
    wgt = torch.randn(24, 11, device=DEV)
    grads = {}
    for dtype in ("fp32", "bf16"):
        model = _rawiq(d, dtype)
        model.train()
        model._core.calls = 5
        x = src.clone().requires_grad_(True)
        (model(x) * wgt).sum().backward()
        grads[dtype] = ({n: p.grad.detach().clone() for n, p in model.named_parameters()}, x.grad.detach().clone())
    (gf, xf), (gb, xb) = grads["fp32"], grads["bf16"]
    assert l2_rel(xb, xf) < 5e-2
    # (the key bias gets an exactly zero gradient, softmax being shift-invariant: both sides are rounding noise)
    worst = max((l2_rel(gb[n], gf[n]), n) for n in gf if not n.endswith("w_k.bias"))
    assert worst[0] < 8e-2, worst
    # the masks are really on: the same bf16 model at another counter value gives other gradients
    model = _rawiq(d, "bf16")
    model.train()
    model._core.calls = 6
    (model(src) * wgt).sum().backward()
    assert max(l2_rel(p.grad, gb[n]) for n, p in model.named_parameters() if not n.endswith("w_k.bias")) > 0.2


@pytest.mark.parametrize("cls_top", [True, False])
def test_staged_backward_equals_one_call(cls_top):
    """amc_model_bwd_ex over [0, L + 2) in one call and stage by stage: the stage of layer l + 1 hands the gradient of
    layer l's norm2 input (dw16 / dw32) to the next stage, and writes layer l's gamma2 / beta2 / b2 gradients."""
    model = _rawiq(128, "bf16", n_layers=3)
    core = model._core
    B = 16
    src = torch.randn(B, 2, 256, device=DEV)
    desc = core.make_desc(src, training=True, module_training=True)
    ws = torch.empty(_lib.workspace_bytes(desc), dtype=torch.uint8, device=DEV)
    T = core.layout.T
    logits = torch.empty(B, 11, device=DEV)
    dlogits = torch.randn(B, 11, device=DEV) * 1e-2
    enc = torch.empty(B, T, 128, device=DEV)
    denc = torch.randn(B, T, 128, device=DEV) * 1e-3
    L = core.n_layers

    def run(ranges):
        _lib.check(_lib.lib.amc_model_fwd(C.byref(desc), src.data_ptr(), core.flat.data_ptr(),
                                          core.pos_buffer().data_ptr(), ws.data_ptr(),
                                          logits.data_ptr() if cls_top else 0, 0 if cls_top else enc.data_ptr(),
                                          stream()), "fwd")
        grads = torch.zeros(core.layout.total, device=DEV)
        dsrc = torch.zeros_like(src)
        for s0, s1 in ranges:
            _lib.check(_lib.lib.amc_model_bwd_ex(C.byref(desc), src.data_ptr(), core.flat.data_ptr(), ws.data_ptr(),
                                                 dlogits.data_ptr() if cls_top else 0,
                                                 0 if cls_top else denc.data_ptr(), grads.data_ptr(),
                                                 dsrc.data_ptr(), s0, s1, stream()), "bwd")
        torch.cuda.synchronize()
        return grads, dsrc

    g1, x1 = run([(0, L + 2)])
    g2, x2 = run([(s, s + 1) for s in range(L + 2)])
    g3, x3 = run([(0, 2), (2, L + 2)])
    assert g1.norm() > 0 and x1.norm() > 0
    for g, x in ((g2, x2), (g3, x3)):
        assert l2_rel(g, g1) < 1e-5
        assert l2_rel(x, x1) < 1e-5
    # the norm2 parameter gradients of every layer below the top one are produced, and by the stage above
    Lo = core.layout
    for l in range(L - 1):
        b = Lo.layer0 + l * Lo.layer_stride
        for off in (Lo.g2, Lo.be2, Lo.b2):
            assert g1[b + off:b + off + 128].norm() > 0
    part = run([(0, 2)])[0]           # head + top layer only: layer L - 2's norm2 gradients are final
    b = Lo.layer0 + (L - 2) * Lo.layer_stride
    for off in (Lo.g2, Lo.be2, Lo.b2):
        assert l2_rel(part[b + off:b + off + 128], g1[b + off:b + off + 128]) < 1e-5

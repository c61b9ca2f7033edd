"""Projected-gradient attacks: the amc_adv_step / amc_adv_init kernels against torch and float64 (adversarial_ref.py),
PGDAttack against the module surface's autograd, attack strength on a trained model, adversarial training through
TrainStep / GraphTrainStep / HostPipeline, robust evaluation, and argument errors."""
import math
import re

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import adversarial_ref as R  # noqa: E402
from conftest import GOLDEN_CASES, load_golden  # noqa: E402

import vit_vs_raw_iq_b200 as amc  # noqa: E402
from vit_vs_raw_iq_b200 import _lib, synth  # noqa: E402
from vit_vs_raw_iq_b200.adversarial import PGDAttack  # noqa: E402
from vit_vs_raw_iq_b200.evaluate import evaluate_model_with_confusion  # noqa: E402
from vit_vs_raw_iq_b200.trainer import GraphTrainStep, HostPipeline, TrainStep  # noqa: E402

DEV = "cuda:0"
STATS = {"i_mean": 0.03, "i_std": 0.8, "q_mean": -0.02, "q_std": 1.3}
LINF, L2 = _lib.NORM_LINF, _lib.NORM_L2


def stream():
    return torch.cuda.current_stream().cuda_stream


def adv_step(x0, g, eps, step_frac, x, norm):
    B, n = x0.shape[0], x0[0].numel()
    _lib.check(_lib.lib.amc_adv_step(B, n, norm, x0.data_ptr(), g.data_ptr(), eps.data_ptr(), step_frac, x.data_ptr(),
                                     stream()), "amc_adv_step")


def adv_init(x0, eps, seed, offset, ctr, x, norm):
    B, n = x0.shape[0], x0[0].numel()
    _lib.check(_lib.lib.amc_adv_init(B, n, norm, x0.data_ptr(), eps.data_ptr(), seed, offset, _lib.ptr(ctr),
                                     x.data_ptr(), stream()), "amc_adv_init")


def frames(B, n, seed, offset=0):
    """x0, x (inside the L-inf ball of eps), g with exact zeros, eps with zero frames; `offset` > 0 gives frames that
    start off the 16-byte grid."""
    gen = torch.Generator(device=DEV).manual_seed(seed)

    def buf(t):
        if not offset:
            return t.contiguous()
        raw = torch.empty(t.numel() + offset, device=DEV)
        v = raw[offset:].view(t.shape)
        v.copy_(t)
        return v

    x0 = torch.randn(B, n, device=DEV, generator=gen)
    eps = 0.05 + 0.2 * torch.rand(B, device=DEV, generator=gen)
    eps[::7] = 0.0
    x = x0 + eps[:, None] * (2 * torch.rand(B, n, device=DEV, generator=gen) - 1)
    g = torch.randn(B, n, device=DEV, generator=gen)
    g[torch.rand(B, n, device=DEV, generator=gen) < 0.1] = 0.0
    return buf(x0), buf(x), buf(g), eps


# ---- 1. L-inf step: bit-identical to the torch formula -------------------------------------------------------------
@pytest.mark.parametrize("n", [1, 6, 2048, 4096, 4098, 32766])
@pytest.mark.parametrize("B", [1, 3, 1000])
def test_linf_step_bit_identical_to_torch(B, n):
    for offset, step_frac in ((0, 0.3), (1, 0.25)):
        x0, x, g, eps = frames(B, n, seed=B * 7 + n, offset=offset)
        a = eps * torch.tensor(step_frac, dtype=torch.float32, device=DEV)
        ref = torch.min(torch.max(x + a[:, None] * g.sign(), x0 - eps[:, None]), x0 + eps[:, None])
        adv_step(x0, g, eps, step_frac, x, LINF)
        assert torch.equal(x, ref)
        assert torch.equal(x[::7], x0[::7])                        # eps = 0 frames: exactly x0


# ---- 2. L2 step: float64 reference within the fp32 bound -----------------------------------------------------------
@pytest.mark.parametrize("n", [1, 6, 2048, 4096, 4098, 8192, 32766])   # 8192: the vector path of the streaming kernel
@pytest.mark.parametrize("B", [3, 200])
def test_l2_step_matches_float64(B, n):
    for offset in (0, 1):
        x0, x, g, eps = frames(B, n, seed=B + n, offset=offset)
        # an L2 budget of 0.3 ||x0|| (so the fp32 rounding of x0 + d is small next to eps); start at 0.8 eps
        eps = 0.3 * x0.norm(dim=1)
        eps[::7] = 0.0
        d = x - x0
        x = (x0 + d * (0.8 * eps / d.norm(dim=1).clamp_min(1e-30))[:, None]).contiguous()
        g[1::5] = 0.0                                             # frames with ||g|| = 0
        x_in = x.clone()
        ref = R.step_l2(x.cpu().numpy(), x0.cpu().numpy(), g.cpu().numpy(), eps.cpu().numpy(), 0.5)
        bound = R.l2_step_bound(x.cpu().numpy(), x0.cpu().numpy(), g.cpu().numpy(), eps.cpu().numpy(), 0.5)
        if offset:
            xo = torch.empty(x.numel() + 1, device=DEV)[1:].view(x.shape)
            xo.copy_(x)
            x = xo
        adv_step(x0, g, eps, 0.5, x, L2)
        got = x.cpu().numpy().astype(np.float64)
        assert (np.abs(got - ref) <= bound).all(), np.abs(got - ref).max()
        zero_g = [b for b in range(1, B, 5) if b % 7]
        assert torch.equal(x[zero_g], x_in[zero_g])               # ||g|| = 0: unchanged
        assert torch.equal(x[::7], x0[::7])                       # eps = 0: exactly x0
        dn = np.linalg.norm(got - x0.cpu().numpy().astype(np.float64), axis=1)
        assert (dn <= eps.cpu().numpy().astype(np.float64) * (1 + 1e-6)).all()


# ---- 3. random start -----------------------------------------------------------------------------------------------
def test_init_linf_inside_ball_and_moments():
    B, n = 512, 2048                                              # 1 M elements
    x0 = torch.zeros(B, n, device=DEV)
    eps = torch.ones(B, device=DEV)
    x = torch.empty_like(x0)
    adv_init(x0, eps, 1234, 7, None, x, LINF)
    u = x.double().cpu().numpy().ravel()                          # = 2u - 1, exact
    N = u.size
    assert np.abs(u).max() <= 1.0
    assert abs(u.mean()) <= 5 * math.sqrt(1 / 3 / N)
    assert abs((u * u).mean() - 1 / 3) <= 5 * math.sqrt(4 / 45 / N)
    # a nonzero centre: inside [x0 - eps, x0 + eps] as fp32 rounds them
    x0, _, _, eps = frames(300, 4098, seed=3)
    x = torch.empty_like(x0)
    adv_init(x0, eps, 1, 2, None, x, LINF)
    assert bool(((x >= x0 - eps[:, None]) & (x <= x0 + eps[:, None])).all())
    assert torch.equal(x[::7], x0[::7])


@pytest.mark.parametrize("n", [6, 2048, 4098])
def test_init_l2_inside_ball_and_radii(n):
    x0, _, _, _ = frames(400, n, seed=n)
    eps = 0.3 * x0.norm(dim=1)
    eps[::7] = 0.0
    x = torch.empty_like(x0)
    adv_init(x0, eps, 99, 0, None, x, L2)
    r = (x.double() - x0.double()).norm(dim=1)
    e = eps.double()
    assert bool((r <= e * (1 + 1e-6)).all())
    assert torch.equal(x[::7], x0[::7])
    if n == 2048:                                                  # radii u^(1/n): all >= 0.99 eps at n = 2048
        keep = e > 0
        assert bool((r[keep] >= 0.99 * e[keep]).all())


@pytest.mark.parametrize("norm", [LINF, L2])
def test_init_keying_and_graph_replay(norm):
    x0, _, _, eps = frames(64, 2048, seed=5)
    eps = eps + 0.1

    def draw(seed, offset, ctr=None):
        x = torch.empty_like(x0)
        adv_init(x0, eps, seed, offset, ctr, x, norm)
        return x

    a = draw(11, 3)
    assert torch.equal(a, draw(11, 3))
    for other in (draw(12, 3), draw(11, 4), draw(11, 3, torch.ones(1, dtype=torch.int32, device=DEV))):
        assert (other != a).float().mean().item() > 0.99
    # a captured graph reads the device counter: replay at counter k = eager draw at offset 3 + k
    ctr = torch.zeros(1, dtype=torch.int32, device=DEV)
    xg = torch.empty_like(x0)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        adv_init(x0, eps, 11, 3, ctr, xg, norm)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        adv_init(x0, eps, 11, 3, ctr, xg, norm)
    for k in (0, 5):
        ctr.fill_(k)
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(xg, draw(11, 3 + k))


# ---- 4. FGSM against the module surface ----------------------------------------------------------------------------
def bf16_supported(kind, kw):
    K = kw["in_channels"] * (kw["patch_size"] ** 2 if kind == "vit" else
                             (1 if kw["embedding_type"] == "conv1d" else kw["segment_size"]))
    return (K % 8 == 0 or (K <= 16 and kw["d_model"] >= 32)) and kw["d_model"] % 8 == 0


def golden_model(name, dtype, drop=0.0):
    kind, kw = GOLDEN_CASES[name]
    cls = amc.RawIQAMCTransformer if kind == "rawiq" else amc.ViTAMCTransformer
    model = cls(**kw, drop_prob=drop, device=DEV, compute_dtype=dtype)
    _, params, _, _ = load_golden(name)
    model.load_state_dict({k: torch.from_numpy(v) for k, v in params.items()}, strict=True)
    return model


def batch(model, B, layout, seed):
    kind, f = model._core.kind, model._core.fields
    gen = torch.Generator(device=DEV).manual_seed(seed)
    if layout == "dataset":
        model.set_raw_input(STATS)
        L = f["seq_len"] if kind == _lib.KIND_RAWIQ else f["img_h"] * f["img_w"] // 2
        shape = (B, L, 2)
    else:
        shape = (B, f["in_ch"], f["seq_len"]) if kind == _lib.KIND_RAWIQ else (B, 1, f["img_h"], f["img_w"])
    x = torch.randn(shape, device=DEV, generator=gen)
    y = torch.randint(0, f["C"], (B,), device=DEV, generator=gen)
    return x, y


@pytest.mark.parametrize("layout", ["model", "dataset"])
@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
@pytest.mark.parametrize("name", ["vit_p16", "vit_p4", "rawiq_seg16", "rawiq_conv1d", "rawiq_meanpool"])
def test_fgsm_matches_module_surface(name, dtype, layout):
    kind, kw = GOLDEN_CASES[name]
    if dtype == "bf16" and not bf16_supported(kind, kw):
        pytest.skip("tiny fixture outside the bf16 path's shapes")
    model = golden_model(name, dtype)
    model.eval()
    x0, y = batch(model, 64, layout, seed=17)
    eps = 0.05
    xr = x0.clone().requires_grad_(True)
    loss = torch.nn.functional.cross_entropy(model(xr), y, reduction="sum")
    (g,) = torch.autograd.grad(loss, xr)
    ref = (x0 + eps * g.sign()).detach()
    got = PGDAttack(model, eps=eps, steps=1, random_start=False, step_frac=1.0)(x0, y)
    assert got.shape == x0.shape and got.device == x0.device
    diff = (got - ref).abs()
    bad = diff > 1e-6
    # a sign flip where |g| sits at round-off (amc_ce_loss and torch's CE differ in the last bits): off by eps or 2 eps
    assert bad.float().mean().item() <= 1e-4, bad.sum().item()
    d = diff[bad]
    assert bool((((d - eps).abs() < 1e-5) | ((d - 2 * eps).abs() < 1e-5)).all())


# ---- 5. PGD properties ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("norm", ["linf", "l2"])
def test_pgd_deterministic_and_in_ball(norm):
    model = golden_model("vit_p16", "bf16")
    x0, y = batch(model, 32, "model", seed=2)
    eps = 0.1 if norm == "linf" else 0.1 * math.sqrt(x0[0].numel())
    for steps in (1, 2, 5):
        atk = PGDAttack(model, norm=norm, eps=eps, steps=steps, random_start=False)
        a = atk(x0, y).clone()
        assert torch.equal(a, atk(x0, y))                         # the frozen chain has no atomics
        d = (a - x0).double().view(32, -1)
        if norm == "linf":
            assert bool(((a >= x0 - eps) & (a <= x0 + eps)).all())
        else:
            assert bool((d.norm(dim=1) <= eps * (1 + 1e-6)).all())


@pytest.mark.parametrize("norm", ["linf", "l2"])
@pytest.mark.parametrize("layout", ["model", "dataset"])
def test_psr_budget_matches_float64(norm, layout):
    model = golden_model("rawiq_seg16", "fp32")
    x0, y = batch(model, 16, layout, seed=4)
    x0 = x0 * torch.linspace(0.2, 3.0, 16, device=DEV).view(16, *([1] * (x0.dim() - 1)))   # frames of unequal power
    x0 = x0.contiguous()
    out = PGDAttack(model, norm=norm, psr_db=-20.0, steps=1, random_start=False, step_frac=1.0)(x0, y)
    ref = R.psr_eps(x0.cpu().numpy(), -20.0, norm)
    d = (out.double() - x0.double()).view(16, -1).cpu().numpy()
    got = np.abs(d).max(1) if norm == "linf" else np.linalg.norm(d, axis=1)
    # fp32: the budget's own rounding, plus x0 + eps rounded to fp32 (ulp(x0) / 2 next to eps >= 0.02 at -20 dB)
    np.testing.assert_allclose(got, ref, rtol=1e-4)


def test_targeted_attack_raises_target_rate():
    model = golden_model("vit_p16", "fp32")
    model.eval()
    x0, _ = batch(model, 256, "model", seed=8)
    with torch.no_grad():
        pred = model(x0).argmax(1)
    target = (pred + 1) % model._core.C
    x = PGDAttack(model, eps=0.5, steps=10, targeted=True)(x0, target)
    with torch.no_grad():
        hit = (model(x).argmax(1) == target).float().mean().item()
    assert hit >= 0.25, hit                                      # 0 before the attack


# ---- 6. attack strength on a trained model -------------------------------------------------------------------------
def test_pgd_is_stronger_than_fgsm_and_noise():
    """A small raw-IQ model trained 300 steps on synthetic frames (fixed seeds), attacked in the dataset layout at a PSR
    of -10 dB (L-inf budget = 0.32 x the frame's RMS amplitude, i.e. the perturbation carries a tenth of the frame's
    power).  Random-sign noise of that budget is white noise at +10 dB SNR on top of the frame; FGSM and PGD-10 must both
    do at least 5 points worse than it, and PGD-10 (random start, 10 steps) may be at most 2 points (20 of the 1024
    held-out frames) above FGSM: its iterates need not dominate FGSM on every frame, but on average a 10-step ascent
    finds at least as high a loss."""
    torch.manual_seed(0)
    X, y, _ = synth.make_frames(4096 + 1024, classes=synth.CLASSES_11, seed=21)
    stats = synth.normalization_stats(X[:4096])
    model = amc.RawIQAMCTransformer(in_channels=2, seq_length=1024, num_classes=11, d_model=64, n_head=4, n_layers=2,
                                    ffn_hidden=128, drop_prob=0.0, device=DEV, segment_size=16, compute_dtype="bf16")
    model.set_raw_input(stats)
    Xt, yt = torch.from_numpy(X).to(DEV), torch.from_numpy(y).to(DEV)
    ts = GraphTrainStep(model, lr=1e-3, weight_decay=1e-2)
    for i in range(300):
        k = (i % 16) * 256
        ts.step(Xt[k:k + 256], yt[k:k + 256])
    xe, ye = Xt[4096:].contiguous(), yt[4096:].contiguous()

    def acc(x):
        with torch.no_grad():
            model.eval()
            return (model(x).argmax(1) == ye).float().mean().item()

    psr = -10.0
    eps = torch.from_numpy(R.psr_eps(xe.cpu().numpy(), psr, "linf").astype(np.float32)).to(DEV)
    gen = torch.Generator(device=DEV).manual_seed(1)
    noise = xe + eps.view(-1, 1, 1) * (torch.randint(0, 2, xe.shape, device=DEV, generator=gen) * 2 - 1)
    clean, a_noise = acc(xe), acc(noise)
    a_fgsm = acc(PGDAttack(model, psr_db=psr, steps=1, random_start=False, step_frac=1.0)(xe, ye))
    a_pgd = acc(PGDAttack(model, psr_db=psr, steps=10)(xe, ye))
    print(f"clean {clean:.3f} noise {a_noise:.3f} fgsm {a_fgsm:.3f} pgd10 {a_pgd:.3f}")
    assert clean > 0.2, clean                                     # the model learned something
    assert a_pgd <= a_fgsm + 0.02
    assert a_fgsm < a_noise - 0.05 and a_pgd < a_noise - 0.05


# ---- 7. adversarial training ---------------------------------------------------------------------------------------
def twin(name, dtype):
    return golden_model(name, dtype), golden_model(name, dtype)


@pytest.mark.parametrize("name,dtype", [("rawiq_seg16", "fp32"), ("vit_p16", "bf16")])
def test_attacked_step_equals_attack_then_plain_step(name, dtype):
    z, _, _, _ = load_golden(name)
    src = torch.from_numpy(z["src"]).to(DEV)
    labels = torch.from_numpy(z["labels"]).to(DEV)
    a, b = twin(name, dtype)
    ts_a = TrainStep(a, lr=1e-3, weight_decay=1e-2, attack=PGDAttack(a, eps=0.1, steps=3))
    ts_b = TrainStep(b, lr=1e-3, weight_decay=1e-2)
    atk_b = PGDAttack(b, eps=0.1, steps=3)
    ts_a.step(src, labels)
    b._core.calls += 1            # the attacked step makes its own descriptor first: align the random-start key
    x_adv = atk_b(src, labels)
    ts_b.step(x_adv, labels)
    (buf,) = ts_a.attack._bufs.values()
    assert torch.equal(buf["x"], x_adv)
    pa, pb = a.flat_parameters(), b.flat_parameters()
    tol = 1e-4 if dtype == "fp32" else 2e-2
    assert (pa - pb).abs().max().item() <= tol * pa.abs().max().item()


def test_zero_budget_attack_is_the_plain_step():
    z, _, _, _ = load_golden("rawiq_seg16")
    src = torch.from_numpy(z["src"]).to(DEV)
    labels = torch.from_numpy(z["labels"]).to(DEV)
    a, b = twin("rawiq_seg16", "fp32")
    ts_a = TrainStep(a, lr=1e-3, weight_decay=1e-2, attack=PGDAttack(a, eps=0.0, steps=2, random_start=False))
    ts_b = TrainStep(b, lr=1e-3, weight_decay=1e-2)
    for _ in range(2):
        ts_a.step(src, labels)
        ts_b.step(src, labels)
    pa, pb = a.flat_parameters(), b.flat_parameters()
    assert (pa - pb).abs().max().item() <= 1e-4 * pa.abs().max().item()
    la, lb = ts_a.read_stats()[0], ts_b.read_stats()[0]
    assert abs(la - lb) <= 5e-3 * abs(la)


@pytest.mark.parametrize("norm", ["linf", "l2"])
def test_graph_train_step_with_attack_follows_eager(norm):
    """Same tolerance as test_gpu_train.py::test_graph_train_step_matches_the_eager_step.  The eager twin keys its
    random starts by the same device counter, advanced once per step as amc_adamw_clip_step_graph does."""
    z, _, _, _ = load_golden("vit_p16")
    src = torch.from_numpy(z["src"]).to(DEV)
    labels = torch.from_numpy(z["labels"]).to(DEV)
    eps = 0.1 if norm == "linf" else 3.0
    a, b = twin("vit_p16", "bf16")
    ts_g = GraphTrainStep(a, lr=1e-3, weight_decay=1e-2, attack=PGDAttack(a, norm=norm, eps=eps, steps=2))
    ts_e = TrainStep(b, lr=1e-3, weight_decay=1e-2, attack=PGDAttack(b, norm=norm, eps=eps, steps=2))
    ctr = torch.zeros(1, dtype=torch.int32, device=DEV)
    b._core.step_counter = ctr
    lg, le = [], []
    for i in range(6):
        ts_g.step(src, labels)
        ts_e.step(src, labels)
        ctr.add_(1)
        if i == 0:
            (xg,) = [v["x"] for v in ts_g.attack._bufs.values()]
            (xe,) = [v["x"] for v in ts_e.attack._bufs.values()]
            assert torch.equal(xg, xe)
        lg.append(ts_g.read_stats()[0])
        le.append(ts_e.read_stats()[0])
    assert ts_g._graph is not None and int(ts_g.counter.item()) == 6
    pg, pe = a.flat_parameters(), b.flat_parameters()
    assert (pg - pe).abs().max().item() <= 2e-2 * pe.abs().max().item()
    assert all(abs(x - y) <= 5e-3 * abs(x) + 1e-5 for x, y in zip(le, lg)), (le, lg)


def test_graph_capture_survives_calls_at_other_shapes():
    """A GraphTrainStep replays kernels that write into the attack's buffers of the training shape.  Calling the same
    attack at another shape between replays (robust evaluation with a short last batch) must leave those buffers alive:
    the trainer keeps following its eager twin, and tensors allocated in between are not written by the replays."""
    z, _, _, _ = load_golden("vit_p16")
    src = torch.from_numpy(z["src"]).to(DEV)
    labels = torch.from_numpy(z["labels"]).to(DEV)
    a, b = twin("vit_p16", "bf16")
    atk_g, atk_e = PGDAttack(a, eps=0.1, steps=2), PGDAttack(b, eps=0.1, steps=2)
    ts_g = GraphTrainStep(a, lr=1e-3, weight_decay=1e-2, attack=atk_g)
    ts_e = TrainStep(b, lr=1e-3, weight_decay=1e-2, attack=atk_e)
    ctr = torch.zeros(1, dtype=torch.int32, device=DEV)
    b._core.step_counter = ctr
    small_src, small_labels = src[:2].contiguous(), labels[:2].contiguous()
    junk = []
    lg, le = [], []
    for _ in range(6):
        ts_g.step(src, labels)
        ts_e.step(src, labels)
        ctr.add_(1)
        lg.append(ts_g.read_stats()[0])
        le.append(ts_e.read_stats()[0])
        for atk in (atk_g, atk_e):
            atk(small_src, small_labels)
        junk += [torch.full_like(src, 7.0) for _ in range(4)] + [torch.full((len(src), 19), 7.0, device=DEV)
                                                                 for _ in range(2)]
    torch.cuda.synchronize()
    assert ts_g._graph is not None and ts_g.replays == 5
    assert all(bool((t == 7.0).all()) for t in junk)
    pg, pe = a.flat_parameters(), b.flat_parameters()
    assert (pg - pe).abs().max().item() <= 2e-2 * pe.abs().max().item()
    assert all(abs(x - y) <= 5e-3 * abs(x) + 1e-5 for x, y in zip(le, lg)), (le, lg)


def test_budget_is_read_only_and_a_tensor_budget_is_read_every_call():
    model = golden_model("rawiq_seg16", "fp32")
    x0, y = batch(model, 4, "model", seed=6)
    atk = PGDAttack(model, eps=0.1)
    for name in ("eps", "psr_db"):
        with pytest.raises(AttributeError):
            setattr(atk, name, 0.2)
    eps = torch.zeros(4, device=DEV)
    fgsm = PGDAttack(model, eps=eps, steps=1, random_start=False, step_frac=1.0)
    assert torch.equal(fgsm(x0, y), x0)
    eps.fill_(0.25)                                               # an eps schedule: update the tensor in place
    d = (fgsm(x0, y) - x0).abs()
    assert abs(d.max().item() - 0.25) < 1e-6


def test_launch_counts():
    """attack=None launches exactly the plain step's kernels; an attacked step adds exactly the attack's."""
    z, _, _, _ = load_golden("vit_p16")
    src = torch.from_numpy(z["src"]).to(DEV)
    labels = torch.from_numpy(z["labels"]).to(DEV)
    count = _lib.lib.amc_launch_count

    def launches(fn):
        fn()
        torch.cuda.synchronize()
        n0 = count()
        fn()
        return count() - n0

    a, b = twin("vit_p16", "bf16")
    atk = PGDAttack(a, eps=0.1, steps=3)
    ts_plain, ts_none = TrainStep(b), TrainStep(b, attack=None)
    n_plain = launches(lambda: ts_plain.step(src, labels))
    assert launches(lambda: ts_none.step(src, labels)) == n_plain
    n_atk = launches(lambda: atk(src, labels))
    ts_atk = TrainStep(a, attack=atk)
    assert launches(lambda: ts_atk.step(src, labels)) == n_plain + n_atk


def test_host_pipeline_with_attacked_trainer():
    z, _, _, _ = load_golden("rawiq_seg16")
    src, labels = torch.from_numpy(z["src"]), torch.from_numpy(z["labels"])
    model = golden_model("rawiq_seg16", "bf16")
    ts = TrainStep(model, lr=1e-3, attack=PGDAttack(model, eps=0.05, steps=1, step_frac=1.25))
    hp = HostPipeline(ts, tuple(src.shape))
    out = [hp.step(src.pin_memory(), labels.pin_memory()) for _ in range(4)] + [hp.flush()]
    assert out[0] is None and all(math.isfinite(v) for v in out[1:])


# ---- 8. robust evaluation ------------------------------------------------------------------------------------------
def test_robust_evaluation_report(tmp_path):
    X, y, snr = synth.make_frames(600, classes=synth.CLASSES_11, seed=9)
    torch.manual_seed(0)
    model = amc.RawIQAMCTransformer(in_channels=2, seq_length=1024, num_classes=11, d_model=64, n_head=4, n_layers=2,
                                    ffn_hidden=128, drop_prob=0.1, device=DEV, segment_size=16, compute_dtype="bf16")
    model.set_raw_input(synth.normalization_stats(X))
    Xt, yt, st = torch.from_numpy(X), torch.from_numpy(y), torch.from_numpy(snr)
    batches = [(Xt[i:i + 256], yt[i:i + 256], st[i:i + 256]) for i in range(0, 600, 256)]
    clean = evaluate_model_with_confusion(model, batches, synth.CLASSES_11, tmp_path / "clean")
    zero = evaluate_model_with_confusion(model, batches, synth.CLASSES_11, tmp_path / "zero",
                                         attack=PGDAttack(model, eps=0.0, steps=3))
    assert open(zero["report_path"], "rb").read() == open(clean["report_path"], "rb").read()
    rob = evaluate_model_with_confusion(model, batches, synth.CLASSES_11, tmp_path / "rob",
                                        attack=PGDAttack(model, psr_db=-10.0, steps=3))
    text = open(rob["report_path"]).read()
    assert float(re.search(r'Overall Accuracy:\s+([\d.]+)%', text).group(1)) == round(rob["overall_accuracy"] * 100, 2)
    snrs = {int(a): float(b) for a, b in re.findall(r'SNR\s+([-+]\d+)\s+dB:\s+([\d.]+)%', text)}
    assert set(snrs) == set(rob["snr_accuracies"])
    rows = [m for m in (re.match(r'^\s*(\w+)\s+([\d.]+)\s+([\d.]+)\s+([\d.]+)\s+(\d+)', line)
                        for line in text.splitlines()) if m]
    assert sum(int(m.group(5)) for m in rows if m.group(1) in synth.CLASSES_11) == 600


# ---- 9. argument errors --------------------------------------------------------------------------------------------
def test_argument_errors():
    model = golden_model("rawiq_seg16", "fp32")
    other = golden_model("rawiq_seg16", "fp32")
    x0, y = batch(model, 4, "model", seed=1)
    n = x0[0].numel()
    g, x, eps = torch.zeros_like(x0), x0.clone(), torch.ones(4, device=DEV)
    lib = _lib.lib

    def step_rc(B=4, n=n, norm=LINF, sf=0.5, ptrs=None):
        p = ptrs or (x0.data_ptr(), g.data_ptr(), eps.data_ptr(), x.data_ptr())
        return lib.amc_adv_step(B, n, norm, p[0], p[1], p[2], sf, p[3], stream())

    assert step_rc() == 0
    for kw in (dict(norm=2), dict(norm=-1), dict(n=0), dict(B=-1), dict(sf=-0.5), dict(sf=float("nan")),
               dict(sf=float("inf")), dict(ptrs=(x0.data_ptr(), 0, eps.data_ptr(), x.data_ptr()))):
        assert step_rc(**kw) < 0, kw
        assert lib.amc_last_error()
    assert lib.amc_adv_init(4, n, 5, x0.data_ptr(), eps.data_ptr(), 0, 0, None, x.data_ptr(), stream()) < 0
    assert lib.amc_adv_init(4, 0, LINF, x0.data_ptr(), eps.data_ptr(), 0, 0, None, x.data_ptr(), stream()) < 0
    assert lib.amc_adv_init(4, n, LINF, 0, eps.data_ptr(), 0, 0, None, x.data_ptr(), stream()) < 0
    assert step_rc(B=0, ptrs=(0, 0, 0, 0)) == 0                  # nothing to do

    with pytest.raises(ValueError, match="norm"):
        PGDAttack(model, norm="l1", eps=0.1)
    with pytest.raises(ValueError, match="exactly one"):
        PGDAttack(model, eps=0.1, psr_db=-10.0)
    with pytest.raises(ValueError, match="exactly one"):
        PGDAttack(model)
    for sf in (-1.0, float("nan")):
        with pytest.raises(ValueError, match="step_frac"):
            PGDAttack(model, eps=0.1, step_frac=sf)
    with pytest.raises(ValueError, match="eps"):
        PGDAttack(model, eps=torch.ones(4))                       # host tensor
    with pytest.raises(ValueError, match="eps"):
        PGDAttack(model, eps=torch.ones(5, device=DEV))(x0, y)    # wrong shape
    with pytest.raises(ValueError, match="bound"):
        TrainStep(model, attack=PGDAttack(other, eps=0.1))
    with pytest.raises(ValueError, match="bound"):
        evaluate_model_with_confusion(model, [], ["a"], "unused", attack=PGDAttack(other, eps=0.1))
    atk = PGDAttack(model, eps=0.1)
    for bad in (y.cpu(), y.int(), y[:3], y.view(2, 2)):
        with pytest.raises(ValueError, match="labels"):
            atk(x0, bad)

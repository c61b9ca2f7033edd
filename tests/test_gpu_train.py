"""GPU tests of the fused training step (TrainStep), dropout consistency and the host pipeline."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from conftest import GOLDEN_CASES, GOLDEN_HP, load_golden  # noqa: E402

import vit_vs_raw_iq_b200 as amc  # noqa: E402
from vit_vs_raw_iq_b200.trainer import GraphTrainStep, HostPipeline, TrainStep, predict  # noqa: E402

DEV = "cuda:0"


def build(name, dtype, drop=0.0):
    kind, kw = GOLDEN_CASES[name]
    cls = amc.RawIQAMCTransformer if kind == "rawiq" else amc.ViTAMCTransformer
    return cls(**kw, drop_prob=drop, device=DEV, compute_dtype=dtype)


@pytest.mark.parametrize("name", ["rawiq_seg16", "rawiq_meanpool", "vit_p4", "vit_p16"])
def test_fused_train_step_matches_reference_step(name):
    """TrainStep.step (CE + backward + clip + AdamW, no autograd) == the reference's step on the golden case."""
    z, params, grads, after = load_golden(name)
    model = build(name, "fp32")
    model.load_state_dict({k: torch.from_numpy(v) for k, v in params.items()}, strict=True)
    ts = TrainStep(model, lr=GOLDEN_HP["lr"], weight_decay=GOLDEN_HP["weight_decay"], betas=GOLDEN_HP["betas"],
                   max_norm=GOLDEN_HP["clip"], label_smoothing=GOLDEN_HP["label_smoothing"])
    src = torch.from_numpy(z["src"]).to(DEV)
    labels = torch.from_numpy(z["labels"]).to(DEV)
    ts.step(src, labels)
    loss, acc = ts.read_stats()
    assert abs(loss - float(z["loss"])) < 1e-4
    ref_acc = float((z["logits"].argmax(1) == z["labels"]).mean())
    assert abs(acc - ref_acc) < 1e-6
    assert abs(ts.norm_ws[1].item() - float(z["grad_norm"])) / float(z["grad_norm"]) < 1e-4
    core = model._core
    for n, p in model.named_parameters():
        if n.endswith("w_k.bias"):
            continue
        upd = p.detach().cpu().numpy() - params[n]
        ref_upd = after[n] - params[n]
        assert np.abs(upd - ref_upd).max() < 1e-5 + 2e-2 * np.abs(ref_upd).max(), n
    # flat gradient blob holds the same gradients as the reference
    for (o, cnt, shape), p, (n, _) in zip(core.slots, core.params, model.named_parameters()):
        pass
    names = {id(p): n for n, p in model.named_parameters()}
    for p, (o, cnt, shape) in zip(core.params, core.slots):
        n = names[id(p)]
        if n.endswith("w_k.bias"):
            continue
        g = ts.grads[o:o + cnt].view(shape).cpu().numpy()
        r = grads[n]
        assert np.linalg.norm(g - r) / (np.linalg.norm(r) + 1e-20) < 1e-3, n


def test_dropout_backward_uses_the_forward_masks():
    """With p>0 the masks are regenerated in backward from (seed, offset): the analytic directional
    derivative must match a central finite difference taken with the *same* masks."""
    torch.manual_seed(0)
    model = amc.RawIQAMCTransformer(in_channels=2, seq_length=128, num_classes=11, d_model=32, n_head=4, n_layers=2,
                                    ffn_hidden=64, drop_prob=0.3, device=DEV, segment_size=16, compute_dtype="fp32")
    model.train()
    core = model._core
    src = torch.randn(6, 2, 128, device=DEV)
    wgt = torch.randn(6, 11, device=DEV)

    def f():
        core.calls = 7          # freeze the dropout counter -> identical masks on every call
        return (model(src) * wgt).sum()

    out1 = f()
    out2 = f()
    assert torch.equal(out1, out2)
    model.zero_grad()
    out1.backward()
    flat = model.flat_parameters()
    g = torch.cat([p.grad.reshape(-1) for p in core.params])
    v = torch.randn_like(g)
    v /= v.norm()
    analytic = float((g * v).sum())
    eps = 3e-3
    saved = [p.detach().clone() for p in core.params]
    with torch.no_grad():
        def shift(sign):
            o = 0
            for p, s in zip(core.params, saved):
                p.copy_(s + sign * eps * v[o:o + p.numel()].view_as(p))
                o += p.numel()
        shift(+1)
        fp = float(f())
        shift(-1)
        fm = float(f())
        shift(0)
    numeric = (fp - fm) / (2 * eps)
    assert abs(analytic - numeric) < 3e-2 * max(abs(analytic), abs(numeric), 1e-3), (analytic, numeric)
    # dropout really is active in train mode and off in eval mode
    model.eval()
    with torch.no_grad():
        e1, e2 = model(src), model(src)
    assert torch.equal(e1, e2)
    model.train()
    with torch.no_grad():
        t1, t2 = model(src), model(src)          # counter advances -> different masks
    assert not torch.equal(t1, t2)
    assert (t1 - e1).abs().max() > 1e-3


def test_dropout_keep_rate_and_scaling():
    """E[dropout(x)] = x: averaging many train-mode encoder embeddings approaches the eval-mode one."""
    torch.manual_seed(1)
    model = amc.ViTAMCTransformer(in_channels=1, img_size_h=32, img_size_w=64, patch_size=16, num_classes=19,
                                  d_model=64, n_head=4, n_layers=0, ffn_hidden=128, drop_prob=0.25, device=DEV,
                                  compute_dtype="fp32")
    src = torch.randn(64, 1, 32, 64, device=DEV)
    with torch.no_grad():
        model.eval()
        ref = model.encoder(src)
        model.train()
        one = model.encoder(src)
        zero_frac = float((one == 0).float().mean())
        acc = torch.zeros_like(ref)
        n = 200
        for _ in range(n):
            acc += model.encoder(src)
    assert abs(zero_frac - 0.25) < 0.02
    kept = one != 0
    assert torch.allclose(one[kept], ref[kept] / 0.75, rtol=1e-5, atol=1e-6)
    err = ((acc / n - ref).abs().mean() / ref.abs().mean()).item()
    assert err < 0.08


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_training_reduces_loss_on_synthetic_iq(dtype):
    """A few hundred fused steps on synthetic modulated IQ must learn (loss falls, accuracy > chance)."""
    from vit_vs_raw_iq_b200 import synth
    torch.manual_seed(0)
    X, y, _ = synth.make_frames(2048, classes=synth.CLASSES_11[:4], seed=3)
    keep = np.ones(len(X), dtype=bool)
    stats = synth.normalization_stats(X)
    model = amc.RawIQAMCTransformer(in_channels=2, seq_length=1024, num_classes=4, d_model=64, n_head=4, n_layers=2,
                                    ffn_hidden=128, drop_prob=0.1, device=DEV, segment_size=16, compute_dtype=dtype)
    model.set_raw_input(stats)
    ts = TrainStep(model, lr=2e-3, weight_decay=1e-4)
    xd, yd = torch.from_numpy(X[keep]).to(DEV), torch.from_numpy(y[keep]).to(DEV)
    losses = []
    for it in range(150):
        i = (it * 256) % (len(xd) - 256)
        ts.step(xd[i:i + 256], yd[i:i + 256])
        if it % 25 == 24:
            losses.append(ts.read_stats()[0])
    assert losses[-1] < losses[0] - 0.1, losses
    pred = predict(model, xd[:1024])
    acc = float((pred == yd[:1024]).float().mean())
    assert acc > 0.4, acc     # chance = 0.25


def test_host_pipeline_step():
    z, params, _, _ = load_golden("vit_p16")
    model = build("vit_p16", "fp32")
    model.load_state_dict({k: torch.from_numpy(v) for k, v in params.items()}, strict=True)
    ts = TrainStep(model, lr=1e-3, weight_decay=1e-2)
    src = torch.from_numpy(z["src"]).pin_memory()
    labels = torch.from_numpy(z["labels"]).pin_memory()
    pipe = HostPipeline(ts, tuple(src.shape))
    assert pipe.step(src, labels) is None            # losses come back one step late (copy/compute overlap)
    l0 = pipe.step(src, labels)
    assert abs(l0 - float(z["loss"])) < 1e-4
    for _ in range(5):
        pipe.step(src, labels)
    l1 = pipe.flush()
    assert l1 < l0
    from vit_vs_raw_iq_b200.trainer import HostPredictor
    hp = HostPredictor(model, tuple(src.shape))
    assert hp.predict(src) is None
    a = hp.predict(src).clone()
    b = hp.flush().clone()
    ref = predict(model, src.to(DEV)).cpu()
    assert torch.equal(a, ref) and torch.equal(b, ref)


def test_thirty_step_trajectory_matches_reference_training_loop():
    """The reference's own loop (30 steps, AdamW + clip + CE ls 0.1) recorded in tests/golden/trajectory_rawiq.npz
    vs the fused TrainStep on the fp32 path: same per-step losses / accuracies and final weights."""
    import os
    from conftest import GOLDEN_DIR
    z = np.load(os.path.join(GOLDEN_DIR, "trajectory_rawiq.npz"))
    params = {k[len("param/"):]: z[k] for k in z.files if k.startswith("param/")}
    final = {k[len("final/"):]: z[k] for k in z.files if k.startswith("final/")}
    model = amc.RawIQAMCTransformer(in_channels=2, seq_length=256, num_classes=4, d_model=32, n_head=4, n_layers=2,
                                    ffn_hidden=64, drop_prob=0.0, device=DEV, use_cls_token=True,
                                    embedding_type="segment", segment_size=16, compute_dtype="fp32")
    model.load_state_dict({k: torch.from_numpy(v) for k, v in params.items()}, strict=True)
    ts = TrainStep(model, lr=2e-3, weight_decay=1e-2, betas=(0.9, 0.99), max_norm=1.0, label_smoothing=0.1)
    X, y = torch.from_numpy(z["X"]).to(DEV), torch.from_numpy(z["y"]).to(DEV)
    N, B = X.shape[0], 32
    for it in range(30):
        i = (it * B) % N
        ts.step(X[i:i + B].contiguous(), y[i:i + B].contiguous())
        loss, acc = ts.read_stats()
        assert abs(loss - float(z["losses"][it])) < 2e-3 * max(1.0, float(z["losses"][it])), (it, loss)
        assert abs(acc - float(z["accs"][it])) <= 1.0 / B + 1e-6, (it, acc)
    worst = 0.0
    for n, p in model.named_parameters():
        if n.endswith("w_k.bias"):
            continue
        ref = final[n]
        moved = np.abs(ref - params[n]).max()
        err = np.abs(p.detach().cpu().numpy() - ref).max()
        worst = max(worst, err / max(moved, 1e-6))
    assert worst < 5e-2, worst       # 30 Adam steps amplify fp32 rounding; updates themselves are ~30*lr


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_thirty_step_vit_trajectory_matches_reference_training_loop(dtype):
    """The ViT family of the headline benchmark (patch 16, T = 9): the reference's loop recorded in
    tests/golden/trajectory_vit.npz vs the fused TrainStep.  fp32: step-for-step; bf16: the losses track the reference
    within bf16 noise while the trajectories are still close (first 10 steps) and the run converges like it."""
    import os
    from conftest import GOLDEN_DIR
    z = np.load(os.path.join(GOLDEN_DIR, "trajectory_vit.npz"))
    params = {k[len("param/"):]: z[k] for k in z.files if k.startswith("param/")}
    final = {k[len("final/"):]: z[k] for k in z.files if k.startswith("final/")}
    model = amc.ViTAMCTransformer(in_channels=1, img_size_h=32, img_size_w=64, patch_size=16, num_classes=4, d_model=64,
                                  n_head=8, n_layers=2, ffn_hidden=128, drop_prob=0.0, device=DEV, compute_dtype=dtype)
    model.load_state_dict({k: torch.from_numpy(v) for k, v in params.items()}, strict=True)
    ts = TrainStep(model, lr=2e-3, weight_decay=1e-2, betas=(0.9, 0.99), max_norm=1.0, label_smoothing=0.1)
    X, y = torch.from_numpy(z["X"]).to(DEV), torch.from_numpy(z["y"]).to(DEV)
    N, B = X.shape[0], 32
    losses = []
    for it in range(30):
        i = (it * B) % N
        ts.step(X[i:i + B].contiguous(), y[i:i + B].contiguous())
        loss, acc = ts.read_stats()
        losses.append(loss)
        ref = float(z["losses"][it])
        if dtype == "fp32":
            assert abs(loss - ref) < 2e-3 * max(1.0, ref), (it, loss, ref)
            assert abs(acc - float(z["accs"][it])) <= 1.0 / B + 1e-6, (it, acc)
        elif it < 10:
            assert abs(loss - ref) < 5e-2 * max(1.0, ref), (it, loss, ref)
    if dtype == "fp32":
        worst = 0.0
        for n, p in model.named_parameters():
            if n.endswith("w_k.bias"):
                continue
            moved = np.abs(final[n] - params[n]).max()
            worst = max(worst, np.abs(p.detach().cpu().numpy() - final[n]).max() / max(moved, 1e-6))
        assert worst < 5e-2, worst
    else:
        assert abs(np.mean(losses[-5:]) - float(np.mean(z["losses"][-5:]))) < 0.1


def test_labels_are_validated_like_cross_entropy_loss():
    """nn.CrossEntropyLoss (R/training/train.py:260) raises on a wrong label dtype / length / device and on a target
    outside [0, C); TrainStep rejects the former up front and the kernel turns the latter into a NaN loss that the host
    raises on when it reads the statistics (ADVICE r1)."""
    z, params, _, _ = load_golden("vit_p16")
    model = build("vit_p16", "fp32")
    model.load_state_dict({k: torch.from_numpy(v) for k, v in params.items()}, strict=True)
    ts = TrainStep(model, lr=1e-3)
    src = torch.from_numpy(z["src"]).to(DEV)
    labels = torch.from_numpy(z["labels"]).to(DEV)
    for bad in (labels.int(), labels[:-1], labels.cpu(), labels.float(), labels.view(-1, 1)):
        with pytest.raises(ValueError):
            ts.step(src, bad)
    ts.step(src, labels)
    loss, _ = ts.read_stats()
    assert abs(loss - float(z["loss"])) < 1e-4
    oob = labels.clone()
    oob[0] = GOLDEN_CASES["vit_p16"][1]["num_classes"]
    ts.step(src, oob)
    with pytest.raises(RuntimeError, match="label outside"):
        ts.read_stats()
    neg = labels.clone()
    neg[1] = -1
    ts.step(src, neg)
    with pytest.raises(RuntimeError, match="label outside"):
        ts.read_stats()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_model_on_a_non_current_device():
    """The reference's plain `.to(device)` usage: model and batch on cuda:1 while cuda:0 is the current device (ADVICE r1:
    the ABI switches to the device that owns the buffers).  bf16 runs the tcgen05 kernels, whose shared-memory attributes are
    per device: a bf16 forward on cuda:0 comes first, so cuda:1 must get them too."""
    z, params, grads, _ = load_golden("vit_p16")
    torch.cuda.set_device(0)
    dev1 = torch.device("cuda", 1)
    kind, kw = GOLDEN_CASES["vit_p16"]
    state = {k: torch.from_numpy(v) for k, v in params.items()}
    model0 = amc.ViTAMCTransformer(**kw, drop_prob=0.0, device=DEV, compute_dtype="bf16")
    model0.load_state_dict(state, strict=True)
    with torch.no_grad():
        model0(torch.from_numpy(z["src"]).to(DEV))
    torch.cuda.synchronize(0)
    for dtype, tol in (("fp32", 1e-4), ("bf16", 2e-2)):
        model = amc.ViTAMCTransformer(**kw, drop_prob=0.0, device=dev1, compute_dtype=dtype)
        model.load_state_dict(state, strict=True)
        src = torch.from_numpy(z["src"]).to(dev1)
        labels = torch.from_numpy(z["labels"]).to(dev1)
        assert torch.cuda.current_device() == 0
        ts = TrainStep(model, lr=1e-3)
        ts.step(src, labels)
        loss, _ = ts.read_stats()
        assert abs(loss - float(z["loss"])) < tol, dtype
        assert torch.cuda.current_device() == 0


@pytest.mark.parametrize("name,dtype", [("rawiq_seg16", "fp32"), ("vit_p16", "bf16")])
def test_graph_train_step_matches_the_eager_step(name, dtype):
    """GraphTrainStep (one CUDA-graph replay per step, step number and dropout counter on the device) follows TrainStep:
    with dropout off the parameters after 6 steps agree to fp32 round-off (the weight-gradient atomics reorder sums)."""
    z, params, _, _ = load_golden(name)
    src = torch.from_numpy(z["src"]).to(DEV)
    labels = torch.from_numpy(z["labels"]).to(DEV)
    outs = []
    for cls in (TrainStep, GraphTrainStep):
        model = build(name, dtype)
        model.load_state_dict({k: torch.from_numpy(v) for k, v in params.items()}, strict=True)
        ts = cls(model, lr=1e-3, weight_decay=1e-2)
        losses = []
        for _ in range(6):
            ts.step(src, labels)
            losses.append(ts.read_stats()[0])
        outs.append((model.flat_parameters().clone(), losses))
        if cls is GraphTrainStep:
            assert ts._graph is not None and int(ts.counter.item()) == 6
    (p0, l0), (p1, l1) = outs
    # (Adam's first steps move every weight by ~lr whatever the gradient's size, so the split-K atomics' summation-order
    # noise in tiny gradient entries shows up at a few 1e-5 of the weight scale after 6 steps of lr = 1e-3)
    tol = 1e-4 if dtype == "fp32" else 2e-2
    assert (p0 - p1).abs().max().item() <= tol * p0.abs().max().item()
    assert all(abs(a - b) <= 5e-3 * abs(a) + 1e-5 for a, b in zip(l0, l1)), (l0, l1)
    assert l0[-1] < l0[0]


def test_graph_train_step_draws_new_dropout_masks_every_replay():
    """The dropout counter lives in device memory, so replays of one captured graph use different masks: with lr = 0 the
    weights never move, yet the training loss of the same batch changes from step to step (and repeats nowhere)."""
    z, params, _, _ = load_golden("vit_p16")
    model = build("vit_p16", "fp32", drop=0.3)
    model.load_state_dict({k: torch.from_numpy(v) for k, v in params.items()}, strict=True)
    ts = GraphTrainStep(model, lr=0.0, weight_decay=0.0)
    src = torch.from_numpy(z["src"]).to(DEV)
    labels = torch.from_numpy(z["labels"]).to(DEV)
    losses = []
    for _ in range(6):
        ts.step(src, labels)
        losses.append(round(ts.read_stats()[0], 6))
    assert len(set(losses)) == len(losses), losses

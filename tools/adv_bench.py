"""Cost of projected-gradient attacks and adversarial training (profiles/adv_bench.txt).

Workloads of tools/input_grad_bench.py (dataset-layout frames [B, L, 2], bf16, budgets at a PSR of -20 dB).  Arms,
timed with CUDA events after warm-up:
  1. PGD-10 L-inf as the autograd loop a user writes on the module surface today (frozen model, torch ops for the step)
  2. PGDAttack (PGD-10 L-inf) eager
  3. PGDAttack (PGD-10 L-inf) captured in one CUDA graph
  4. TrainStep / GraphTrainStep without an attack
  5. TrainStep / GraphTrainStep with FGSM-RS (steps=1, step_frac=1.25, random start)
  6. TrainStep / GraphTrainStep with PGD-7 L-inf
A profiled eager PGD-10 call then gives the adv_step kernel class's algorithmic bytes over its time, an effective rate
that may include L2 hits, against the device-to-device copy peak measured on a B200 (6.55 TB/s, DESIGN.md).

    python tools/adv_bench.py [--steps N] [--warmup W]
"""
import argparse
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch

import bench
import vit_vs_raw_iq_b200 as amc
from vit_vs_raw_iq_b200 import _lib, synth
from vit_vs_raw_iq_b200.adversarial import PGDAttack
from vit_vs_raw_iq_b200.trainer import GraphTrainStep, TrainStep

WORKLOADS = [("vit_p16_d256_L6", 32768), ("rawiq_sps1_seg8_d256_L6", 1024), ("rawiq_seg16_d128_L6", 256)]
PSR_DB = -20.0
COPY_PEAK_TBS = 6.55


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown (nvidia-smi failed)"


def time_ms(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def autograd_pgd(model, x0, y, steps=10):
    """The loop on the module surface: uniform start, autograd input gradient, sign step, clamp to the ball."""
    n = x0[0].numel()
    eps = (x0.view(len(x0), -1).norm(dim=1) * (10.0 ** (PSR_DB / 20.0) / n ** 0.5)).view(-1, *([1] * (x0.dim() - 1)))
    a = 2.5 / steps * eps
    loss_fn = torch.nn.CrossEntropyLoss(reduction="sum")

    def run():
        x = x0 + eps * (2 * torch.rand_like(x0) - 1)
        for _ in range(steps):
            xg = x.detach().requires_grad_(True)
            (g,) = torch.autograd.grad(loss_fn(model(xg), y), xg)
            x = torch.min(torch.max(x + a * g.sign(), x0 - eps), x0 + eps)
        return x
    return run


def graphed(fn):
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        fn()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        fn()
    return g.replay


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("adv_bench.py measures on the GPU; no CUDA device found")
    dev = torch.device("cuda", 0)
    print(f"GPU (name, power limit, max SM clock): {gpu_info()}")
    print(f"CUDA events, {a.warmup} warm-up + {a.steps} timed calls per arm; bf16; dataset-layout frames; "
          f"budgets at PSR {PSR_DB:g} dB")
    for wname, B in WORKLOADS:
        w = bench.WORKLOADS[wname]
        cls = amc.ViTAMCTransformer if w["kind"] == "vit" else amc.RawIQAMCTransformer
        classes = synth.CLASSES_19 if w["kw"]["num_classes"] == 19 else synth.CLASSES_11
        X, Y, _ = synth.make_frames(1024, classes=classes, sps=w.get("sps", 1), seed=42)
        idx = np.arange(B) % len(X)
        x = torch.from_numpy(X[idx]).to(dev)
        y = torch.from_numpy(Y[idx]).to(dev)
        stats = synth.normalization_stats(X)

        def fresh():
            torch.manual_seed(0)
            m = cls(**w["kw"], device=dev, compute_dtype="bf16")
            m.set_raw_input(stats)
            return m

        print(f"\n== {wname}  B = {B}  input {tuple(x.shape)}  frame n = {x[0].numel()}")
        ms = {}
        model = fresh()
        model.eval()
        for p in model.parameters():
            p.requires_grad_(False)
        ms["1 PGD-10 autograd loop (module surface)"] = time_ms(autograd_pgd(model, x, y), a.steps, a.warmup)
        for p in model.parameters():
            p.requires_grad_(True)
        atk = PGDAttack(model, psr_db=PSR_DB, steps=10)
        ms["2 PGDAttack PGD-10 eager"] = time_ms(lambda: atk(x, y), a.steps, a.warmup)
        ms["3 PGDAttack PGD-10 CUDA graph"] = time_ms(graphed(lambda: atk(x, y)), a.steps, a.warmup)
        _lib.profile(True)
        try:
            atk(x, y)
            table = _lib.profile_dump()
        finally:
            _lib.profile(False)
        del atk, model
        for label, kw in (("4 no attack", None), ("5 FGSM-RS", dict(steps=1, step_frac=1.25)),
                          ("6 PGD-7", dict(steps=7))):
            for tcls in (TrainStep, GraphTrainStep):
                model = fresh()
                ts = tcls(model, attack=None if kw is None else PGDAttack(model, psr_db=PSR_DB, **kw))
                ms[f"{label} {tcls.__name__}"] = time_ms(lambda: ts.step(x, y), a.steps, max(a.warmup, 2))
                del ts, model
        base = ms["2 PGDAttack PGD-10 eager"]
        for arm, t in ms.items():
            print(f"  {arm:42s} {t:9.3f} ms/call  {B / t * 1e3:12.0f} frames/s  ({t / base:.3f} x arm 2)")
        tot = sum(r["ms"] for r in table.values())
        print(f"  -- profile classes, one eager PGD-10 call (events around every launch site; {tot:.3f} ms in total)")
        print(f"     {'class':24s} {'launches':>8s} {'ms':>9s} {'GB':>9s} {'share':>7s}")
        for name, r in sorted(table.items(), key=lambda kv: -kv[1]["ms"]):
            print(f"     {name:24s} {r['n']:8d} {r['ms']:9.3f} {r['bytes'] / 1e9:9.3f} {r['ms'] / tot:7.1%}")
        s = table["adv_step"]
        tbs = s["bytes"] / (s["ms"] / s["n"] * 1e-3) / s["n"] / 1e12
        # an effective rate, not HBM bandwidth: g was written by frontend_bwd_dsrc just before, and whatever part of it
        # (and of x, read by that backward) is still in the 126 MB L2 is not read from HBM
        print(f"  adv_step: {s['bytes'] / s['n'] / 1e6:.1f} MB per launch algorithmic (16 B / element), "
              f"{s['ms'] / s['n'] * 1e3:.1f} us per launch -> {tbs:.2f} TB/s effective = {tbs / COPY_PEAK_TBS:.0%} "
              f"of the {COPY_PEAK_TBS} TB/s copy peak (may include L2 hits on g and x, written / read by the "
              f"backward just before); {s['ms'] / tot:.1%} of the attack's kernel time")
        del x, y
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()

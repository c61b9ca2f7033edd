"""Cost of Integrated Gradients on the device (model.integrated_gradients) against the host loop a user would write.

Per workload, bf16, model.eval(), on synthetic dataset frames (the workloads of tools/attn_maps_bench.py plus the
reference's batch, raw-IQ seg16 d128 L6 at 256 frames):
  * integrated_gradients(x, steps=32) with the default pass size;
  * the autograd host loop at the same 32 Gauss-Legendre nodes: per node a frozen forward of x' + a_k (x - x') and
    torch.autograd.grad of the target logits, summed on the host (the target taken once from a forward of x);
  * one FGSM step of the same batch (frozen forward + input gradient of the cross-entropy loss);
  * the launch-site profile classes of one integrated_gradients call;
  * at 256 frames, integrated_gradients with 1, 4, 8, 16 and 32 path points per pass (internal_batch_size).
Calls are timed with CUDA events over --steps calls after --warmup warm-up calls.

    python tools/ig_bench.py [--steps N] [--warmup W] [--out profiles/ig_bench.txt]
"""
import argparse
import io
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import numpy as np
import torch

import bench
import vit_vs_raw_iq_b200 as amc
from attn_maps_bench import WORKLOADS, gpu_info, time_calls
from vit_vs_raw_iq_b200 import _lib, synth

NODES = 32


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None, help="also write the report to this file")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ig_bench.py measures on the GPU; no CUDA device found")
    buf = io.StringIO()

    def say(s=""):
        print(s, flush=True)
        buf.write(s + "\n")

    dev = torch.device("cuda", 0)
    say(f"GPU (name, power limit, max SM clock): {gpu_info()}")
    say(f"bf16; {NODES} Gauss-Legendre nodes, zero baseline, argmax target; CUDA events over {a.steps} calls after "
        f"{a.warmup} warm-up; model.eval()")
    alpha, wts = np.polynomial.legendre.leggauss(NODES)
    alpha, wts = (alpha + 1.0) / 2.0, wts / 2.0
    summary = []
    for wname, B in [(w, b) for w, b, _ in WORKLOADS] + [("rawiq_seg16_d128_L6", 256)]:
        w = bench.WORKLOADS[wname]
        kw = {k: v for k, v in w["kw"].items() if k != "drop_prob"}
        torch.manual_seed(0)
        cls = amc.ViTAMCTransformer if w["kind"] == "vit" else amc.RawIQAMCTransformer
        model = cls(**kw, drop_prob=0.0, device=dev, compute_dtype="bf16").eval()
        T = model._core.layout.T
        classes = synth.CLASSES_19 if kw["num_classes"] == 19 else synth.CLASSES_11
        X, Y, _ = synth.make_frames(1024, classes=classes, sps=w.get("sps", 1), seed=42)
        model.set_raw_input(synth.normalization_stats(X))
        idx = np.arange(B) % len(X)
        x = torch.from_numpy(X[idx]).to(dev)
        y = torch.from_numpy(np.asarray(Y)[idx].astype(np.int64)).to(dev)
        base = torch.zeros_like(x)
        per_pass = max(1, model.IG_TOKEN_BUDGET // (B * T))
        chunk = -(-NODES // -(-NODES // per_pass))
        desc = model._core._desc(B=B, dtype=_lib.BF16, training=True)
        ws_gb = _lib.ig_workspace_bytes(desc, chunk) / 1e9
        say(f"\n== {wname}  B = {B}  T = {T}  ({chunk} points a pass, workspace {ws_gb:.2f} GB)")

        loss_fn = torch.nn.CrossEntropyLoss()
        rows = torch.arange(B, device=dev)

        def ig():
            model.integrated_gradients(x)

        def fgsm():
            xg = x.detach().requires_grad_(True)
            torch.autograd.grad(loss_fn(model(xg), y), xg)

        def loop():
            with torch.no_grad():
                t = model(x).argmax(1)
            total = torch.zeros_like(x)
            for ak, wk in zip(alpha, wts):
                xk = (base + float(ak) * (x - base)).requires_grad_(True)
                (g,) = torch.autograd.grad(model(xk)[rows, t].sum(), xk)
                total += float(wk) * g
            return (x - base) * total

        t_ig = time_calls(ig, a.steps, a.warmup)
        for p in model.parameters():
            p.requires_grad_(False)
        t_loop = time_calls(loop, a.steps, a.warmup)
        t_g = time_calls(fgsm, a.steps, a.warmup)
        a_dev = model.integrated_gradients(x)
        a_loop = loop()
        err = float((a_dev - a_loop).norm() / a_loop.norm())
        for p in model.parameters():
            p.requires_grad_(True)
        say(f"  FGSM step (frozen fwd+dsrc)      {t_g:9.3f} ms/call")
        say(f"  autograd host loop, {NODES} nodes    {t_loop:9.3f} ms/call = {t_loop / t_g:.2f} x the FGSM step")
        say(f"  integrated_gradients, {NODES} nodes  {t_ig:9.3f} ms/call = {t_ig / t_g:.2f} x the FGSM step, "
            f"{t_loop / t_ig:.2f} x faster than the host loop (L2-rel difference {err:.2e})")
        summary.append((wname, B, t_g, t_loop, t_ig))
        if B == 256:
            for n in (1, 4, 8, 16, 32):
                t_n = time_calls(lambda: model.integrated_gradients(x, internal_batch_size=n * B), a.steps, a.warmup)
                say(f"    internal_batch_size = {n:2d} x B      {t_n:9.3f} ms/call")
        _lib.profile(True)
        try:
            model.integrated_gradients(x)
            tab = _lib.profile_dump()
        finally:
            _lib.profile(False)
        say("  -- profile classes, one integrated_gradients call (events around every launch site)")
        for name, r in sorted(tab.items(), key=lambda kv: -kv[1]["ms"]):
            bw = f"  {r['bytes'] / (r['ms'] * 1e-3) / 1e12:6.2f} TB/s" if r["bytes"] > 0 and r["ms"] > 0 else ""
            say(f"     {name:24s} {r['n']:8d} {r['ms']:9.3f} ms{bw}")
        del model, x
        torch.cuda.empty_cache()

    say("\nsummary: workload, B, FGSM ms, host loop ms, integrated_gradients ms, loop / IG")
    for s in summary:
        say(f"  {s[0]:26s} {s[1]:6d} {s[2]:9.3f} {s[3]:9.3f} {s[4]:9.3f} {s[3] / s[4]:6.2f}")
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(buf.getvalue())


if __name__ == "__main__":
    main()

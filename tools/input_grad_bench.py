"""Cost of the input gradient (saliency maps, FGSM / PGD adversarial examples) against the training backward.

For each workload, four arms through the nn.Module surface, timed with CUDA events after warm-up:
  1. eval forward (torch.no_grad)
  2. forward + backward with parameter gradients (the training backward)
  3. frozen model (requires_grad_(False)): forward + input-gradient backward, i.e. one FGSM / PGD step
  4. forward + backward with both parameter and input gradients
All arms run the model in .eval() (dropout off), so they differ only in the gradients they compute; input frames are
dataset-layout [B, L, 2] (the z-score is fused into the front end, and the input gradient is w.r.t. the raw frames).
A second, profiled pass prints the amc_profile_dump class table of each arm.

    python tools/input_grad_bench.py [--steps N] [--warmup W]
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

# the default bench workload; raw-IQ at SPS 1 (T = 129); the reference's own batch of 256 frames
WORKLOADS = [("vit_p16_d256_L6", 32768), ("rawiq_sps1_seg8_d256_L6", 1024), ("rawiq_seg16_d128_L6", 256)]
ARMS = ["eval_forward", "fwd_bwd_params", "fwd_bwd_input_frozen", "fwd_bwd_params_and_input"]


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown (nvidia-smi failed)"


def make_arm(model, x, y, arm):
    loss_fn = torch.nn.CrossEntropyLoss()
    params = list(model.parameters())

    def eval_forward():
        with torch.no_grad():
            model(x)

    def fwd_bwd_params():
        model.zero_grad(set_to_none=True)
        loss_fn(model(x), y).backward()

    def fwd_bwd_input_frozen():
        xg = x.detach().requires_grad_(True)
        torch.autograd.grad(loss_fn(model(xg), y), xg)

    def fwd_bwd_params_and_input():
        model.zero_grad(set_to_none=True)
        xg = x.detach().requires_grad_(True)
        loss_fn(model(xg), y).backward()
        return xg.grad

    frozen = arm == "fwd_bwd_input_frozen"
    for p in params:
        p.requires_grad_(not frozen)
    return dict(eval_forward=eval_forward, fwd_bwd_params=fwd_bwd_params, fwd_bwd_input_frozen=fwd_bwd_input_frozen,
                fwd_bwd_params_and_input=fwd_bwd_params_and_input)[arm]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("input_grad_bench.py measures on the GPU; no CUDA device found")
    dev = torch.device("cuda", 0)
    print(f"GPU (name, power limit, max SM clock): {gpu_info()}")
    print(f"CUDA events, {a.warmup} warm-up + {a.steps} timed calls per arm; bf16; model.eval() (dropout off)")
    for wname, B in WORKLOADS:
        w = bench.WORKLOADS[wname]
        torch.manual_seed(0)
        cls = amc.ViTAMCTransformer if w["kind"] == "vit" else amc.RawIQAMCTransformer
        model = cls(**w["kw"], device=dev, compute_dtype="bf16")
        model.eval()
        classes = synth.CLASSES_19 if w["kw"]["num_classes"] == 19 else synth.CLASSES_11
        X, Y, _ = synth.make_frames(1024, classes=classes, sps=w.get("sps", 1), seed=42)
        model.set_raw_input(synth.normalization_stats(X))
        idx = np.arange(B) % len(X)
        x = torch.from_numpy(X[idx]).to(dev)
        y = torch.from_numpy(Y[idx]).to(dev)
        print(f"\n== {wname}  B = {B}  input {tuple(x.shape)}")
        ms = {}
        tables = {}
        for arm in ARMS:
            fn = make_arm(model, x, y, arm)
            for _ in range(a.warmup):
                fn()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(a.steps):
                fn()
            e1.record()
            torch.cuda.synchronize()
            ms[arm] = e0.elapsed_time(e1) / a.steps
            _lib.profile(True)
            try:
                fn()
                tables[arm] = _lib.profile_dump()
            finally:
                _lib.profile(False)
        for arm in ARMS:
            rel = f"  ({ms[arm] / ms['fwd_bwd_params']:.3f} x arm 2)" if arm != "eval_forward" else ""
            print(f"  {arm:26s} {ms[arm]:9.3f} ms/call  {B / ms[arm] * 1e3:12.0f} frames/s{rel}")
        for arm in ARMS:
            print(f"  -- profile classes, {arm} (one call; events around every launch site)")
            print(f"     {'class':24s} {'launches':>8s} {'ms':>9s} {'GB':>9s} {'TFLOP':>9s}")
            for name, r in sorted(tables[arm].items(), key=lambda kv: -kv[1]["ms"]):
                print(f"     {name:24s} {r['n']:8d} {r['ms']:9.3f} {r['bytes'] / 1e9:9.3f} {r['flops'] / 1e12:9.4f}")
        del model, x, y
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()

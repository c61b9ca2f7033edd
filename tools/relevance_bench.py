"""Cost of the class-specific attention relevance (amc_attention_relevance_step, model.attention_relevance).

Per workload, bf16, model.eval(), the five workloads of tools/attn_maps_bench.py:
  * per-launch time of amc_attention_relevance_step against amc_attention_rollout_step on the same random qkv of the
    workload's attention shape, both with a dense v_in (as below the top layer), and of the relevance step with
    v_in = e_0 (the top layer of a CLS model).  Each launch is timed alone with CUDA events after a 256 MB memset that
    evicts L2, median of --steps launches.  The goal is a dense relevance step of at most 2x the dense rollout step;
  * model.attention_relevance(x) against a plain eval forward model(x) and against one FGSM step of the same batch
    (frozen model: forward + input-gradient backward), CUDA events over --steps calls after --warmup;
  * the launch-site profile classes of one attention_relevance call.

    python tools/relevance_bench.py [--steps N] [--warmup W] [--out profiles/relevance_bench.txt]
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
from attn_maps_bench import WORKLOADS, gpu_info, time_calls, time_launches
from vit_vs_raw_iq_b200 import _lib, synth


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the report to this file")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("relevance_bench.py measures on the GPU; no CUDA device found")
    buf = io.StringIO()

    def say(s=""):
        print(s, flush=True)
        buf.write(s + "\n")

    dev = torch.device("cuda", 0)
    say(f"GPU (name, power limit, max SM clock): {gpu_info()}")
    say(f"bf16; kernels: median of {a.steps} single launches, each after a 256 MB L2-evicting memset; "
        f"model calls: CUDA events over {a.steps} calls after {a.warmup} warm-up; model.eval()")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream
    summary = []
    for wname, B, _ in WORKLOADS:
        w = bench.WORKLOADS[wname]
        kw = {k: v for k, v in w["kw"].items() if k != "drop_prob"}
        torch.manual_seed(0)
        cls = amc.ViTAMCTransformer if w["kind"] == "vit" else amc.RawIQAMCTransformer
        model = cls(**kw, drop_prob=0.0, device=dev, compute_dtype="bf16").eval()
        T, h, d = model._core.layout.T, kw["n_head"], kw["d_model"]
        dh = d // h
        say(f"\n== {wname}  B = {B}  T = {T}  h = {h}  dh = {dh}")

        # ---- kernels on a random qkv / dO of the workload's shape
        qkv = (torch.randn(B * T, 3 * d, device=dev) * 1.5).to(torch.bfloat16)
        dout = (torch.randn(B * T, d, device=dev) * 0.1).to(torch.bfloat16)
        v = torch.rand(B, T, device=dev)
        v /= v.sum(1, keepdim=True)
        e0 = torch.zeros(B, T, device=dev)
        e0[:, 0] = 1.0
        vo = torch.empty(B, T, device=dev)

        def roll():
            _lib.check(_lib.lib.amc_attention_rollout_step(_lib.BF16, B, T, h, dh, qkv.data_ptr(), v.data_ptr(),
                                                           vo.data_ptr(), stream))

        def rel(vin):
            return lambda: _lib.check(_lib.lib.amc_attention_relevance_step(
                _lib.BF16, B, T, h, dh, qkv.data_ptr(), dout.data_ptr(), vin.data_ptr(), vo.data_ptr(), stream))

        t_roll = time_launches(roll, a.steps, a.warmup, flush)
        t_rel = time_launches(rel(v), a.steps, a.warmup, flush)
        t_rel0 = time_launches(rel(e0), a.steps, a.warmup, flush)
        ratio = t_rel / t_roll
        say(f"  rollout step   (dense v_in) {t_roll * 1e3:9.1f} us/launch")
        say(f"  relevance step (dense v_in) {t_rel * 1e3:9.1f} us/launch  = {ratio:.2f} x the rollout step "
            f"({'meets' if ratio <= 2.0 else 'misses'} the 2x goal)")
        say(f"  relevance step (v_in = e_0) {t_rel0 * 1e3:9.1f} us/launch")
        del qkv, dout

        # ---- whole calls through the module surface on synthetic dataset frames
        classes = synth.CLASSES_19 if kw["num_classes"] == 19 else synth.CLASSES_11
        X, Y, _ = synth.make_frames(1024, classes=classes, sps=w.get("sps", 1), seed=42)
        model.set_raw_input(synth.normalization_stats(X))
        idx = np.arange(B) % len(X)
        x = torch.from_numpy(X[idx]).to(dev)
        y = torch.from_numpy(np.asarray(Y)[idx].astype(np.int64)).to(dev)

        def fwd():
            with torch.no_grad():
                model(x)

        loss_fn = torch.nn.CrossEntropyLoss()

        def fgsm():
            xg = x.detach().requires_grad_(True)
            torch.autograd.grad(loss_fn(model(xg), y), xg)

        t_f = time_calls(fwd, a.steps, a.warmup)
        t_r = time_calls(lambda: model.attention_relevance(x), a.steps, a.warmup)
        for p in model.parameters():
            p.requires_grad_(False)
        t_g = time_calls(fgsm, a.steps, a.warmup)
        for p in model.parameters():
            p.requires_grad_(True)
        say(f"  eval forward                {t_f:9.3f} ms/call")
        say(f"  FGSM step (frozen fwd+dsrc) {t_g:9.3f} ms/call")
        say(f"  attention_relevance         {t_r:9.3f} ms/call  = {t_r / t_f:.2f} x the eval forward, "
            f"{t_r / t_g:.2f} x the FGSM step")
        summary.append((wname, t_roll, t_rel, ratio, t_rel0, t_r / t_f, t_r / t_g))
        _lib.profile(True)
        try:
            model.attention_relevance(x)
            tab = _lib.profile_dump()
        finally:
            _lib.profile(False)
        say("  -- profile classes, one attention_relevance call (events around every launch site)")
        for name, r in sorted(tab.items(), key=lambda kv: -kv[1]["ms"]):
            say(f"     {name:24s} {r['n']:8d} {r['ms']:9.3f} ms")
        del model, x
        torch.cuda.empty_cache()

    say("\nsummary: workload, rollout step us, relevance step us, ratio, e_0 step us, call / eval fwd, call / FGSM")
    for s in summary:
        say(f"  {s[0]:26s} {s[1] * 1e3:9.1f} {s[2] * 1e3:9.1f} {s[3]:6.2f} {s[4] * 1e3:9.1f} {s[5]:6.2f} {s[6]:6.2f}")
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(buf.getvalue())


if __name__ == "__main__":
    main()

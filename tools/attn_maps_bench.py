"""Cost of the attention maps (amc_attention_probs) and of the attention rollout (amc_attention_rollout_step,
model.attention_rollout).

Per workload, bf16, model.eval():
  * per-launch time of amc_attention_probs and of amc_attention_rollout_step (a dense v_in, as below the top layer, and
    v_in = e_0, the top layer of a CLS model) on a random qkv of the workload's attention shape.  Each launch is timed
    alone with CUDA events after a 256 MB memset that evicts L2, median of --steps launches;
  * the probs kernel's bytes (fp32 P written, q and k read) over its time, against the 6.55 TB/s copy peak (DESIGN §5);
  * the rollout step's time against its larger lower bound: S = Q K^T once on the tensor pipe (2 B h T^2 dh FLOP at
    the 2.25 PFLOP/s dense bf16 data-sheet rate) or one ex2 per score at 16 per clock per SM (148 SMs at the max SM
    clock read below);
  * model.attention_rollout(x) against a plain eval forward model(x) of the same batch (CUDA events over --steps calls).

    python tools/attn_maps_bench.py [--steps N] [--warmup W]
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

COPY_PEAK = 6.55e12       # bytes/s, DESIGN §5
BF16_PEAK = 2.25e15       # FLOP/s dense, one B200
# (bench workload, batch for the rollout / forward comparison and the kernels, batch for the maps or None = same)
WORKLOADS = [("vit_p4_d128_L6", 1024, None), ("rawiq_sps1_seg8_d256_L6", 1024, None),
             ("rawiq_sps2_seg8_d256_L6", 512, None), ("vit_p16_d256_L6", 32768, None),
             ("rawiq_conv1d_d128_L6", 128, 16)]


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown (nvidia-smi failed)"


def max_sm_clock_hz(info):
    try:
        return float(info.split(",")[2].strip().split()[0]) * 1e6
    except (IndexError, ValueError):
        return float("nan")


def time_launches(fn, steps, warmup, flush):
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(steps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(np.median(ts))


def time_calls(fn, steps, warmup):
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("attn_maps_bench.py measures on the GPU; no CUDA device found")
    dev = torch.device("cuda", 0)
    info = gpu_info()
    clk = max_sm_clock_hz(info)
    print(f"GPU (name, power limit, max SM clock): {info}")
    print(f"bf16; kernels: median of {a.steps} single launches, each after a 256 MB L2-evicting memset; "
          f"model calls: CUDA events over {a.steps} calls after {a.warmup} warm-up; model.eval()")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream
    for wname, B, Bmaps in WORKLOADS:
        w = bench.WORKLOADS[wname]
        kw = {k: v for k, v in w["kw"].items() if k != "drop_prob"}
        torch.manual_seed(0)
        cls = amc.ViTAMCTransformer if w["kind"] == "vit" else amc.RawIQAMCTransformer
        model = cls(**kw, drop_prob=0.0, device=dev, compute_dtype="bf16").eval()
        T, h, d = model._core.layout.T, kw["n_head"], kw["d_model"]
        dh = d // h
        Bm = Bmaps or B
        print(f"\n== {wname}  B = {B}  T = {T}  h = {h}  dh = {dh}" + (f"  (maps at B = {Bm})" if Bmaps else ""))

        # ---- kernels on a random qkv of the workload's shape
        qkv = (torch.randn(B * T, 3 * d, device=dev) * 1.5).to(torch.bfloat16)
        probs = torch.empty(Bm * h * T * T, dtype=torch.float32, device=dev)
        v = torch.rand(B, T, device=dev)
        v /= v.sum(1, keepdim=True)
        e0 = torch.zeros(B, T, device=dev)
        e0[:, 0] = 1.0
        vo = torch.empty(B, T, device=dev)

        def run_probs():
            _lib.check(_lib.lib.amc_attention_probs(_lib.BF16, Bm, T, h, dh, qkv.data_ptr(), probs.data_ptr(), stream))

        def run_roll(vin):
            return lambda: _lib.check(_lib.lib.amc_attention_rollout_step(_lib.BF16, B, T, h, dh, qkv.data_ptr(),
                                                                          vin.data_ptr(), vo.data_ptr(), stream))

        t_p = time_launches(run_probs, a.steps, a.warmup, flush)
        by = 4.0 * Bm * h * T * T + 2.0 * Bm * T * 2 * d
        print(f"  attn_probs            {t_p * 1e3:9.1f} us/launch  {by / 1e9:8.3f} GB  {by / t_p / 1e9:7.3f} TB/s  "
              f"= {by / t_p / 1e9 / (COPY_PEAK / 1e12):.3f} of the 6.55 TB/s copy peak")
        for name, vin in (("dense v_in", v), ("v_in = e_0", e0)):
            t_r = time_launches(run_roll(vin), a.steps, a.warmup, flush)
            rows = B * T if vin is v else B
            fl = 2.0 * rows * h * T * dh
            t_mma, t_ex2 = fl / BF16_PEAK, rows * h * T / (16 * 148 * clk)
            bound, what = (t_mma, "tensor pipe") if t_mma > t_ex2 else (t_ex2, "ex2")
            print(f"  attn_rollout ({name:10s}) {t_r * 1e3:9.1f} us/launch  bound {bound * 1e6:8.1f} us ({what}) "
                  f"-> {bound * 1e3 / t_r:.3f} of it")
        del qkv, probs

        # ---- whole calls through the module surface on synthetic dataset frames
        classes = synth.CLASSES_19 if kw["num_classes"] == 19 else synth.CLASSES_11
        X, _, _ = synth.make_frames(1024, classes=classes, sps=w.get("sps", 1), seed=42)
        model.set_raw_input(synth.normalization_stats(X))
        x = torch.from_numpy(X[np.arange(B) % len(X)]).to(dev)

        def fwd():
            with torch.no_grad():
                model(x)

        t_f = time_calls(fwd, a.steps, a.warmup)
        t_ro = time_calls(lambda: model.attention_rollout(x), a.steps, a.warmup)
        print(f"  eval forward          {t_f:9.3f} ms/call")
        print(f"  attention_rollout     {t_ro:9.3f} ms/call  = {t_ro / t_f:.2f} x the eval forward")
        if Bmaps:
            xm = x[:Bm].contiguous()
            t_m = time_calls(lambda: model.attention_maps(xm, layers=[0]), a.steps, a.warmup)
            print(f"  attention_maps(layers=[0]) at B = {Bm}: {t_m:9.3f} ms/call")
        _lib.profile(True)
        try:
            model.attention_rollout(x)
            tab = _lib.profile_dump()
        finally:
            _lib.profile(False)
        print(f"  -- profile classes, one attention_rollout call (events around every launch site)")
        for name, r in sorted(tab.items(), key=lambda kv: -kv[1]["ms"]):
            print(f"     {name:24s} {r['n']:8d} {r['ms']:9.3f} ms")
        del model, x
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""bench.py -- IQ frames/s of the encoder hot path (BASELINE.json metric) on N B200s.

    python bench.py --gpus N --steps K --warmup W            # our arm (CUDA, sm_100a)
    python bench.py --impl reference --steps K --warmup W     # reference arm: the unmodified reference (oracle/_ref) on the host cores
    python bench.py ... --dump-outputs DIR                    # also write the last timed step's outputs as DIR/*.npy

A "step" is one training step (zero_grad -> forward -> CE(label_smoothing) -> backward -> clip -> AdamW,
R/training/train.py:258-271) over one batch of synthetic RadioML-shaped frames (random-init weights).
Workload at N=1: BASELINE.json configs[1] = ViT, 32x64 IQ image, patch 16, d=256, 6 layers, bf16.
  value : whole-job training frames/s with the input batches already resident in HBM
  e2e   : same step driven from pinned HOST buffers: H2D of the raw dataset-layout frames + labels and a
          D2H read of the loss every step are inside the timed region
Both are timed with CUDA events, barrier + synchronize on both sides, max over ranks.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # BASELINE.json configs[1]; 19 classes / dropout 0.1 / lr 1e-4 / wd 1e-3 from V/training/train.py:59-93
    # batch: frames per GPU per step.  32768 (301k token rows) keeps every kernel of the step above ~100 us, where the
    # bandwidth-bound ones get within 15-25 % of the copy peak; 8192 gives 1.59 M frames/s, 32768 1.87 M.
    "vit_p16_d256_L6": dict(kind="vit", batch=32768, eager_batch=8192, lr=1e-4, wd=1e-3,
                            kw=dict(in_channels=1, img_size_h=32, img_size_w=64, patch_size=16, num_classes=19,
                                    d_model=256, n_head=8, n_layers=6, ffn_hidden=1024, drop_prob=0.1)),
    # BASELINE.json configs[0] shape (R/training/train.py:84-95, 11 classes)
    "rawiq_seg16_d128_L6": dict(kind="rawiq", batch=2048, lr=1e-4, wd=1e-4,
                                kw=dict(in_channels=2, seq_length=1024, num_classes=11, d_model=128, n_head=8,
                                        n_layers=6, ffn_hidden=1024, drop_prob=0.2, use_cls_token=True,
                                        embedding_type="segment", segment_size=16)),
    # production ViT (V/training/train.py:83-88)
    "vit_p4_d128_L6": dict(kind="vit", batch=1024, lr=1e-4, wd=1e-3,
                           kw=dict(in_channels=1, img_size_h=32, img_size_w=64, patch_size=4, num_classes=19,
                                   d_model=128, n_head=8, n_layers=6, ffn_hidden=512, drop_prob=0.1)),
    # BASELINE.json configs[2]: raw-IQ across SPS modes, d256 h8 L6 F1024 (SURVEY §8d table row 3)
    "rawiq_sps1_seg8_d256_L6": dict(kind="rawiq", batch=1024, lr=1e-4, wd=1e-4, sps=1,
                                    kw=dict(in_channels=2, seq_length=1024, num_classes=11, d_model=256, n_head=8,
                                            n_layers=6, ffn_hidden=1024, drop_prob=0.2, use_cls_token=True,
                                            embedding_type="segment", segment_size=8)),
    "rawiq_sps2_seg16_d256_L6": dict(kind="rawiq", batch=1024, lr=1e-4, wd=1e-4, sps=2,
                                     kw=dict(in_channels=2, seq_length=2048, num_classes=11, d_model=256, n_head=8,
                                             n_layers=6, ffn_hidden=1024, drop_prob=0.2, use_cls_token=True,
                                             embedding_type="segment", segment_size=16)),
    "rawiq_sps2_seg8_d256_L6": dict(kind="rawiq", batch=512, lr=1e-4, wd=1e-4, sps=2,
                                    kw=dict(in_channels=2, seq_length=2048, num_classes=11, d_model=256, n_head=8,
                                            n_layers=6, ffn_hidden=1024, drop_prob=0.2, use_cls_token=True,
                                            embedding_type="segment", segment_size=8)),
    # BASELINE.json configs[4] corner: the largest point of the hyper-parameter grid (d512, 12 layers, F=4d)
    "rawiq_seg16_d512_L12": dict(kind="rawiq", batch=1024, lr=1e-4, wd=1e-4,
                                 kw=dict(in_channels=2, seq_length=1024, num_classes=11, d_model=512, n_head=8,
                                         n_layers=12, ffn_hidden=2048, drop_prob=0.2, use_cls_token=True,
                                         embedding_type="segment", segment_size=16)),
    # the reference Encoder's default embedding (R/models/encoder.py:26,34-41): Conv1d(2, d, 1), one token per
    # IQ sample -> T = 1025, long-sequence attention (attn_long.cu) + small-K embedding; train.py's other defaults
    "rawiq_conv1d_d128_L6": dict(kind="rawiq", batch=128, lr=1e-4, wd=1e-4,
                                 kw=dict(in_channels=2, seq_length=1024, num_classes=11, d_model=128, n_head=8,
                                         n_layers=6, ffn_hidden=1024, drop_prob=0.2, use_cls_token=True,
                                         embedding_type="conv1d", segment_size=64)),
}
DEFAULT_WORKLOAD = "vit_p16_d256_L6"


def geometry(w):
    kw = w["kw"]
    if w["kind"] == "vit":
        ttok = (kw["img_size_h"] // kw["patch_size"]) * (kw["img_size_w"] // kw["patch_size"])
        kemb = kw["in_channels"] * kw["patch_size"] ** 2
        T = ttok + 1
    else:
        seg = 1 if kw.get("embedding_type", "segment") == "conv1d" else kw["segment_size"]
        ttok = kw["seq_length"] // seg
        kemb = kw["in_channels"] * seg
        T = ttok + (1 if kw.get("use_cls_token", True) else 0)
    return T, ttok, kemb


def flops_per_frame(w):
    """Algorithmic forward FLOPs per frame (BASELINE.md §4); training = 3x."""
    kw = w["kw"]
    T, ttok, kemb = geometry(w)
    d, F, L, C = kw["d_model"], kw["ffn_hidden"], kw["n_layers"], kw["num_classes"]
    return L * T * (8 * d * d + 4 * d * F + 4 * T * d) + 2 * ttok * kemb * d + 2 * d * C


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        j = json.load(open(p))
        return dict(hbm_gbs=j["hbm_gbs"], tf_burst=j["bf16_tflops"], tf_sustained=j["bf16_tflops_sustained"],
                    source="measured")
    return dict(hbm_gbs=6650.0, tf_burst=1590.0, tf_sustained=1400.0, source="fallback")


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU while the timed region runs (NVML)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.samples, self.reasons, self.max_mhz = index, False, [], set(), None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {getattr(nv, k): k for k in dir(nv) if k.startswith("nvmlClocksEventReason") or
                 k.startswith("nvmlClocksThrottleReason")}
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if isinstance(bit, int) and bit and (r & bit) == bit and bin(bit).count("1") == 1:
                        short = name.replace("nvmlClocksEventReason", "").replace("nvmlClocksThrottleReason", "")
                        if short not in ("GpuIdle", "None", "All"):
                            self.reasons.add(short)
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons)}


# ------------------------------------------------------------------------------------------------
# Reference arm / CPU baseline: the unmodified reference modules (oracle/_ref, vendored by oracle/make_ref.py) on the host
# cores; when they did not travel, the PyTorch-eager port of the reference path (oracle/amc_torch_port.py: the same ATen
# operators the reference's modules issue, dropout included)
# ------------------------------------------------------------------------------------------------
def port_setup(w, sample_frames, device="cpu", seed=0):
    import torch
    from oracle import amc_oracle as O
    from oracle import amc_torch_port as TP
    kw = {k: v for k, v in w["kw"].items() if k != "drop_prob"}
    cfg = O.Config(kind=w["kind"], **kw)
    params = TP.make_params(cfg, seed, device)
    g = torch.Generator().manual_seed(seed)
    shape = (sample_frames, 1, 32, 64) if w["kind"] == "vit" else (sample_frames, 2, kw["seq_length"])
    src = torch.randn(shape, generator=g).to(device)
    labels = torch.randint(0, cfg.num_classes, (sample_frames,), generator=g).to(device)
    ts = TP.TrainStep(params, cfg, drop_prob=w["kw"]["drop_prob"], lr=w["lr"], weight_decay=w["wd"],
                      betas=(0.9, 0.99), max_norm=1.0, label_smoothing=0.1)
    return ts, src, labels


class ReferenceStep:
    """The reference's own training step on its own, unmodified modules (vendored into oracle/_ref by oracle/make_ref.py):
    R/training/train.py:258-271 verbatim -- zero_grad, model(x), CrossEntropyLoss(label_smoothing=0.1), backward,
    clip_grad_norm_(1.0), AdamW(betas (0.9, 0.99)).step() -- model.train(), dropout as configured."""

    def __init__(self, w, device="cpu", seed=0):
        import torch
        from oracle.make_ref import load_reference
        classes = load_reference()
        if classes is None:
            raise FileNotFoundError("oracle/_ref is absent (python oracle/make_ref.py in the build container)")
        RawIQ, ViT = classes
        torch.manual_seed(seed)
        self.model = (ViT if w["kind"] == "vit" else RawIQ)(**w["kw"], device=device).to(device)
        self.model.train()
        self.criterion = torch.nn.CrossEntropyLoss(label_smoothing=0.1)
        self.opt = torch.optim.AdamW(self.model.parameters(), lr=w["lr"], weight_decay=w["wd"], betas=(0.9, 0.99))
        self.torch = torch

    def step(self, images, labels):
        self.opt.zero_grad()
        outputs = self.model(images)
        loss = self.criterion(outputs, labels)
        loss.backward()
        self.torch.nn.utils.clip_grad_norm_(self.model.parameters(), max_norm=1.0)
        self.opt.step()
        return loss


def reference_available():
    return os.path.exists(os.path.join(ROOT, "oracle", "_ref", "MANIFEST.json"))


def cpu_train_frames_per_s(w, sample_frames, steps, warmup):
    """Train steps on all host threads -> (frames/s, s/step, threads, kind): the unmodified reference when oracle/_ref
    travelled with the snapshot ("reference"), else the torch port of its operator sequence ("port")."""
    import torch
    n = os.cpu_count() or 1
    torch.set_num_threads(n)
    if reference_available():
        kind = "reference"
        kw = w["kw"]
        g = torch.Generator().manual_seed(0)
        shape = (sample_frames, 1, 32, 64) if w["kind"] == "vit" else (sample_frames, 2, kw["seq_length"])
        src = torch.randn(shape, generator=g)
        labels = torch.randint(0, kw["num_classes"], (sample_frames,), generator=g)
        ref = ReferenceStep(w)
        step = lambda: ref.step(src, labels)
    else:
        kind = "port"
        ts, src, labels = port_setup(w, sample_frames)
        step = lambda: ts.step(src, labels)[0]
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        loss = step()
        loss.item()                                   # the reference reads loss.item() every step
        if it >= warmup:
            times.append(time.perf_counter() - t0)
    return sample_frames * len(times) / sum(times), sum(times) / len(times), torch.get_num_threads(), kind


KIND_NOTE = {"reference": "the unmodified reference modules (oracle/_ref) and its train step (R/training/train.py:258-271): "
                          "fp32, dropout on, torch CPU eager, all host threads",
             "port": "PyTorch-eager CPU port (oracle/amc_torch_port.py) of the reference train step: same ATen operators, "
                     "dropout on, fp32, all host threads (oracle/_ref was not vendored)"}


def gpu_eager_port_frames_per_s(w, frames, dev, steps=5, warmup=2):
    """The same port in PyTorch eager on the GPU (TF32 on, as R/training/train.py:359-360 sets it)."""
    import torch
    tf32 = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = True
    try:
        ts, src, labels = port_setup(w, frames, dev)
        for _ in range(warmup):
            ts.step(src, labels)
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            loss, _, _ = ts.step(src, labels)
            loss.item()
        e1.record()
        torch.cuda.synchronize(dev)
        ms = e0.elapsed_time(e1) / steps
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = tf32
        del ts, src, labels
        torch.cuda.empty_cache()
    return frames / (ms / 1e3), ms


def run_reference_arm(args, w, wname):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sample = args.batch or args.cpu_sample       # --batch runs the reference arm at a stated per-step batch
    fps, sec, cores, kind = cpu_train_frames_per_s(w, sample, args.steps, max(args.warmup, 1))
    line = {
        "impl": "reference", "metric": "train_frames_per_sec", "value": fps, "unit": "frames/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": wname, "frames_per_step": sample, "note": KIND_NOTE[kind]},
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores, "kind": kind,
                         "sample": f"{args.steps} train steps of {sample} frames, torch CPU eager on {cores} threads"},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
def ncu_traffic(table, workload, kernel_class, frames, default_frames):
    """DRAM bytes per launch of `kernel_class` from profiles/ncu_traffic.json -> (bytes or None, where they come from).
    An entry records the frames per launch of its `ncu --set full` capture (absent = the workload's bench batch); when this
    run's batch differs the figure is scaled linearly (every kernel class here moves bytes in proportion to the frames)."""
    ent = table.get(workload, {}).get(kernel_class, {})
    traffic = ent.get("dram_bytes_per_launch")
    if traffic is None:
        return None, None
    cap = ent.get("frames") or default_frames
    if cap != frames:
        return traffic * frames / cap, f"ncu capture at {cap} frames per launch, scaled by {frames}/{cap}"
    return traffic, f"ncu capture at this launch size ({ent.get('report')})"


# --dump-outputs: elements kept per array (float32), 64 MB in all
DUMP_ELEMS = {"logits": 4 << 20, "parameters": 12 << 20}


def dump_outputs(out_dir, trainer):
    """Writes what the last training step handed its caller to out_dir/<name>.npy (float32): `logits`, the [B, classes]
    output of its forward pass, and `parameters`, the model's parameters after its AdamW update (named_parameters order,
    flattened and concatenated).  An array with more elements than DUMP_ELEMS allows is replaced by a fixed, seeded
    sample of them (sorted flat indices, the same for every run with the same arguments), so the outputs of two builds
    can be compared element for element.  Compare them with a tolerance: the weight-gradient GEMMs add split-K partial
    sums with atomics, so two runs of one build already differ in the last bits, and training steps amplify that (bf16,
    default workload, 25 steps: logits 2e-3 and parameters 5e-4 of their largest magnitude, measured on a B200 at 1000 W)."""
    import numpy as np
    import torch
    arrays = {"logits": trainer._logits,
              "parameters": torch.cat([p.detach().reshape(-1) for p in trainer.model.parameters()])}
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        a = t.float().cpu().numpy()
        if a.size > DUMP_ELEMS[name]:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, DUMP_ELEMS[name], replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0, help="frames per GPU per step (default: workload's)")
    ap.add_argument("--global-batch", type=int, default=0,
                    help="strong scaling: total frames per step, split evenly over the GPUs (overrides --batch)")
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--cpu-sample", type=int, default=256, help="frames per CPU-baseline step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--gpu-eager", action="store_true",
                    help="also time the reference port in PyTorch eager on the GPU (reported beside; off by default: the "
                         "default run touches oracle/ only for the CPU baseline)")
    ap.add_argument("--no-gpu-eager", action="store_true", help=argparse.SUPPRESS)   # accepted, now the default
    ap.add_argument("--graph", action="store_true",
                    help="single GPU: drive the step as one CUDA-graph replay (GraphTrainStep) -- the launch-bound small batches")
    ap.add_argument("--profile-out", default="")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write the logits and updated parameters of the last timed training step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    w = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference_arm(args, w, args.workload)
        return
    if args.warmup < 3:
        args.warmup = 3

    import numpy as np
    import torch
    import torch.distributed as dist
    import vit_vs_raw_iq_b200 as amc
    from vit_vs_raw_iq_b200 import _lib, synth
    from vit_vs_raw_iq_b200.trainer import GraphTrainStep, HostPipeline, HostPredictor, TrainStep, predict

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    B = args.batch or w["batch"]
    if args.global_batch:
        if args.global_batch % world:
            raise SystemExit("--global-batch must be divisible by the number of GPUs")
        B = args.global_batch // world
    kw = dict(w["kw"])
    T, ttok, kemb = geometry(w)

    torch.manual_seed(0)
    cls = amc.ViTAMCTransformer if w["kind"] == "vit" else amc.RawIQAMCTransformer
    model = cls(**kw, device=dev, compute_dtype=args.dtype)
    classes = synth.CLASSES_19 if kw["num_classes"] == 19 else synth.CLASSES_11

    # synthetic dataset-layout frames [n, 1024, 2]; a small pool is tiled to the batch (content does not
    # change the arithmetic; a 64 MB batch is far larger than... the activations it produces are >> L2)
    pool_n = 2048
    sps = w.get("sps", 1)
    if sps > 1:
        pool_n = 1024
    X, y, _ = synth.make_frames(pool_n, classes=classes, sps=sps, seed=42 + rank)
    stats = synth.normalization_stats(X)
    model.set_raw_input(stats)
    n_batches = 3
    reps = (B + pool_n - 1) // pool_n
    host_x, host_y = [], []
    for i in range(n_batches):
        perm = np.random.default_rng(100 + i + 10 * rank).permutation(pool_n * reps)[:B] % pool_n
        host_x.append(torch.from_numpy(X[perm]).pin_memory())
        host_y.append(torch.from_numpy(y[perm]).pin_memory())
    dev_x = [t.to(dev) for t in host_x]
    dev_y = [t.to(dev) for t in host_y]

    step_cls = GraphTrainStep if (args.graph and world == 1) else TrainStep
    trainer = step_cls(model, lr=w["lr"], weight_decay=w["wd"], betas=(0.9, 0.99), max_norm=1.0,
                       label_smoothing=0.1)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(ms):
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return ms

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(i)
        e1.record()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1))

    # ---- device-resident training throughput (value) ------------------------------------------------
    for i in range(args.warmup):
        trainer.step(dev_x[i % n_batches], dev_y[i % n_batches])
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = _lib.lib.amc_launch_count()
    replays0 = getattr(trainer, "replays", 0)
    ms_train = timed(lambda i: trainer.step(dev_x[i % n_batches], dev_y[i % n_batches]), args.steps)
    launches = _lib.lib.amc_launch_count() - launches0
    if step_cls is GraphTrainStep:      # kernels of the library launched by the graph replays of the timed region
        launches += (trainer.replays - replays0) * trainer.kernels_per_replay
    loss, acc = trainer.read_stats()
    if args.dump_outputs and rank == 0:     # before the steps below train the model further
        dump_outputs(args.dump_outputs, trainer)

    # ---- end to end from host buffers (e2e) -----------------------------------------------------------
    pipe = HostPipeline(trainer, tuple(host_x[0].shape))
    for i in range(3):
        pipe.step(host_x[i % n_batches], host_y[i % n_batches])
    pipe.flush()

    def e2e_step(i):
        pipe.step(host_x[i % n_batches], host_y[i % n_batches])   # returns the previous step's loss (host float)
        if i == args.steps - 1:
            pipe.flush()                                            # ... and the last one inside the timed region
    ms_e2e = timed(e2e_step, args.steps)
    sampler.stop_flag = True
    sampler.join(timeout=2)

    # ---- inference (R/training/utils.py:311-320) -------------------------------------------------------
    preds = torch.empty(B, dtype=torch.int64, device=dev)
    for i in range(3):
        predict(model, dev_x[i % n_batches], preds)
    ms_inf = timed(lambda i: predict(model, dev_x[i % n_batches], preds), args.steps)
    hp = HostPredictor(model, tuple(host_x[0].shape))

    def infer_host(i):
        hp.predict(host_x[i % n_batches])                           # previous batch's predictions (pinned int64)
        if i == args.steps - 1:
            hp.flush()
    for i in range(3):
        hp.predict(host_x[i % n_batches])
    hp.flush()
    ms_inf_e2e = timed(infer_host, args.steps)

    # ---- in-situ kernel-class timing for the roofline --------------------------------------------------
    _lib.profile(True)
    prof_steps = 3
    for i in range(prof_steps):            # (the in-library events need real launches: graph mode runs these steps eagerly)
        (trainer._run if step_cls is GraphTrainStep else trainer.step)(dev_x[i % n_batches], dev_y[i % n_batches])
    prof = _lib.profile_dump()
    _lib.profile(False)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = load_peaks()
    fl_frame = flops_per_frame(w)
    frames = B * world
    train_fps = frames * args.steps / (ms_train / 1e3)
    tot_ms = sum(v["ms"] for v in prof.values())
    peak_tf = peaks["tf_sustained"] if args.dtype == "bf16" else None     # fp32 mode runs on the FMA pipe

    def class_roofline(name, v):
        """Roofline of one kernel class: algorithmic FLOPs / bytes per launch over its CUDA-event time (events are
        recorded inside the library on the launch stream, amc_profile_enable/dump)."""
        ms = v["ms"] / max(v["n"], 1)
        tf = v["flops"] / max(v["ms"], 1e-9) / 1e9
        gbs = v["bytes"] / max(v["ms"], 1e-9) / 1e6
        t_tensor = v["flops"] / (peak_tf * 1e12) if peak_tf and v["flops"] else 0.0
        t_hbm = v["bytes"] / (peaks["hbm_gbs"] * 1e9)
        bound = "tensor" if t_tensor > t_hbm else "hbm"
        r = {"kernel": name, "bound": bound, "launches_per_step": v["n"] / prof_steps, "avg_launch_ms": ms,
             "share_of_step": v["ms"] / tot_ms if tot_ms else None}
        if bound == "tensor":
            r.update(achieved=tf, peak=peak_tf, unit="TFLOP/s", frac=tf / peak_tf, hbm_GBps=gbs)
        else:
            r.update(achieved=gbs, peak=peaks["hbm_gbs"], unit="GB/s", frac=gbs / peaks["hbm_gbs"], tflops=tf)
        return r

    table = [class_roofline(k, v) for k, v in sorted(prof.items(), key=lambda kv: -kv[1]["ms"]) if v["bytes"] or v["flops"]]
    dom = table[0]
    traffic, traffic_note = None, None
    tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")      # written by tools/ncu_summary.py from `ncu --set full`
    if os.path.exists(tpath):
        traffic, traffic_note = ncu_traffic(json.load(open(tpath)), args.workload, dom["kernel"], B, w["batch"])
    roofline = {k: dom[k] for k in ("kernel", "bound", "achieved", "peak", "unit", "frac")}
    if traffic is not None:
        roofline["traffic_source"] = traffic_note
    roofline.update(traffic=traffic, peak_source=peaks["source"] + (" (sustained)" if dom["bound"] == "tensor" else ""),
                    launches_per_step=dom["launches_per_step"], avg_launch_ms=dom["avg_launch_ms"],
                    share_of_step=dom["share_of_step"],
                    algorithmic_per_launch={"flops": prof[dom["kernel"]]["flops"] / max(prof[dom["kernel"]]["n"], 1),
                                            "bytes": prof[dom["kernel"]]["bytes"] / max(prof[dom["kernel"]]["n"], 1)})
    gemm = {k: v for k, v in prof.items() if k.startswith("gemm")}
    g_ms = sum(v["ms"] for v in gemm.values())
    g_fl = sum(v["flops"] for v in gemm.values())
    g_by = sum(v["bytes"] for v in gemm.values())
    roofline["all_gemms"] = {"tflops": g_fl / max(g_ms, 1e-9) / 1e9, "frac_of_tensor_peak": g_fl / max(g_ms, 1e-9) / 1e9 / peaks["tf_sustained"],
                             "algorithmic_GBps": g_by / max(g_ms, 1e-9) / 1e6,
                             "frac_of_hbm_peak": g_by / max(g_ms, 1e-9) / 1e6 / peaks["hbm_gbs"],
                             "share_of_step": g_ms / tot_ms if tot_ms else None}
    classes_ms = {k: round(v["ms"] / prof_steps, 4) for k, v in sorted(prof.items(), key=lambda kv: -kv[1]["ms"])}

    line = {
        "metric": "train_frames_per_sec", "value": train_fps, "unit": "frames/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_train / args.steps,
        "higher_is_better": True, "scaling": "strong" if args.global_batch else "weak", "vs_baseline": None,
        "dtype": args.dtype, "data": "synthetic",
        "config": {"workload": args.workload, "frames_per_gpu_per_step": B, "global_batch": frames, "tokens": T,
                   **{k: kw[k] for k in ("d_model", "n_head", "n_layers", "ffn_hidden", "num_classes", "drop_prob")},
                   "parallelism": f"dp{world}", "optimizer": "clip1.0+AdamW", "label_smoothing": 0.1,
                   "step_driver": "cuda_graph_replay" if step_cls is GraphTrainStep else "stream_launches",
                   "l2_policy": "inputs+activations per step (>1 GB) exceed the 126 MB L2; 3 batches rotate",
                   "input": f"raw [B,{X.shape[1]},2] fp32 frames, z-score+framing fused in the front end"},
        "model_tflops": train_fps * 3 * fl_frame / 1e12,
        "model_tflops_frac_of_bf16_peak": train_fps * 3 * fl_frame / 1e12 / (peaks["tf_sustained"] * world),
        "e2e": {"value": frames * args.steps / (ms_e2e / 1e3), "unit": "frames/s",
                "h2d_bytes_per_step": pipe.h2d_bytes, "d2h_bytes_per_step": pipe.d2h_bytes,
                "ms_per_step": ms_e2e / args.steps},
        "infer": {"value": frames * args.steps / (ms_inf / 1e3), "unit": "frames/s",
                  "e2e_value": frames * args.steps / (ms_inf_e2e / 1e3),
                  "e2e_h2d_bytes_per_step": host_x[0].numel() * 4, "e2e_d2h_bytes_per_step": B * 8},
        "gpu_launches": int(launches),
        "clocks": sampler.summary(),
        "roofline": roofline,
        "rooflines": [{k: (round(v, 4) if isinstance(v, float) else v) for k, v in r.items()} for r in table],
        "kernel_ms_per_step": classes_ms,
        "train_loss": loss, "train_acc": acc,
    }
    if world == 1 and args.gpu_eager and not args.no_gpu_eager:
        del trainer, pipe, hp, model
        torch.cuda.empty_cache()
        ef, ems = gpu_eager_port_frames_per_s(w, min(B, w.get("eager_batch", B)), dev)
        line["gpu_eager_port"] = {"value": ef, "unit": "frames/s", "ms_per_step": ems, "note":
                                  "the reference's operator sequence in PyTorch eager on this GPU (TF32 on as the "
                                  "reference sets it, fp32 weights, dropout on); reported beside, not the target"}
    if not args.no_cpu_baseline:
        t0 = time.perf_counter()
        fps, sec, cores, kind = cpu_train_frames_per_s(w, args.cpu_sample, 2, 1)
        n_steps = max(2, min(40, int(12.0 / max(sec, 1e-3))))
        fps, sec, cores, kind = cpu_train_frames_per_s(w, args.cpu_sample, n_steps, 1)
        line["cpu_baseline"] = {"value": fps, "unit": "frames/s", "cores": cores, "kind": kind,
                                "sample": f"{n_steps} train steps of {args.cpu_sample} frames ({KIND_NOTE[kind]}), "
                                          f"{time.perf_counter() - t0:.0f} s total"}
    print(json.dumps(line), flush=True)
    if args.profile_out:
        with open(args.profile_out, "w") as f:
            json.dump({"prof_steps": prof_steps, "classes": prof, "line": line}, f, indent=1)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

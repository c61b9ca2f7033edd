"""The training step and the inference loop of the reference, fused around the flat blobs.

``TrainStep.step`` is R/training/train.py:258-271 (zero_grad -> forward -> CrossEntropyLoss(label
smoothing) -> backward -> clip_grad_norm_ -> AdamW.step) without the autograd round trip: gradients
accumulate straight into one flat fp32 blob, the loss / accuracy counters stay on the device
(the reference's two ``.item()`` calls per step, train.py:274-277, are what serialise it), and under
data parallelism the flat gradient is all-reduced in per-stage buckets that overlap the rest of
backward (NCCL over NVLink; SURVEY §8e).  ``predict`` is the loop of R/training/utils.py:311-320.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Tuple

import torch

from . import _lib
from .modules import _AMCBase, _DTYPES


def _check_labels(labels, B: int, dev: torch.device) -> None:
    # the kernel reads `labels` as B contiguous int64 on the model's device: anything else is an out-of-bounds or
    # garbage device read (nn.CrossEntropyLoss raises in these cases too)
    if not (isinstance(labels, torch.Tensor) and labels.is_cuda and labels.device == dev):
        raise ValueError(f"labels must be a CUDA tensor on {dev}")
    if labels.dtype != torch.int64 or labels.dim() != 1 or labels.numel() != B or not labels.is_contiguous():
        raise ValueError(f"labels must be a contiguous int64 tensor of shape [{B}], got {labels.dtype} "
                         f"{tuple(labels.shape)}")


class TrainStep:
    def __init__(self, model: _AMCBase, lr: float = 1e-4, weight_decay: float = 1e-4, betas=(0.9, 0.99),
                 eps: float = 1e-8, max_norm: float = 1.0, label_smoothing: float = 0.1,
                 process_group=None, layers_per_bucket: int = 2, data_parallel: bool = True, attack=None):
        """``data_parallel=False``: train this model on this rank alone even though ``torch.distributed`` is initialised
        (rank-sharded hyper-parameter search: every rank holds DIFFERENT models, so no collective may be issued).

        ``attack`` (an ``adversarial.PGDAttack`` on this model): adversarial training.  Each step first replaces the batch
        by ``attack(src, labels)`` against the current parameters, reusing the step's workspace, then runs the unchanged
        step on it (PGD training; ``steps=1, step_frac=1.25`` with a random start is "fast" FGSM-RS training)."""
        if attack is not None and attack.model is not model:
            raise ValueError("the attack must be bound to the model this TrainStep trains")
        self.attack = attack
        self.model = model
        self.core = model._core
        self.lr, self.wd, self.betas, self.eps = lr, weight_decay, betas, eps
        self.max_norm, self.ls = max_norm, label_smoothing
        self.pg = process_group
        self.world = 1
        if data_parallel and (process_group is not None or
                              (torch.distributed.is_available() and torch.distributed.is_initialized())):
            self.world = torch.distributed.get_world_size(process_group)
        flat = model.flat_parameters()
        if not flat.is_cuda:
            raise RuntimeError("TrainStep needs the model on a CUDA device (no CPU fallback)")
        self.dev = flat.device
        n = flat.numel()
        self.grads = torch.zeros(n, dtype=torch.float32, device=self.dev)
        self.exp_avg = torch.zeros_like(self.grads)
        self.exp_avg_sq = torch.zeros_like(self.grads)
        self.stats = torch.zeros(2, dtype=torch.float32, device=self.dev)     # [sum loss, #correct]
        self.norm_ws = torch.zeros(2, dtype=torch.float32, device=self.dev)
        self.step_count = 0
        self.frames_seen = 0
        if self.world > 1:
            # replicas start identical whatever each rank's seed or checkpoint was (only gradients are reduced afterwards),
            # and every rank draws its own dropout masks
            for t in (flat.data, self.exp_avg, self.exp_avg_sq):
                torch.distributed.broadcast(t, src=torch.distributed.get_global_rank(process_group, 0)
                                            if process_group is not None else 0, group=process_group)
            self.core.rank_salt = torch.distributed.get_rank(process_group)
        self._ws: Optional[torch.Tensor] = None
        self._ws_key = None
        self._logits = self._dlogits = None
        self.buckets = self._make_buckets(layers_per_bucket)

    # gradient buckets: (stage_begin, stage_end, blob_lo, blob_hi) in backward order
    def _make_buckets(self, per: int) -> List[Tuple[int, int, int, int]]:
        L, nl = self.core.layout, self.core.n_layers
        head_lo = L.head_ln_w if L.head_ln_w >= 0 else L.head_w
        out = []
        s = 1
        first = True
        while s <= nl:
            e = min(nl + 1, s + per)
            lo = L.layer0 + (nl - (e - 1)) * L.layer_stride          # lowest layer index in this bucket
            hi = L.layer0 + (nl - (s - 1)) * L.layer_stride
            if first:                                                # head rides with the top layers
                out.append((0, e, lo, hi))
                out.append((-1, -1, head_lo, L.total))
                first = False
            else:
                out.append((s, e, lo, hi))
            s = e
        if first:
            out.append((0, 1, head_lo, L.total))
        out.append((nl + 1, nl + 2, 0, L.layer0))
        return out

    def _buffers(self, B: int, desc):
        key = (B, desc.dtype, desc.p_drop > 0)
        if self._ws_key != key:
            self._ws = torch.empty(_lib.workspace_bytes(desc), dtype=torch.uint8, device=self.dev)
            self._logits = torch.empty((B, self.core.C), dtype=torch.float32, device=self.dev)
            self._dlogits = torch.empty_like(self._logits)
            self._ws_key = key
        return self._ws, self._logits, self._dlogits

    def step(self, src: torch.Tensor, labels: torch.Tensor) -> None:
        """One optimisation step on device tensors; statistics accumulate in ``self.stats``."""
        core = self.core
        self.model.train()
        desc = core.make_desc(src, training=True, module_training=True)
        B = desc.B
        _check_labels(labels, B, self.dev)
        if src.device != self.dev:
            raise ValueError(f"src is on {src.device}, the model on {self.dev}")
        ws, logits, dlogits = self._buffers(B, desc)
        if self.attack is not None:               # stream order: the attack is done before the forward reuses `ws`
            src = self.attack._run(src, labels, ws)
        flat = self.model.flat_parameters()
        st = torch.cuda.current_stream(self.dev).cuda_stream
        lib = _lib.lib
        _lib.check(lib.amc_zero(self.grads.data_ptr(), self.grads.numel() * 4, st), "amc_zero")     # optimizer.zero_grad()
        _lib.check(lib.amc_model_fwd(C.byref(desc), src.data_ptr(), flat.data_ptr(), core.pos_buffer().data_ptr(),
                                     ws.data_ptr(), logits.data_ptr(), 0, st), "amc_model_fwd")
        gb = B * self.world
        _lib.check(lib.amc_ce_loss(B, core.C, logits.data_ptr(), labels.data_ptr(), self.ls, 1.0 / gb, 1.0,
                                   dlogits.data_ptr(), self.stats.data_ptr(), st), "amc_ce_loss")
        works = []
        for (s0, s1, lo, hi) in self.buckets:
            if s0 >= 0:
                _lib.check(lib.amc_model_bwd(C.byref(desc), src.data_ptr(), flat.data_ptr(), ws.data_ptr(),
                                             dlogits.data_ptr(), 0, self.grads.data_ptr(), s0, s1, st),
                           "amc_model_bwd")
            if self.world > 1:
                # NCCL runs on its own stream after the kernels enqueued so far; later stages overlap it
                works.append(torch.distributed.all_reduce(self.grads[lo:hi], group=self.pg, async_op=True))
        for w in works:
            w.wait()
        self.step_count += 1
        self.frames_seen += B
        _lib.check(lib.amc_adamw_clip_step(flat.numel(), flat.data_ptr(), self.grads.data_ptr(),
                                           self.exp_avg.data_ptr(), self.exp_avg_sq.data_ptr(), self.lr,
                                           self.betas[0], self.betas[1], self.eps, self.wd, self.max_norm, 1.0,
                                           self.step_count, self.norm_ws.data_ptr(), st), "amc_adamw_clip_step")

    def read_stats(self, reset: bool = True) -> Tuple[float, float]:
        """(mean loss per frame, accuracy) since the last reset -- one device->host read."""
        s = self.stats.tolist()
        n = max(self.frames_seen, 1)
        if reset:
            self.stats.zero_()
            self.frames_seen = 0
        _check_loss(s[0])
        return s[0] / n, s[1] / n


def _check_loss(loss_sum: float) -> None:
    """amc_ce_loss turns a frame's loss into NaN when its label is outside [0, num_classes) -- the case in which
    nn.CrossEntropyLoss raises (R/training/train.py:260); a diverged model shows up here the same way."""
    if loss_sum != loss_sum:
        raise RuntimeError("training loss is NaN: a label outside [0, num_classes) (nn.CrossEntropyLoss would have "
                           "raised 'Target out of bounds') or a diverged model")


class GraphTrainStep(TrainStep):
    """``TrainStep`` for a fixed batch shape as ONE CUDA-graph launch per step.

    At the reference's own batch (256 frames, R/training/train.py:94) a step is ~110 kernels of a few microseconds each:
    launch- and host-bound.  Everything in it is static for a fixed shape -- kernel parameters, tensor maps, workspace --
    except two scalars that change every step: the AdamW step number (bias corrections) and the dropout counter.  Both
    live in one device word here (``AmcDesc.step_counter`` / ``amc_adamw_clip_step_graph``), so the step is captured once
    and replayed.  The first call runs eagerly (one-time set-up must not happen inside a capture), the second captures.
    Single process only: data-parallel runs use ``TrainStep`` (its NCCL buckets overlap backward on their own stream)."""

    def __init__(self, model: _AMCBase, *args, **kwargs):
        super().__init__(model, *args, **kwargs)
        if self.world > 1:
            raise RuntimeError("GraphTrainStep is single-process; use TrainStep under torch.distributed")
        self.counter = torch.zeros(1, dtype=torch.int32, device=self.dev)
        self.core.step_counter = self.counter
        self._graph = None
        self._gkey = None
        self._gsrc = self._glabels = None
        self.kernels_per_replay = 0
        self.replays = 0

    def _run(self, src: torch.Tensor, labels: torch.Tensor) -> None:
        core = self.core
        desc = core.make_desc(src, training=True, module_training=True)
        B = desc.B
        ws, logits, dlogits = self._buffers(B, desc)
        if self.attack is not None:               # captured too: the random start reads the device step counter
            src = self.attack._run(src, labels, ws)
        flat = self.model.flat_parameters()
        st = torch.cuda.current_stream(self.dev).cuda_stream
        lib = _lib.lib
        _lib.check(lib.amc_zero(self.grads.data_ptr(), self.grads.numel() * 4, st), "amc_zero")     # optimizer.zero_grad()
        _lib.check(lib.amc_model_fwd(C.byref(desc), src.data_ptr(), flat.data_ptr(), core.pos_buffer().data_ptr(),
                                     ws.data_ptr(), logits.data_ptr(), 0, st), "amc_model_fwd")
        _lib.check(lib.amc_ce_loss(B, core.C, logits.data_ptr(), labels.data_ptr(), self.ls, 1.0 / B, 1.0,
                                   dlogits.data_ptr(), self.stats.data_ptr(), st), "amc_ce_loss")
        _lib.check(lib.amc_model_bwd(C.byref(desc), src.data_ptr(), flat.data_ptr(), ws.data_ptr(), dlogits.data_ptr(),
                                     0, self.grads.data_ptr(), 0, core.n_layers + 2, st), "amc_model_bwd")
        _lib.check(lib.amc_adamw_clip_step_graph(flat.numel(), flat.data_ptr(), self.grads.data_ptr(),
                                                 self.exp_avg.data_ptr(), self.exp_avg_sq.data_ptr(), self.lr,
                                                 self.betas[0], self.betas[1], self.eps, self.wd, self.max_norm, 1.0,
                                                 self.counter.data_ptr(), self.norm_ws.data_ptr(), st),
                   "amc_adamw_clip_step_graph")

    def step(self, src: torch.Tensor, labels: torch.Tensor) -> None:
        self.model.train()
        B = int(src.shape[0])
        _check_labels(labels, B, self.dev)
        key = (tuple(src.shape), src.dtype, self.core.compute_dtype, self.core.drop_prob > 0)
        if self._gkey != key:                              # new shape: this call runs eagerly, the next one captures
            self._graph, self._gkey = None, key
            self._gsrc, self._glabels = torch.empty_like(src), torch.empty_like(labels)
            self._gsrc.copy_(src)
            self._glabels.copy_(labels)
            self._run(self._gsrc, self._glabels)
        else:
            self._gsrc.copy_(src, non_blocking=True)
            self._glabels.copy_(labels, non_blocking=True)
            if self._graph is None:
                torch.cuda.synchronize(self.dev)
                g = torch.cuda.CUDAGraph()
                n0 = _lib.lib.amc_launch_count()
                with torch.cuda.graph(g):
                    self._run(self._gsrc, self._glabels)
                self.kernels_per_replay = _lib.lib.amc_launch_count() - n0    # library kernels inside one replay
                self._graph = g
            self._graph.replay()
            self.replays += 1
        self.step_count += 1
        self.frames_seen += B


class HostPipeline:
    """End-to-end step from HOST buffers: pinned host frames -> async H2D on a copy stream (double buffered)
    -> TrainStep.step -> loss read back every step.  This is the loop of train.py:254-277
    (.to(device, non_blocking=True) ... loss.item()) with one change: ``step`` returns the loss of the
    PREVIOUS step, so the H2D copy of step i overlaps the compute of step i-1 instead of waiting for it.
    ``flush()`` returns the last one."""

    def __init__(self, trainer: TrainStep, src_shape):
        self.t = trainer
        dev = trainer.dev
        self.copy_stream = torch.cuda.Stream(device=dev)
        self.bufs = [(torch.empty(src_shape, dtype=torch.float32, device=dev),
                      torch.empty((src_shape[0],), dtype=torch.int64, device=dev)) for _ in range(2)]
        self.ready = [torch.cuda.Event() for _ in range(2)]
        self.free = [torch.cuda.Event() for _ in range(2)]
        self.loss_evt = [torch.cuda.Event() for _ in range(2)]
        self.loss_host = [torch.zeros(2, dtype=torch.float32).pin_memory() for _ in range(2)]
        self.h2d_bytes = self.bufs[0][0].numel() * 4 + self.bufs[0][1].numel() * 8
        self.d2h_bytes = 8
        self.i = 0
        self.batch = src_shape[0]

    def step(self, src_host: torch.Tensor, labels_host: torch.Tensor, sync: bool = False):
        """``sync=True``: wait for THIS step and return its loss (the reference's ``loss.item()`` semantics, train.py:274);
        the default returns the previous step's loss so that the next batch's H2D copy overlaps this step's compute."""
        k = self.i & 1
        xs, ys = self.bufs[k]
        cur = torch.cuda.current_stream(self.t.dev)
        with torch.cuda.stream(self.copy_stream):
            self.copy_stream.wait_event(self.free[k])          # the step that last used this buffer is done
            xs.copy_(src_host, non_blocking=True)
            ys.copy_(labels_host, non_blocking=True)
            self.ready[k].record(self.copy_stream)
        cur.wait_event(self.ready[k])
        self.t.step(xs, ys)
        self.free[k].record(cur)
        self.loss_host[k].copy_(self.t.stats, non_blocking=True)
        _lib.check(_lib.lib.amc_zero(self.t.stats.data_ptr(), 8, cur.cuda_stream), "amc_zero")
        self.t.frames_seen = 0
        self.loss_evt[k].record(cur)
        if sync:
            self.loss_evt[k].synchronize()
            _check_loss(float(self.loss_host[k][0]))
            self.i += 1
            return float(self.loss_host[k][0]) / self.batch
        prev = None
        if self.i > 0:
            self.loss_evt[1 - k].synchronize()
            _check_loss(float(self.loss_host[1 - k][0]))
            prev = float(self.loss_host[1 - k][0]) / self.batch
        self.i += 1
        return prev

    def flush(self):
        if self.i == 0:
            return None
        k = (self.i - 1) & 1
        self.loss_evt[k].synchronize()
        _check_loss(float(self.loss_host[k][0]))
        return float(self.loss_host[k][0]) / self.batch


class HostPredictor:
    """Inference from HOST buffers (R/training/utils.py:311-320: images.to(device) -> model(x).max(1) ->
    predicted.cpu()), double buffered: ``predict`` returns the PREVIOUS batch's class indices (pinned int64
    tensor, valid until the next-but-one call); ``flush()`` returns the last."""

    def __init__(self, model: _AMCBase, src_shape):
        self.model = model
        dev = model.flat_parameters().device
        self.dev = dev
        self.copy_stream = torch.cuda.Stream(device=dev)
        self.x = [torch.empty(src_shape, dtype=torch.float32, device=dev) for _ in range(2)]
        self.p = [torch.empty((src_shape[0],), dtype=torch.int64, device=dev) for _ in range(2)]
        self.p_host = [torch.empty((src_shape[0],), dtype=torch.int64).pin_memory() for _ in range(2)]
        self.ready = [torch.cuda.Event() for _ in range(2)]
        self.free = [torch.cuda.Event() for _ in range(2)]
        self.done = [torch.cuda.Event() for _ in range(2)]
        self.h2d_bytes = self.x[0].numel() * 4
        self.d2h_bytes = src_shape[0] * 8
        self.i = 0

    def predict(self, src_host: torch.Tensor):
        k = self.i & 1
        cur = torch.cuda.current_stream(self.dev)
        with torch.cuda.stream(self.copy_stream):
            self.copy_stream.wait_event(self.free[k])
            self.x[k].copy_(src_host, non_blocking=True)
            self.ready[k].record(self.copy_stream)
        cur.wait_event(self.ready[k])
        predict(self.model, self.x[k], self.p[k])
        self.free[k].record(cur)
        self.p_host[k].copy_(self.p[k], non_blocking=True)
        self.done[k].record(cur)
        prev = None
        if self.i > 0:
            self.done[1 - k].synchronize()
            prev = self.p_host[1 - k]
        self.i += 1
        return prev

    def flush(self):
        if self.i == 0:
            return None
        k = (self.i - 1) & 1
        self.done[k].synchronize()
        return self.p_host[k]


class GraphPredictor:
    """The inference loop for a fixed batch shape as ONE CUDA-graph launch: eval forward + argmax are captured
    once (all kernel parameters, tensor maps and the workspace are static for a fixed shape) and replayed.
    At the reference's interactive batch sizes (1..256 frames, compare_models.py / evaluate.py) the forward is
    ~40 short kernels and launch-bound; the replay removes the per-kernel launch and host set-up cost.
    ``predict`` accepts a device or (pinned) host tensor of the captured shape and returns the static int64 result
    tensor (valid until the next call)."""

    def __init__(self, model: _AMCBase, src_shape, warmup: int = 2):
        self.model = model
        dev = model.flat_parameters().device
        self.dev = dev
        self.x = torch.zeros(src_shape, dtype=torch.float32, device=dev)
        self.out = torch.empty((src_shape[0],), dtype=torch.int64, device=dev)
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):                       # lazy one-time set-up must not happen inside the capture
            for _ in range(max(warmup, 1)):
                predict(model, self.x, self.out)
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            predict(model, self.x, self.out)

    def predict(self, src: torch.Tensor) -> torch.Tensor:
        self.x.copy_(src, non_blocking=True)
        self.graph.replay()
        return self.out


@torch.no_grad()
def predict(model: _AMCBase, src: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """argmax class per frame (R/training/utils.py:311-317: model.eval(); model(x).max(1))."""
    model.eval()
    logits = model(src)
    if not logits.is_cuda:
        raise RuntimeError("predict needs the model on a CUDA device (no CPU fallback)")
    B, ncls = logits.shape
    if out is None:
        out = torch.empty(B, dtype=torch.int64, device=logits.device)
    elif out.dtype != torch.int64 or out.numel() != B or not out.is_contiguous() or out.device != logits.device:
        raise ValueError(f"out must be a contiguous int64 tensor of shape [{B}] on {logits.device}")
    _lib.check(_lib.lib.amc_argmax(B, ncls, logits.data_ptr(), out.data_ptr(),
                                   torch.cuda.current_stream(logits.device).cuda_stream), "amc_argmax")
    return out

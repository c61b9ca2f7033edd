"""Projected-gradient adversarial attacks on the fused path: FGSM and PGD in an L-inf or L2 ball.

``PGDAttack`` crafts adversarial frames for robustness evaluation (accuracy against the perturbation-to-signal ratio,
the usual second axis after clean accuracy per SNR in modulation classification) and for adversarial training
(``TrainStep(..., attack=...)``).  Every iteration is four library calls and no autograd: the forward with activations
kept (dropout off), ``amc_ce_loss``, the frozen-model backward to the input frames (``amc_model_bwd_ex`` without a
gradient blob) and ``amc_adv_step`` (ascent step + projection onto the ball around the clean frames).  All buffers are
cached per shape, so after the first call at a shape a call allocates nothing and never synchronises with the host,
and can be captured in a CUDA graph.

The attack works in whatever layout the model reads: model layout ([B, C, L] / [B, 1, H, W]), or dataset layout
([B, L, 2], ``set_raw_input``), in which case the perturbation is on the physical, un-normalised IQ samples.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Optional, Union

import torch

from . import _lib
from .modules import _AMCBase
from .trainer import _check_labels

_NORMS = {"linf": _lib.NORM_LINF, "l2": _lib.NORM_L2}


class PGDAttack:
    """``x_adv = PGDAttack(model, ...)(src, labels)``.

    norm         "linf" or "l2".
    eps          budget per frame: a float, or a device fp32 tensor [B] (its values are not checked: that would need a
                 host synchronisation).
    psr_db       budget relative to each clean frame x0 instead (pass exactly one of eps / psr_db): the perturbation-
                 to-signal ratio in dB.  L2: eps_b = 10^(psr/20) * ||x0_b||_2; L-inf: the same divided by sqrt(n), i.e.
                 relative to the frame's RMS amplitude.
    steps        ascent steps; step_frac (default 2.5 / steps, Madry et al.) is the step length as a fraction of eps.
    random_start start from a uniform (L-inf) or uniform-in-ball (L2) draw around x0, keyed by the model's dropout seed
                 (rank salt included) and call counter, or its device step counter under ``GraphTrainStep``.
    targeted     ``labels`` are targets: the steps descend the targets' cross-entropy.

    FGSM is ``steps=1, random_start=False, step_frac=1``; "fast" FGSM-RS training uses ``steps=1, step_frac=1.25``.
    The returned tensor has the shape, layout and device of ``src`` and is a buffer reused by the next call at that shape.
    The buffers of every shape the attack has seen are kept for the attack's lifetime (a CUDA graph that captured a call,
    e.g. ``GraphTrainStep(attack=...)``, keeps writing into them).  The budget is fixed at construction (``eps`` and
    ``psr_db`` are read-only); for a budget schedule pass a device tensor ``eps`` and update it in place, which eager calls
    and graph replays both read.
    """

    def __init__(self, model: _AMCBase, norm: str = "linf", eps: Union[float, torch.Tensor, None] = None,
                 psr_db: Optional[float] = None, steps: int = 10, step_frac: Optional[float] = None,
                 random_start: bool = True, targeted: bool = False):
        if not isinstance(model, _AMCBase):
            raise TypeError("PGDAttack needs a RawIQAMCTransformer or ViTAMCTransformer")
        if norm not in _NORMS:
            raise ValueError(f"norm must be one of {sorted(_NORMS)}, got {norm!r}")
        if (eps is None) == (psr_db is None):
            raise ValueError("pass exactly one of eps and psr_db")
        if isinstance(eps, torch.Tensor):
            if not eps.is_cuda or eps.dtype != torch.float32 or eps.dim() != 1 or not eps.is_contiguous():
                raise ValueError("an eps tensor must be a contiguous CUDA float32 tensor [B]")
        elif eps is not None:
            eps = float(eps)
            if not (math.isfinite(eps) and eps >= 0.0):
                raise ValueError(f"eps must be finite and >= 0, got {eps}")
        if psr_db is not None:
            psr_db = float(psr_db)
            if not math.isfinite(psr_db):
                raise ValueError(f"psr_db must be finite, got {psr_db}")
        if int(steps) != steps or steps < 1:
            raise ValueError(f"steps must be an integer >= 1, got {steps}")
        step_frac = 2.5 / steps if step_frac is None else float(step_frac)
        if not (math.isfinite(step_frac) and step_frac >= 0.0):
            raise ValueError(f"step_frac must be finite and >= 0, got {step_frac}")
        self.model = model
        self.norm = norm
        self._eps, self._psr_db = eps, psr_db
        self.steps, self.step_frac = int(steps), step_frac
        self.random_start, self.targeted = bool(random_start), bool(targeted)
        self._bufs = {}

    @property
    def eps(self):
        return self._eps

    @property
    def psr_db(self):
        return self._psr_db

    def __call__(self, src: torch.Tensor, labels: torch.Tensor) -> torch.Tensor:
        return self._run(src, labels, None)

    def _buffers(self, src: torch.Tensor, desc, ws: Optional[torch.Tensor]):
        core = self.model._core
        key = (tuple(src.shape), desc.dtype, src.device)
        b = self._bufs.get(key)
        if b is None:
            B, dev = desc.B, src.device
            b = dict(ws_bytes=_lib.workspace_bytes(desc),
                     logits=torch.empty((B, core.C), dtype=torch.float32, device=dev),
                     g=torch.empty_like(src), x=torch.empty_like(src),
                     eps=(torch.full((B,), self.eps, dtype=torch.float32, device=dev) if isinstance(self.eps, float)
                          else None if isinstance(self.eps, torch.Tensor)
                          else torch.empty(B, dtype=torch.float32, device=dev)))
            b["dlogits"] = torch.empty_like(b["logits"])
            self._bufs[key] = b
        if ws is None:
            if b.get("ws") is None:
                b["ws"] = torch.empty(b["ws_bytes"], dtype=torch.uint8, device=src.device)
            ws = b["ws"]
        else:
            # the caller's step workspace (TrainStep): amc_model_workspace does not depend on p_drop
            assert ws.numel() == b["ws_bytes"], (ws.numel(), b["ws_bytes"])
        return b, ws

    def _run(self, src: torch.Tensor, labels: torch.Tensor, ws: Optional[torch.Tensor]) -> torch.Tensor:
        core = self.model._core
        # training=1 keeps the activations the backward needs; dropout stays off whatever model.training is
        desc = core.make_desc(src, training=True, module_training=False)
        B = desc.B
        dev = src.device
        _check_labels(labels, B, dev)
        b, ws = self._buffers(src, desc, ws)
        if isinstance(self.eps, torch.Tensor):
            if self.eps.device != dev or self.eps.numel() != B:
                raise ValueError(f"eps must be a tensor of shape [{B}] on {dev}, got {tuple(self.eps.shape)} on "
                                 f"{self.eps.device}")
            eps = self.eps
        elif self.psr_db is not None:
            eps = b["eps"]
            n = src[0].numel()
            scale = 10.0 ** (self.psr_db / 20.0) / (math.sqrt(n) if self.norm == "linf" else 1.0)
            torch.linalg.vector_norm(src.view(B, -1), dim=1, out=eps)
            eps.mul_(scale)
        else:
            eps = b["eps"]
        x, g, logits, dlogits = b["x"], b["g"], b["logits"], b["dlogits"]
        n = src[0].numel()
        norm = _NORMS[self.norm]
        flat = self.model.flat_parameters()
        pos = core.pos_buffer()
        st = torch.cuda.current_stream(dev).cuda_stream
        lib = _lib.lib
        if self.random_start:
            _lib.check(lib.amc_adv_init(B, n, norm, src.data_ptr(), eps.data_ptr(), desc.seed, desc.offset,
                                        desc.step_counter, x.data_ptr(), st), "amc_adv_init")
        else:
            x.copy_(src)
        gscale = -1.0 if self.targeted else 1.0
        for _ in range(self.steps):
            _lib.check(lib.amc_model_fwd(C.byref(desc), x.data_ptr(), flat.data_ptr(), pos.data_ptr(), ws.data_ptr(),
                                         logits.data_ptr(), 0, st), "amc_model_fwd")
            _lib.check(lib.amc_ce_loss(B, core.C, logits.data_ptr(), labels.data_ptr(), 0.0, gscale, 1.0,
                                       dlogits.data_ptr(), 0, st), "amc_ce_loss")
            _lib.check(lib.amc_model_bwd_ex(C.byref(desc), x.data_ptr(), flat.data_ptr(), ws.data_ptr(),
                                            dlogits.data_ptr(), 0, 0, g.data_ptr(), 0, core.n_layers + 2, st),
                       "amc_model_bwd_ex")
            _lib.check(lib.amc_adv_step(B, n, norm, src.data_ptr(), g.data_ptr(), eps.data_ptr(), self.step_frac,
                                        x.data_ptr(), st), "amc_adv_step")
        return x

"""Host-side mirror of the reference's operator API for the encoder path.

The reference exposes the path as two ``nn.Module`` classes both called ``AMCTransformer``
(R/models/transformer_rawIQ.py:7-98, V/models/amc_transformer.py:5-31).  The classes here keep
their constructor kwargs, ``forward`` signatures, attribute names and ``state_dict`` keys, so
``train.py`` / ``evaluate.py`` / ``test_model.py`` of the reference run against them unchanged,
and ``torch.manual_seed(s)`` gives bit-identical initial weights (sub-modules are created in the
reference's order with the same torch constructors).

Behind that surface there is no PyTorch arithmetic: ``forward`` is one ``torch.autograd.Function``
that calls the sm_100a library through the C ABI (include/amc_b200.h).  All parameters are views
into one flat fp32 blob whose layout the library defines (``amc_param_layout``), which is what
lets w_q / w_k / w_v stay three ``state_dict`` tensors while the kernel reads one [3d, d] matrix.
"""
from __future__ import annotations

import ctypes as C
import operator
import os
from typing import List, Optional, Tuple

import numpy as np
import torch
from torch import nn

from . import _lib
from ._lib import AmcDesc

_DTYPES = {"fp32": _lib.F32, "float32": _lib.F32, "bf16": _lib.BF16, "bfloat16": _lib.BF16}


def default_compute_dtype() -> str:
    return os.environ.get("AMC_B200_DTYPE", "bf16")


# ----------------------------------------------------------------------------------------------
# leaf modules: parameter containers with the reference's names.  Their arithmetic lives in the
# fused kernels; calling them stand-alone is not part of the path (fails loudly, no fallback).
# ----------------------------------------------------------------------------------------------
class _ParamContainer(nn.Module):
    def forward(self, *a, **k):  # pragma: no cover - deliberate
        raise NotImplementedError(
            f"{type(self).__name__} is fused into the B200 encoder kernels; call AMCTransformer.forward / "
            "Encoder.forward (there is no unfused PyTorch fallback).")


class LayerNorm(_ParamContainer):
    """R/models/layers/layers_norm.py:4-19 (gamma/beta names, eps=1e-12)."""

    def __init__(self, d_model, eps=1e-12):
        super().__init__()
        self.gamma = nn.Parameter(torch.ones(d_model))
        self.beta = nn.Parameter(torch.zeros(d_model))
        self.eps = eps


class ScaleDotProductAttention(_ParamContainer):
    """R/models/layers/scale_dot_product_attention.py (no parameters)."""


class MultiHeadAttention(_ParamContainer):
    """R/models/layers/multi_head_attention.py:6-14."""

    def __init__(self, d_model, n_head):
        super().__init__()
        self.n_head = n_head
        self.attention = ScaleDotProductAttention()
        self.w_q = nn.Linear(d_model, d_model)
        self.w_k = nn.Linear(d_model, d_model)
        self.w_v = nn.Linear(d_model, d_model)
        self.w_concat = nn.Linear(d_model, d_model)


class PositionwiseFeedForward(_ParamContainer):
    """R/models/layers/position_wise_feed_forward.py:3-10 (ReLU, D1)."""

    def __init__(self, d_model, hidden, drop_prob=0.1):
        super().__init__()
        self.linear1 = nn.Linear(d_model, hidden)
        self.linear2 = nn.Linear(hidden, d_model)
        self.relu = nn.ReLU()
        self.dropout = nn.Dropout(p=drop_prob)


class EncoderLayer(_ParamContainer):
    """R/models/blocks/encoder_layer.py:7-16 (post-LN)."""

    def __init__(self, d_model, ffn_hidden, n_head, drop_prob):
        super().__init__()
        self.attention = MultiHeadAttention(d_model=d_model, n_head=n_head)
        self.norm1 = LayerNorm(d_model=d_model)
        self.dropout1 = nn.Dropout(p=drop_prob)
        self.ffn = PositionwiseFeedForward(d_model=d_model, hidden=ffn_hidden, drop_prob=drop_prob)
        self.norm2 = LayerNorm(d_model=d_model)
        self.dropout2 = nn.Dropout(p=drop_prob)


class SequenceEmbedding(_ParamContainer):
    """R/models/embedding/patch_embedding.py:5-45."""

    def __init__(self, in_channels=2, embedding_dim=256, method="conv1d", segment_size=None):
        super().__init__()
        self.in_channels, self.embedding_dim, self.method, self.segment_size = (
            in_channels, embedding_dim, method, segment_size)
        if method == "conv1d":
            self.projection = nn.Conv1d(in_channels, embedding_dim, kernel_size=1)
        elif method == "segment":
            if segment_size is None:
                raise ValueError("segment_size is required for 'segment' method")
            self.projection = nn.Conv1d(in_channels, embedding_dim, kernel_size=segment_size, stride=segment_size)
        else:
            raise ValueError(f"Unknown method: {method}. Use 'conv1d' or 'segment'")


class PatchEmbedding(_ParamContainer):
    """V/models/embedding/patch_embedding.py:3-9."""

    def __init__(self, in_channels, patch_size, embedding_dim):
        super().__init__()
        self.projection = nn.Conv2d(in_channels, embedding_dim, kernel_size=patch_size, stride=patch_size)


class PositionalEncoding(_ParamContainer):
    """Sinusoidal table as a persistent buffer ``encoding`` (D10): the raw-IQ and ViT trees build it
    with different float32 formulas (R/.../positional_encoding.py:28-47 vs V/.../positional_encoding.py:9-19);
    the kernels read the buffer and never regenerate it."""

    def __init__(self, d_model, max_len=5000, device="cpu", dropout=0.0, style="rawiq"):
        super().__init__()
        import math
        if style == "rawiq":
            encoding = torch.zeros(max_len, d_model)
            position = torch.arange(0, max_len, dtype=torch.float32).unsqueeze(1)
            div_term = torch.exp(torch.arange(0, d_model, 2, dtype=torch.float32) * -(math.log(10000.0) / d_model))
            encoding[:, 0::2] = torch.sin(position * div_term)
            encoding[:, 1::2] = torch.cos(position * div_term)
        else:
            encoding = torch.zeros(max_len, d_model)
            pos = torch.arange(0, max_len).float().unsqueeze(dim=1)
            _2i = torch.arange(0, d_model, step=2).float()
            denominator = torch.pow(10000.0, _2i / d_model)
            encoding[:, 0::2] = torch.sin(pos / denominator)
            encoding[:, 1::2] = torch.cos(pos / denominator)
        self.register_buffer("encoding", encoding)
        self.dropout = nn.Dropout(p=dropout) if dropout > 0 else None


# ----------------------------------------------------------------------------------------------
# the autograd boundary
# ----------------------------------------------------------------------------------------------
class _EncoderPathFn(torch.autograd.Function):
    """forward = amc_model_fwd, backward = amc_model_bwd_ex.  ``params`` are passed only so autograd
    routes gradients to them; the kernels read the flat blob they are views of.  The input gradient (``src.grad``,
    saliency maps, adversarial examples) comes out of the same backward; when no parameter needs a gradient (a frozen
    model) the backward runs the data-gradient chain alone, without weight-gradient GEMMs or a gradient blob."""

    @staticmethod
    def forward(ctx, owner, src, want_logits, need_grad, *params):
        core = owner._core
        desc = core.make_desc(src, training=need_grad, module_training=owner.training)
        B = desc.B
        dev = src.device
        ws = torch.empty(_lib.workspace_bytes(desc), dtype=torch.uint8, device=dev)
        logits = torch.empty((B, core.C), dtype=torch.float32, device=dev) if want_logits else None
        enc = None if want_logits else torch.empty((B, core.layout.T, core.d), dtype=torch.float32, device=dev)
        stream = torch.cuda.current_stream(dev).cuda_stream
        _lib.check(_lib.lib.amc_model_fwd(C.byref(desc), src.data_ptr(), core.flat.data_ptr(),
                                          core.pos_buffer().data_ptr(), ws.data_ptr(), _lib.ptr(logits),
                                          _lib.ptr(enc), stream), "amc_model_fwd")
        if need_grad:
            ctx.owner, ctx.desc, ctx.ws, ctx.src, ctx.want_logits = owner, desc, ws, src, want_logits
        return logits if want_logits else enc

    @staticmethod
    def backward(ctx, dout):
        core = ctx.owner._core
        dout = dout.contiguous().float()
        # a partially frozen model still gets every parameter gradient; only a fully frozen one skips them
        want_params = any(ctx.needs_input_grad[4:])
        grads = torch.zeros(core.layout.total, dtype=torch.float32, device=dout.device) if want_params else None
        dsrc = torch.empty_like(ctx.src) if ctx.needs_input_grad[1] else None
        stream = torch.cuda.current_stream(dout.device).cuda_stream
        dl = dout.data_ptr() if ctx.want_logits else 0
        de = 0 if ctx.want_logits else dout.data_ptr()
        _lib.check(_lib.lib.amc_model_bwd_ex(C.byref(ctx.desc), ctx.src.data_ptr(), core.flat.data_ptr(),
                                             ctx.ws.data_ptr(), dl, de, _lib.ptr(grads), _lib.ptr(dsrc), 0,
                                             core.n_layers + 2, stream), "amc_model_bwd_ex")
        ctx.ws = None
        views = [grads[o:o + n].view(shape) for (o, n, shape) in core.slots] if want_params else [None] * len(core.slots)
        return (None, dsrc, None, None, *views)


class _Core:
    """Flat-blob bookkeeping shared by the two model classes."""

    def __init__(self, owner: nn.Module, kind: int, fields: dict, drop_prob: float, compute_dtype: Optional[str]):
        self.kind = kind
        self.fields = fields
        self.drop_prob = float(drop_prob)
        self.compute_dtype = compute_dtype or default_compute_dtype()
        if self.compute_dtype not in _DTYPES:
            raise ValueError(f"compute_dtype must be one of {sorted(_DTYPES)}")
        self.d, self.C, self.n_layers = fields["d"], fields["C"], fields["n_layers"]
        self.layout = _lib.param_layout(self._desc(B=0, dtype=_lib.F32))
        self.flat: Optional[torch.Tensor] = None
        self.slots: List[Tuple[int, int, torch.Size]] = []
        self.params: List[nn.Parameter] = []
        self.calls = 0
        self.seed = int(torch.initial_seed()) & 0xFFFFFFFFFFFF
        self.norm_stats = (0.0, 1.0, 0.0, 1.0)
        self.input_layout = _lib.INPUT_MODEL

    def _desc(self, B: int, dtype: int, training: bool = False, p_drop: float = 0.0) -> AmcDesc:
        f = self.fields
        d = AmcDesc()
        d.kind, d.dtype, d.B = self.kind, dtype, B
        d.d, d.h, d.F, d.C, d.n_layers = f["d"], f["h"], f["F"], f["C"], f["n_layers"]
        d.in_ch, d.seq_len, d.seg = f.get("in_ch", 1), f.get("seq_len", 0), f.get("seg", 1)
        d.img_h, d.img_w, d.patch = f.get("img_h", 0), f.get("img_w", 0), f.get("patch", 1)
        d.has_cls, d.head_ln = f["has_cls"], f["head_ln"]
        d.input_layout = getattr(self, "input_layout", _lib.INPUT_MODEL)
        d.training = 1 if training else 0
        d.p_drop = p_drop
        d.ln_eps, d.head_ln_eps = 1e-12, 1e-5
        ns = getattr(self, "norm_stats", (0.0, 1.0, 0.0, 1.0))
        for i in range(4):
            d.norm[i] = ns[i]
        # dropout key: (seed, per-call counter); data-parallel ranks fold their rank in (TrainStep sets rank_salt) so that
        # the shards do not share one mask
        d.seed = (getattr(self, "seed", 0) ^ (getattr(self, "rank_salt", 0) * 0x9E3779B97F4A7C15)) & 0xFFFFFFFFFFFFFFFF
        d.offset = getattr(self, "calls", 0)
        ctr = getattr(self, "step_counter", None)          # device int32 tensor (CUDA-graph training): offset lives there
        if ctr is not None:
            d.offset = 0
            d.step_counter = ctr.data_ptr()
        return d

    # ---- parameter blob ---------------------------------------------------------------------
    def bind(self, owner: nn.Module) -> None:
        """Order the owner's parameters by blob offset and remember (offset, numel, shape)."""
        L, enc = self.layout, owner.encoder
        emb = enc.sequence_embedding if self.kind == _lib.KIND_RAWIQ else enc.patch_embedding
        table = [(L.emb_w, emb.projection.weight), (L.emb_b, emb.projection.bias)]
        if L.cls >= 0:
            table.append((L.cls, enc.cls_token))
        for i, lay in enumerate(enc.layers):
            b = L.layer0 + i * L.layer_stride
            a, f = lay.attention, lay.ffn
            table += [(b + L.wq, a.w_q.weight), (b + L.wk, a.w_k.weight), (b + L.wv, a.w_v.weight),
                      (b + L.bq, a.w_q.bias), (b + L.bk, a.w_k.bias), (b + L.bv, a.w_v.bias),
                      (b + L.wo, a.w_concat.weight), (b + L.bo, a.w_concat.bias),
                      (b + L.g1, lay.norm1.gamma), (b + L.be1, lay.norm1.beta),
                      (b + L.w1, f.linear1.weight), (b + L.b1, f.linear1.bias),
                      (b + L.w2, f.linear2.weight), (b + L.b2, f.linear2.bias),
                      (b + L.g2, lay.norm2.gamma), (b + L.be2, lay.norm2.beta)]
        if L.head_ln_w >= 0:
            table += [(L.head_ln_w, owner.mlp_head[0].weight), (L.head_ln_b, owner.mlp_head[0].bias),
                      (L.head_w, owner.mlp_head[1].weight), (L.head_b, owner.mlp_head[1].bias)]
        else:
            table += [(L.head_w, owner.mlp_head.weight), (L.head_b, owner.mlp_head.bias)]
        self.params = [p for _, p in table]
        self.slots = [(int(o), p.numel(), p.shape) for o, p in table]
        assert len({id(p) for p in self.params}) == len(list(owner.parameters())), "unbound parameter"
        self.owner_pos = enc.positional_encoding
        self.flatten()

    def is_flat(self) -> bool:
        if self.flat is None:
            return False
        base = self.flat.data_ptr()
        return all(p.data_ptr() == base + 4 * o and p.device == self.flat.device and p.dtype == torch.float32
                   for p, (o, _, _) in zip(self.params, self.slots))

    def flatten(self) -> None:
        """(Re)build the blob on the parameters' current device and make every parameter a view of it.
        Called after construction and whenever .to()/.cuda()/load_state_dict replaced storage."""
        dev = self.params[0].device
        flat = torch.zeros(self.layout.total, dtype=torch.float32, device=dev)
        with torch.no_grad():
            for p, (o, n, shape) in zip(self.params, self.slots):
                flat[o:o + n].copy_(p.detach().reshape(-1).to(device=dev, dtype=torch.float32))
                p.data = flat[o:o + n].view(shape)
        self.flat = flat

    def pos_buffer(self) -> torch.Tensor:
        enc = self.owner_pos.encoding
        if enc.dtype != torch.float32 or not enc.is_contiguous():
            raise RuntimeError("positional encoding buffer must be contiguous float32")
        return enc

    # ---- per-call description -----------------------------------------------------------------
    def make_desc(self, src: torch.Tensor, training: bool, module_training: bool) -> AmcDesc:
        if not src.is_cuda:
            raise RuntimeError("the B200 encoder path needs CUDA tensors (there is no CPU fallback); "
                               f"got input on {src.device}")
        if src.dtype != torch.float32 or not src.is_contiguous():
            raise RuntimeError("input must be a contiguous float32 tensor")
        if not self.is_flat() or self.flat.device != src.device:
            if self.params[0].device != src.device:
                raise RuntimeError(f"model parameters are on {self.params[0].device}, input on {src.device}")
            self.flatten()
        f = self.fields
        if self.input_layout == _lib.INPUT_RAW:
            n = f["seq_len"] if self.kind == _lib.KIND_RAWIQ else f["img_h"] * f["img_w"] // 2
            ok = src.dim() == 3 and tuple(src.shape[1:]) == (n, 2)
            expect = f"[B, {n}, 2]"
        elif self.kind == _lib.KIND_RAWIQ:
            ok = src.dim() == 3 and tuple(src.shape[1:]) == (f["in_ch"], f["seq_len"])
            expect = f"[B, {f['in_ch']}, {f['seq_len']}]"
        else:
            ok = src.dim() == 4 and tuple(src.shape[1:]) == (f["in_ch"], f["img_h"], f["img_w"])
            expect = f"[B, {f['in_ch']}, {f['img_h']}, {f['img_w']}]"
        if not ok:
            raise RuntimeError(f"expected input of shape {expect}, got {tuple(src.shape)}")
        T = self.layout.T
        if T > self.pos_buffer().size(0):  # R/models/embedding/positional_encoding.py:65-69
            raise ValueError(f"Sequence length {T} exceeds maximum length {self.pos_buffer().size(0)}. "
                             "Increase max_len parameter.")
        self.calls += 1
        p = self.drop_prob if module_training else 0.0
        return self._desc(B=int(src.shape[0]), dtype=_DTYPES[self.compute_dtype], training=training, p_drop=p)


class _AMCBase(nn.Module):
    _core: _Core

    def _finish_init(self, kind, fields, drop_prob, compute_dtype):
        object.__setattr__(self, "_core", _Core(self, kind, fields, drop_prob, compute_dtype))
        self._core.bind(self)

    # .to()/.cuda()/.float() replace parameter storage: rebuild the blob afterwards
    def _apply(self, fn, *a, **k):
        out = super()._apply(fn, *a, **k)
        if getattr(self, "_core", None) is not None and self._core.params:
            self._core.flatten()
        return out

    def load_state_dict(self, *a, **k):
        out = super().load_state_dict(*a, **k)
        if not self._core.is_flat():
            self._core.flatten()
        return out

    @property
    def compute_dtype(self) -> str:
        return self._core.compute_dtype

    def set_compute_dtype(self, name: str) -> "_AMCBase":
        if name not in _DTYPES:
            raise ValueError(f"compute_dtype must be one of {sorted(_DTYPES)}")
        self._core.compute_dtype = name
        return self

    def set_raw_input(self, norm_stats=None) -> "_AMCBase":
        """Feed dataset-layout frames [B, L, 2] (interleaved I/Q, un-normalised) instead of the model layout;
        the dataset z-score (i_mean, i_std, q_mean, q_std) and the framing are fused into the front end
        (R/dataloader/dataset.py:215-222, V/dataloader/dataset.py:211-224).  ``None`` restores model layout."""
        if norm_stats is None:
            self._core.input_layout = _lib.INPUT_MODEL
        else:
            self._core.input_layout = _lib.INPUT_RAW
            self._core.norm_stats = tuple(float(norm_stats[k]) for k in ("i_mean", "i_std", "q_mean", "q_std"))
        return self

    def flat_parameters(self) -> torch.Tensor:
        if not self._core.is_flat():
            self._core.flatten()
        return self._core.flat

    @torch.no_grad()
    def _attention(self, src, mask: int, want_rollout: bool):
        core = self._core
        # training=1 keeps every layer's qkv in the workspace; module_training=False turns dropout off
        desc = core.make_desc(src, training=True, module_training=False)
        dev = src.device
        T, h = core.layout.T, core.fields["h"]
        ws = torch.empty(_lib.workspace_bytes(desc), dtype=torch.uint8, device=dev)
        probs = torch.empty((bin(mask).count("1"), desc.B, h, T, T), dtype=torch.float32, device=dev) if mask else None
        roll = torch.empty((desc.B, T), dtype=torch.float32, device=dev) if want_rollout else None
        _lib.check(_lib.lib.amc_model_attention(C.byref(desc), src.data_ptr(), core.flat.data_ptr(),
                                                core.pos_buffer().data_ptr(), ws.data_ptr(), mask, _lib.ptr(probs),
                                                _lib.ptr(roll), torch.cuda.current_stream(dev).cuda_stream),
                   "amc_model_attention")
        return probs, roll

    def attention_maps(self, src, layers=None) -> List[torch.Tensor]:
        """The attention probabilities softmax(q k^T / sqrt(d_head)) of the requested encoder layers: the ``score`` that
        the reference's ``ScaleDotProductAttention`` returns (R/models/layers/scale_dot_product_attention.py:26-39).

        ``src`` is what ``forward`` takes (either input layout, see ``set_raw_input``).  ``layers`` is a sequence of
        layer indices in ``[0, n_layers)`` (any integer type), or ``None`` for all of them.  Returns one fp32
        tensor ``[B, n_head, T, T]`` per requested layer, in the order requested (a repeated layer is a separate copy); T counts the CLS token when the model has one.

        Runs under ``torch.no_grad()`` with dropout off whatever ``self.training`` is, in the model's compute dtype.
        The maps take ``4 B h T^2`` bytes per layer (3.3 GB for all 6 layers at B = 1024, T = 129, h = 8)."""
        n = self._core.n_layers
        idx = []
        for l in (range(n) if layers is None else layers):
            try:
                i = operator.index(l)             # any integer type (int, numpy / torch integer scalars), not bool
            except TypeError:
                i = None
            if isinstance(l, (bool, np.bool_)) or i is None or not 0 <= i < min(n, 32):
                raise ValueError(f"layers must hold encoder layer indices in [0, {min(n, 32)}), got {l!r}")
            idx.append(i)
        if not idx:
            raise ValueError("layers is empty")
        uniq = sorted(set(idx))
        probs, _ = self._attention(src, sum(1 << l for l in uniq), False)
        # a layer asked for twice comes back as two tensors that do not share storage
        seen = set()
        out = []
        for l in idx:
            t = probs[uniq.index(l)]
            out.append(t.clone() if l in seen else t)
            seen.add(l)
        return out

    def attention_rollout(self, src) -> torch.Tensor:
        """Attention rollout (Abnar & Zuidema, 2020) of the whole encoder: ``u^T A_{L-1} ... A_0`` with
        ``A_l = 0.5 * mean_heads(P_l) + 0.5 * I`` (the residual path counted as half of each layer), and ``u`` the head's
        read-out of the top layer: the CLS row (``e_0``) or, for mean pooling, ``1/T`` on every token.  Returns fp32
        ``[B, T]``; every row is non-negative and sums to 1.  Computed on the device without materialising any ``P``.

        Columns (S = segment_size, p = patch_size):
          * column 0 is the CLS token (when the model has one);
          * raw-IQ ``embedding_type='segment'``: column t >= 1 covers samples ``[(t-1)*S, t*S)`` of both I and Q;
          * raw-IQ ``embedding_type='conv1d'``: column t >= 1 is sample t - 1;
          * ViT: column t >= 1 is patch ``divmod(t-1, 64 // p)`` (patch row, patch column) of the ``[1, 32, 64]`` image,
            whose rows 0-15 hold I and rows 16-31 hold Q;
          * without a CLS token (mean pooling): column t is token t (the same segment / sample without the shift).

        ``src`` is what ``forward`` takes (either input layout).  Runs under ``torch.no_grad()`` with dropout off
        whatever ``self.training`` is, in the model's compute dtype."""
        _, roll = self._attention(src, 0, True)
        return roll

    @torch.no_grad()
    def attention_relevance(self, src, target=None) -> torch.Tensor:
        """Class-specific attention relevance: the gradient-weighted rollout of Chefer, Gur & Wolf, "Generic
        Attention-model Explainability" (ICCV 2021).  Where ``attention_rollout`` gives one map per frame, this answers
        "which tokens made the model score class t?".

        ``r = u^T (I + A_{L-1}) ... (I + A_0)`` with ``A_l = mean_heads(relu(dy_t/dP_l * P_l))``: ``P_l`` the attention
        probabilities of layer l, ``y_t`` the logit of the target class (not the loss and not the softmax), and ``u`` the
        head's read-out of the top layer, ``e_0`` for a CLS model or ``1/T`` on every token for mean pooling.  The
        gradient comes from a frozen backward on the device; no ``[B, h, T, T]`` tensor is materialised.

        ``target`` is ``None`` (each frame's predicted class, the first maximum of its logits) or a contiguous int64
        CUDA tensor ``[B]`` on the model's device with values in ``[0, num_classes)``; anything else raises
        ``ValueError``.  Returns fp32 ``[B, T]``; columns as in ``attention_rollout`` (column 0 is the CLS token when the
        model has one).  Every entry is non-negative and ``r >= u`` elementwise, so ``r[:, 0] >= 1`` for CLS models.
        Rows are not normalised: divide by the row sum, or subtract ``u``, to compare frames.

        ``src`` is what ``forward`` takes (either input layout).  Runs under ``torch.no_grad()`` with dropout off whatever
        ``self.training`` is, in the model's compute dtype; parameters, their ``.grad`` and ``training`` are left as they
        are.  Memory: the training-mode workspace of the batch plus ``[B, T]`` and ``[B, num_classes]`` fp32."""
        core = self._core
        self._check_target(src, target)
        # training=1 keeps every layer's activations for the backward; module_training=False turns dropout off
        desc = core.make_desc(src, training=True, module_training=False)
        dev = src.device
        ws = torch.empty(_lib.workspace_bytes(desc), dtype=torch.uint8, device=dev)
        logits = torch.empty((desc.B, core.C), dtype=torch.float32, device=dev)
        rel = torch.empty((desc.B, core.layout.T), dtype=torch.float32, device=dev)
        _lib.check(_lib.lib.amc_model_relevance(C.byref(desc), src.data_ptr(), core.flat.data_ptr(),
                                                core.pos_buffer().data_ptr(), ws.data_ptr(), _lib.ptr(target),
                                                logits.data_ptr(), rel.data_ptr(),
                                                torch.cuda.current_stream(dev).cuda_stream),
                   "amc_model_relevance")
        return rel

    def _check_target(self, src, target) -> None:
        """ValueError unless ``target`` is None or a contiguous int64 tensor [B] on the model's device with values in
        [0, num_classes)."""
        if target is None:
            return
        core = self._core
        B = int(src.shape[0]) if src.dim() >= 1 else -1
        if not isinstance(target, torch.Tensor):
            raise ValueError(f"target must be None or an int64 CUDA tensor [B], got {type(target).__name__}")
        if target.dtype != torch.int64 or target.dim() != 1 or target.shape[0] != B or not target.is_contiguous():
            raise ValueError(f"target must be a contiguous int64 tensor of shape [{B}], got {target.dtype} "
                             f"{tuple(target.shape)}")
        if target.device != core.params[0].device:
            raise ValueError(f"target is on {target.device}, the model on {core.params[0].device}")
        if B > 0:
            lo, hi = torch.aminmax(target)
            lo, hi = int(lo), int(hi)
            if lo < 0 or hi >= core.C:
                raise ValueError(f"target values must lie in [0, {core.C}), got [{lo}, {hi}]")

    # token rows (frames x tokens per frame) per device pass of integrated_gradients when internal_batch_size is None:
    # measured at 256 frames of raw-IQ seg16 (T = 65), doubling a pass from 2^18 to 2^19 rows gains 3 % for twice the
    # workspace (DESIGN §8.1)
    IG_TOKEN_BUDGET = 1 << 18

    @torch.no_grad()
    def integrated_gradients(self, src, target=None, baseline=None, steps=32, internal_batch_size=None,
                             return_delta=False):
        """Integrated Gradients (Sundararajan, Taly & Yan, "Axiomatic Attribution for Deep Networks", ICML 2017) of
        the target-class logit w.r.t. every input sample:

            IG_t(x) = (x - x') * integral_0^1 dy_t/dx (x' + a (x - x')) da

        with ``y_t`` the logit of class t (not the loss and not the softmax) and ``x'`` the baseline.  The integral is
        the ``steps``-point Gauss-Legendre rule on [0, 1].  Completeness: ``attr[b].sum()`` approaches
        ``y_t(x_b) - y_t(x'_b)`` as ``steps`` grows.

        ``src`` is what ``forward`` takes, in either input layout; after ``set_raw_input`` the attribution is w.r.t. the
        un-normalised dataset frames, as ``src.grad`` is.  ``baseline`` is ``None`` (zeros in that layout) or an fp32
        tensor of the shape of ``src`` on its device.  ``target`` is ``None`` (each frame's predicted class at ``x``,
        the first maximum of its logits, from the same forward) or a contiguous int64 CUDA tensor ``[B]`` with values
        in ``[0, num_classes)``.  Returns fp32 with the shape and layout of ``src``; with ``return_delta=True`` also
        ``delta`` fp32 ``[B]``, ``attr[b].sum() - (y_t(x_b) - y_t(x'_b))``, the convergence check.

        All on the device: one forward of ``[x; x']``, then chunks of path points, each a blend of the two endpoint
        embeddings (the front end is affine in ``src``), the layers, the seed ``w_k e_t`` and the frozen backward down
        to the embedding; their gradients are summed in fp32 in a fixed order (repeated calls are bit-identical) and
        the embedding dgrad and the scatter times ``x - x'`` run once.

        ``internal_batch_size`` caps the frames per device pass: a pass takes at most
        ``max(1, internal_batch_size // B)`` path points, ``n_c * B`` frames (never fewer than one point's B frames),
        and the points are spread evenly over the fewest passes.  ``None`` caps a pass at ``IG_TOKEN_BUDGET`` = 2^18
        token rows (frames x tokens per frame), so large batches run one point per pass.  Memory: the training-mode
        workspace of ``max(2, n_c) * B`` frames plus fp32 copies of ``[x; x']``, of both endpoints' embeddings
        ``[2B, T, d]`` and of the gradient sum: 7.1 GB for raw-IQ seg16 d128 L6 at B = 256 in bf16 (11 points a
        pass), 17 GB for SPS-1 seg8 d256 L6 at B = 1024 (DESIGN §8.1).  Results for different
        ``internal_batch_size`` agree to fp32 summation order.

        Runs under ``torch.no_grad()`` with dropout off whatever ``self.training`` is, in the model's compute dtype;
        parameters, their ``.grad`` and ``training`` are left as they are.  Raises ``ValueError`` for a bad
        ``target``, ``baseline``, ``steps < 1`` or ``internal_batch_size < 1``."""
        core = self._core
        self._check_target(src, target)
        if baseline is None:
            baseline = torch.zeros_like(src)
        else:
            if not isinstance(baseline, torch.Tensor):
                raise ValueError(f"baseline must be None or a tensor, got {type(baseline).__name__}")
            if baseline.shape != src.shape or baseline.dtype != torch.float32 or baseline.device != src.device:
                raise ValueError(f"baseline must be float32 {tuple(src.shape)} on {src.device}, got {baseline.dtype} "
                                 f"{tuple(baseline.shape)} on {baseline.device}")
            baseline = baseline.contiguous()
        steps = self._positive_int("steps", steps)
        ibs = None if internal_batch_size is None else self._positive_int("internal_batch_size", internal_batch_size)
        desc = core.make_desc(src, training=True, module_training=False)
        B, dev = desc.B, src.device
        per_pass = max(1, ibs // max(B, 1) if internal_batch_size is not None else
                       self.IG_TOKEN_BUDGET // max(B * core.layout.T, 1))
        passes = -(-steps // per_pass)
        chunk = -(-steps // passes)
        x, w = np.polynomial.legendre.leggauss(steps)
        alpha = torch.tensor((x + 1.0) / 2.0, dtype=torch.float32, device=dev)
        weight = torch.tensor(w / 2.0, dtype=torch.float32, device=dev)
        ws = torch.empty(_lib.ig_workspace_bytes(desc, chunk), dtype=torch.uint8, device=dev)
        logits = torch.empty((2, B, core.C), dtype=torch.float32, device=dev)
        attr = torch.empty_like(src)
        stream = torch.cuda.current_stream(dev).cuda_stream
        _lib.check(_lib.lib.amc_model_integrated_gradients(C.byref(desc), src.data_ptr(), baseline.data_ptr(),
                                                           core.flat.data_ptr(), core.pos_buffer().data_ptr(),
                                                           ws.data_ptr(), _lib.ptr(target), steps, alpha.data_ptr(),
                                                           weight.data_ptr(), chunk, logits.data_ptr(),
                                                           attr.data_ptr(), stream),
                   "amc_model_integrated_gradients")
        if not return_delta:
            return attr
        t = target
        if t is None:
            t = torch.empty(B, dtype=torch.int64, device=dev)
            _lib.check(_lib.lib.amc_argmax(B, core.C, logits.data_ptr(), t.data_ptr(), stream), "amc_argmax")
        y = logits.gather(2, t.view(1, B, 1).expand(2, B, 1)).squeeze(2).double()
        delta = attr.reshape(B, -1).double().sum(1) - (y[0] - y[1])
        return attr, delta.float()

    @staticmethod
    def _positive_int(name, v) -> int:
        try:
            i = operator.index(v)
        except TypeError:
            i = None
        if isinstance(v, (bool, np.bool_)) or i is None or i < 1:
            raise ValueError(f"{name} must be an integer >= 1, got {v!r}")
        return i

    def _run(self, src, want_logits):
        # grad mode is switched off inside Function.forward, so decide here whether to keep activations
        need_grad = torch.is_grad_enabled() and (src.requires_grad or any(p.requires_grad for p in self._core.params))
        return _EncoderPathFn.apply(self, src, want_logits, need_grad, *self._core.params)


class _EncoderBase(nn.Module):
    """``model.encoder(src)`` -> [B, T, d] (R/models/encoder.py:86-117, V/models/encoder.py:34-53)."""

    def _set_owner(self, owner):
        object.__setattr__(self, "_owner", owner)

    def forward(self, src, src_mask=None):
        if src_mask is not None:
            raise NotImplementedError("src_mask is never used by the reference call paths (SURVEY §3.2); "
                                      "the fused attention kernel has no mask input")
        return self._owner._run(src, False)


# ----------------------------------------------------------------------------------------------
# raw-IQ model
# ----------------------------------------------------------------------------------------------
class RawIQEncoder(_EncoderBase):
    """R/models/encoder.py:16-84."""

    def __init__(self, in_channels, seq_length, d_model, ffn_hidden, n_head, n_layers, drop_prob, device,
                 use_cls_token=True, embedding_type="conv1d", segment_size=64):
        super().__init__()
        self.device = device
        self.use_cls_token = use_cls_token
        self.embedding_type = embedding_type
        if embedding_type == "conv1d":
            self.sequence_embedding = SequenceEmbedding(in_channels=in_channels, embedding_dim=d_model,
                                                        method="conv1d")
            num_tokens = seq_length
        elif embedding_type == "segment":
            if seq_length % segment_size != 0:
                raise ValueError(f"seq_length ({seq_length}) must be divisible by segment_size ({segment_size})")
            self.sequence_embedding = SequenceEmbedding(in_channels=in_channels, embedding_dim=d_model,
                                                        segment_size=segment_size, method="segment")
            num_tokens = seq_length // segment_size
        else:
            raise ValueError(f"Unknown embedding_type: {embedding_type}")
        max_len = num_tokens + (1 if use_cls_token else 0)
        self.positional_encoding = PositionalEncoding(d_model=d_model, max_len=max_len, device=device, dropout=0.0,
                                                      style="rawiq")
        if use_cls_token:
            self.cls_token = nn.Parameter(torch.randn(1, 1, d_model))
        self.layers = nn.ModuleList([EncoderLayer(d_model=d_model, ffn_hidden=ffn_hidden, n_head=n_head,
                                                  drop_prob=drop_prob) for _ in range(n_layers)])
        self.dropout = nn.Dropout(p=drop_prob)

    def get_cls_token_output(self, src, src_mask=None):
        if not self.use_cls_token:
            raise ValueError("CLS token is not enabled. Set use_cls_token=True")
        return self.forward(src, src_mask)[:, 0, :]

    def get_sequence_output(self, src, src_mask=None):
        x = self.forward(src, src_mask)
        return x[:, 1:, :] if self.use_cls_token else x


class RawIQAMCTransformer(_AMCBase):
    """Drop-in for R/models/transformer_rawIQ.py::AMCTransformer."""

    def __init__(self, in_channels, seq_length, num_classes, d_model, n_head, n_layers, ffn_hidden, drop_prob,
                 device, use_cls_token=True, embedding_type="segment", segment_size=64, compute_dtype=None):
        super().__init__()
        self.use_cls_token = use_cls_token
        self.d_model = d_model
        if d_model % n_head != 0:  # R/training/train.py:132-133
            raise ValueError(f"D_MODEL ({d_model}) must be divisible by N_HEAD ({n_head})")
        self.encoder = RawIQEncoder(in_channels=in_channels, seq_length=seq_length, d_model=d_model, n_head=n_head,
                                    ffn_hidden=ffn_hidden, drop_prob=drop_prob, n_layers=n_layers, device=device,
                                    use_cls_token=use_cls_token, embedding_type=embedding_type,
                                    segment_size=segment_size)
        self.mlp_head = nn.Sequential(nn.LayerNorm(d_model), nn.Linear(d_model, num_classes))
        fields = dict(d=d_model, h=n_head, F=ffn_hidden, C=num_classes, n_layers=n_layers, in_ch=in_channels,
                      seq_len=seq_length, seg=(1 if embedding_type == "conv1d" else segment_size),
                      has_cls=1 if use_cls_token else 0, head_ln=1)
        self._finish_init(_lib.KIND_RAWIQ, fields, drop_prob, compute_dtype)
        self.encoder._set_owner(self)
        if device is not None and str(device) != "cpu":
            self.to(device)

    def forward(self, src):
        """src [B, in_channels, seq_length] fp32 -> logits [B, num_classes] (transformer_rawIQ.py:72-98)."""
        return self._run(src, True)


# ----------------------------------------------------------------------------------------------
# ViT model
# ----------------------------------------------------------------------------------------------
class ViTEncoder(_EncoderBase):
    """V/models/encoder.py:11-32."""

    def __init__(self, in_channels, img_size_h, img_size_w, patch_size, d_model, ffn_hidden, n_head, n_layers,
                 drop_prob, device):
        super().__init__()
        self.device = device
        self.patch_embedding = PatchEmbedding(in_channels=in_channels, patch_size=patch_size, embedding_dim=d_model)
        num_patches = (img_size_h // patch_size) * (img_size_w // patch_size)
        self.positional_encoding = PositionalEncoding(d_model=d_model, max_len=num_patches + 1, device=device,
                                                      style="vit")
        self.cls_token = nn.Parameter(torch.randn(1, 1, d_model))
        self.layers = nn.ModuleList([EncoderLayer(d_model=d_model, ffn_hidden=ffn_hidden, n_head=n_head,
                                                  drop_prob=drop_prob) for _ in range(n_layers)])
        self.dropout = nn.Dropout(p=drop_prob)


class ViTAMCTransformer(_AMCBase):
    """Drop-in for V/models/amc_transformer.py::AMCTransformer."""

    def __init__(self, in_channels, img_size_h, img_size_w, patch_size, num_classes, d_model, n_head, n_layers,
                 ffn_hidden, drop_prob, device, compute_dtype=None):
        super().__init__()
        if d_model % n_head != 0:
            raise ValueError(f"D_MODEL ({d_model}) must be divisible by N_HEAD ({n_head})")
        self.encoder = ViTEncoder(in_channels=in_channels, img_size_h=img_size_h, img_size_w=img_size_w,
                                  patch_size=patch_size, d_model=d_model, n_head=n_head, ffn_hidden=ffn_hidden,
                                  drop_prob=drop_prob, n_layers=n_layers, device=device)
        self.mlp_head = nn.Linear(d_model, num_classes)
        fields = dict(d=d_model, h=n_head, F=ffn_hidden, C=num_classes, n_layers=n_layers, in_ch=in_channels,
                      img_h=img_size_h, img_w=img_size_w, patch=patch_size, has_cls=1, head_ln=0)
        self._finish_init(_lib.KIND_VIT, fields, drop_prob, compute_dtype)
        self.encoder._set_owner(self)
        if device is not None and str(device) != "cpu":
            self.to(device)

    def forward(self, src):
        """src [B, in_channels, H, W] fp32 -> logits [B, num_classes] (amc_transformer.py:26-31)."""
        return self._run(src, True)

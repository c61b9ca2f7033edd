"""The kernels around the encoder, element by element against float64 references of the same operation
(tests/isolated_ref.py): the embedding front end and its backward, dropout at the positional-encoding site, the
classifier head, and the cross-entropy, argmax, clip + AdamW, IQ-statistics and generic-epilogue GEMM calls.

A model with n_layers = 0 is a valid description: its forward returns the front end's x0 as enc_out and the head's
logits on it, and its backward runs only the head and the embedding backward.  The bf16 references use the operands
the kernels round (bf16_rne), so what remains is fp32 accumulation and every bound is derived from that arithmetic
(see the docstrings of isolated_ref.py).  Every check is per element and prints its worst error-to-bound ratio."""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

import isolated_ref as R  # noqa: E402
from oracle import amc_oracle as O  # noqa: E402

from vit_vs_raw_iq_b200 import _lib  # noqa: E402

DEV = "cuda:0"
STATS = {"i_mean": 0.03, "i_std": 0.8, "q_mean": -0.02, "q_std": 1.3}
U = R.U


def stream():
    return torch.cuda.current_stream().cuda_stream


def cuda(a, dtype=torch.float32):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV, dtype)


def check(what, got, ref, bound):
    """|got - ref| <= bound element by element (a zero bound demands exact equality)."""
    got = np.asarray(got, dtype=np.float64)
    ref = np.asarray(ref, dtype=np.float64)
    bound = np.broadcast_to(np.asarray(bound, dtype=np.float64), ref.shape)
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    err = np.abs(got - ref)
    bad = ~(err <= bound)
    pos = bound > 0
    worst = float((err[pos] / bound[pos]).max()) if pos.any() else 0.0
    print(f"  {what}: worst err/bound {worst:.3g}")
    if bad.any():
        i = np.unravel_index(np.argmax(bad), ref.shape)
        raise AssertionError(f"{what}: {int(bad.sum())} of {ref.size} elements out of bound; first at {i}: "
                             f"got {got[i]!r} ref {ref[i]!r} bound {bound[i]!r}")
    return worst


# ---------------------------------------------------------------------------------------------------------------------
# 0-layer models through the C ABI
# ---------------------------------------------------------------------------------------------------------------------
def geometry(g):
    """O.Config of a geometry spec: ("rawiq", seq_len, seg | "conv1d", has_cls) or ("vit", H, W, patch)."""
    if g[0] == "rawiq":
        _, L, seg, has_cls = g
        conv = seg == "conv1d"
        return O.Config(kind="rawiq", n_layers=0, seq_length=L, use_cls_token=bool(has_cls),
                        embedding_type="conv1d" if conv else "segment", segment_size=64 if conv else seg)
    _, H, W, p = g
    return O.Config(kind="vit", n_layers=0, in_channels=1, img_size_h=H, img_size_w=W, patch_size=p)


class ZeroLayer:
    """A 0-layer model: descriptor, random parameters in the flat blob, a random positional table, a workspace."""

    def __init__(self, geo, dtype, B, d, C=11, head_ln=None, layout="model", p_drop=0.0, seed=1, offset=0, rng=0,
                 w_scale=None, b_shift=0.0):
        cfg = geometry(geo)
        cfg.d_model, cfg.num_classes = d, C
        self.cfg, self.B, self.layout = cfg, B, layout
        self.head_ln = (cfg.kind == "rawiq") if head_ln is None else head_ln
        D = _lib.AmcDesc()
        D.kind = _lib.KIND_RAWIQ if cfg.kind == "rawiq" else _lib.KIND_VIT
        D.dtype = _lib.BF16 if dtype == "bf16" else _lib.F32
        D.B, D.d, D.h, D.F, D.C, D.n_layers = B, d, max(1, d // 64), 8, C, 0
        if cfg.kind == "rawiq":
            D.in_ch, D.seq_len = 2, cfg.seq_length
            D.seg = 1 if cfg.embedding_type == "conv1d" else cfg.segment_size
        else:
            D.in_ch, D.img_h, D.img_w, D.patch = 1, cfg.img_size_h, cfg.img_size_w, cfg.patch_size
        D.has_cls, D.head_ln = int(cfg.has_cls), int(self.head_ln)
        D.input_layout = _lib.INPUT_RAW if layout == "dataset" else _lib.INPUT_MODEL
        D.training, D.p_drop, D.ln_eps, D.head_ln_eps = 1, p_drop, 1e-12, 1e-5
        for i, k in enumerate(("i_mean", "i_std", "q_mean", "q_std")):
            D.norm[i] = STATS[k]
        D.seed, D.offset = seed, offset
        self.desc = D
        self.L = _lib.param_layout(D)
        L = self.L
        T, K = L.T, L.K_embed
        g = np.random.default_rng(rng)
        blob = np.zeros(L.total, dtype=np.float32)
        p = {}

        def put(off, name, shape, a):
            blob[off:off + a.size] = a.ravel()
            p[name] = a.astype(np.float32).reshape(shape)

        ek = R.emb_key(cfg)
        put(L.emb_w, ek + ".weight", (d, K), g.standard_normal((d, K)) * (w_scale or 1 / np.sqrt(K)))
        put(L.emb_b, ek + ".bias", (d,), g.standard_normal(d) * 0.1 + b_shift)
        if cfg.has_cls:
            put(L.cls, "encoder.cls_token", (d,), g.standard_normal(d) * 0.5 + b_shift)
        kw, kb, kg, kbeta = R.head_keys(cfg, self.head_ln)
        if self.head_ln:
            put(L.head_ln_w, kg, (d,), 1 + 0.2 * g.standard_normal(d))
            put(L.head_ln_b, kbeta, (d,), 0.1 * g.standard_normal(d))
        put(L.head_w, kw, (C, d), g.standard_normal((C, d)) / np.sqrt(d))
        put(L.head_b, kb, (C,), 0.1 * g.standard_normal(C))
        self.p = p
        self.pos = (0.5 * g.standard_normal((T, d))).astype(np.float32)
        self.params = cuda(blob)
        self.pos_d = cuda(self.pos)
        self.ws = torch.empty(_lib.workspace_bytes(D), dtype=torch.uint8, device=DEV)
        if layout == "dataset":
            n = cfg.seq_length if cfg.kind == "rawiq" else cfg.img_size_h * cfg.img_size_w // 2
            self.x = (g.standard_normal((B, n, 2)) * 0.7 + 0.05).astype(np.float32)
        else:
            shape = (B, 2, cfg.seq_length) if cfg.kind == "rawiq" else (B, 1, cfg.img_size_h, cfg.img_size_w)
            self.x = g.standard_normal(shape).astype(np.float32)
        self.src = cuda(self.x)
        self.bf16 = dtype == "bf16"

    def forward(self):
        """(x0 [B, T, d], logits [B, C], profiled kernel classes)"""
        T, d = self.L.T, self.desc.d
        x0 = torch.empty((self.B, T, d), device=DEV)
        logits = torch.empty((self.B, self.desc.C), device=DEV)
        torch.cuda.synchronize()
        _lib.profile(True)
        try:
            _lib.check(_lib.lib.amc_model_fwd(C.byref(self.desc), self.src.data_ptr(), self.params.data_ptr(),
                                              self.pos_d.data_ptr(), self.ws.data_ptr(), logits.data_ptr(),
                                              x0.data_ptr(), stream()), "amc_model_fwd")
            classes = _lib.profile_dump()
        finally:
            _lib.profile(False)
        return x0.cpu().numpy(), logits.cpu().numpy(), classes

    def backward(self, dlogits=None, denc=None):
        """(parameter-gradient blob, dsrc) for dL/dlogits and / or dL/dx0"""
        grads = torch.zeros(self.L.total, device=DEV)
        dsrc = torch.full(self.src.shape, float("nan"), device=DEV)
        dl = cuda(dlogits) if dlogits is not None else None
        de = cuda(denc) if denc is not None else None
        _lib.check(_lib.lib.amc_model_bwd_ex(C.byref(self.desc), self.src.data_ptr(), self.params.data_ptr(),
                                             self.ws.data_ptr(), _lib.ptr(dl), _lib.ptr(de), grads.data_ptr(),
                                             dsrc.data_ptr(), 0, 2, stream()), "amc_model_bwd_ex")
        return grads.cpu().numpy().astype(np.float64), dsrc.cpu().numpy()

    def grad(self, blob, name):
        L, d, K = self.L, self.desc.d, self.L.K_embed
        off, shape = {"emb_w": (L.emb_w, (d, K)), "emb_b": (L.emb_b, (d,)), "cls": (L.cls, (d,)),
                      "head_w": (L.head_w, (self.desc.C, d)), "head_b": (L.head_b, (self.desc.C,)),
                      "ln_w": (L.head_ln_w, (d,)), "ln_b": (L.head_ln_b, (d,))}[name]
        return blob[off:off + int(np.prod(shape))].reshape(shape)

    def ref(self):
        return R.frontend_ref(self.x, self.p, self.pos, self.cfg, self.layout, STATS, self.bf16)


def check_frontend_bwd(m, got_blob, dsrc, ref, extra=None):
    """emb_w / emb_b / cls gradients and dsrc against a frontend_bwd_ref result (plus an optional propagated bound)."""
    for name in ("emb_w", "emb_b", "cls"):
        if ref[name] is None:
            continue
        b = ref[name + "_bound"] + (extra[name] if extra is not None else 0.0)
        check(name, m.grad(got_blob, name), ref[name], b)
    if dsrc is not None:
        check("dsrc", dsrc, ref["dsrc"], ref["dsrc_bound"])


# ---------------------------------------------------------------------------------------------------------------------
# front end: every path, both layouts, x0 and the embedding gradients
# ---------------------------------------------------------------------------------------------------------------------
FUSED, GEMM, SMALLK = ("frontend_fused",), ("patchify", "gemm_embed"), ("patchify", "embed_smallk")
FRONT_CASES = [
    # geometry, d, B, dtype -> path
    (("vit", 32, 64, 16), 64, 129, "bf16", FUSED),
    (("vit", 32, 64, 8), 384, 127, "bf16", FUSED),
    (("vit", 32, 64, 4), 32, 128, "bf16", FUSED),
    (("rawiq", 256, 4, 1), 128, 1000, "bf16", FUSED),
    (("rawiq", 1024, 8, 1), 256, 1, "bf16", FUSED),
    (("rawiq", 2048, 16, 1), 512, 33, "bf16", FUSED),
    (("rawiq", 1024, 32, 0), 96, 129, "bf16", FUSED),
    (("rawiq", 1024, 64, 1), 128, 127, "bf16", GEMM),       # K = 128
    (("rawiq", 768, 16, 1), 64, 1000, "bf16", GEMM),        # 48 tokens: not a power of two
    (("vit", 36, 68, 8), 64, 5, "bf16", GEMM),              # image sides not multiples of the patch: uncovered samples
    (("rawiq", 512, "conv1d", 1), 128, 129, "bf16", SMALLK),  # K = 2
    (("rawiq", 768, 3, 0), 32, 31, "bf16", SMALLK),         # K = 6
    (("vit", 32, 64, 16), 64, 129, "fp32", GEMM),
    (("rawiq", 768, 16, 1), 64, 1000, "fp32", GEMM),
    (("rawiq", 512, "conv1d", 1), 128, 129, "fp32", GEMM),
    (("vit", 36, 68, 8), 64, 5, "fp32", GEMM),
]


def front_id(c):
    return f"{c[3]}-{'_'.join(map(str, c[0]))}-d{c[1]}-B{c[2]}"


@pytest.mark.parametrize("layout", ["model", "dataset"])
@pytest.mark.parametrize("case", FRONT_CASES, ids=[front_id(c) for c in FRONT_CASES])
def test_frontend_forward_and_backward(case, layout):
    geo, d, B, dtype, path = case
    m = ZeroLayer(geo, dtype, B, d, layout=layout, rng=d + B)
    x0, _, classes = m.forward()
    for k in path:
        assert k in classes, (path, sorted(classes))
    if path == FUSED:
        assert "patchify" not in classes
    ref, A, bound = m.ref()
    check("x0", x0, ref, bound)
    G = np.random.default_rng(5).standard_normal(x0.shape).astype(np.float32)
    blob, dsrc = m.backward(denc=G)
    rb = R.frontend_bwd_ref(G, A, m.p, m.cfg, layout, STATS, m.bf16)
    check_frontend_bwd(m, blob, dsrc, rb)
    if geo[0] == "vit" and (geo[1] % geo[3] or geo[2] % geo[3]):
        assert (rb["dsrc_bound"] == 0).any()       # the uncovered samples were checked to be exactly 0


# ---------------------------------------------------------------------------------------------------------------------
# dropout at the positional-encoding site
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype,geo", [("bf16", ("rawiq", 1024, 16, 1)), ("fp32", ("vit", 32, 64, 4))])
@pytest.mark.parametrize("p", [0.1, 0.5])
def test_pe_dropout_mask_scale_and_regeneration(dtype, geo, p):
    # bias and CLS around 3, |A W| and |pe| well below: the reference x0 is never 0, so a dropped element is an exact 0
    B = 128 if geo[0] == "rawiq" else 64
    m = ZeroLayer(geo, dtype, B, 128, layout="dataset", p_drop=p, seed=1234, offset=7, w_scale=0.05, b_shift=3.0)
    ref, A, bound = m.ref()
    assert np.abs(ref).min() > 100 * bound.max()
    x0, _, _ = m.forward()
    assert x0.size >= 10 ** 6
    s = R.keep_scale(p)
    kept = x0 != 0
    # a kept element is the reference times the fp32 scale: one more rounding
    check("x0 kept", np.where(kept, x0, ref * s), ref * s, (bound + 2 * U * np.abs(ref)) * s)
    pe = R.p_effective(p)
    frac = kept.mean()
    sigma = np.sqrt(pe * (1 - pe) / kept.size)
    print(f"  kept fraction {frac:.6f}, expected {1 - pe:.6f} +- {sigma:.2e}")
    assert abs(frac - (1 - pe)) <= 5 * sigma
    assert kept[:, 0].any() and not kept[:, 0].all()        # the CLS row is dropped too

    m.desc.offset = 8
    x0b, _, _ = m.forward()
    differ = ((x0b != 0) != kept).mean()
    print(f"  offset 7 vs 8: masks differ in {differ:.4f} of the elements")
    assert differ > pe * (1 - pe)                 # independent masks differ in 2 p (1 - p)

    m.desc.offset = 7                             # backward regenerates the mask of (seed, offset) = (1234, 7)
    G = np.random.default_rng(6).standard_normal(x0.shape).astype(np.float32)
    blob, dsrc = m.backward(denc=G)
    rb = R.frontend_bwd_ref(G, A, m.p, m.cfg, "dataset", STATS, m.bf16, mult=kept * s)
    check_frontend_bwd(m, blob, dsrc, rb)


# ---------------------------------------------------------------------------------------------------------------------
# classifier head
# ---------------------------------------------------------------------------------------------------------------------
HEAD_CASES = [
    # has_cls, head_ln, tokens, d, C, B
    (1, 1, 16, 32, 1, 1),
    (1, 0, 16, 96, 2, 31),
    (1, 1, 16, 256, 11, 32),
    (1, 1, 8, 512, 24, 33),
    (1, 0, 8, 96, 25, 1000),
    (1, 1, 4, 96, 48, 4097),
    (1, 0, 4, 32, 49, 4097),
    (1, 1, 8, 512, 64, 1000),
    (0, 1, 257, 32, 25, 33),
    (0, 0, 257, 96, 64, 31),
    (0, 1, 1025, 32, 49, 32),
    (0, 0, 1025, 256, 11, 1),
    (0, 1, 257, 512, 24, 129),
]


@pytest.mark.parametrize("case", HEAD_CASES, ids=[f"cls{c[0]}-ln{c[1]}-T{c[2]}-d{c[3]}-C{c[4]}-B{c[5]}" for c in HEAD_CASES])
def test_head_forward_and_backward(case):
    has_cls, head_ln, tokens, d, Cn, B = case
    m = ZeroLayer(("rawiq", tokens, "conv1d", has_cls), "fp32", B, d, C=Cn, head_ln=bool(head_ln), rng=B + Cn)
    x0, logits, classes = m.forward()
    assert "head" in classes
    ref_logits, cache, lb = R.head_ref(x0, m.p, m.cfg, bool(head_ln))
    check("logits", logits, ref_logits, lb)
    dl = np.random.default_rng(9).standard_normal((B, Cn)).astype(np.float32)
    blob, _ = m.backward(dlogits=dl)
    hb = R.head_bwd_ref(dl, cache)
    check("head_w", m.grad(blob, "head_w"), hb["head_w"], hb["head_w_bound"])
    check("head_b", m.grad(blob, "head_b"), hb["head_b"], hb["head_b_bound"])
    if head_ln:
        check("mlp_head.0.weight", m.grad(blob, "ln_w"), hb["ln_w"], hb["ln_w_bound"])
        check("mlp_head.0.bias", m.grad(blob, "ln_b"), hb["ln_b"], hb["ln_b_bound"])
    # dx0 reaches the embedding gradients (fp32: no rounding of demb); its bound propagates linearly
    _, A, _ = m.ref()
    rb = R.frontend_bwd_ref(hb["dx0"], A, m.p, m.cfg)
    eb = R.frontend_bwd_ref(hb["dx0_bound"], np.abs(A), m.p, m.cfg)
    check_frontend_bwd(m, blob, None, rb, extra=eb)


# ---------------------------------------------------------------------------------------------------------------------
# cross-entropy and argmax
# ---------------------------------------------------------------------------------------------------------------------
def ce_call(z, labels, ls, grad_scale=1.0, loss_scale=1.0, want_dl=True, want_stats=True):
    B, Cn = z.shape
    zl = cuda(z)
    lab = cuda(labels, torch.int64)
    dl = torch.full((B, Cn), float("nan"), device=DEV) if want_dl else None
    st = torch.zeros(2, device=DEV) if want_stats else None
    _lib.check(_lib.lib.amc_ce_loss(B, Cn, zl.data_ptr(), lab.data_ptr(), ls, grad_scale, loss_scale, _lib.ptr(dl),
                                    _lib.ptr(st), stream()), "amc_ce_loss")
    return (dl.cpu().numpy() if want_dl else None), (st.cpu().numpy() if want_stats else None)


def ce_bounds(z, labels, ls, gs):
    """fp32 bounds of the per-frame loss and of dlogits: logp = z - max - log(sum exp) carries the C-term sum, expf and
    logf (a few ulp each); the loss sums C weighted logp terms; dlogits = (exp(logp) - target) * grad_scale."""
    z = np.asarray(z, dtype=np.float64)
    B, Cn = z.shape
    loss, dl = R.ce_ref(z, labels, ls)
    mx = z.max(1, keepdims=True)
    lse = np.log(np.exp(z - mx).sum(1, keepdims=True))
    logp = z - mx - lse
    e_logp = R.C_ACC * (Cn + 4) * U * (1 + np.abs(mx) + np.abs(z).max(1, keepdims=True) + np.abs(lse))
    tgt = np.exp(logp) - dl
    e_loss = (e_logp + R.C_ACC * (Cn + 2) * U * (np.abs(tgt * logp).sum(1, keepdims=True) + np.abs(logp).sum(1, keepdims=True) * ls / Cn)).ravel()
    prob = np.exp(logp)
    # (+ 2^-126: expf of a logit far below the row maximum underflows to 0 or a subnormal)
    e_dl = gs * (prob * (e_logp + 4 * U) + 2 * U * (prob + np.abs(tgt)) + 2.0 ** -126) + U * np.abs(dl * gs)
    return loss, dl, e_loss, e_dl


@pytest.mark.parametrize("B", [1, 127, 128, 129, 100000])
@pytest.mark.parametrize("Cn", [1, 2, 11, 33, 64])
@pytest.mark.parametrize("ls", [0.0, 0.1, 0.3])
def test_ce_loss(ls, Cn, B):
    g = np.random.default_rng(B * 7 + Cn)
    z = (g.standard_normal((B, Cn)) * 4).astype(np.float32)
    z[::7] = np.where(g.random((len(z[::7]), Cn)) < 0.5, 80.0, -80.0)      # logits of +-80
    z[3::11] = np.round(z[3::11])                                         # exact ties among small integers
    labels = g.integers(0, Cn, B)
    gs, lsc = 1.0 / 3.0, 0.25
    loss, dl, e_loss, e_dl = ce_bounds(z, labels, ls, gs)
    got_dl, st = ce_call(z, labels, ls, gs, lsc)
    check("dlogits", got_dl, dl * gs, e_dl)
    # stats[0] += sum_b loss_b * loss_scale: B terms through warp sums and one fp32 atomic per warp
    check("stats[0]", st[0], loss.sum() * lsc, lsc * (e_loss.sum() + R.C_ACC * (B + 1) * U * np.abs(loss).sum()))
    assert st[1] == (R.argmax_ref(z) == labels).sum()
    # NULL outputs: each of the two may be left out
    got_dl2, _ = ce_call(z, labels, ls, gs, lsc, want_stats=False)
    assert np.array_equal(got_dl2, got_dl)
    _, st2 = ce_call(z, labels, ls, gs, lsc, want_dl=False)
    check("stats[0] without dlogits", st2[0], loss.sum() * lsc,
          lsc * (e_loss.sum() + R.C_ACC * (B + 1) * U * np.abs(loss).sum()))
    assert st2[1] == st[1]


def test_ce_loss_out_of_range_label_poisons_only_the_loss():
    g = np.random.default_rng(4)
    B, Cn, ls = 64, 11, 0.1
    z = g.standard_normal((B, Cn)).astype(np.float32)
    z[5, 3] = z[6, 3] = z[7, 3] = 10.0                  # argmax 3 on the frames with bad labels
    labels = g.integers(0, Cn, B)
    labels[5], labels[6], labels[7] = Cn, -1, 2 ** 32 + 3   # 2^32 + 3 truncates to class 3 in 32 bits
    _, dl, _, e_dl = ce_bounds(z, labels, ls, 1.0)
    got_dl, st = ce_call(z, labels, ls)
    assert np.isnan(st[0])
    ok = (labels >= 0) & (labels < Cn)
    assert st[1] == ((R.argmax_ref(z) == labels) & ok).sum()
    check("dlogits (bad rows: all-smoothing target)", got_dl, dl, e_dl)


@pytest.mark.parametrize("B", [1, 127, 129, 1000])
@pytest.mark.parametrize("Cn", [1, 11, 64])
def test_argmax(Cn, B):
    g = np.random.default_rng(Cn + B)
    z = np.round(g.standard_normal((B, Cn)) * 2).astype(np.float32)       # many exact ties
    if B > 8 and Cn > 1:
        z[1] = 3.0                                                        # all equal
        z[2, Cn // 2] = np.nan                                            # NaN: its index
        z[3, 0] = np.nan
        z[3, Cn - 1] = np.nan                                             # the first NaN
        z[4] = -np.inf
        z[5, -1] = np.inf
    out = torch.empty(B, dtype=torch.int64, device=DEV)
    _lib.check(_lib.lib.amc_argmax(B, Cn, cuda(z).data_ptr(), out.data_ptr(), stream()), "amc_argmax")
    assert np.array_equal(out.cpu().numpy(), R.argmax_ref(z))


# ---------------------------------------------------------------------------------------------------------------------
# clip + AdamW
# ---------------------------------------------------------------------------------------------------------------------
F32 = lambda v: float(np.float32(v))  # noqa: E731  (the kernels see the fp32 values of the hyperparameters)
HP = dict(lr=F32(1e-3), beta1=F32(0.9), beta2=F32(0.99), eps=F32(1e-8))
GRID = 148 * 8 * 256                 # the kernels' grid-stride: n above it loops


def n_chain(n):
    blocks = min((n + 255) // 256, 148 * 8)
    return -(-n // GRID) + 5 + 3 + blocks


def adam_state(n, gnorm, seed):
    g = np.random.default_rng(seed)
    p = g.standard_normal(n).astype(np.float32)
    gr = g.standard_normal(n)
    gr = (gr * gnorm / np.linalg.norm(gr)).astype(np.float32)
    m = (g.standard_normal(n) * gnorm / np.sqrt(n)).astype(np.float32)
    v = (g.random(n) * gnorm ** 2 / n).astype(np.float32)
    return p, gr, m, v


def check_adam(tag, got, state, step, wd, max_norm, gs, ws):
    p, g, m, v = state
    n = p.size
    rp, rm, rv, norm = R.adamw_ref(p, g, m, v, step, HP["lr"], HP["beta1"], HP["beta2"], HP["eps"], wd, max_norm, gs)
    ep, em, ev, e_norm = R.adamw_bound(p, g, m, v, step, HP["lr"], HP["beta1"], HP["beta2"], HP["eps"], wd, max_norm, gs,
                                       n_chain(n))
    check(f"{tag} exp_avg", got[2], rm, em)
    check(f"{tag} exp_avg_sq", got[3], rv, ev)
    check(f"{tag} param", got[0], rp, ep)
    if max_norm > 0:
        check(f"{tag} norm_ws[1]", ws[1], norm, norm * e_norm)
    else:                               # clipping disabled: the scratch is neither read nor written
        assert np.isnan(ws).all()


ADAM_CASES = [
    # max_norm, grad norm, grad_scale, weight decay, step
    (F32(1e-4), 1e-3, 1.0, 0.0, 1),   # clip active at a small norm (the 1e-6 of the coefficient matters: 1e-3 relative)
    (F32(1e-4), 1e-3, 0.5, F32(0.01), 10000),
    (1e6, 2.0, 0.25, F32(0.01), 1),    # clip inactive
    (0.0, 2.0, 2.0, 0.0, 10000),       # clip disabled
]


@pytest.mark.parametrize("n", [1, 255, 257, GRID + 3, 10 ** 7])
@pytest.mark.parametrize("case", ADAM_CASES, ids=[f"clip{c[0]:g}-g{c[1]:g}-gs{c[2]:g}-wd{c[3]:g}-step{c[4]}" for c in ADAM_CASES])
def test_adamw_clip_step(case, n):
    max_norm, gnorm, gs, wd, step = case
    state = adam_state(n, gnorm, n % 1000 + step)
    t = [cuda(a) for a in state]
    ws = torch.full((2,), float("nan"), device=DEV)
    _lib.check(_lib.lib.amc_adamw_clip_step(n, t[0].data_ptr(), t[1].data_ptr(), t[2].data_ptr(), t[3].data_ptr(),
                                            HP["lr"], HP["beta1"], HP["beta2"], HP["eps"], wd, max_norm, gs, step,
                                            ws.data_ptr(), stream()), "amc_adamw_clip_step")
    got = [a.cpu().numpy() for a in t]
    assert np.array_equal(got[1], state[1])            # the gradients are read, not scaled in place
    check_adam("plain", got, state, step, wd, max_norm, gs, ws.cpu().numpy())


@pytest.mark.parametrize("max_norm", [1e-4, 0.0])
def test_adamw_graph_variant_matches_plain_eager_and_replayed(max_norm):
    n, gs, wd = GRID + 3, 0.5, F32(0.01)
    max_norm = F32(max_norm)
    state0 = adam_state(n, 1e-3, 3)
    lr, b1, b2, eps = HP["lr"], HP["beta1"], HP["beta2"], HP["eps"]

    def run(kind):
        t = [cuda(a) for a in state0]
        ws = torch.full((2,), float("nan"), device=DEV)
        ctr = torch.zeros(1, dtype=torch.int32, device=DEV)
        args = lambda: (n, t[0].data_ptr(), t[1].data_ptr(), t[2].data_ptr(), t[3].data_ptr(), lr, b1, b2, eps, wd,  # noqa
                        max_norm, gs)
        graph = None
        if kind == "graph":          # one captured update, replayed five times: the counter advances the step
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                _lib.check(_lib.lib.amc_adamw_clip_step_graph(*args(), ctr.data_ptr(), ws.data_ptr(),
                                                              torch.cuda.current_stream().cuda_stream), "capture")
            torch.cuda.synchronize()
            assert int(ctr.item()) == 0
        for step in range(1, 6):
            prev = [a.cpu().numpy() for a in t]
            ws.fill_(float("nan"))
            if kind == "plain":
                _lib.check(_lib.lib.amc_adamw_clip_step(*args(), step, ws.data_ptr(), stream()), "plain")
            elif kind == "eager":
                _lib.check(_lib.lib.amc_adamw_clip_step_graph(*args(), ctr.data_ptr(), ws.data_ptr(), stream()), "eager")
            else:
                graph.replay()
            torch.cuda.synchronize()
            if kind != "plain":
                assert int(ctr.item()) == step
            got = [a.cpu().numpy() for a in t]
            check_adam(f"{kind} step {step}", got, prev, step, wd, max_norm, gs, ws.cpu().numpy())

    # each variant is checked step by step against the float64 step from its own previous state, so the two
    # agree within the AdamW bound of each step (not bit for bit: fp32 atomics of the norm, device-side pow)
    for kind in ("plain", "eager", "graph"):
        run(kind)


# ---------------------------------------------------------------------------------------------------------------------
# IQ statistics
# ---------------------------------------------------------------------------------------------------------------------
def iq_call(x, acc=None, offset_floats=0):
    n_frames, frame_len = x.shape[0], x.shape[1]
    buf = torch.empty(x.size + 4, device=DEV)
    buf[offset_floats:offset_floats + x.size] = cuda(x.ravel())
    acc = torch.zeros(4, dtype=torch.float64, device=DEV) if acc is None else acc
    rc = _lib.lib.amc_iq_stats(n_frames, frame_len, buf.data_ptr() + 4 * offset_floats, acc.data_ptr(), stream())
    return rc, acc


@pytest.mark.parametrize("shape,mean,std", [((3, 1001), 0.0, 1.0), ((157, 2049), 0.5, 2.0),
                                            ((700, 1024), 1e3, 1e-2)])
def test_iq_stats_sums(shape, mean, std):
    x = (np.random.default_rng(shape[1]).standard_normal(shape + (2,)) * std + mean).astype(np.float32)
    ref, bound = R.iq_stats_ref(x)
    rc, acc = iq_call(x)
    assert rc == 0
    check("sums", acc.cpu().numpy(), ref, bound)
    rc, acc = iq_call(x, acc)                    # a second call accumulates
    assert rc == 0
    check("sums after two calls", acc.cpu().numpy(), 2 * ref, 2 * bound + 2 * U * U * np.abs(ref))
    if mean == 1e3:                              # the unbiased std survives the cancellation
        s = acc.cpu().numpy() / 2
        n = x.size // 2
        var = (s[1] - s[0] ** 2 / n) / (n - 1)
        assert abs(np.sqrt(var) - x[..., 0].astype(np.float64).std(ddof=1)) < 1e-4 * std


def test_iq_stats_alignment():
    x = np.random.default_rng(0).standard_normal((5, 33, 2)).astype(np.float32)
    ref, bound = R.iq_stats_ref(x)
    rc, acc = iq_call(x, offset_floats=2)        # 8-byte but not 16-byte aligned
    assert rc == 0
    check("sums (8-byte aligned)", acc.cpu().numpy(), ref, bound)
    rc, _ = iq_call(x, offset_floats=1)          # 4-byte aligned: refused
    assert rc < 0 and b"aligned" in _lib.lib.amc_last_error()


# ---------------------------------------------------------------------------------------------------------------------
# amc_gemm: the generic-epilogue tcgen05 kernel (gemm_tc_kernel<BN, 0>, behind the unfused embedding)
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("M,N,K,lda,ldd16,ldd32", [(300, 40, 64, 64, 0, 40), (257, 200, 96, 104, 208, 204),
                                                   (129, 384, 128, 136, 392, 388), (1000, 512, 256, 256, 512, 512)])
def test_gemm_generic_epilogue(M, N, K, lda, ldd16, ldd32):
    g = np.random.default_rng(M + N)
    A = R.bf16_rne(g.standard_normal((M, lda)).astype(np.float32))
    Bm = R.bf16_rne((g.standard_normal((N, K)) / np.sqrt(K)).astype(np.float32))
    bias = g.standard_normal(N).astype(np.float32)
    Ad, Bd, bd = cuda(A, torch.bfloat16), cuda(Bm, torch.bfloat16), cuda(bias)
    D16 = torch.zeros((M, ldd16), dtype=torch.bfloat16, device=DEV) if ldd16 else None
    D32 = torch.full((M, ldd32), 7.0, device=DEV)
    _lib.check(_lib.lib.amc_gemm(_lib.BF16, M, N, K, Ad.data_ptr(), lda, 0, Bd.data_ptr(), K, 0, bd.data_ptr(), None, 0,
                                 0, _lib.ptr(D16), ldd16, D32.data_ptr(), ldd32, 0, stream()), "amc_gemm")
    a = A[:, :K].astype(np.float64)
    ref = a @ Bm.T.astype(np.float64) + bias
    bound = R.C_ACC * (K + 1) * U * (np.abs(a) @ np.abs(Bm.T.astype(np.float64)) + np.abs(bias))
    d32 = D32.cpu().numpy()
    check("D32", d32[:, :N], ref, bound)
    assert (d32[:, N:] == 7.0).all()                      # the row padding is not written
    if D16 is not None:
        d16 = D16.float().cpu().numpy()
        assert np.array_equal(d16[:, :N], R.bf16_rne(d32[:, :N]))   # D16 is the RNE of the same fp32 value
        assert (d16[:, N:] == 0).all()

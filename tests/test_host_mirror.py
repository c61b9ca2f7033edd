"""CPU-side checks of the drop-in boundary: constructor signatures, state_dict keys, flat blob,
error behaviour, and that the C-ABI library exports every symbol the header declares."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from conftest import GOLDEN_CASES, GOLDEN_DIR, ROOT, load_golden
from oracle import amc_oracle as O

import vit_vs_raw_iq_b200 as amc
from vit_vs_raw_iq_b200 import _lib


def build_ours(name, **extra):
    kind, kw = GOLDEN_CASES[name]
    cls = amc.RawIQAMCTransformer if kind == "rawiq" else amc.ViTAMCTransformer
    return cls(**kw, drop_prob=0.0, device="cpu", **extra)


@pytest.mark.parametrize("name", list(GOLDEN_CASES))
def test_state_dict_keys_shapes_order_match_reference(name):
    kind, kw = GOLDEN_CASES[name]
    model = build_ours(name)
    sd = model.state_dict()
    shapes = O.param_shapes(O.Config(kind=kind, **kw))
    assert list(sd) == list(shapes)
    for k, v in sd.items():
        assert tuple(v.shape) == shapes[k], k
    assert sum(p.numel() for p in model.parameters()) == O.param_count(O.Config(kind=kind, **kw))


@pytest.mark.parametrize("name", list(GOLDEN_CASES))
def test_strict_load_of_reference_state_dict_and_flat_views(name):
    _, params, _, _ = load_golden(name)
    model = build_ours(name)
    model.load_state_dict({k: torch.from_numpy(v) for k, v in params.items()}, strict=True)
    core = model._core
    assert core.is_flat()
    flat = model.flat_parameters()
    for p, (o, n, shape) in zip(core.params, core.slots):
        assert p.data_ptr() == flat.data_ptr() + 4 * o
    for k, v in model.state_dict().items():
        assert np.array_equal(v.numpy(), params[k]), k
    # q/k/v adjacency: the fused QKV GEMM reads one [3d,d] matrix
    L = core.layout
    d = core.d
    assert (L.wk - L.wq, L.wv - L.wk, L.bk - L.bq, L.bv - L.bk) == (d * d, d * d, d, d)
    # in-place optimiser updates must land in the blob
    with torch.no_grad():
        model.encoder.layers[0].attention.w_k.weight.add_(1.0)
    o = L.layer0 + L.wk
    assert torch.equal(flat[o:o + d * d].view(d, d), model.encoder.layers[0].attention.w_k.weight)


def test_known_answer_param_counts():
    m = amc.RawIQAMCTransformer(in_channels=2, seq_length=1024, num_classes=11, d_model=128, n_head=8, n_layers=2,
                                ffn_hidden=512, drop_prob=0.1, device="cpu", use_cls_token=True,
                                embedding_type="segment", segment_size=64)
    assert sum(p.numel() for p in m.parameters()) == 414_859            # R/test_model.py:71-75
    m = amc.ViTAMCTransformer(in_channels=1, img_size_h=32, img_size_w=64, patch_size=4, num_classes=19,
                              d_model=256, n_head=16, n_layers=6, ffn_hidden=1024, drop_prob=0.15, device="cpu")
    assert sum(p.numel() for p in m.parameters()) == 4_748_051          # V/main.ipynb:772
    assert sum(p.numel() for p in m.encoder.layers[0].parameters()) == 789_760


@pytest.mark.parametrize("kind", ["rawiq", "vit"])
def test_same_seed_gives_reference_initial_weights(kind):
    """The reference's modules constructed after torch.manual_seed(s) (tests/golden/make_golden.py trajectory_case /
    trajectory_vit_case: seed 5 / 6, dropout 0) stored their initial state_dict as the trajectories' param/*; ours
    must draw the same weights from the same seed.  Dropout has no parameters and draws nothing at construction, so
    building ours with dropout on must not change them."""
    if kind == "rawiq":
        seed, golden = 5, "trajectory_rawiq.npz"
        kw = dict(in_channels=2, seq_length=256, num_classes=4, d_model=32, n_head=4, n_layers=2, ffn_hidden=64,
                  drop_prob=0.1, device="cpu", use_cls_token=True, embedding_type="segment", segment_size=16)
        ours_cls = amc.RawIQAMCTransformer
    else:
        seed, golden = 6, "trajectory_vit.npz"
        kw = dict(in_channels=1, img_size_h=32, img_size_w=64, patch_size=16, num_classes=4, d_model=64, n_head=8,
                  n_layers=2, ffn_hidden=128, drop_prob=0.1, device="cpu")
        ours_cls = amc.ViTAMCTransformer
    z = np.load(os.path.join(GOLDEN_DIR, golden))
    rsd = {k[len("param/"):]: z[k] for k in z.files if k.startswith("param/")}
    torch.manual_seed(seed)
    osd = ours_cls(**kw).state_dict()
    assert list(rsd) == list(osd)
    for k in rsd:
        assert np.array_equal(rsd[k], osd[k].numpy()), k


def test_constructor_errors_match_reference():
    base = dict(in_channels=2, num_classes=11, d_model=32, n_head=4, n_layers=1, ffn_hidden=64, drop_prob=0.0,
                device="cpu")
    with pytest.raises(ValueError, match="must be divisible by segment_size"):     # R/models/encoder.py:45-48
        amc.RawIQAMCTransformer(seq_length=100, segment_size=16, **base)
    with pytest.raises(ValueError, match="Unknown embedding_type"):               # R/models/encoder.py:57
        amc.RawIQAMCTransformer(seq_length=128, embedding_type="bogus", **base)
    m = amc.RawIQAMCTransformer(seq_length=128, segment_size=16, use_cls_token=False, **base)
    with pytest.raises(ValueError, match="CLS token is not enabled"):             # R/models/encoder.py:131-132
        m.encoder.get_cls_token_output(torch.zeros(1, 2, 128))


def test_no_cpu_fallback():
    m = build_ours("rawiq_seg16")
    with pytest.raises(RuntimeError, match="CUDA"):
        m(torch.zeros(2, 2, 256))
    with pytest.raises(NotImplementedError):
        m.encoder.layers[0](torch.zeros(1, 17, 32), None)


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "amc_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(amc_[a-z0-9_]+)\s*\(", hdr))
    assert declared, "no declarations parsed"
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} declared in include/amc_b200.h but not exported"
    assert set(_lib.EXPORTS) == declared, (set(_lib.EXPORTS) ^ declared)
    assert lib.amc_abi_version() == _lib.ABI_VERSION
    m = re.search(r"#define AMC_ABI_VERSION (\d+)", hdr)
    assert int(m.group(1)) == _lib.ABI_VERSION


def test_layout_and_workspace_host_calls():
    core = build_ours("vit_p16")._core
    L = core.layout
    assert (L.T, L.Ttok, L.K_embed) == (9, 8, 256)
    assert L.total % 64 == 0 and L.cls >= 0 and L.head_ln_w == -1
    d32 = core._desc(B=8, dtype=_lib.F32, training=True)
    d16 = core._desc(B=8, dtype=_lib.BF16, training=True)
    assert _lib.workspace_bytes(d32) > 0 and _lib.workspace_bytes(d16) > 0
    bad = core._desc(B=8, dtype=_lib.F32)
    bad.h = 7
    with pytest.raises(ValueError, match="divisible"):
        _lib.param_layout(bad)


def test_conv1d_embedding_envelope_host_calls():
    """embedding_type='conv1d' (the reference Encoder's default, R/models/encoder.py:26): one token per IQ sample -> T = seq_length + 1, K = 2.  Both
    arithmetic modes accept it (long-sequence attention + small-K embedding); past 16384 tokens the layout call refuses."""
    m = amc.RawIQAMCTransformer(in_channels=2, seq_length=1024, num_classes=11, d_model=128, n_head=8, n_layers=2,
                                ffn_hidden=256, drop_prob=0.1, device="cpu", embedding_type="conv1d")
    core = m._core
    L = core.layout
    assert (L.T, L.Ttok, L.K_embed) == (1025, 1024, 2)
    assert m.encoder.sequence_embedding.projection.weight.shape == (128, 2, 1)          # Conv1d(2, d, kernel_size=1)
    assert m.encoder.positional_encoding.encoding.shape == (1025, 128)
    for dt in (_lib.F32, _lib.BF16):
        assert _lib.workspace_bytes(core._desc(B=4, dtype=dt, training=True)) > _lib.workspace_bytes(
            core._desc(B=4, dtype=dt, training=False)) > 0
    too_long = core._desc(B=1, dtype=_lib.BF16)
    too_long.seq_len = 20000
    with pytest.raises(ValueError, match="tokens per frame unsupported"):
        _lib.param_layout(too_long)
    odd = core._desc(B=1, dtype=_lib.BF16)
    odd.in_ch, odd.seg = 3, 7                                                            # K = 21: neither % 8 nor <= 16
    odd.seq_len = 1022
    with pytest.raises(ValueError, match="patch width"):
        _lib.param_layout(odd)


def test_error_text_is_thread_local():
    """SURVEY §8b: autograd calls backward from its own thread, so the error text behind a non-zero return must belong
    to the calling thread (`amc_last_error` is thread-local)."""
    import threading
    core = build_ours("vit_p16")._core
    seen = {}
    barrier = threading.Barrier(2)

    def worker(tag, mutate, expect):
        d = core._desc(B=2, dtype=_lib.F32)
        mutate(d)
        out = _lib.AmcParamLayout()
        for _ in range(200):
            rc = _lib.lib.amc_param_layout(ctypes.byref(d), ctypes.byref(out))
            barrier.wait()
            msg = _lib.lib.amc_last_error().decode()
            if rc == 0 or expect not in msg:
                seen[tag] = msg
                barrier.abort()
                return
        seen[tag] = "ok"

    a = threading.Thread(target=worker, args=("a", lambda d: setattr(d, "h", 7), "divisible by n_head"))
    b = threading.Thread(target=worker, args=("b", lambda d: setattr(d, "kind", 99), "unknown model kind"))
    a.start(); b.start(); a.join(); b.join()
    assert seen == {"a": "ok", "b": "ok"}, seen

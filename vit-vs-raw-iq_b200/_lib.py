"""ctypes binding of the C ABI in include/amc_b200.h.

The shared library is built in-tree by ``__graft_entry__.build()`` (nvcc, sm_100a).  There is
no fallback: if the library is missing the import fails, and every call that returns non-zero
raises ``RuntimeError(amc_last_error())``.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libamc_b200.so")

ABI_VERSION = 8
KIND_RAWIQ, KIND_VIT = 0, 1
F32, BF16 = 0, 1
INPUT_MODEL, INPUT_RAW = 0, 1
NORM_LINF, NORM_L2 = 0, 1


class AmcDesc(C.Structure):
    _fields_ = [
        ("kind", C.c_int32), ("dtype", C.c_int32), ("B", C.c_int32), ("d", C.c_int32), ("h", C.c_int32),
        ("F", C.c_int32), ("C", C.c_int32), ("n_layers", C.c_int32), ("in_ch", C.c_int32),
        ("seq_len", C.c_int32), ("seg", C.c_int32), ("img_h", C.c_int32), ("img_w", C.c_int32),
        ("patch", C.c_int32), ("has_cls", C.c_int32), ("head_ln", C.c_int32), ("input_layout", C.c_int32),
        ("training", C.c_int32), ("p_drop", C.c_float), ("ln_eps", C.c_float), ("head_ln_eps", C.c_float),
        ("norm", C.c_float * 4), ("seed", C.c_uint64), ("offset", C.c_uint64), ("step_counter", C.c_void_p),
    ]


_LAYOUT_I64 = ["total", "emb_w", "emb_b", "cls", "layer0", "layer_stride", "wq", "wk", "wv", "bq", "bk", "bv", "wo",
               "bo", "g1", "be1", "w1", "b1", "w2", "b2", "g2", "be2", "head_ln_w", "head_ln_b", "head_w", "head_b"]


class AmcParamLayout(C.Structure):
    _fields_ = [(n, C.c_int64) for n in _LAYOUT_I64] + [("T", C.c_int32), ("Ttok", C.c_int32),
                                                        ("K_embed", C.c_int32), ("pad_", C.c_int32)]


class AmcWorkspaceInfo(C.Structure):
    _fields_ = [("bytes", C.c_size_t), ("saved_bytes", C.c_size_t)]


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: the sm_100a CUDA library has not been built. "
            "Run `python -c 'import __graft_entry__ as g; g.build()'` at the repo root. "
            "There is no CPU or PyTorch fallback for this path.")
    lib = C.CDLL(LIB_PATH)
    vp, i32, i64, f32 = C.c_void_p, C.c_int, C.c_int64, C.c_float
    lib.amc_abi_version.restype = C.c_int
    lib.amc_last_error.restype = C.c_char_p
    lib.amc_launch_count.restype = C.c_longlong
    lib.amc_launch_count.argtypes = []
    sigs = {
        "amc_param_layout": [C.POINTER(AmcDesc), C.POINTER(AmcParamLayout)],
        "amc_model_workspace": [C.POINTER(AmcDesc), C.POINTER(AmcWorkspaceInfo)],
        "amc_model_fwd": [C.POINTER(AmcDesc), vp, vp, vp, vp, vp, vp, vp],
        "amc_model_bwd": [C.POINTER(AmcDesc), vp, vp, vp, vp, vp, vp, i32, i32, vp],
        "amc_model_bwd_ex": [C.POINTER(AmcDesc), vp, vp, vp, vp, vp, vp, vp, i32, i32, vp],
        "amc_ce_loss": [i32, i32, vp, vp, f32, f32, f32, vp, vp, vp],
        "amc_argmax": [i32, i32, vp, vp, vp],
        "amc_zero": [vp, C.c_size_t, vp],
        "amc_adamw_clip_step": [i64, vp, vp, vp, vp, f32, f32, f32, f32, f32, f32, f32, i64, vp, vp],
        "amc_adamw_clip_step_graph": [i64, vp, vp, vp, vp, f32, f32, f32, f32, f32, f32, f32, vp, vp, vp],
        "amc_iq_stats": [i64, i64, vp, vp, vp],
        "amc_adv_step": [i64, i64, i32, vp, vp, vp, f32, vp, vp],
        "amc_adv_init": [i64, i64, i32, vp, vp, C.c_uint64, C.c_uint64, vp, vp, vp],
        "amc_gemm": [i32, i32, i32, i32, vp, i32, i32, vp, i32, i32, vp, vp, i32, i32, vp, i32, vp, i32, i32, vp],
        "amc_gemm_ln": [i32, i32, i32, vp, i32, vp, i32, vp, vp, vp, vp, f32, vp, vp, vp, vp, vp],
        "amc_gemm_relu_mask": [i32, i32, i32, vp, i32, vp, i32, vp, f32, vp, vp],
        "amc_attention_fwd": [i32, i32, i32, i32, i32, vp, vp, vp, vp],
        "amc_attention_bwd": [i32, i32, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp],
        "amc_attention_cls_fwd": [i32, i32, i32, i32, vp, vp, vp],
        "amc_attention_cls_bwd": [i32, i32, i32, i32, vp, vp, vp, vp, vp],
        "amc_layernorm_fwd": [i32, i32, i32, vp, vp, vp, f32, vp, vp, vp, vp, vp],
        "amc_layernorm_bwd": [i32, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp],
        "amc_frontend_fwd": [C.POINTER(AmcDesc), vp, vp, vp, vp, vp, vp, C.c_size_t, vp, vp],
        "amc_profile_enable": [i32],
        "amc_profile_dump": [C.c_char_p, C.c_size_t],
    }
    for name, args in sigs.items():
        fn = getattr(lib, name)
        fn.argtypes = args
        fn.restype = C.c_int
    if lib.amc_abi_version() != ABI_VERSION:
        raise ImportError(f"{LIB_PATH}: ABI version {lib.amc_abi_version()} != expected {ABI_VERSION}; rebuild")
    return lib, sorted(sigs) + ["amc_abi_version", "amc_last_error", "amc_launch_count"]


lib, EXPORTS = _load()


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = lib.amc_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"{what or 'amc_b200'} failed (rc={rc}): {msg}")


def ptr(t) -> int:
    """Device/host address of a torch tensor (None -> NULL)."""
    return 0 if t is None else t.data_ptr()


def param_layout(desc: AmcDesc) -> AmcParamLayout:
    out = AmcParamLayout()
    rc = lib.amc_param_layout(C.byref(desc), C.byref(out))
    if rc != 0:
        # constructor-time validation mirrors the reference's ValueError (R/models/encoder.py:45-48)
        raise ValueError(lib.amc_last_error().decode("utf-8", "replace"))
    return out


def workspace_bytes(desc: AmcDesc) -> int:
    out = AmcWorkspaceInfo()
    check(lib.amc_model_workspace(C.byref(desc), C.byref(out)), "amc_model_workspace")
    return int(out.bytes)


def profile(enable: bool) -> None:
    check(lib.amc_profile_enable(1 if enable else 0), "amc_profile_enable")


def profile_dump() -> dict:
    """{class: dict(n=launches, ms=total_ms, flops=..., bytes=...)} since the last dump (synchronises)."""
    buf = C.create_string_buffer(1 << 16)
    check(lib.amc_profile_dump(buf, len(buf)), "amc_profile_dump")
    out = {}
    for line in buf.value.decode().splitlines():
        name, n, ms, fl, by = line.split()
        out[name] = dict(n=int(n), ms=float(ms), flops=float(fl), bytes=float(by))
    return out


def device_norm_stats(x) -> dict:
    """i_mean / i_std / q_mean / q_std of device-resident interleaved frames [N, L, 2] (fp32), computed on the
    GPU with fp64 accumulation (the reference subsamples <= 5000 frames on the host: dataset.py:115-157)."""
    import torch
    if not (x.is_cuda and x.dtype == torch.float32 and x.is_contiguous() and x.dim() == 3 and x.shape[2] == 2):
        raise RuntimeError("device_norm_stats expects a contiguous CUDA float32 tensor [N, L, 2]")
    acc = torch.zeros(4, dtype=torch.float64, device=x.device)
    check(lib.amc_iq_stats(x.shape[0], x.shape[1], x.data_ptr(), acc.data_ptr(),
                           torch.cuda.current_stream(x.device).cuda_stream), "amc_iq_stats")
    si, ssi, sq, ssq = acc.tolist()
    n = float(x.shape[0] * x.shape[1])
    out = {}
    for name, s1, s2 in (("i", si, ssi), ("q", sq, ssq)):
        mean = s1 / n
        var = max((s2 - s1 * s1 / n) / max(n - 1.0, 1.0), 0.0)
        out[name + "_mean"] = mean
        out[name + "_std"] = max(var ** 0.5, 1e-8)
    return out

"""bench.py contract checks: the reference arm prints one well-formed JSON line; --dump-outputs (the end-to-end run of
our arm needs a GPU)."""
import json
import math
import os
import subprocess
import sys

import pytest

from conftest import ROOT


def test_reference_arm_prints_contract_line():
    env = dict(os.environ, OMP_NUM_THREADS="4")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "1", "--cpu-sample", "16", "--workload", "vit_p16_d256_L6"],
                         capture_output=True, text=True, timeout=300, env=env, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "train_frames_per_sec" and line["unit"] == "frames/s"
    assert line["higher_is_better"] is True and line["value"] > 0
    # the unmodified reference when oracle/_ref has been vendored (oracle/make_ref.py, run by build()), else the port
    import bench
    assert line["cpu_baseline"]["kind"] == ("reference" if bench.reference_available() else "port")
    assert line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"] == {"value": line["value"], "unit": "frames/s", "h2d_bytes_per_step": 0,
                           "d2h_bytes_per_step": 0}
    assert line["config"]["workload"] == "vit_p16_d256_L6"


def test_reference_arm_other_ranks_exit_silently():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "1"], capture_output=True, text=True, timeout=120, env=env, cwd=ROOT)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_algorithmic_flops_match_the_survey_table():
    """SURVEY §8(d) table: forward GFLOP per frame of the BASELINE configs (the numerators of every roofline figure)."""
    import bench
    expect = {"rawiq_seg16_d128_L6": 0.2691, "vit_p16_d256_L6": 0.0865, "vit_p4_d128_L6": 0.3560,
              "rawiq_sps1_seg8_d256_L6": 1.3207, "rawiq_sps2_seg8_d256_L6": 2.8333}
    for name, gf in expect.items():
        got = bench.flops_per_frame(bench.WORKLOADS[name]) / 1e9
        assert abs(got - gf) / gf < 5e-3, (name, got, gf)
    # conv1d embedding: one token per IQ sample (T = 1025, K = 2); the §8(d) formula L*T*(8d^2 + 4dF + 4Td) + 2*Ttok*K*d + 2dC
    w = bench.WORKLOADS["rawiq_conv1d_d128_L6"]
    assert bench.geometry(w) == (1025, 1024, 2)
    d, F, T = 128, 1024, 1025
    assert bench.flops_per_frame(w) == 6 * T * (8 * d * d + 4 * d * F + 4 * T * d) + 2 * 1024 * 2 * d + 2 * d * 11


def test_ncu_launch_list_summary_parses_the_committed_capture(tmp_path):
    """tools/ncu_summary.py turns the ncu CSV launch list into the per-kernel share table under profiles/."""
    src = os.path.join(ROOT, "profiles", "r1_launches_train.csv")
    out = tmp_path / "launches.md"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "ncu_summary.py"), "launches", src, str(out)],
                       capture_output=True, text=True, timeout=60)
    assert r.returncode == 0, r.stderr
    text = out.read_text()
    assert "gemm_tc_kernel<256, 1, 0>" in text and "frontend_tc_kernel<256>" in text
    shares = [float(l.split("|")[-2].strip().rstrip("%")) for l in text.splitlines() if l.startswith("| `")]
    assert abs(sum(shares) - 100.0) < 1.0


# A stand-in for the reference's model code with its layout (Transformer_Thesis/{transformer_rawIQ,ViT}/models/**.py,
# sub-packages without __init__.py) and two files make_ref.py must leave behind: a non-Python file and a script outside
# models/.  The classes take the reference's constructor arguments.
_STAND_IN_MODELS = {
    "transformer_rawIQ/models/transformer_rawIQ.py": (
        "import torch\nfrom .blocks.head import head\n\n\nclass AMCTransformer(torch.nn.Module):\n"
        "    def __init__(self, in_channels, seq_length, num_classes, device='cpu', **kw):\n"
        "        super().__init__()\n        self.head = head(in_channels * seq_length, num_classes)\n\n"
        "    def forward(self, x):\n        return self.head(x.flatten(1))\n"),
    "transformer_rawIQ/models/blocks/head.py": "import torch\n\n\ndef head(k, n):\n    return torch.nn.Linear(k, n)\n",
    "ViT/models/amc_transformer.py": (
        "import torch\n\n\nclass AMCTransformer(torch.nn.Module):\n"
        "    def __init__(self, in_channels, img_size_h, img_size_w, num_classes, device='cpu', **kw):\n"
        "        super().__init__()\n        self.head = torch.nn.Linear(in_channels * img_size_h * img_size_w, num_classes)\n\n"
        "    def forward(self, x):\n        return self.head(x.flatten(1))\n"),
}
_STAND_IN_OTHER = {"transformer_rawIQ/models/notes.txt": "not Python\n", "ViT/training/train.py": "raise SystemExit\n"}


def _forget_vendored_modules():
    from oracle import make_ref
    for k in [k for k in sys.modules if k.split(".")[0] in make_ref.PACKAGES]:
        del sys.modules[k]


def _run_reference_steps(bench, torch):
    for name, x, n_cls in (("rawiq_seg16_d128_L6", torch.randn(4, 2, 1024), 11),
                           ("vit_p16_d256_L6", torch.randn(4, 1, 32, 64), 19)):
        ref = bench.ReferenceStep(bench.WORKLOADS[name])
        y = torch.randint(0, n_cls, (4,))
        l0 = ref.step(x, y).item()
        l1 = ref.step(x, y).item()
        assert math.isfinite(l0) and math.isfinite(l1)
        yield name, ref


def test_vendored_reference_is_a_byte_copy_and_runs(tmp_path, monkeypatch):
    """oracle/make_ref.py copies the reference's model code unmodified (sha256 manifest) and the copy is importable; the
    reference arm's train step is the reference's own loop body (R/training/train.py:258-271).  The copy is made from a
    stand-in tree; where the reference itself has been vendored into oracle/_ref, that copy is run too."""
    import hashlib

    import torch
    import bench
    from oracle import make_ref
    if bench.reference_available():
        _forget_vendored_modules()
        for name, ref in _run_reference_steps(bench, torch):
            if name == "rawiq_seg16_d128_L6":
                assert sum(p.numel() for p in ref.model.parameters()) == 1985163     # SURVEY §8d cross-check for cfg-1
        _forget_vendored_modules()

    src = tmp_path / "src"
    for rel, text in {**_STAND_IN_MODELS, **_STAND_IN_OTHER}.items():
        f = src / "Transformer_Thesis" / rel
        f.parent.mkdir(parents=True, exist_ok=True)
        f.write_text(text)
    dst = tmp_path / "_ref"
    m = make_ref.vendor(str(src), str(dst))
    assert sorted(m) == sorted(_STAND_IN_MODELS)
    for rel, digest in m.items():
        data = (src / "Transformer_Thesis" / rel).read_bytes()
        assert (dst / rel).read_bytes() == data and digest == hashlib.sha256(data).hexdigest()
    assert json.loads((dst / "MANIFEST.json").read_text())["files"] == m
    assert not (dst / "transformer_rawIQ" / "models" / "notes.txt").exists() and not (dst / "ViT" / "training").exists()
    make_ref.vendor(str(src), str(dst), check=True)
    edited = dst / "ViT" / "models" / "amc_transformer.py"
    edited.write_text(_STAND_IN_MODELS["ViT/models/amc_transformer.py"] + "# edited\n")
    with pytest.raises(SystemExit, match="differs from the reference"):
        make_ref.vendor(str(src), str(dst), check=True)
    edited.write_text(_STAND_IN_MODELS["ViT/models/amc_transformer.py"])

    monkeypatch.setattr(make_ref, "HERE", str(tmp_path))            # load_reference() -> <tmp_path>/_ref
    monkeypatch.setattr(sys, "path", list(sys.path))
    _forget_vendored_modules()
    try:
        for _, ref in _run_reference_steps(bench, torch):
            assert os.path.dirname(sys.modules[type(ref.model).__module__].__file__).startswith(str(dst))
    finally:
        _forget_vendored_modules()


def test_roofline_traffic_is_scaled_to_the_run_batch():
    """`roofline.traffic` comes from an ncu capture that may have been taken at another batch: bench.py scales it and says so."""
    import bench
    table = {"vit_p16_d256_L6": {"gemm_wgrad": {"dram_bytes_per_launch": 100.0, "report": "a.csv", "frames": None},
                                 "attn_fwd": {"dram_bytes_per_launch": 50.0, "report": "b.csv", "frames": 8192}}}
    assert bench.ncu_traffic(table, "vit_p16_d256_L6", "gemm_wgrad", 32768, 32768) == (100.0, "ncu capture at this launch size (a.csv)")
    got, note = bench.ncu_traffic(table, "vit_p16_d256_L6", "attn_fwd", 32768, 32768)
    assert got == 200.0 and "8192" in note and "scaled" in note
    got, note = bench.ncu_traffic(table, "vit_p16_d256_L6", "gemm_wgrad", 4096, 32768)      # --batch 4096 run
    assert got == 12.5 and "scaled" in note
    assert bench.ncu_traffic(table, "vit_p16_d256_L6", "ln_bwd", 32768, 32768) == (None, None)
    assert bench.ncu_traffic(table, "other", "gemm_wgrad", 1, 1) == (None, None)


def test_ncu_full_summary_reads_the_raw_csv_made_on_the_gpu_box(tmp_path, monkeypatch):
    """tools/ncu_summary.py full: per-kernel aggregation of the `ncu --page raw --csv` text (the reports themselves are too
    big to bring back from the GPU box) and the class table bench.py reads; a new capture replaces a class's old entry."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import importlib
    ns = importlib.import_module("ncu_summary")
    csv_text = (
        '"ID","Kernel Name","gpu__time_duration.sum","dram__bytes_read.sum","dram__bytes_write.sum","launch__registers_per_thread"\n'
        '"","","us","Mbyte","Mbyte","register/thread"\n'
        '"0","void amc::<unnamed>::gemm_tc_kernel<256, 1, 0>(CUtensorMap_st, int)","100","300","100","128"\n'
        '"1","void amc::<unnamed>::gemm_tc_kernel<256, 1, 0>(CUtensorMap_st, int)","120","320","80","128"\n'
        '"2","void amc::<unnamed>::attn_tc5_bwd_kernel<2>(CUtensorMap_st)","300","340","170","156"\n')
    src = tmp_path / "cap.csv"
    src.write_text(csv_text)
    monkeypatch.setattr(ns, "ROOT", str(tmp_path))
    os.makedirs(tmp_path / "profiles")
    (tmp_path / "profiles" / "ncu_traffic.json").write_text(json.dumps(
        {"w": {"gemm_wgrad": {"dram_bytes_per_launch": 1.0, "launches": 9, "kernels": ["old"], "report": "old.ncu-rep"}}}))
    out = tmp_path / "sum.json"
    ns.full(str(src), str(out), "w", 4096)
    res = json.loads(out.read_text())["kernels"]
    k = res["gemm_tc_kernel<256, 1, 0>"]
    assert k["launches"] == 2 and abs(k["duration_us_per_launch"] - 110.0) < 1e-6
    assert abs(k["dram_bytes_per_launch"] - 400e6) < 1.0
    tj = json.loads((tmp_path / "profiles" / "ncu_traffic.json").read_text())["w"]
    assert tj["gemm_wgrad"]["report"] == "cap.csv" and tj["gemm_wgrad"]["launches"] == 2 and tj["gemm_wgrad"]["frames"] == 4096
    assert abs(tj["gemm_wgrad"]["dram_bytes_per_launch"] - 400e6) < 1.0
    assert tj["attn_bwd"]["kernels"] == ["attn_tc5_bwd_kernel<2>"] and abs(tj["attn_bwd"]["dram_bytes_per_launch"] - 510e6) < 1.0


def test_dump_outputs_writes_float32_arrays_and_samples_the_large_ones(tmp_path, monkeypatch):
    """--dump-outputs: the last step's logits and updated parameters as DIR/<name>.npy; an array over its element budget
    becomes the same seeded sample of its elements on every run."""
    import types

    import numpy as np
    import torch
    import bench
    model = torch.nn.Sequential(torch.nn.Linear(8, 6), torch.nn.Linear(6, 3))
    logits = torch.randn(5, 3, dtype=torch.float64)
    trainer = types.SimpleNamespace(model=model, _logits=logits)
    bench.dump_outputs(str(tmp_path / "a"), trainer)
    flat = torch.cat([p.detach().reshape(-1) for p in model.parameters()]).numpy()
    got = {n: np.load(tmp_path / "a" / f"{n}.npy") for n in ("logits", "parameters")}
    assert got["logits"].dtype == np.float32 and np.array_equal(got["logits"], logits.float().numpy())
    assert got["parameters"].dtype == np.float32 and np.array_equal(got["parameters"], flat)
    assert sum(bench.DUMP_ELEMS.values()) * 4 <= 64 << 20
    monkeypatch.setitem(bench.DUMP_ELEMS, "parameters", 20)
    bench.dump_outputs(str(tmp_path / "b"), trainer)
    bench.dump_outputs(str(tmp_path / "c"), trainer)
    b, c = np.load(tmp_path / "b" / "parameters.npy"), np.load(tmp_path / "c" / "parameters.npy")
    assert b.shape == (20,) and np.array_equal(b, c) and np.isin(b, flat).all()
    assert np.array_equal(np.load(tmp_path / "b" / "logits.npy"), got["logits"])


@pytest.mark.gpu
def test_bench_dump_outputs_end_to_end(tmp_path):
    """bench.py --steps 3 --dump-outputs DIR on the GPU: the JSON line reports the 3 timed steps and DIR holds the last
    step's logits [batch, classes] and every parameter of the workload's model as finite float32."""
    import numpy as np
    import bench
    from oracle import amc_oracle as O
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "3", "--warmup", "3", "--batch", "512",
                          "--no-cpu-baseline", "--dump-outputs", str(tmp_path)], capture_output=True, text=True,
                         timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == 3 and line["config"]["frames_per_gpu_per_step"] == 512
    w = bench.WORKLOADS[bench.DEFAULT_WORKLOAD]
    logits = np.load(tmp_path / "logits.npy")
    params = np.load(tmp_path / "parameters.npy")
    assert logits.dtype == params.dtype == np.float32
    assert logits.shape == (512, w["kw"]["num_classes"]) and np.isfinite(logits).all()
    kw = {k: v for k, v in w["kw"].items() if k != "drop_prob"}
    assert params.shape == (O.param_count(O.Config(kind=w["kind"], **kw)),) and np.isfinite(params).all()

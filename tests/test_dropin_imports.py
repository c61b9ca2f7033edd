"""The zero-edit switch-over of dropin/: with one shim directory on PYTHONPATH the reference's own import statements
(R/training/train.py:26-29, V/training/train.py:25-28: sys.path.append(root); from models.X import AMCTransformer)
resolve to the B200 modules, while the reference's other packages keep resolving to its own files."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

CASES = {
    "rawiq": ("transformer_rawIQ", "from models.transformer_rawIQ import AMCTransformer", "RawIQAMCTransformer",
              "AMCTransformer(in_channels=2, seq_length=1024, num_classes=11, d_model=128, n_head=8, n_layers=2, "
              "ffn_hidden=512, drop_prob=0.1, device='cpu', use_cls_token=True, embedding_type='segment', segment_size=64)",
              414859),                                                     # R/test_model.py:71-75
    "vit": ("ViT", "from models.amc_transformer import AMCTransformer", "ViTAMCTransformer",
            "AMCTransformer(in_channels=1, img_size_h=32, img_size_w=64, patch_size=4, num_classes=19, d_model=256, "
            "n_head=16, n_layers=6, ffn_hidden=1024, drop_prob=0.15, device='cpu')", 4748051),   # V/main.ipynb:772
}


def _reference_layout(root, kind):
    """A stand-in for the reference's project directory with the layout dropin/README.md describes: ``models/`` has no
    ``__init__.py`` (a namespace package) and holds a module of the name the reference's scripts import -- one that fails
    if it is ever imported instead of the shim -- next to the reference's own ``training/``."""
    sub, stmt = CASES[kind][:2]
    base = root / sub
    (base / "models").mkdir(parents=True)
    (base / "models" / (stmt.split()[1].split(".")[1] + ".py")).write_text(
        "raise ImportError('the reference module was imported instead of the shim')\n")
    (base / "training").mkdir()
    (base / "training" / "train.py").write_text("")
    return str(base)


def _run(kind, cwd, reference_root=None):
    sub, stmt, cls, ctor, n_params = CASES[kind]
    code = "import sys\n"
    if reference_root:
        # what the reference scripts do before importing (train.py: sys.path.append(str(Path(__file__).parent.parent)))
        code += f"sys.path.append({reference_root!r})\n"
    code += (f"{stmt}\nm = {ctor}\n"
             "print(type(m).__module__, type(m).__name__, sum(p.numel() for p in m.parameters()))\n")
    if reference_root:
        code += "import training\nprint(list(training.__path__)[0])\n"
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([ROOT, os.path.join(ROOT, "dropin", kind)]))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, cwd=cwd, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    return r.stdout.strip().splitlines()


@pytest.mark.parametrize("kind", ["rawiq", "vit"])
def test_shim_resolves_the_reference_import_statement(kind, tmp_path):
    out = _run(kind, tmp_path)
    mod, cls, n = out[0].split()
    assert mod.startswith("vit_vs_raw_iq_b200") and cls == CASES[kind][2] and int(n) == CASES[kind][4]


@pytest.mark.parametrize("kind", ["rawiq", "vit"])
def test_shim_wins_over_the_reference_namespace_package(kind, tmp_path):
    ref_root = _reference_layout(tmp_path / "Transformer_Thesis", kind)
    out = _run(kind, tmp_path, reference_root=ref_root)
    mod, cls, n = out[0].split()
    assert mod.startswith("vit_vs_raw_iq_b200") and cls == CASES[kind][2] and int(n) == CASES[kind][4]
    assert out[1].startswith(ref_root)          # training.* is still the reference's

"""vit-vs-raw-iq_b200 -- B200-native (sm_100a) transformer-encoder path of aliftffd/ViT-vs-Raw-IQ.

Import name: ``vit_vs_raw_iq_b200`` (see ``/vit_vs_raw_iq_b200.py`` at the repo root, which maps the
importable name onto this directory).  Importing this package loads the in-tree CUDA library
``lib/libamc_b200.so`` and fails loudly if it has not been built.
"""
from . import _lib  # noqa: F401  (loads the shared library; raises ImportError if missing)
from .modules import (RawIQAMCTransformer, ViTAMCTransformer, default_compute_dtype)  # noqa: F401
from .adversarial import PGDAttack  # noqa: F401

__all__ = ["RawIQAMCTransformer", "ViTAMCTransformer", "default_compute_dtype", "PGDAttack"]

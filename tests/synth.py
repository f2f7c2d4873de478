"""Test-side alias of the package's synthetic weights / inputs (multimodal-rare-disease_b200/synthetic.py)."""

import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import mrd_b200  # noqa: E402,F401  (alias of the hyphenated package)
from importlib import import_module  # noqa: E402

_s = import_module("multimodal-rare-disease_b200.synthetic")
build_model = _s.build_model
sensitise = _s.sensitise
train_weights = _s.train_weights
checksum = _s.checksum
make_inputs = _s.make_inputs
make_global_rows = _s.make_global_rows
tensor_digest = _s.tensor_digest

GOLD = os.path.join(ROOT, "tests", "golden")


def load_train_golden(name):
    """A training-step fixture (oracle/make_golden_train.py).  The post-AdamW parameter samples are stored
    in <name>.post.pt beside <name>.pt, which keeps every fixture file under 1 MB."""
    import torch

    fix = torch.load(os.path.join(GOLD, name + ".pt"))
    fix["post"] = torch.load(os.path.join(GOLD, name + ".post.pt"))
    return fix

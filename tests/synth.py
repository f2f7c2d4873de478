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


def packed(lib, cuda, B, S, seed, lens=None):
    """Token packing of a right-padded batch by mrd_compact_tokens: (live row count n, its device copy, seq_off,
    row_tok, mask, row_bias).  Without `lens` the lengths are uniform in [1, S] (about half the tokens live) and
    n % 64 != 0.  A length of 0 is a sample whose mask is all zero: its CLS row is kept with key bias -inf."""
    import torch

    if lens is None:
        g = torch.Generator().manual_seed(seed)
        lens = torch.randint(1, S + 1, (B,), generator=g)
        if int(lens.sum()) % 64 == 0:
            lens[-1] = lens[-1] - 1 if lens[-1] > 1 else 2
        assert int(lens.sum()) % 64 != 0
    else:
        lens = torch.as_tensor(lens)
        assert lens.numel() == B
    mask = (torch.arange(S)[None, :] < lens[:, None]).long().to(cuda)
    seq_off = torch.zeros(B + 1, device=cuda, dtype=torch.int32)
    # row_tok past the live count keeps valid but unrelated token indices: nothing may use them
    row_tok = torch.randint(0, B * S, (B * S,), device=cuda, dtype=torch.int32)
    row_bias = torch.zeros(B * S, device=cuda)
    n_rows = torch.zeros(1, device=cuda, dtype=torch.int32)
    scratch = torch.zeros(B, device=cuda, dtype=torch.int32)
    rc = lib.mrd_compact_tokens(mask.data_ptr(), 0, B, S, 0, seq_off.data_ptr(), row_tok.data_ptr(),
                                row_bias.data_ptr(), n_rows.data_ptr(), scratch.data_ptr(),
                                torch.cuda.current_stream().cuda_stream)
    assert rc == 0, (rc, lib.mrd_last_error())
    n = int(n_rows.item())
    assert n == int(lens.clamp_min(1).sum())
    return n, n_rows, seq_off, row_tok, mask, row_bias


def load_train_golden(name):
    """A training-step fixture (oracle/make_golden_train.py).  The post-AdamW parameter samples are stored
    in <name>.post.pt beside <name>.pt, which keeps every fixture file under 1 MB."""
    import torch

    fix = torch.load(os.path.join(GOLD, name + ".pt"))
    fix["post"] = torch.load(os.path.join(GOLD, name + ".post.pt"))
    return fix

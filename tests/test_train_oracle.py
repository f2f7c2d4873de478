"""Pins oracle/train_oracle.py (the restated training step) to the reference itself: the fixtures
tests/golden/train_*.pt hold loss, gradients and post-AdamW parameters of the UNMODIFIED reference model
run through one src/train.py-style step with dropout p = 0 (oracle/make_golden_train.py).  CPU only."""

import pytest
import torch

import synth
from oracle import train_oracle as T


def _sample(t, stride):
    return t.detach().float().flatten()[::stride]


@pytest.fixture(scope="module")
def sens():
    return synth.train_weights(0)


@pytest.mark.parametrize("name", ["train_p0_bn_eval_b4_s32", "train_p0_bn_train_b4_s32"])
def test_train_oracle_matches_reference_step(sens, name):
    fix = synth.load_train_golden(name)
    images, ids, mask = synth.make_inputs(fix["B"], fix["S"], fix["seed"], fix["lengths"], H=fix["H"], W=fix["W"])
    labels = torch.tensor(fix["labels"])
    stats = {} if fix["bn_train"] else None
    loss, logits, grads = T.loss_and_grads(sens, images, ids, mask, labels, bn_train=fix["bn_train"], stats=stats)
    assert abs(loss.item() - fix["loss"]) <= 1e-4 * max(1.0, abs(fix["loss"]))
    assert (logits - fix["logits"]).abs().max().item() <= 1e-3 * fix["logits"].abs().max().item()
    # the same parameters receive gradients; the pooler receives none in the reference either
    assert set(grads) == set(fix["grads"])
    assert all(".pooler." in k for k in fix["none_grad"])
    worst = 0.0
    for k, g in grads.items():
        ref = fix["grads"][k]
        assert g.numel() == ref["numel"]
        if ref["norm"] == 0.0:   # query/key projections of the length-1 cross attention: exactly zero
            assert g.abs().max().item() == 0.0, k
            continue
        if ref["norm"] < 1e-5:   # key biases: softmax is shift-invariant, the gradient is rounding noise
            assert g.norm().item() < 1e-5, k
            continue
        err = (_sample(g, ref["stride"]) - ref["sample"]).norm().item() / max(ref["sample"].norm().item(), 1e-20)
        worst = max(worst, err)
        assert abs(g.norm().item() - ref["norm"]) <= 2e-3 * ref["norm"], k
        assert err <= 5e-3, (k, err)
    total = torch.sqrt(sum((g.double() ** 2).sum() for g in grads.values())).item()
    assert abs(total - fix["total_norm"]) <= 1e-3 * fix["total_norm"]
    post = T.clip_and_adamw(sens, grads, lr=fix["lr"], weight_decay=fix["weight_decay"])
    # The first AdamW step moves every element by lr * g / (|g| + eps): ~ +-lr wherever |g| >> eps = 1e-8, and
    # anywhere in between for gradient elements at the rounding-noise level.  So the parameter DELTA is
    # compared in relative L2 (SURVEY.md 8(c)(5)), plus an absolute bound of lr per element.
    worst_delta = 0.0
    for k, p in post.items():
        ref = fix["post"][k]
        pre = _sample(sens[k], ref["stride"])
        d_ref, d_got = ref["sample"] - pre, _sample(p, ref["stride"]) - pre
        assert (d_got - d_ref).abs().max().item() <= 1.05 * fix["lr"], k
        if fix["grads"][k]["norm"] < 1e-5:
            continue
        rel = (d_got - d_ref).norm().item() / max(d_ref.norm().item(), 1e-20)
        worst_delta = max(worst_delta, rel)
        assert rel <= 2e-2, (k, rel)
    if fix["bn_train"]:
        for k, v in fix["running"].items():
            assert torch.allclose(stats[k], v, rtol=1e-4, atol=1e-6), k
    print(name, "worst sampled gradient rel err", worst, "worst parameter-delta rel err", worst_delta)

"""Generates tests/golden/train_*.pt by running the UNMODIFIED reference model (from /root/reference)
through one training step, exactly as src/train.py:247-321 does it:

    model.train(); optimizer.zero_grad(); loss = CrossEntropyLoss()(model(...)["logits"], labels)
    loss.backward(); clip_grad_norm_(model.parameters(), 1.0); AdamW(lr=5e-5, weight_decay=0.05).step()

with every dropout probability set to 0 (the reference's Philox dropout stream cannot be reproduced by
another implementation; SURVEY.md 8(c)(5)).  Two BatchNorm variants: the frozen backbone in eval mode
(running statistics) and in train mode (batch statistics + running-stat update, what a bare
model.train() gives).  Build container only; the GPU box reads the fixtures.

    python oracle/make_golden_train.py
"""

from __future__ import annotations

import os
import sys

import torch
import torch.nn as nn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "oracle"))

import synth  # noqa: E402
from make_golden import build_reference  # noqa: E402

N_SAMPLE = 1024
CASES = {
    # name: (B, S, lengths, H, W, seed, labels, backbone in train mode)
    "train_p0_bn_eval_b4_s32": (4, 32, [32, 20, 7, 1], 64, 64, 41, [3, 1, 7, 3], False),
    "train_p0_bn_train_b4_s32": (4, 32, [32, 20, 7, 1], 64, 64, 41, [3, 1, 7, 3], True),
}


def sample(t: torch.Tensor):
    f = t.detach().float().flatten()
    stride = max(1, f.numel() // N_SAMPLE)
    return {"norm": f.norm().item(), "stride": stride, "sample": f[::stride].clone(), "numel": f.numel()}


def main():
    out_dir = os.path.join(ROOT, "tests", "golden")
    # plain random-init weights: |logits| ~ 0.1, so d(loss)/d(logits) = softmax - onehot is well conditioned.
    # (The sensitised set has |logits| ~ 14: a 1 % forward difference moves the softmax tail by 20 %, which
    # would turn a gradient comparison into a comparison of forward rounding.)  LayerNorm parameters are
    # still sensitised so their gradients are not the trivial gamma = 1 / beta = 0 case.
    mine = synth.build_model(0)
    plain = mine.state_dict()
    full = synth.sensitise(plain, 1)
    sens = {k: (full[k] if ("LayerNorm" in k or "layer_norm" in k) else v.clone()) for k, v in plain.items()}
    torch.set_num_threads(os.cpu_count() or 1)
    for name, (B, S, lengths, H, W, seed, labels, bn_train) in CASES.items():
        ref = build_reference()
        ref.load_state_dict(sens, strict=True)
        for m in ref.modules():
            if isinstance(m, nn.Dropout):
                m.p = 0.0
        ref.train()
        if not bn_train:
            ref.cnn_encoder.backbone.eval()
        images, ids, mask = synth.make_inputs(B, S, seed, lengths, H=H, W=W)
        y = torch.tensor(labels)
        opt = torch.optim.AdamW(ref.parameters(), lr=5e-5, weight_decay=0.05)
        opt.zero_grad()
        out = ref(images, ids, mask)
        loss = nn.CrossEntropyLoss()(out["logits"], y)
        loss.backward()
        named = dict(ref.named_parameters())
        grads = {k: sample(p.grad) for k, p in named.items() if p.grad is not None}
        none_grad = sorted(k for k, p in named.items() if p.requires_grad and p.grad is None)
        total_norm = nn.utils.clip_grad_norm_(ref.parameters(), 1.0)
        opt.step()
        post = {k: sample(p) for k, p in named.items() if p.grad is not None}
        fix = {"weights": "plain+ln", "B": B, "S": S, "lengths": lengths, "H": H, "W": W, "seed": seed,
               "labels": labels, "bn_train": bn_train, "loss": loss.item(), "logits": out["logits"].detach().clone(),
               "grads": grads, "none_grad": none_grad, "total_norm": float(total_norm), "post": post,
               "lr": 5e-5, "weight_decay": 0.05}
        if bn_train:
            sd = ref.state_dict()
            fix["running"] = {k: sd[k].clone() for k in ("cnn_encoder.backbone.bn1.running_mean",
                                                         "cnn_encoder.backbone.bn1.running_var",
                                                         "cnn_encoder.backbone.layer1.0.bn3.running_var",
                                                         "cnn_encoder.backbone.layer3.2.bn2.running_mean",
                                                         "cnn_encoder.backbone.layer4.2.bn3.running_var",
                                                         "cnn_encoder.backbone.layer4.0.downsample.1.running_mean")}
            fix["num_batches_tracked"] = int(sd["cnn_encoder.backbone.bn1.num_batches_tracked"])
        # two files, each under 1 MB: tests/synth.py load_train_golden() joins them
        torch.save(fix.pop("post"), os.path.join(out_dir, name + ".post.pt"))
        torch.save(fix, os.path.join(out_dir, name + ".pt"))
        print(name, "loss", loss.item(), "grad norm", float(total_norm), "params with grad", len(grads),
              "requires_grad but None:", len(none_grad))


if __name__ == "__main__":
    main()

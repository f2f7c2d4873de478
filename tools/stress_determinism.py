#!/usr/bin/env python
"""Run-to-run determinism of the forward as shipped: the same 1024-sample batch is pushed through the model `reps`
times and the logits digests are compared (the forward has no atomics whose result depends on order - red.max is
order-independent - so any difference is a synchronisation bug).

    python tools/stress_determinism.py [reps] [batch]
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import mrd_b200  # noqa: E402,F401
from importlib import import_module  # noqa: E402

synth = import_module("multimodal-rare-disease_b200.synthetic")
reps = int(sys.argv[1]) if len(sys.argv) > 1 else 12
batch = int(sys.argv[2]) if len(sys.argv) > 2 else 1024
dev = torch.device("cuda:0")
images, ids, mask = (t.to(dev) for t in synth.make_global_rows(0, batch))
model = synth.build_model(0).to(dev)
digests = {}
first = None
for r in range(reps):
    with torch.no_grad():
        out = model(images, ids, mask)["logits"].clone()
    torch.cuda.synchronize()
    d = synth.tensor_digest(out)[:12]
    digests[d] = digests.get(d, 0) + 1
    if first is None:
        first = out
    elif d != synth.tensor_digest(first)[:12]:
        diff = (out - first).abs()
        rows = (diff.max(dim=1).values > 0).nonzero().flatten().tolist()
        print(f"   rep {r}: {len(rows)} rows differ (first {rows[:8]}), max |diff| {diff.max().item():.3e}")
ok = len(digests) == 1
print("deterministic" if ok else "NOT deterministic", digests)
sys.exit(0 if ok else 1)

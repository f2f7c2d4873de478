#!/usr/bin/env python
"""Input saliency (images.grad through the frozen ResNet50 backbone) against the plain eval forward, B = 64, 224 x 224,
128 tokens.

    python tools/bench_saliency.py [--json OUT.json]

Times (CUDA events, after warm-up) the benchmarked eval forward under torch.no_grad() and forward + logits[:, c].sum()
.backward() with images.requires_grad, reports saliency maps per second, then - in a separate profiled pass - the
device time of every data-gradient label of mrd_ctx_profile with its achieved TFLOP/s (FLOPs from the shapes: 2 x
output elements x input channels x taps for the GEMM launches; the stem's data gradient 2 x 112*112*64 x 3*49 per
image)."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch  # noqa: E402

import synth  # noqa: E402


def timed_ms(fn, reps, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--json", default=None, help="also write the results to this file")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--batch", type=int, default=64)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark needs a GPU"
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    res = {"device": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit": smi[0] if smi else None}
    print("device:", res["device"], "|", res["nvidia_smi_name_power_limit"])
    dev = torch.device("cuda:0")
    B = args.batch
    model = synth.build_model(0).to(dev).eval()
    images, ids, mask = synth.make_inputs(B, 128, 11)
    images, ids, mask = images.to(dev), ids.to(dev), mask.to(dev)
    cls = torch.randint(0, model.num_classes, (B,), generator=torch.Generator().manual_seed(3)).to(dev)

    def plain():
        with torch.no_grad():
            model(images, ids, mask)

    def saliency():
        x = images.clone().requires_grad_(True)
        logits = model(x, ids, mask)["logits"]
        logits.gather(1, cls[:, None]).sum().backward()
        return x.grad

    t_plain = timed_ms(plain, args.reps)
    t_sal = timed_ms(saliency, args.reps)
    res.update({"B": B, "H": 224, "W": 224, "S": 128, "eval_forward_ms": t_plain, "forward_plus_images_grad_ms": t_sal,
                "saliency_maps_per_s": B / t_sal * 1e3, "eval_forward_samples_per_s": B / t_plain * 1e3})
    print(f"B={B}: eval forward {t_plain:.2f} ms ({B / t_plain * 1e3:.0f} samples/s); forward + images.grad "
          f"{t_sal:.2f} ms ({B / t_sal * 1e3:.0f} saliency maps/s)")

    eng = model._engine(allow_training=True)
    torch.cuda.synchronize()
    eng.profile(True)
    saliency()
    torch.cuda.synchronize()
    rows = eng.profile_report()
    eng.profile(False)
    stem_flops = 2.0 * B * 112 * 112 * 64 * 3 * 49
    agg = {}
    for r in rows:
        if not r["label"].startswith("dgrad"):
            continue
        a = agg.setdefault(r["label"], {"launches": 0, "ms": 0.0, "flops": 0.0})
        a["launches"] += r["launches"]
        a["ms"] += r["ms"]
        a["flops"] += stem_flops if r["label"] == "dgrad.stem" else r["flops"]
    fwd_ms = sum(a["ms"] for k, a in agg.items() if k.startswith("dgrad_fwd"))
    bwd_ms = sum(a["ms"] for k, a in agg.items() if not k.startswith("dgrad_fwd"))
    res["profile"] = {}
    print(f"{'label':28s} {'launches':>8s} {'ms':>8s} {'TFLOP/s':>8s}")
    for k, a in sorted(agg.items(), key=lambda kv: -kv[1]["ms"]):
        tf = a["flops"] / a["ms"] / 1e9 if a["ms"] > 0 and a["flops"] > 0 else None
        res["profile"][k] = dict(a, tflops=tf)
        print(f"{k:28s} {a['launches']:8d} {a['ms']:8.3f} {tf if tf is not None else float('nan'):8.1f}")
    res["saving_forward_ms"] = fwd_ms
    res["backbone_backward_ms"] = bwd_ms
    print(f"profiled: saving forward of the backbone {fwd_ms:.2f} ms, backbone data-gradient backward {bwd_ms:.2f} ms")
    if args.json:
        with open(args.json, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()

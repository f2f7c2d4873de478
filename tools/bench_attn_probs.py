#!/usr/bin/env python
"""Write bandwidth of the attention-probabilities kernel (mrd_attention_probs_bf16) at shapes whose output is larger
than the 126 MB L2, and TextEncoder.get_attention_weights against get_all_hidden_states end to end.

    python tools/bench_attn_probs.py [--json OUT.json]

Bytes counted per call: the written probabilities (B*heads*S*S*4) plus the Q block and the sample's keys that every
(sample, head, 128-query block) reads (2 * B*S*heads*64 * (1 + ceil(S/128)) bytes of bf16)."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import mrd_b200  # noqa: E402,F401
from importlib import import_module  # noqa: E402


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
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark needs a GPU"
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    res = {"device": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit": smi[0] if smi else None,
           "kernel": [], "module": {}}
    print("device:", res["device"], "|", res["nvidia_smi_name_power_limit"])

    lib = import_module("multimodal-rare-disease_b200._lib").load()
    dev = torch.device("cuda:0")
    H = 12
    for B, S in ((256, 128), (32, 512)):
        g = torch.Generator(device="cuda").manual_seed(S)
        qkv = (torch.randn(B * S, 3 * H * 64, device=dev, generator=g) * 0.5).to(torch.bfloat16)
        lens = torch.randint(S // 2, S + 1, (B,), device=dev, generator=g)
        bias = torch.where(torch.arange(S, device=dev)[None, :] < lens[:, None], 0.0, float("-inf")).float()
        probs = torch.empty(B, H, S, S, device=dev)
        stream = torch.cuda.current_stream().cuda_stream

        def call():
            rc = lib.mrd_attention_probs_bf16(qkv.data_ptr(), bias.data_ptr(), B, S, H, probs.data_ptr(), stream)
            assert rc == 0, lib.mrd_last_error()

        ms = timed_ms(call, args.reps)
        out_bytes = B * H * S * S * 4
        in_bytes = 2 * B * S * H * 64 * (1 + (S + 127) // 128)
        row = {"B": B, "S": S, "heads": H, "ms": ms, "out_MB": out_bytes / 1e6, "in_MB": in_bytes / 1e6,
               "TB_per_s": (out_bytes + in_bytes) / ms / 1e9}
        res["kernel"].append(row)
        print(f"mrd_attention_probs_bf16 B={B} S={S} H={H}: {ms * 1e3:.1f} us, {row['out_MB']:.0f} MB written, "
              f"{row['TB_per_s']:.2f} TB/s")
        del qkv, probs

    te_mod = import_module("multimodal-rare-disease_b200.text_encoder")
    te = te_mod.TextEncoder(random_init=True).to(dev).eval()
    B, S = 64, 128
    g = torch.Generator().manual_seed(7)
    ids = torch.randint(1, 28000, (B, S), generator=g)
    ids[:, 0] = 101
    lens = torch.randint(16, S + 1, (B,), generator=g)
    mask = (torch.arange(S)[None, :] < lens[:, None]).long()
    ids, mask = ids.to(dev), mask.to(dev)
    te.encoder.set_attn_implementation("eager")
    with torch.no_grad():
        t_attn = timed_ms(lambda: te.get_attention_weights(ids, mask), 10)
        t_hidden = timed_ms(lambda: te.get_all_hidden_states(ids, mask), 10)
        t_fwd = timed_ms(lambda: te(ids, mask), 10)
    L = len(te.encoder.encoder.layer)
    res["module"] = {"B": B, "S": S, "get_attention_weights_ms": t_attn, "get_all_hidden_states_ms": t_hidden,
                     "forward_ms": t_fwd, "attentions_MB": L * B * H * S * S * 4 / 1e6,
                     "hidden_states_MB": (L + 1) * B * S * 768 * 4 / 1e6}
    print(f"B={B} S={S}: get_attention_weights {t_attn:.3f} ms ({res['module']['attentions_MB']:.0f} MB out), "
          f"get_all_hidden_states {t_hidden:.3f} ms ({res['module']['hidden_states_MB']:.0f} MB out), "
          f"forward {t_fwd:.3f} ms")
    if args.json:
        with open(args.json, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()

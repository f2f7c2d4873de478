#!/usr/bin/env python
"""Benchmark of the hot path: batched MultimodalClassifier forward (BASELINE.json configs[3]).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU forward (oracle port)

Workload ("step"): one full multimodal inference pass over a GLOBAL batch of 4096 synthetic samples
(224x224 fp32 images + 128 tokens with padding masks L ~ U{16..128}), sharded data-parallel over the
N GPUs of one box (4096/N samples per rank, replicated random-init weights), followed by the NCCL
all-gather of the [4096,10] logits.  Total work is fixed as N grows -> "scaling": "strong".

value  = samples/s with the inputs already resident in HBM, timed with CUDA events over exactly K
         steps (barrier + synchronize on both sides, max over ranks).  The per-rank inputs
         (>= 308 MB even at N=8) exceed the 126 MB L2, so no L2 flush is needed between steps.
e2e    = the same metric through the public module API starting from pinned HOST buffers: every step
         copies this rank's images/ids/mask host->device and reads the gathered logits back.
roofline = the dominant kernel family (tcgen05 implicit-GEMM: all convolutions and linears), measured
         in a separate profiled step with CUDA events around every launch on the launching stream.
cpu_baseline = the oracle port of the reference forward (oracle/forward_oracle.py, fp32, all host
         threads) timed on a bounded sample of the same workload, rank 0, N=1 only.

--dump-outputs DIR writes what the last timed step returned, so that two builds can be compared output for
output on the same seeded inputs: DIR/logits.npy (the gathered [global_batch, 10] logits) and, unless
--no-e2e, DIR/e2e_logits.npy (the same through the host path), float32.
"""

from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "fused fwd samples/sec (224² img+128 tok) @1/2/4/8 B200; % tensor-pipe peak"
UNIT = "samples/s"
FLOP_PER_SAMPLE = 30.53e9  # BASELINE.md section 2: full multimodal forward, S=128
SEQ = 128
IMG = 224
DUMP_LIMIT = 64 << 20  # bytes of --dump-outputs in all


def _peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            p = json.load(fh)
        return {"src": "measured", "bf16_burst": p.get("bf16_tflops", 1590.0),
                "bf16_sustained": p.get("bf16_tflops_sustained", 1400.0), "hbm": p.get("hbm_gbs", 6650.0)}
    return {"src": "fallback", "bf16_burst": 1590.0, "bf16_sustained": 1400.0, "hbm": 6650.0}


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled every 200 ms while the timed region runs."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
            except (ValueError, IndexError):
                continue
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx,
                "samples": len(sm), "reasons": sorted(reasons)}


def _ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel family, from the
    committed ncu capture of this same command (profiles/rNN_traffic.json, newest round); None when absent."""
    for name in ("r02_traffic.json", "r01_traffic.json"):
        path = os.path.join(ROOT, "profiles", name)
        if os.path.exists(path):
            with open(path) as fh:
                return json.load(fh)
    return None


def _synthetic():
    import mrd_b200  # noqa: F401  (alias of the hyphenated package)
    from importlib import import_module

    return import_module("multimodal-rare-disease_b200.synthetic")


def make_shard(lo, hi, device=None, pin=False):
    """Rows [lo, hi) of the GLOBAL synthetic batch (SURVEY.md 8(d) cfg 4: randn images, ids with [CLS] first
    and 0 on the padded tail, prefix masks with L ~ U{16..128}).  Generated by global sample index
    (synthetic.make_global_rows), so the union over the ranks is the same batch at every world size."""
    images, ids, mask = _synthetic().make_global_rows(lo, hi, SEQ, IMG, 16, 1234)
    if pin:
        return images.pin_memory(), ids.pin_memory(), mask.pin_memory()
    if device is not None:
        return images.to(device), ids.to(device), mask.to(device)
    return images, ids, mask


def dump_outputs(out_dir, arrays):
    """Writes out_dir/<name>.npy for each [rows, ...] float32 array (all with the same rows).  Above DUMP_LIMIT
    bytes in all, every array keeps the same fixed, seeded sample of rows, listed in rows.npy (float64)."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    n = next(iter(arrays.values())).shape[0]
    keep = (DUMP_LIMIT - 4096) // (sum(a[:1].nbytes for a in arrays.values()) + 8)  # 4096: room for the npy headers
    if n > keep:
        rows = np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
        arrays = {k: a[rows] for k, a in arrays.items()}
        arrays["rows"] = rows.astype(np.float64)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def cpu_forward_timer(samples: int, iters: int, warmup: int):
    """Times the oracle port (the reference's algorithm, fp32, ATen CPU kernels, all host threads)."""
    import torch

    from oracle import forward_oracle as oracle

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    model = _synthetic().build_model(0)
    sd = {k: v.float() for k, v in model.state_dict().items() if v.is_floating_point()}
    images, ids, mask = make_shard(0, samples)
    times = []
    for i in range(warmup + iters):
        t0 = time.perf_counter()
        oracle.multimodal_forward(sd, images, ids, mask)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    return samples / statistics.mean(times), statistics.mean(times), cores, torch.get_num_threads()


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    samples = args.cpu_samples
    value, sec, cores, threads = cpu_forward_timer(samples, args.steps, args.warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": _config(args, 1),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": f"{samples} samples of the workload per step (oracle/forward_oracle.py, "
                                   f"fp32, {threads} threads of {cores} host cores)"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


def _config(args, world):
    return {"workload": "configs[3]: full multimodal inference (ResNet50 + BioBERT-base + attention fusion + "
                        f"head), global batch {args.global_batch} data-parallel, 224x224 fp32 images, "
                        f"{SEQ} tokens, padding masks L~U{{16..128}}, logits all-gather",
            "global_batch": args.global_batch, "per_gpu_batch": -(-args.global_batch // world),
            "seq_len": SEQ, "image": IMG, "parallelism": f"dp{world}",
            "l2": "per-rank inputs exceed L2 (>= 308 MB vs 126 MB); no flush between steps",
            # 0 = the engine's defaults: up to 2048 images per ResNet pass, 524288 tokens per BERT pass
            "img_chunk": args.img_chunk, "tok_chunk": args.tok_chunk, "engine_opts": args.engine_opt}


def _timed_ms(fn, iters, warmup):
    import torch

    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def other_configs(model, dev, peaks, iters=10, warmup=3):
    """Short CUDA-event timings of the other BASELINE.json configs on one GPU (inputs resident in HBM, L2 not
    flushed: every case's inputs + activations exceed the 126 MB L2).  They are reported in the N=1 line so the
    driver's BENCH record holds them; the bench metric itself is configs[3].
      configs[1] image_only : CNNEncoder forward, batch 256, 224x224 bf16 NCHW input
      configs[2] text_only  : TextEncoder forward, batch 256 x 512 tokens, masks L~U{64..512} and all-live
      configs[4] training   : fwd + bwd + clip + AdamW, batch 64, 128 tokens (L~U{16..128}), default freeze
                              configuration; the reference's loop with torch.optim.AdamW and with FusedAdamW"""
    import copy

    import torch
    import torch.nn as nn

    import mrd_b200

    burst = peaks["bf16_burst"] * 1e12
    out = {}
    g = torch.Generator().manual_seed(99)
    sampler = ClockSampler(dev.index or 0)
    sampler.start()
    with torch.no_grad():
        B = 256
        images = torch.randn(B, 3, IMG, IMG, generator=g).to(dev, torch.bfloat16)
        ms = _timed_ms(lambda: model.cnn_encoder(images), iters, warmup)
        out["image_only_b256_bf16"] = {"value": B / (ms * 1e-3), "unit": "img/s", "ms": ms,
                                       "tensor_peak_frac": B / (ms * 1e-3) * 8.1769e9 / burst}
        del images
        for name, lo_len in (("text_only_b256_s512_padded", 64), ("text_only_b256_s512_all_live", 512)):
            S = 512
            ids = torch.randint(1, 28996, (B, S), generator=g)
            lengths = torch.randint(lo_len, S + 1, (B,), generator=g)
            mask = (torch.arange(S).unsqueeze(0) < lengths.unsqueeze(1)).long()
            ids = ids * mask
            ids[:, 0] = 101
            ids, mask = ids.to(dev), mask.to(dev)
            ms = _timed_ms(lambda: model.text_encoder(ids, mask), iters, warmup)
            f_dense = 169.869e6 * S + 36864.0 * S * S
            out[name] = {"value": B / (ms * 1e-3), "unit": "seq/s", "ms": ms,
                         "live_token_fraction": float(mask.float().mean()),
                         "tensor_peak_frac": B / (ms * 1e-3) * f_dense / burst}
    # ---- configs[4]: the reference's training loop body (src/train.py:247-321) on a copy of the model
    Bt, S = 64, SEQ
    images, ids, mask = make_shard(0, Bt, device=dev)
    labels = torch.randint(0, 10, (Bt,), generator=g).to(dev)
    crit = nn.CrossEntropyLoss()
    for name, native in (("train_b64_torch_adamw", False), ("train_b64_fused_adamw", True)):
        m = copy.deepcopy(model).train()
        if native:
            opt = mrd_b200.FusedAdamW(m.parameters(), lr=5e-5, weight_decay=0.05, max_grad_norm=1.0)
        else:
            opt = torch.optim.AdamW(m.parameters(), lr=5e-5, weight_decay=0.05)

        def step():
            opt.zero_grad(set_to_none=True)
            loss = crit(m(images, ids, mask)["logits"], labels)
            loss.backward()
            if not native:
                nn.utils.clip_grad_norm_(m.parameters(), 1.0)
            opt.step()
            return loss

        first = step().item()
        ms = _timed_ms(step, 2 * iters, warmup)
        last = step().item()
        out[name] = {"value": Bt / (ms * 1e-3), "unit": "samples/s", "ms": ms, "loss_first_last": [first, last],
                     "optimizer": "mrd_b200.FusedAdamW(max_grad_norm=1)" if native
                     else "clip_grad_norm_ + torch.optim.AdamW", "bn": "batch statistics (bare model.train())"}
        del m, opt
    out["clocks"] = sampler.stop()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--global-batch", type=int, default=4096)
    ap.add_argument("--img-chunk", type=int, default=0)
    ap.add_argument("--tok-chunk", type=int, default=0)
    ap.add_argument("--cpu-samples", type=int, default=128,
                    help="samples per CPU pass: the reference arm's step, and (x2) the cpu_baseline leg")
    ap.add_argument("--micro-batch", type=int, default=2048)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--profile-out", default="")
    ap.add_argument("--engine-opt", action="append", default=[], metavar="KEY=VALUE",
                    help="mrd_ctx_set_option switches for A/B runs, e.g. fuse_ds=0")
    ap.add_argument("--no-other-configs", action="store_true",
                    help="skip the short timings of configs[1], [2] and [4] in the N=1 line")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write the logits of the last timed step as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 path")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        return run_reference(args)

    # dump all stacks and exit instead of hanging a GPU box (a healthy run takes 1-2 minutes)
    import faulthandler

    faulthandler.dump_traceback_later(int(os.environ.get("MRD_BENCH_WATCHDOG", "1500")), exit=True)
    import torch
    import torch.distributed as dist

    import mrd_b200

    synth = _synthetic()
    # torchrun pins OMP_NUM_THREADS=1; the synthetic host data (randn of the image shard) and the
    # model construction are CPU work outside the timed region - give them the rank's share of cores
    torch.set_num_threads(max(1, (os.cpu_count() or 1) // max(1, int(os.environ.get("LOCAL_WORLD_SIZE", "1")))))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the B200 path has no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    total = args.global_batch
    lo, hi = mrd_b200.shard_bounds(total, world, rank)
    n_local = hi - lo
    model = synth.build_model(0).to(dev)
    model.configure_b200(args.img_chunk, args.tok_chunk)
    eng = model._engine()
    for kv in args.engine_opt:
        k, v = kv.split("=", 1)
        eng.set_option(k, float(v))
    dp = mrd_b200.DataParallelForward(
        lambda im, i, m, out: model(im, i, m, logits_out=out), model.num_classes)

    # ---------------------------------------------------------------- value: inputs resident in HBM
    images, ids, mask = make_shard(lo, hi, device=dev)

    def step():
        with torch.no_grad():
            return dp.forward_shard(images, ids, mask, total)

    for _ in range(args.warmup):
        step()
    barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    l0 = eng.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        logits = step()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    launches = eng.launch_count - l0
    clocks = sampler.stop() if sampler else None
    # tokens the packed BERT path actually processes (mask != 0, CLS always kept) vs the dense count
    live = ((mask != 0) | (torch.arange(SEQ, device=dev) == 0))
    live_frac = float(live.float().mean().item())
    # attention work on live tokens only: sum_b L_b^2 against B*S^2
    live_sq_frac = float((live.sum(1).double() ** 2).sum().item() / (mask.shape[0] * SEQ * SEQ))
    t = torch.tensor([ms, float(launches)], device=dev, dtype=torch.float64)
    if world > 1:
        tmax = t.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        ms, launches = tmax[0].item(), int(t[1].item())
    ms_per_step = ms / args.steps
    value = total / (ms_per_step * 1e-3)
    assert logits.shape == (total, model.num_classes) and bool(torch.isfinite(logits).all())
    # bit-exact digest of the gathered logits: inputs are generated by global sample index and no op of the
    # forward mixes samples, so this is the same string at N = 1, 2, 4, 8 (SURVEY.md section 4(iv))
    logits_digest = synth.tensor_digest(logits) if rank == 0 else None
    # host copy now: the e2e path below writes into the same gather buffer
    dumps = {"logits": logits.float().cpu().numpy()} if rank == 0 and args.dump_outputs else None

    # ---------------------------------------------------------------- e2e: host buffers -> logits on host
    e2e = None
    if not args.no_e2e:
        h_images, h_ids, h_mask = make_shard(lo, hi, pin=True)
        h_logits = torch.empty(total, model.num_classes, dtype=torch.float32).pin_memory()

        def e2e_step():
            with torch.no_grad():
                out = dp.forward_shard_host(
                    lambda im, i, m, o: model.forward_host(im, i, m, micro_batch=args.micro_batch, logits_out=o,
                                                           next_batch=(im, i, m)),
                    h_images, h_ids, h_mask, total, dev)
                h_logits.copy_(out, non_blocking=True)

        for _ in range(args.warmup):
            e2e_step()
        barrier()
        e0.record()
        for _ in range(args.steps):
            e2e_step()
        e1.record()
        barrier()
        ems = e0.elapsed_time(e1)
        if world > 1:
            tt = torch.tensor([ems], device=dev, dtype=torch.float64)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            ems = tt.item()
        if dumps is not None:
            dumps["e2e_logits"] = h_logits.numpy().copy()
        h2d = sum(x.numel() * x.element_size() for x in (h_images, h_ids, h_mask))
        e2e = {"value": total / (ems / args.steps * 1e-3), "unit": UNIT,
               "logits_sha256": synth.tensor_digest(h_logits) if rank == 0 else None,
               "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": h_logits.numel() * 4,
               "ms_per_step": ems / args.steps,
               "path": "pinned host tensors -> MultimodalClassifier.forward_host (H2D of micro-batch i+1 on a copy "
                       f"stream under the kernels of micro-batch i, micro_batch={args.micro_batch}; the first micro-batch of the next "
                       f"step is copied under the last one of this step, as a loader that holds the next batch would) -> logits "
                       "all-gather -> pinned host"}

    # ---------------------------------------------------------------- roofline: profiled step (rank 0)
    roofline, families = None, None
    peaks = _peaks()
    if rank == 0:
        eng.profile(True)
        with torch.no_grad():
            model(images, ids, mask)  # local shard only: no collective, the other ranks are not in this step
        rows = eng.profile_report()
        eng.profile(False)
        # executed work: the token-packed BERT GEMMs run on the live rows only (their plans - and so the
        # library's per-launch FLOP figures - are sized for the dense B*S rows), attention on L_b^2 per sample
        packed = ("bert.qkv", "bert.attn_out+res", "bert.attn_out+res+ln", "bert.ffn1+gelu", "bert.ffn2+res",
                  "bert.ffn2+res+ln")
        for r in rows:
            r["flops_exec"] = r["flops"] * (live_frac if r["label"] in packed else
                                            live_sq_frac if r["label"] == "bert.attention" else 1.0)
        tens = [r for r in rows if r["cat"] == "tensor"]
        t_ms = sum(r["ms"] for r in tens)
        t_fl = sum(r["flops"] for r in tens)
        t_fx = sum(r["flops_exec"] for r in tens)
        n_l = sum(r["launches"] for r in tens)
        all_ms = sum(r["ms"] for r in rows)
        achieved = t_fl / (t_ms * 1e-3) / 1e12 if t_ms > 0 else 0.0
        executed = t_fx / (t_ms * 1e-3) / 1e12 if t_ms > 0 else 0.0
        exec_flop_per_sample = sum(r["flops_exec"] for r in rows) / max(n_local, 1)
        roofline = {"bound": "tensor", "kernel": "conv_gemm_kernel (tcgen05 implicit-GEMM: 53 convs + all linears)",
                    "achieved": achieved, "peak": peaks["bf16_sustained"], "unit": "TFLOP/s",
                    "frac": achieved / peaks["bf16_sustained"],
                    # the hardware number: FLOPs the launches really executed (live tokens only) per second
                    "achieved_executed": executed, "frac_executed": executed / peaks["bf16_sustained"],
                    "peak_source": peaks["src"] + " (sustained: timed inside a long step)",
                    "launches_per_step": n_l, "avg_launch_ms": t_ms / max(n_l, 1),
                    "flops_per_launch_avg": t_fl / max(n_l, 1), "flops_executed_per_launch_avg": t_fx / max(n_l, 1),
                    "share_of_step": t_ms / all_ms if all_ms else None,
                    # DRAM bytes per launch of this kernel family (dram__bytes_read.sum + dram__bytes_write.sum, ncu);
                    # the capture it comes from is described in traffic_detail
                    "traffic": (_ncu_traffic() or {}).get("dram_bytes_per_launch"),
                    "traffic_detail": _ncu_traffic(),
                    "note": "achieved / frac count ALGORITHMIC flops (dense, as the reference executes; SURVEY 8(d)); "
                            "achieved_executed / frac_executed count what the kernels ran: the BERT launches skip padded "
                            f"tokens (live fraction {live_frac:.3f} of B*S) and the last layer's post-attention half runs on "
                            "CLS rows only."}
        fam = {}
        for r in rows:
            f = fam.setdefault(r["cat"], {"ms": 0.0, "flops": 0.0, "bytes": 0.0, "launches": 0})
            f["ms"] += r["ms"]; f["flops"] += r["flops"]; f["bytes"] += r["bytes"]; f["launches"] += r["launches"]
        families = {k: {"ms": round(v["ms"], 3), "launches": v["launches"],
                        "tflops": round(v["flops"] / (v["ms"] * 1e-3) / 1e12, 1) if v["ms"] else 0,
                        "gbs": round(v["bytes"] / (v["ms"] * 1e-3) / 1e9, 1) if v["ms"] else 0}
                    for k, v in fam.items()}
        if args.profile_out:
            with open(args.profile_out, "w") as fh:
                fh.write("label,category,launches,total_ms,tflops,tflops_executed,gbs,share\n")
                for r in sorted(rows, key=lambda r: -r["ms"]):
                    sec = r["ms"] * 1e-3
                    fh.write(f'{r["label"]},{r["cat"]},{r["launches"]},{r["ms"]:.4f},'
                             f'{r["flops"] / sec / 1e12 if sec else 0:.1f},'
                             f'{r["flops_exec"] / sec / 1e12 if sec else 0:.1f},'
                             f'{r["bytes"] / sec / 1e9 if sec else 0:.1f},'
                             f'{r["ms"] / all_ms:.4f}\n')

    # ---------------------------------------------------------------- CPU baseline (rank 0, N=1)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        n_cpu = 2 * args.cpu_samples   # ~6 s per pass on 16 cores: 1 warm-up + 2 timed passes = ~20 s of CPU work
        v, sec, cores, threads = cpu_forward_timer(n_cpu, 2, 1)
        cpu = {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
               "sample": f"{n_cpu} samples of the same workload, 1 warm-up + 2 timed passes, "
                         f"{sec:.2f} s per pass (oracle/forward_oracle.py, fp32, {threads} threads of {cores} host cores)"}

    others = None
    if rank == 0 and world == 1 and not args.no_other_configs:
        others = other_configs(model, dev, peaks)

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": _config(args, world),
            "tensor_peak_frac": value * FLOP_PER_SAMPLE / (world * peaks["bf16_burst"] * 1e12),
            "tensor_peak_tflops": peaks["bf16_burst"], "flop_per_sample": FLOP_PER_SAMPLE,
            # the same with the FLOPs the kernels executed (padded tokens and the CLS-only tail not counted)
            "tensor_peak_frac_executed": (value * exec_flop_per_sample / (world * peaks["bf16_burst"] * 1e12)
                                          if roofline else None),
            "flop_per_sample_executed": exec_flop_per_sample if roofline else None,
            "logits_sha256": logits_digest,
            "e2e_logits_match": (e2e["logits_sha256"] == logits_digest) if e2e else None,
            "other_configs": others,
            "e2e": e2e, "gpu_launches": launches, "clocks": clocks, "roofline": roofline,
            "kernel_families": families, "cpu_baseline": cpu, "bert_live_token_fraction": live_frac,
            "device_bytes": eng.device_bytes,
        }
        if dumps is not None:
            dump_outputs(args.dump_outputs, dumps)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())

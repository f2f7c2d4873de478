#!/usr/bin/env python
"""Timing of single GEMM launches at the BERT shapes of the benchmark (74 k live tokens per pass).
    python tools/bench_gemm_shapes.py [M]"""
import ctypes as C
import math
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import mrd_b200  # noqa: E402,F401
from importlib import import_module  # noqa: E402

lib = import_module("multimodal-rare-disease_b200._lib").load()
dev = torch.device("cuda:0")
BF = torch.bfloat16
M = int(sys.argv[1]) if len(sys.argv) > 1 else 74000
s = lambda: C.c_void_p(torch.cuda.current_stream().cuda_stream)  # noqa: E731
print("env:", {k: v for k, v in os.environ.items() if k.startswith("MRD_DEBUG")})
for name, N, K, act, res in (("qkv", 2304, 768, 0, False), ("attn_out+res", 768, 768, 0, True),
                             ("ffn1+gelu", 3072, 768, 2, False), ("ffn2+res", 768, 3072, 0, True),
                             ("ffn2 no res", 768, 3072, 0, False), ("l3.conv3+res", 1024, 256, 1, True)):
    g = torch.Generator(device="cuda").manual_seed(K + N)
    A = torch.randn(M, K, device=dev, generator=g).to(BF)
    W = (torch.randn(N, K, device=dev, generator=g) / math.sqrt(K)).to(BF)
    bias = torch.randn(N, device=dev, generator=g)
    R = torch.randn(M, N, device=dev, generator=g).to(BF) if res else None
    Cc = torch.empty(M, N, device=dev, dtype=BF)

    def run():
        assert lib.mrd_gemm_bf16(A.data_ptr(), K, M, K, W.data_ptr(), N, bias.data_ptr(), Cc.data_ptr(), N,
                                 R.data_ptr() if res else None, N, None, 0, act, s()) == 0, lib.mrd_last_error()
    for _ in range(3):
        run()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(20):
        run()
    e1.record()
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) / 20 * 1e3
    print(f"{name:14s} M={M} N={N} K={K}: {us:8.1f} us  {2.0 * M * N * K / us / 1e6:7.0f} TFLOP/s", flush=True)

#!/usr/bin/env python
"""Timing of dense + residual + LayerNorm: one launch (mrd_gemm_ln_bf16) against the plain GEMM followed by the
LayerNorm launch, at BERT shapes.    python tools/bench_gemm_ln.py [M]"""
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


def timed(fn, reps=20):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps * 1e3


for K in (768, 3072):
    N = 768
    g = torch.Generator(device="cuda").manual_seed(K)
    A = torch.randn(M, K, device=dev, generator=g).to(BF)
    W = (torch.randn(N, K, device=dev, generator=g) / math.sqrt(K)).to(BF)
    bias = torch.randn(N, device=dev, generator=g)
    R = torch.randn(M, N, device=dev, generator=g).to(BF)
    gamma = torch.rand(N, device=dev, generator=g) + 0.5
    beta = torch.randn(N, device=dev, generator=g)
    T = torch.empty(M, N, device=dev, dtype=BF)
    Cc = torch.empty(M, N, device=dev, dtype=BF)

    def plain():
        assert lib.mrd_gemm_bf16(A.data_ptr(), K, M, K, W.data_ptr(), N, bias.data_ptr(), T.data_ptr(), N, R.data_ptr(), N,
                                 None, 0, 0, s()) == 0
        assert lib.mrd_layernorm_residual(T.data_ptr(), N, None, 0, gamma.data_ptr(), beta.data_ptr(), C.c_float(1e-12), M, N,
                                      Cc.data_ptr(), N, None, 0, s()) == 0, lib.mrd_last_error()

    def gemm_only():
        assert lib.mrd_gemm_bf16(A.data_ptr(), K, M, K, W.data_ptr(), N, bias.data_ptr(), T.data_ptr(), N, R.data_ptr(), N,
                                 None, 0, 0, s()) == 0

    ws = torch.zeros(lib.mrd_gemm_ln_ws_bytes(M), device=dev, dtype=torch.uint8)

    def fused():
        assert lib.mrd_gemm_ln_bf16(A.data_ptr(), K, M, K, W.data_ptr(), N, bias.data_ptr(), Cc.data_ptr(), N, R.data_ptr(),
                                    N, gamma.data_ptr(), beta.data_ptr(), C.c_float(1e-12), ws.data_ptr(), s()) == 0, lib.mrd_last_error()

    tg, tp, tf = timed(gemm_only), timed(plain), timed(fused)
    fl = 2.0 * M * N * K
    print(f"M={M} K={K}: gemm {tg:7.1f} us ({fl / tg / 1e6:6.0f} TF/s) | gemm + layernorm {tp:7.1f} us | fused "
          f"{tf:7.1f} us ({fl / tf / 1e6:6.0f} TF/s)", flush=True)

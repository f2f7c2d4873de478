#!/usr/bin/env python
"""Small-shape pass over every hand-written kernel for compute-sanitizer (memcheck / racecheck / synccheck /
initcheck): the unit tests of tests/test_kernels_gpu.py at reduced sizes, one tiny multimodal forward and one
tiny training step,
and the training-step kernel tests of tests/test_train_kernels_gpu.py at their smaller shapes.  Each case also checks its result, so a sanitizer run doubles as a correctness run.

    compute-sanitizer --tool memcheck  python tools/sanitize_kernels.py
    compute-sanitizer --tool racecheck python tools/sanitize_kernels.py
    compute-sanitizer --tool synccheck python tools/sanitize_kernels.py
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torch  # noqa: E402

import mrd_b200  # noqa: E402,F401
import synth  # noqa: E402
import test_kernels_gpu as K  # noqa: E402
import test_train_kernels_gpu as TK  # noqa: E402
from importlib import import_module  # noqa: E402

lib = import_module("multimodal-rare-disease_b200._lib").load()
cuda = torch.device("cuda:0")
quick = "--quick" in sys.argv

cases = [
    ("gemm", lambda: K.test_gemm(lib, cuda, 300, 768, 768, 0, True, False)),
    ("gemm gelu f32", lambda: K.test_gemm(lib, cuda, 256, 128, 128, 1, False, True)),
    ("gemm narrow", lambda: K.test_gemm(lib, cuda, 1000, 64, 256, 1, False, False)),
    ("conv 3x3 s2", lambda: K._conv_case(lib, cuda, 2, 28, 28, 128, 128, 3, 2, 1, False)),
    ("conv 1x1 res", lambda: K._conv_case(lib, cuda, 3, 7, 7, 512, 2048, 1, 1, 1, True)),
    ("conv 3x3 flat", lambda: K.test_conv3x3_flat(lib, cuda, 2, 28, 28, 128, 128, 1)),
    ("conv 1x1 dual s1", lambda: K.test_conv1x1_dual(lib, cuda, 1, 56, 56, 64, 64, 256, 1)),
    ("conv 1x1 dual s2", lambda: K.test_conv1x1_dual(lib, cuda, 2, 14, 14, 256, 512, 1024, 2)),
    ("stem", lambda: K.test_stem(lib, cuda, 1, 64, 96)),
    ("maxpool", lambda: K.test_maxpool(lib, cuda)),
    ("avgpool", lambda: K.test_avgpool(lib, cuda)),
    ("layernorm", lambda: K.test_layernorm(lib, cuda, 77, 512, False, 1e-5)),
    ("bert embed", lambda: K.test_bert_embed(lib, cuda)),
    ("attention S<=128", lambda: K.test_attention(lib, cuda, "tcgen05", 3, 128, 12, [128, 70, 1])),
    ("attention S>128", lambda: K.test_attention(lib, cuda, "tcgen05", 2, 384, 12, [384, 257])),
    ("attention varlen", lambda: K.test_attention_varlen(lib, cuda, "tcgen05", [128, 70, 1, 64, 65], 12)),
    ("attention varlen long", lambda: K.test_attention_varlen(lib, cuda, "tcgen05", [512, 64, 300], 12)),
    ("compact tokens", lambda: K.test_compact_tokens(lib, cuda, 7, 128, 0)),
    ("dropout bf16 strided", lambda: TK.test_dropout_bf16(lib, cuda, 0.1, True)),
    ("dropout f32 family", lambda: TK.test_dropout_f32_family(lib, cuda, 0.1)),
    ("drop + add + layernorm", lambda: TK.test_drop_add_layernorm(lib, cuda, 768, 0.1, False)),
    ("layernorm f32 fwd / bwd", lambda: TK.test_layernorm_f32_forward_backward(lib, cuda, 300, 64, 1)),
    ("transpose pad2", lambda: TK.test_transpose_pad2(lib, cuda, 768, 768, 65, True)),
    ("colsum f32 + relu bwd", lambda: TK.test_colsum_f32_and_relu_bwd(lib, cuda)),
    ("cls gather / scatter", lambda: TK.test_cls_gather_scatter(lib, cuda)),
    ("embed layernorm bwd", lambda: TK.test_embed_layernorm_backward(lib, cuda, 8, 512)),
    ("bn batch stats", lambda: TK.test_batchnorm_batch_statistics(lib, cuda, 3136, 2048, "identity_relu")),
    ("bn running update", lambda: TK.test_batchnorm_running_update(lib, cuda)),
]


def forward_and_step():
    model = synth.build_model(0).to(cuda)
    images, ids, mask = synth.make_inputs(2, 32, 7, [32, 9], H=64, W=64)
    images, ids, mask = images.to(cuda), ids.to(cuda), mask.to(cuda)
    with torch.no_grad():
        out = model(images, ids, mask)["logits"]
    assert bool(torch.isfinite(out).all())
    model.train()
    model.cnn_encoder.backbone.eval()
    opt = mrd_b200.FusedAdamW(model.parameters(), lr=5e-5, weight_decay=0.05, max_grad_norm=1.0)
    loss = torch.nn.functional.cross_entropy(model(images, ids, mask)["logits"], torch.tensor([1, 2], device=cuda))
    loss.backward()
    opt.step()
    torch.cuda.synchronize()
    assert bool(torch.isfinite(loss))


if not quick:
    cases.append(("multimodal forward + training step", forward_and_step))

failed = 0
for name, fn in cases:
    try:
        fn()
        torch.cuda.synchronize()
        print("ok  ", name, flush=True)
    except Exception as e:  # noqa: BLE001
        failed += 1
        print("FAIL", name, repr(e)[:300], flush=True)
print(f"{len(cases) - failed}/{len(cases)} cases passed")
sys.exit(1 if failed else 0)

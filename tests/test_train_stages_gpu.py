"""The staged training backward on one GPU.

A data-parallel step runs the backward one stage at a time (mrd_train_backward_begin, then
mrd_train_backward_stages once per stage: head + fusion + image projection, every BERT layer from the last to the
first, the embeddings) and hands each finished bucket of the flat gradient buffer to the all-reduce.  The plain step
runs all stages in one call.  Both must launch the same kernels and compute the same gradients; the
bucket callbacks must tile the flat buffer in order.  With the text encoder frozen, stage 0 stops after the image
projection's d_pooled and the later stages run nothing.
"""

import pytest
import torch
import torch.nn as nn

import synth

pytestmark = pytest.mark.gpu

B, S, H, W = 4, 64, 64, 64
SEED = 1234


def _model(cuda, frozen_text):
    m = synth.build_model(0)
    m.load_state_dict(synth.train_weights(0))
    for mod in m.modules():
        if isinstance(mod, nn.Dropout):
            mod.p = 0.0
    mc = m.text_encoder.model_config
    mc.hidden_dropout_prob = mc.attention_probs_dropout_prob = 0.0
    m = m.to(cuda)
    m.train()
    m.cnn_encoder.backbone.eval()
    if frozen_text:
        m.text_encoder.requires_grad_(False)
    return m


def _step(eng, inputs, nc, named, dlogits, staged):
    """One train-mode forward + backward with the library profiler on: logits, gradients, per-label launch counts,
    the engine's launch count of the step, the bucket slices (staged only) and the flat gradient buffer."""
    images, ids, mask = inputs
    buckets = []
    eng.profile(True)
    n0 = eng.launch_count
    logits = eng.train_forward(images, ids, mask, nc, SEED)
    grads = eng.train_backward(dlogits, named, on_bucket=buckets.append if staged else None)
    torch.cuda.synchronize()
    counts = {r["label"]: r["launches"] for r in eng.profile_report()}
    launches = eng.launch_count - n0
    eng.profile(False)
    return logits.clone(), [g.clone() for g in grads], counts, launches, buckets, eng.last_flat_grad


def _maxdiff(a, b):
    return (a.float() - b.float()).abs().max().item() if a.numel() else 0.0


@pytest.mark.parametrize("frozen_text", [False, True])
def test_staged_backward_matches_one_call(cuda, frozen_text):
    model = _model(cuda, frozen_text)
    images, ids, mask = synth.make_inputs(B, S, 17, [64, 40, 9, 57], H=H, W=W)
    inputs = (images.to(cuda), ids.to(cuda), mask.to(cuda))
    model(*inputs)   # applies the train-mode options and hands the weights over
    eng = model._engine(allow_training=True)
    named = [(n, tuple(p.shape)) for n, p in model._trainable()]
    assert any(n.startswith("text_encoder.") for n, _ in named) != frozen_text
    nc = model.num_classes
    dlogits = torch.randn(B, nc, generator=torch.Generator().manual_seed(3)).to(cuda)

    ref = _step(eng, inputs, nc, named, dlogits, staged=False)
    stg = _step(eng, inputs, nc, named, dlogits, staged=True)
    reps = [_step(eng, inputs, nc, named, dlogits, staged=False) for _ in range(2)]

    # the same kernels, the same number of times
    assert stg[2] == ref[2]
    assert stg[3] == ref[3]
    for r in reps:
        assert r[2] == ref[2] and r[3] == ref[3]

    # one bucket per stage that completes a gradient, tiling the flat buffer from its start, in order
    n_layers = int(eng.lib.mrd_train_backward_num_stages(eng._ctx)) - 2
    stages = {eng._backward_stage_of(n, n_layers) for n, _ in named}
    assert stages == ({0} if frozen_text else set(range(n_layers + 2)))
    buckets, flat = stg[4], stg[5]
    assert len(buckets) == len(stages)
    pos = 0
    for b in buckets:
        assert b.dim() == 1 and b.numel() > 0
        assert b.data_ptr() == flat.data_ptr() + 4 * pos
        pos += b.numel()
    assert pos == sum((torch.Size(sh).numel() + 3) // 4 * 4 for _, sh in named)

    # Split-K SIMT GEMMs and atomics (colsums, LayerNorm parameter gradients, embedding scatter) make repeated runs
    # differ in the last bits, and a last-bit difference can move a bf16 rounding further down the backward.  The
    # staged run must be no further from the first one-call run than the repeated one-call runs are; the floor
    # (about 80 fp32 ulps of the tensor's largest entry) covers tensors the repeats happened to reproduce exactly.
    worst = 0.0
    for k, (name, _) in enumerate([("logits", None)] + named):
        a = ref[0] if k == 0 else ref[1][k - 1]
        s = stg[0] if k == 0 else stg[1][k - 1]
        rs = [r[0] if k == 0 else r[1][k - 1] for r in reps]
        assert bool(torch.isfinite(s).all()), name
        spread = max(_maxdiff(r, a) for r in rs)
        floor = 1e-5 * a.float().abs().max().item() if a.numel() else 0.0
        d = _maxdiff(s, a)
        worst = max(worst, d / (2 * spread + floor) if d else 0.0)
        assert d <= 2 * spread + floor, (name, d, spread, floor)
    print(f"frozen_text={frozen_text}: {len(named)} gradients, {len(buckets)} buckets, {stg[3]} launches, "
          f"worst staged difference / allowance {worst:.3f}")

"""Attention probabilities: mrd_attention_probs_bf16 (attention_probs_kernel) and TextEncoder.get_attention_weights.

The reference for the module is the reference's own stack: a CPU copy of the HF BertModel holding the same
weights, switched to the eager attention backend and run with output_attentions=True
(HF:models/bert/modeling_bert.py:115-140).  The kernel is checked against an fp64 softmax(Q K^T + bias) of the
same bf16 qkv.

Bars of the bf16 module path (every layer, every query row, padded positions included): max-abs <= 2e-2 and per-row
total variation 1/2 sum_k |dp| <= 3e-2, on the plain and the sensitised weights.  The measured errors per layer are
printed (pytest -s) and recorded in DESIGN.md section 6.  A sample with no attended key gets all-zero rows (the
library's attention output for it is zero too); HF's uniform 1/S rows for it are deliberately not matched.
"""

import copy
import pytest
import torch

import mrd_b200  # noqa: F401
import synth

pytestmark = pytest.mark.gpu

HEADS = 12


def _check(lib, rc):
    assert rc == 0, lib.mrd_last_error().decode(errors="replace")


def _ref_probs(qkv, bias, B, S, H):
    x = qkv.double().view(B, S, 3, H, 64)
    q, k = x[:, :, 0].transpose(1, 2), x[:, :, 1].transpose(1, 2)
    s = q @ k.transpose(-1, -2)
    if bias is not None:
        s = s + bias.double().view(B, 1, 1, S)
    return torch.softmax(s, -1)


def _run_kernel(lib, qkv, bias, B, S, H):
    probs = torch.full((B, H, S, S), float("nan"), dtype=torch.float32, device=qkv.device)
    _check(lib, lib.mrd_attention_probs_bf16(qkv.data_ptr(), None if bias is None else bias.data_ptr(), B, S, H,
                                             probs.data_ptr(), torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    return probs


@pytest.mark.parametrize("S", [1, 5, 16, 31, 64, 100, 128, 129, 200, 256, 300, 512])
def test_probs_kernel_vs_fp64_softmax(cuda, lib, S):
    """Per-sample lengths (full, 1, about 2/3), a sample whose key 0 is masked, a sample with no attended key,
    and mask_bias = NULL.  Every element is written (the buffer starts as NaN)."""
    g = torch.Generator().manual_seed(1000 + S)
    B, H = 5, HEADS
    qkv = torch.randn(B * S, 3 * H * 64, generator=g)
    qkv[:, : H * 64] *= 0.25                   # Q pre-scaled (1/8 folded into W_q): scores of a few units
    qkv = qkv.to(torch.bfloat16).to(cuda)
    live = torch.zeros(B, S, dtype=torch.bool)
    live[0] = True
    live[1, 0] = True
    live[2, : max(1, (2 * S + 2) // 3)] = True
    live[3, 1:] = True                         # key 0 masked (for S = 1: no attended key at all)
    # sample 4: no attended key
    bias = torch.where(live, 0.0, float("-inf")).float().to(cuda)
    got = _run_kernel(lib, qkv, bias, B, S, H).cpu()
    ref = _ref_probs(qkv.cpu(), bias.cpu(), B, S, H)
    assert torch.isfinite(got).all()
    has_key = live.any(1)
    for b in range(B):
        if not has_key[b]:
            assert bool((got[b] == 0).all()), f"sample {b} without attended keys must be all zeros"
            continue
        err = (got[b].double() - ref[b]).abs().max().item()
        assert err <= 1e-5, f"S={S} sample {b}: max-abs {err:.3g}"
        rs = (got[b].double().sum(-1) - 1).abs().max().item()
        assert rs <= 1e-5, f"S={S} sample {b}: row sums off by {rs:.3g}"
        assert bool((got[b][:, :, ~live[b]] == 0).all()), "masked keys must be exactly 0"

    # mask_bias = NULL: every key attended
    got = _run_kernel(lib, qkv[: 2 * S], None, 2, S, H).cpu()
    ref = _ref_probs(qkv[: 2 * S].cpu(), None, 2, S, H)
    assert (got.double() - ref).abs().max().item() <= 1e-5
    assert (got.double().sum(-1) - 1).abs().max().item() <= 1e-5


# ---------------------------------------------------------------------------------------------- module level
@pytest.fixture(scope="module")
def enc(cuda):
    model = synth.build_model(0)
    plain = {k: v.clone() for k, v in model.state_dict().items()}
    sens = synth.sensitise(plain, 1)
    te = model.text_encoder.to(cuda).eval()

    def sub(sd):
        return {k[len("text_encoder."):]: v for k, v in sd.items() if k.startswith("text_encoder.")}

    return {"te": te, "plain": sub(plain), "sens": sub(sens)}


def _load(enc, which):
    te = enc["te"]
    te.load_state_dict(enc[which], strict=True)
    return te


def _set_backend(te, impl):
    te.encoder.set_attn_implementation(impl)
    assert te.encoder.config._attn_implementation == impl


def _hf_eager(te, ids, mask):
    ref = copy.deepcopy(te.encoder).cpu().float().eval()
    ref.set_attn_implementation("eager")
    with torch.no_grad():
        out = ref(input_ids=ids, attention_mask=mask, output_attentions=True)
    return out.attentions


def _errors(got, ref):
    """per layer: (max-abs, mean-abs, max / p99 per-row total variation)"""
    rows = []
    for g, r in zip(got, ref):
        d = (g.float().cpu() - r).abs()
        tv = 0.5 * d.sum(-1).flatten()
        rows.append((d.max().item(), d.mean().item(), tv.max().item(), tv.quantile(0.99).item()))
    return rows


def _print(tag, rows):
    print(f"\n[attn probs] {tag}: layer max-abs / mean-abs / max TV / p99 TV")
    for i, (a, m, t, t99) in enumerate(rows):
        print(f"  layer {i:2d}: {a:.3e} {m:.3e} {t:.3e} {t99:.3e}")


CASES = [(3, 40, [40, 13, 27], 77), (3, 200, [200, 77, 129], 78)]


@pytest.mark.parametrize("which", ["plain", "sens"])
@pytest.mark.parametrize("B,S,lens,seed", CASES)
def test_module_bf16_vs_hf_eager(cuda, enc, which, B, S, lens, seed):
    """S = 40 reads the blocked qkv layout of the short plans, S = 200 the long path's."""
    te = _load(enc, which)
    _, ids, mask = synth.make_inputs(B, S, seed, lens, H=32, W=32)
    _set_backend(te, "eager")
    try:
        with torch.no_grad():
            emb, attn = te.get_attention_weights(ids.to(cuda), mask.to(cuda))
    finally:
        _set_backend(te, "sdpa")
    torch.cuda.synchronize()
    ref = _hf_eager(te, ids, mask)
    assert len(attn) == len(ref) == 12
    assert all(a.shape == (B, HEADS, S, S) and a.dtype == torch.float32 and a.device == cuda for a in attn)
    rows = _errors(attn, ref)
    _print(f"bf16 {which} B={B} S={S} lens={lens}", rows)
    for i, (a, _, t, _) in enumerate(rows):
        assert a <= 2e-2, f"layer {i}: max-abs {a:.3g}"
        assert t <= 3e-2, f"layer {i}: max row total variation {t:.3g}"


@pytest.mark.parametrize("which", ["plain", "sens"])
@pytest.mark.parametrize("B,S,lens,seed", CASES + [(2, 512, [512, 300], 79)])
def test_module_fp32_check_vs_hf_eager(cuda, enc, which, B, S, lens, seed):
    te = _load(enc, which)
    _, ids, mask = synth.make_inputs(B, S, seed, lens, H=32, W=32)
    _set_backend(te, "eager")
    te.configure_b200(fp32_check=True)
    try:
        with torch.no_grad():
            emb, attn = te.get_attention_weights(ids.to(cuda), mask.to(cuda))
            fwd = te(ids.to(cuda), mask.to(cuda))
    finally:
        te.configure_b200(fp32_check=False)
        _set_backend(te, "sdpa")
    torch.cuda.synchronize()
    assert torch.equal(emb, fwd)
    ref = _hf_eager(te, ids, mask)
    rows = _errors(attn, ref)
    _print(f"fp32 check {which} B={B} S={S} lens={lens}", rows)
    for i, (a, _, _, _) in enumerate(rows):
        assert a <= 1e-5, f"layer {i}: max-abs {a:.3g}"


def test_module_structure(cuda, enc):
    """Masked keys are 0, rows sum to 1, the embedding is forward()'s, calls are deterministic, and micro-batched
    runs reproduce one pass bit for bit; mask=None attends every key."""
    te = _load(enc, "sens")
    B, S = 5, 40
    lens = [40, 1, 17, 33, 8]
    _, ids, mask = synth.make_inputs(B, S, 81, lens, H=32, W=32)
    ids, mask = ids.to(cuda), mask.to(cuda)
    _set_backend(te, "eager")
    try:
        with torch.no_grad():
            emb, attn = te.get_attention_weights(ids, mask)
            emb2, attn2 = te.get_attention_weights(ids, mask)
            fwd = te(ids, mask)
            te.configure_b200(seq_chunk_tokens=2 * S)
            try:
                emb3, attn3 = te.get_attention_weights(ids, mask)
            finally:
                te.configure_b200(seq_chunk_tokens=524288)
            _, attn_nomask = te.get_attention_weights(ids, None)
    finally:
        _set_backend(te, "sdpa")
    torch.cuda.synchronize()
    assert torch.equal(emb, fwd)
    assert torch.equal(emb, emb2) and all(torch.equal(a, b) for a, b in zip(attn, attn2))
    assert torch.equal(emb, emb3) and all(torch.equal(a, b) for a, b in zip(attn, attn3))
    assert attn[1].data_ptr() - attn[0].data_ptr() == B * HEADS * S * S * 4   # views of one [L,B,H,S,S] buffer
    stack = torch.stack(attn)
    keymask = (mask == 0).view(1, B, 1, 1, S).expand_as(stack)
    assert bool((stack[keymask] == 0).all())
    assert (stack.double().sum(-1) - 1).abs().max().item() <= 1e-5
    nm = torch.stack(attn_nomask)
    assert (nm.double().sum(-1) - 1).abs().max().item() <= 1e-5


def test_default_backend_returns_empty_tuple(cuda, enc):
    te = _load(enc, "plain")
    _, ids, mask = synth.make_inputs(2, 24, 82, [24, 9], H=32, W=32)
    ids, mask = ids.to(cuda), mask.to(cuda)
    assert te.encoder.config._attn_implementation == "sdpa"
    with torch.no_grad():
        fwd = te(ids, mask)
        emb, attn = te.get_attention_weights(ids, mask)
        assert attn == () and torch.equal(emb, fwd)
        _set_backend(te, "eager")
        _, attn = te.get_attention_weights(ids, mask)
        assert len(attn) == 12
        _set_backend(te, "sdpa")
        emb, attn = te.get_attention_weights(ids, mask)
        assert attn == () and torch.equal(emb, fwd)


@pytest.mark.parametrize("impl", ["sdpa", "eager"])
def test_train_mode_raises(cuda, enc, impl):
    te = _load(enc, "plain")
    _, ids, mask = synth.make_inputs(2, 16, 83, [16, 5], H=32, W=32)
    _set_backend(te, impl)
    te.train()
    try:
        with pytest.raises(NotImplementedError):
            te.get_attention_weights(ids.to(cuda), mask.to(cuda))
    finally:
        te.eval()
        _set_backend(te, "sdpa")

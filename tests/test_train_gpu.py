"""Training step on the B200 path (SURVEY.md 8(f).1, BASELINE.json configs[4]) against the reference.

Comparators: tests/golden/train_*.pt (one src/train.py-style step of the UNMODIFIED reference with
dropout p = 0: loss, gradients, post-AdamW parameters) and oracle/train_oracle.py (pinned to the same
fixtures by tests/test_train_oracle.py) for the runs with dropout, whose masks are exported from the
library (mrd_dropout_mask) and fed to the oracle.
Bars actually applied (SURVEY.md 8(c)(5) asked for 5e-2 on the weight deltas; measured, no bf16 step of a
random-init BERT meets that - stock PyTorch bf16 autocast is 16-25 % off fp32 on the query/key gradients):
  * fp32 check mode (plain-fp32 forward and backward of the library): loss 1e-5, every parameter gradient within
    1e-4 relative L2 of the unmodified reference's (test_fp32_check_backward_vs_reference_fixture) - the structural
    gate;
  * bf16 step against those fp32 gradients at FIXED bars (BF16_BARS: 5e-2 global / 1e-1 per tensor on the
    well-conditioned linear-loss case, 1.1e-1 / 2.5e-1 on the cross-entropy fixture);
  * additionally, per case, no worse than 1.3x the bf16-autocast oracle's own error + 5e-2 (the floor any bf16
    implementation has), and the loss within 2e-3 relative.
"""

import ctypes as C

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

import mrd_b200
import synth
from oracle import train_oracle as T

pytestmark = pytest.mark.gpu
GRAD_TOL = 5e-2


def _sample(t, stride):
    return t.detach().float().flatten()[::stride].cpu()


def _p(t):
    return C.c_void_p(t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _zero_dropout(model):
    for m in model.modules():
        if isinstance(m, nn.Dropout):
            m.p = 0.0
    mc = model.text_encoder.model_config
    mc.hidden_dropout_prob = 0.0
    mc.attention_probs_dropout_prob = 0.0


# --------------------------------------------------------------------------------------- kernels
def _attention_ref(qkv, bias, B, S, heads, dctx, mask=None, p=0.0):
    """fp32 autograd reference on the bf16-rounded inputs.  qkv [B*S, 3*heads*64] (Q pre-scaled)."""
    x = qkv.float().clone().requires_grad_(True)
    q, k, v = x.view(B, S, 3, heads, 64).permute(2, 0, 3, 1, 4)
    s = q @ k.transpose(-1, -2)
    if bias is not None:
        s = s + bias.view(B, 1, 1, S)
    pr = torch.softmax(s, dim=-1)
    if mask is not None:
        pr = pr * mask.view(B, heads, S, S) / (1.0 - p)
    o = (pr @ v).permute(0, 2, 1, 3).reshape(B * S, heads * 64)
    o.backward(dctx.float())
    return o.detach(), x.grad


@pytest.mark.parametrize("B,S,lens,p", [(3, 128, [128, 77, 5], 0.0), (4, 48, [48, 48, 17, 1], 0.0),
                                        (2, 128, [128, 100], 0.1), (5, 32, [32, 9, 32, 20, 31], 0.25),
                                        # > 128 tokens: tiled backward (fp32 dK/dV accumulation), mma.sync forward
                                        (3, 256, [256, 130, 3], 0.0), (2, 200, [200, 129], 0.1),
                                        (2, 512, [512, 385], 0.0), (1, 384, [300], 0.2)])
def test_attention_backward_vs_autograd(cuda, lib, B, S, lens, p):
    heads = 12
    g = torch.Generator().manual_seed(5)
    qkv = (torch.randn(B * S, 3 * heads * 64, generator=g) * 0.7).to(cuda, torch.bfloat16)
    dctx = torch.randn(B * S, heads * 64, generator=g).to(cuda, torch.bfloat16)
    bias = torch.zeros(B, S)
    for b, L in enumerate(lens):
        bias[b, L:] = float("-inf")
    bias = bias.to(cuda)
    seed, site = 1234567, 7
    mask = None
    if p > 0:
        mask = torch.empty(B * heads * S * S, device=cuda)
        assert lib.mrd_dropout_mask(C.c_ulonglong(seed), site, p, mask.numel(), _p(mask), _stream()) == 0
        assert abs(mask.mean().item() - (1 - p)) < 0.01
    # forward with the same mask (tcgen05 kernel), then the backward kernel
    out = torch.empty(B * S, heads * 64, device=cuda, dtype=torch.bfloat16)
    assert lib.mrd_attention_train_bf16(_p(qkv), _p(bias), B, S, heads, C.c_ulonglong(seed), site, p, _p(out),
                                        _stream()) == 0, lib.mrd_last_error()
    o_ref, d_ref = _attention_ref(qkv, bias, B, S, heads, dctx, mask, p)
    live = (bias > float("-inf")).view(B * S)
    err_o = (out.float()[live] - o_ref[live]).norm() / o_ref[live].norm()
    assert err_o.item() <= 1e-2, err_o.item()
    dqkv = torch.zeros_like(qkv)
    acc = torch.zeros(B * S, 2 * heads * 64, device=cuda) if S > 128 else None
    assert lib.mrd_attention_bwd_bf16(_p(qkv), _p(out), _p(dctx), _p(bias), None, B, S, heads, C.c_ulonglong(seed),
                                      site, p, _p(dqkv), None if acc is None else _p(acc), B * S,
                                      _stream()) == 0, lib.mrd_last_error()
    torch.cuda.synchronize()
    # padded QUERY rows are outputs nobody reads: the engine never feeds them a gradient; here they do get
    # one, so compare everything (keys beyond the length receive exactly zero dK/dV in both)
    for name, sl in (("dQ", slice(0, 768)), ("dK", slice(768, 1536)), ("dV", slice(1536, 2304))):
        a, r = dqkv.float()[:, sl], d_ref[:, sl]
        err = ((a - r).norm() / r.norm()).item()
        assert err <= 2e-2, (name, err)


def test_attention_backward_packed_layout(cuda, lib):
    """Token-packed rows (seq_off) give the same gradients as the dense layout with a key bias."""
    B, S, heads, lens = 4, 64, 12, [64, 30, 1, 47]
    g = torch.Generator().manual_seed(6)
    qkv = (torch.randn(B * S, 2304, generator=g) * 0.7).to(cuda, torch.bfloat16)
    dctx = torch.randn(B * S, 768, generator=g).to(cuda, torch.bfloat16)
    ctx = torch.randn(B * S, 768, generator=g).to(cuda, torch.bfloat16)
    rows = torch.cat([torch.arange(L) + b * S for b, L in enumerate(lens)]).to(cuda)
    off = torch.tensor([0] + list(torch.tensor(lens).cumsum(0)), dtype=torch.int32, device=cuda)
    bias = torch.zeros(B, S)
    for b, L in enumerate(lens):
        bias[b, L:] = float("-inf")
    bias = bias.to(cuda)
    dctx[(bias == float("-inf")).view(B * S).cpu()] = 0   # padded queries do not exist in the packed layout
    d_dense = torch.zeros_like(qkv)
    assert lib.mrd_attention_bwd_bf16(_p(qkv), _p(ctx), _p(dctx), _p(bias), None, B, S, heads, C.c_ulonglong(1), 0,
                                      0.0, _p(d_dense), None, B * S, _stream()) == 0
    pq, pc, pd = qkv[rows].contiguous(), ctx[rows].contiguous(), dctx[rows].contiguous()
    d_pack = torch.zeros_like(pq)
    assert lib.mrd_attention_bwd_bf16(_p(pq), _p(pc), _p(pd), None, _p(off), B, S, heads, C.c_ulonglong(1), 0, 0.0,
                                      _p(d_pack), None, pq.shape[0], _stream()) == 0
    torch.cuda.synchronize()
    assert torch.equal(d_pack, d_dense[rows])


@pytest.mark.parametrize("M,N,K,live", [(768, 3072, 2048, None), (3072, 768, 4096, 2560), (2304, 768, 1024, 700),
                                        (768, 768, 512, 64), (256, 64, 8192, None)])
def test_splitk_weight_gradient_gemm(cuda, lib, M, N, K, live):
    """dW = dY^T X: split-K tcgen05 GEMM with fp32 partial sums reduced in L2, bounded by the live K on the device."""
    g = torch.Generator().manual_seed(11)
    A = torch.randn(M, K, generator=g).to(cuda, torch.bfloat16)
    W = torch.randn(N, K, generator=g).to(cuda, torch.bfloat16)
    dyn = None
    if live is not None:
        up = (live + 63) // 64 * 64
        A[:, live:up] = 0          # the staging transposes zero-fill up to the next K block ...
        W[:, live:up] = 0
        A[:, up:] = float("nan")   # ... and nothing beyond it may be read
        W[:, up:] = float("nan")
        dyn = torch.tensor([live], dtype=torch.int32, device=cuda)
    out = torch.zeros(M, N, device=cuda)
    assert lib.mrd_gemm_splitk_f32(_p(A), K, M, K, _p(W), N, _p(out), N, None if dyn is None else _p(dyn),
                                   _stream()) == 0, lib.mrd_last_error()
    kk = K if live is None else live
    ref = A[:, :kk].float() @ W[:, :kk].float().T
    torch.cuda.synchronize()
    assert torch.isfinite(out).all()
    assert ((out - ref).norm() / ref.norm()).item() <= 3e-5   # bf16 products are exact in fp32; only the order differs
    # accumulation semantics: a second launch adds on top
    assert lib.mrd_gemm_splitk_f32(_p(A), K, M, K, _p(W), N, _p(out), N, None if dyn is None else _p(dyn),
                                   _stream()) == 0
    torch.cuda.synchronize()
    assert ((out - 2 * ref).norm() / ref.norm()).item() <= 6e-5


@pytest.mark.parametrize("rows,width", [
    pytest.param(1000, 768, id="768"), pytest.param(1000, 512, id="512"),
    # 8192 rows (the training benchmark's B*S) against a grid of 296 blocks x 8 warps: 3-4 rows per warp
    (8192, 256), (8192, 768), (8192, 1024), (1000, 1024)])
def test_layernorm_backward_vs_autograd(cuda, lib, rows, width):
    g = torch.Generator().manual_seed(8)
    s_in = (torch.randn(rows, width, generator=g) * 2 + 0.3).to(cuda, torch.bfloat16)
    dy = torch.randn(rows, width, generator=g).to(cuda, torch.bfloat16)
    gamma = (0.5 + torch.rand(width, generator=g)).to(cuda)
    x = s_in.float().requires_grad_(True)
    gm = gamma.clone().requires_grad_(True)
    bt = torch.zeros(width, device=cuda, requires_grad=True)
    F.layer_norm(x, (width,), gm, bt, 1e-12).backward(dy.float())
    dx = torch.full_like(s_in, float("nan"))
    dg, db = torch.zeros(width, device=cuda), torch.zeros(width, device=cuda)
    assert lib.mrd_layernorm_bwd_bf16(_p(s_in), _p(dy), _p(gamma), 1e-12, rows, width, _p(dx), _p(dg), _p(db),
                                      _stream()) == 0, lib.mrd_last_error()
    torch.cuda.synchronize()
    assert ((dx.float() - x.grad).norm() / x.grad.norm()).item() <= 1e-2
    assert ((dg - gm.grad).norm() / gm.grad.norm()).item() <= 1e-4
    assert ((db - bt.grad).norm() / bt.grad.norm()).item() <= 1e-4


def test_dropout_mask_statistics(cuda, lib):
    n = 1 << 20
    m = torch.empty(n, device=cuda)
    for p in (0.1, 0.3, 0.5):
        assert lib.mrd_dropout_mask(C.c_ulonglong(99), 3, p, n, _p(m), _stream()) == 0
        assert abs(m.mean().item() - (1 - p)) < 3e-3
        m2 = torch.empty(n, device=cuda)
        assert lib.mrd_dropout_mask(C.c_ulonglong(99), 4, p, n, _p(m2), _stream()) == 0
        # different sites are independent: agreement rate = (1-p)^2 + p^2
        assert abs((m == m2).float().mean().item() - ((1 - p) ** 2 + p ** 2)) < 5e-3
    assert lib.mrd_dropout_mask(C.c_ulonglong(99), 3, 0.0, n, _p(m), _stream()) == 0
    assert bool((m == 1).all())


# --------------------------------------------------------------------------------------- full step
def _oracle_grads_gpu(sd, images, ids, mask, labels=None, R=None, masks=None, autocast=False, bn_train=False):
    """Gradients of the (reference-pinned) training oracle, evaluated with torch on the GPU: fp32, or under
    bf16 autocast - the latter is the rounding-noise floor a stock PyTorch bf16 run of the reference has on
    the same case, the yardstick the B200 step is held to."""
    names = set(T.trainable_names(sd))
    work = {k: (v.detach().clone().float().cuda().requires_grad_(k in names) if v.is_floating_point() else v.cuda())
            for k, v in sd.items()}
    mk = None if masks is None else {k: v.cuda() for k, v in masks.items()}
    tf32 = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
    torch.set_default_device("cuda")
    try:
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
            logits = T.train_forward(work, images.cuda(), ids.cuda(), mask.cuda(), mk, bn_train)
        loss = F.cross_entropy(logits.float(), labels.cuda()) if R is None else (logits.float() * R.cuda()).sum()
        loss.backward()
    finally:
        torch.set_default_device("cpu")
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = tf32
    return loss.item(), {k: (work[k].grad.detach().float().cpu() if work[k].grad is not None
                             else torch.zeros_like(work[k]).cpu()) for k in names}


def _compare_with_floor(got, ref, floor, what, per_tensor=True):
    """got / ref / floor: {name: gradient}.  Every tensor of `got` must be as close to `ref` (fp32) as the
    bf16-autocast oracle `floor` is (x1.3 + GRAD_TOL headroom), and so must the concatenation of all of them."""
    tot = torch.sqrt(sum((g.double() ** 2).sum() for g in ref.values())).item()
    rows, n_got, n_floor = [], 0.0, 0.0
    for k, r in ref.items():
        if r.norm().item() < 1e-5 * tot:
            assert got[k].norm().item() <= 1e-2 * tot, k
            continue
        eg = ((got[k] - r).norm() / r.norm()).item()
        ef = ((floor[k] - r).norm() / r.norm()).item()
        n_got += (got[k] - r).double().pow(2).sum().item()
        n_floor += (floor[k] - r).double().pow(2).sum().item()
        rows.append((eg, ef, k))
    rows.sort(reverse=True)
    g_got, g_floor = n_got ** 0.5 / tot, n_floor ** 0.5 / tot
    print(f"{what}: global rel-L2 ours {g_got:.4f} vs bf16-autocast oracle {g_floor:.4f}; worst:",
          [(round(a, 4), round(b, 4), k) for a, b, k in rows[:4]])
    assert g_got <= 1.3 * g_floor + GRAD_TOL, (g_got, g_floor)
    for eg, ef, k in rows:
        if per_tensor:
            assert eg <= 1.3 * ef + GRAD_TOL, (k, eg, ef)
    return g_got, g_floor

@pytest.fixture(scope="module")
def sens():
    """Weights of the training fixtures: plain random init + sensitised LayerNorm parameters (small logits, so
    softmax - onehot is well conditioned; see oracle/make_golden_train.py)."""
    return synth.train_weights(0)


def _train_model(sens, zero_dropout=True):
    model = synth.build_model(0)
    model.load_state_dict(sens)
    if zero_dropout:
        _zero_dropout(model)
    model = model.to("cuda:0")
    model.train()
    model.cnn_encoder.backbone.eval()   # frozen backbone on running statistics
    return model


def test_train_step_vs_reference_fixture(cuda, sens):
    """One src/train.py-style step through the module API: loss.backward() fills .grad through the library's
    backward; clip_grad_norm_ and torch.optim.AdamW stay the caller's, as in the reference."""
    fix = synth.load_train_golden("train_p0_bn_eval_b4_s32")
    model = _train_model(sens)
    images, ids, mask = synth.make_inputs(fix["B"], fix["S"], fix["seed"], fix["lengths"], H=fix["H"], W=fix["W"])
    labels = torch.tensor(fix["labels"]).cuda()
    before = {k: v.detach().clone() for k, v in model.named_parameters()}
    opt = torch.optim.AdamW(model.parameters(), lr=fix["lr"], weight_decay=fix["weight_decay"])
    opt.zero_grad()
    out = model(images.cuda(), ids.cuda(), mask.cuda())
    assert out["logits"].requires_grad and out["probs"].shape == (fix["B"], 10)
    loss = nn.CrossEntropyLoss()(out["logits"], labels)
    loss.backward()
    torch.cuda.synchronize()
    assert abs(loss.item() - fix["loss"]) <= 2e-3 * abs(fix["loss"]), (loss.item(), fix["loss"])
    named = dict(model.named_parameters())
    got = {k for k, p in named.items() if p.grad is not None}
    assert got == set(fix["grads"]), (sorted(got ^ set(fix["grads"]))[:5])
    report = []
    for k, ref in fix["grads"].items():
        g = named[k].grad
        assert g.dtype == torch.float32 and g.shape == named[k].shape
        if ref["norm"] == 0.0:
            assert g.abs().max().item() == 0.0, k
            continue
        if ref["norm"] < 1e-5:   # key biases (softmax shift invariance): noise in both implementations
            assert g.norm().item() <= 1e-2 * fix["total_norm"], k
            continue
        if ref["sample"].norm().item() < 1e-3 * ref["norm"]:   # sparse gradient (word embeddings): norm only
            assert abs(g.norm().item() - ref["norm"]) <= GRAD_TOL * ref["norm"], k
            continue
        err = (_sample(g, ref["stride"]) - ref["sample"]).norm().item() / ref["sample"].norm().item()
        report.append((err, k, g.norm().item() / ref["norm"]))
    report.sort(reverse=True)
    print("worst gradients vs the reference fixture (rel err, name, norm ratio):", report[:4])
    # random-init BERT is an ill-conditioned case for ANY bf16 step (tests/diag_train_noise.py: stock PyTorch
    # bf16 autocast of the same model is 16-25 % off fp32 on the query/key gradients), so the per-tensor bar is
    # the bf16-autocast oracle's own error on this very case, not a fixed 5 %.
    _, g32 = _oracle_grads_gpu(sens, images, ids, mask, labels=torch.tensor(fix["labels"]))
    _, g16 = _oracle_grads_gpu(sens, images, ids, mask, labels=torch.tensor(fix["labels"]), autocast=True)
    ours = {k: named[k].grad.float().cpu() for k in g32}
    _compare_with_floor(ours, g32, g16, "fixture step")
    for err, k, ratio in report:   # and against the reference's own numbers: same bar, sampled elements
        r = fix["grads"][k]
        floor = (_sample(g16[k], r["stride"]) - r["sample"]).norm().item() / r["sample"].norm().item()
        assert err <= 1.3 * floor + GRAD_TOL, (k, err, floor, ratio)
    total = nn.utils.clip_grad_norm_(model.parameters(), 1.0)
    assert abs(total.item() - fix["total_norm"]) <= 3e-2 * fix["total_norm"]
    opt.step()
    torch.cuda.synchronize()
    # parameter deltas of the AdamW step, relative L2 per parameter group
    groups = {}
    for k, ref in fix["post"].items():
        if fix["grads"][k]["norm"] < 1e-5:
            continue
        pre = _sample(before[k], ref["stride"])
        d_ref, d_got = ref["sample"] - pre, _sample(named[k], ref["stride"]) - pre
        a = groups.setdefault(k.split(".")[0], [0.0, 0.0])
        a[0] += (d_got - d_ref).norm().item() ** 2
        a[1] += d_ref.norm().item() ** 2
    rel = {k: (v[0] / v[1]) ** 0.5 for k, v in groups.items()}
    # the same step taken from the bf16-autocast oracle's gradients: Adam's first step is ~ lr * sign(g), so
    # gradient noise flips small elements; the bar is again what stock bf16 does
    post16 = T.clip_and_adamw(sens, g16, lr=fix["lr"], weight_decay=fix["weight_decay"])
    fl = {}
    for k, ref in fix["post"].items():
        if fix["grads"][k]["norm"] < 1e-5:
            continue
        pre = _sample(before[k], ref["stride"])
        d_ref, d_16 = ref["sample"] - pre, _sample(post16[k], ref["stride"]) - pre
        a = fl.setdefault(k.split(".")[0], [0.0, 0.0])
        a[0] += (d_16 - d_ref).norm().item() ** 2
        a[1] += d_ref.norm().item() ** 2
    floor = {k: (v[0] / v[1]) ** 0.5 for k, v in fl.items()}
    print("AdamW delta rel-L2 per group: ours", rel, "bf16-autocast oracle", floor)
    for k, v in rel.items():
        assert v <= 1.3 * floor[k] + GRAD_TOL, (k, v, floor[k])
    # the next forward sees the updated parameters (packed weights are refreshed)
    out2 = model(images.cuda(), ids.cuda(), mask.cuda())
    assert not torch.equal(out2["logits"], out["logits"])


def _export_masks(lib, model, seed, B, S, opts):
    """The masks mrd_train_forward drew for `seed`, in the layout oracle.train_oracle expects
    (csrc/rng.cuh / engine_train.cuh: site ids and element indexing; all-ones attention mask, so packed row
    r = b*S + j)."""
    dev = torch.device("cuda:0")

    def mk(site, p, shape):
        n = 1
        for d in shape:
            n *= d
        m = torch.empty(n, device=dev)
        assert lib.mrd_dropout_mask(C.c_ulonglong(seed), site, p, n, _p(m), _stream()) == 0
        return (m.view(shape) / (1.0 - p)).cpu() if p > 0 else None

    ph, pa = opts["train.p_bert_hidden"], opts["train.p_bert_attn"]
    masks = {"emb": mk(1000, ph, (B, S, 768)), "text_out": mk(1001, opts["train.p_text_out"], (B, 768)),
             "cnn_proj": mk(1002, opts["train.p_cnn_proj"], (B, 512)),
             "i2t": mk(1003, opts["train.p_fusion"], (B, 8)), "t2i": mk(1004, opts["train.p_fusion"], (B, 8)),
             "fusion_mlp": mk(1005, opts["train.p_fusion"], (B, 512)),
             "head.0": mk(1010, opts["train.p_head"], (B, 256)), "head.1": mk(1011, opts["train.p_head"], (B, 128))}
    for l in range(12):
        masks[f"attn.{l}"] = mk(16 * l, pa, (B, 12, S, S))
        masks[f"attn_out.{l}"] = mk(16 * l + 1, ph, (B, S, 768))
        masks[f"ffn_out.{l}"] = mk(16 * l + 2, ph, (B, S, 768))
    return {k: v for k, v in masks.items() if v is not None}


def test_train_step_with_dropout_vs_oracle(cuda, lib, sens):
    """Dropout active at the reference's default probabilities; the oracle receives the library's own masks."""
    B, S = 3, 32
    model = _train_model(sens, zero_dropout=False)
    images, ids, mask = synth.make_inputs(B, S, 51, None, H=64, W=64)
    labels = torch.tensor([2, 9, 4])
    torch.manual_seed(77)
    seed = int(torch.randint(0, 2 ** 62, (1,)).item())
    torch.manual_seed(77)
    out = model(images.cuda(), ids.cuda(), mask.cuda())
    loss = F.cross_entropy(out["logits"], labels.cuda())
    loss.backward()
    torch.cuda.synchronize()
    masks = _export_masks(lib, model, seed, B, S, model._train_options())
    assert len(masks) == 8 + 36
    ref_loss, g32 = _oracle_grads_gpu(sens, images, ids, mask, labels=labels, masks=masks)
    _, g16 = _oracle_grads_gpu(sens, images, ids, mask, labels=labels, masks=masks, autocast=True)
    assert abs(loss.item() - ref_loss) <= 2e-3 * abs(ref_loss), (loss.item(), ref_loss)
    named = dict(model.named_parameters())
    _compare_with_floor({k: named[k].grad.float().cpu() for k in g32}, g32, g16, "dropout step")
    # a different seed gives different masks, hence different logits
    out2 = model(images.cuda(), ids.cuda(), mask.cuda())
    assert not torch.equal(out2["logits"], out["logits"])


def test_backward_only_linear_loss_sensitised(cuda):
    """Backward in isolation on the sensitised weights (|logits| ~ 14): a loss that is LINEAR in the logits
    makes d(loss)/d(logits) identical for both implementations, so the gradient error measured here is the
    backward pass's own (plus the forward activations it reuses), not the softmax's conditioning."""
    sd = synth.sensitise(synth.build_model(0).state_dict(), 1)
    model = _train_model(sd)
    B, S = 5, 64
    images, ids, mask = synth.make_inputs(B, S, 71, [64, 33, 64, 2, 17], H=96, W=64)
    R = torch.randn(B, 10, generator=torch.Generator().manual_seed(9))
    out = model(images.cuda(), ids.cuda(), mask.cuda())
    (out["logits"] * R.cuda()).sum().backward()
    torch.cuda.synchronize()
    _, g32 = _oracle_grads_gpu(sd, images, ids, mask, R=R)
    _, g16 = _oracle_grads_gpu(sd, images, ids, mask, R=R, autocast=True)
    named = dict(model.named_parameters())
    g_got, _ = _compare_with_floor({k: named[k].grad.float().cpu() for k in g32}, g32, g16, "linear loss")
    assert g_got <= GRAD_TOL   # a well-conditioned case: the fixed 5 % bar holds globally


# the unmodified reference on this batch, dropout 0, lr 2e-4 (oracle/ref_train_loop.py)
REF_LOOP = [2.289, 2.268, 2.241, 2.212, 2.176, 2.161, 2.111, 2.054, 1.997, 1.932, 1.914, 1.827, 1.829, 1.706,
            1.645, 1.562, 1.869, 1.583, 1.462, 1.384]


def test_train_step_long_sequences(cuda, sens):
    """256 tokens (what the reference's multimodal trainer tokenises to, src/train_multimodal.py:53): mma.sync
    forward with dropout-capable probabilities, tiled attention backward; dropout on, library masks to the oracle."""
    B, S = 2, 256
    model = _train_model(sens, zero_dropout=False)
    images, ids, mask = synth.make_inputs(B, S, 81, None, H=64, W=64)
    labels = torch.tensor([5, 0])
    torch.manual_seed(78)
    seed = int(torch.randint(0, 2 ** 62, (1,)).item())
    torch.manual_seed(78)
    out = model(images.cuda(), ids.cuda(), mask.cuda())
    loss = F.cross_entropy(out["logits"], labels.cuda())
    loss.backward()
    torch.cuda.synchronize()
    masks = _export_masks(lib_handle(), model, seed, B, S, model._train_options())
    ref_loss, g32 = _oracle_grads_gpu(sens, images, ids, mask, labels=labels, masks=masks)
    _, g16 = _oracle_grads_gpu(sens, images, ids, mask, labels=labels, masks=masks, autocast=True)
    assert abs(loss.item() - ref_loss) <= 2e-3 * abs(ref_loss), (loss.item(), ref_loss)
    named = dict(model.named_parameters())
    _compare_with_floor({k: named[k].grad.float().cpu() for k in g32}, g32, g16, "256-token step")
    # padded variant: 2 sequences of 200 / 131 tokens in a 256-token batch, no dropout, vs the fp32 oracle
    model2 = _train_model(sens)
    images, ids, mask = synth.make_inputs(B, S, 82, [200, 131], H=64, W=64)
    out = model2(images.cuda(), ids.cuda(), mask.cuda())
    F.cross_entropy(out["logits"], labels.cuda()).backward()
    _, g32 = _oracle_grads_gpu(sens, images, ids, mask, labels=labels)
    _, g16 = _oracle_grads_gpu(sens, images, ids, mask, labels=labels, autocast=True)
    named = dict(model2.named_parameters())
    _compare_with_floor({k: named[k].grad.float().cpu() for k in g32}, g32, g16, "256-token padded step")


def lib_handle():
    from importlib import import_module
    return import_module("multimodal-rare-disease_b200._lib").load()


def test_training_loop_follows_reference(cuda):
    """20 steps of the reference's loop shape (zero_grad / forward / CrossEntropyLoss / backward /
    clip_grad_norm_ / AdamW.step) on a fixed padded batch: the loss follows the reference's own trajectory."""
    torch.manual_seed(3)
    model = synth.build_model(0)
    _zero_dropout(model)
    model = model.to("cuda:0")
    model.train()
    model.cnn_encoder.backbone.eval()
    images, ids, mask = synth.make_inputs(8, 48, 61, [48, 30, 12, 48, 7, 25, 40, 3], H=64, W=64)
    labels = torch.tensor([0, 1, 2, 3, 4, 5, 6, 7]).cuda()
    images, ids, mask = images.cuda(), ids.cuda(), mask.cuda()
    opt = torch.optim.AdamW(model.parameters(), lr=2e-4, weight_decay=0.05)
    crit = nn.CrossEntropyLoss()
    losses = []
    for _ in range(20):
        opt.zero_grad()
        loss = crit(model(images, ids, mask)["logits"], labels)
        loss.backward()
        nn.utils.clip_grad_norm_(model.parameters(), 1.0)
        opt.step()
        losses.append(loss.item())
    print("losses", [round(x, 3) for x in losses])
    assert all(x == x for x in losses)
    for i in range(4):   # identical start, then trajectories drift apart chaotically (bf16 vs fp32)
        assert abs(losses[i] - REF_LOOP[i]) <= 0.02, (i, losses[i], REF_LOOP[i])
    # (bf16 vs fp32 trajectories of a 12-layer transformer decorrelate after a dozen steps; measured end-of-run
    # averages: 1.41-1.42 here vs 1.57 for the reference)
    assert abs(sum(losses[-5:]) / 5 - sum(REF_LOOP[-5:]) / 5) <= 0.4
    assert losses[-1] < losses[0] - 0.5
    # eval mode afterwards uses the updated weights on the inference path
    model.eval()
    with torch.no_grad():
        pred = model(images, ids, mask)["logits"]
    assert torch.isfinite(pred).all()


def test_train_step_batchnorm_batch_statistics(cuda, sens):
    """A bare model.train() (what the reference's trainers call, src/train.py:240): the frozen backbone's
    BatchNorm layers use batch statistics and update their running buffers (TV:143-163 in train mode)."""
    fix = synth.load_train_golden("train_p0_bn_train_b4_s32")
    model = synth.build_model(0)
    model.load_state_dict(sens)
    _zero_dropout(model)
    model = model.to("cuda:0")
    model.train()
    images, ids, mask = synth.make_inputs(fix["B"], fix["S"], fix["seed"], fix["lengths"], H=fix["H"], W=fix["W"])
    labels = torch.tensor(fix["labels"])
    out = model(images.cuda(), ids.cuda(), mask.cuda())
    loss = F.cross_entropy(out["logits"], labels.cuda())
    loss.backward()
    torch.cuda.synchronize()
    assert abs(loss.item() - fix["loss"]) <= 5e-3 * abs(fix["loss"]), (loss.item(), fix["loss"])
    sd = model.state_dict()
    rels = {}
    for k, v in fix["running"].items():
        got = sd[k].cpu()
        rels[k] = ((got - v).norm() / (v - sens[k]).norm().clamp_min(1e-12)).item()   # error relative to the UPDATE
    print("running-stat update rel err:", {k.replace("cnn_encoder.backbone.", ""): round(r, 4) for k, r in rels.items()})
    for k, r in rels.items():
        # 4 images of 64x64: layer4 statistics are taken over 16 values per channel after 50 bf16 conv+BN
        # layers; the stem is exact to bf16 rounding
        assert r <= (2e-2 if ".bn1.running" in k and "layer" not in k else 1.5e-1), (k, r)
    assert int(sd["cnn_encoder.backbone.bn1.num_batches_tracked"]) == fix["num_batches_tracked"] == 1
    assert int(sd["cnn_encoder.backbone.layer4.2.bn3.num_batches_tracked"]) == 1
    _, g32 = _oracle_grads_gpu(sens, images, ids, mask, labels=labels, bn_train=True)
    _, g16 = _oracle_grads_gpu(sens, images, ids, mask, labels=labels, bn_train=True, autocast=True)
    named = dict(model.named_parameters())
    # 4 images make the batch statistics of layer3/4 so noisy that EVERY bf16 run is ~45 % off fp32 here (ours
    # and stock autocast alike): only the aggregate is meaningful, single tensors scatter around their floor
    _compare_with_floor({k: named[k].grad.float().cpu() for k in g32}, g32, g16, "batch-stat BN step",
                        per_tensor=False)
    # and against the reference's own sampled gradients for the image branch (the part BN feeds)
    for k in ("cnn_encoder.projection.0.weight", "cnn_encoder.projection.3.weight", "fusion.fusion_layer.image_proj.weight"):
        r = fix["grads"][k]
        err = (_sample(named[k].grad, r["stride"]) - r["sample"]).norm().item() / r["sample"].norm().item()
        floor = (_sample(g16[k], r["stride"]) - r["sample"]).norm().item() / r["sample"].norm().item()
        assert err <= 1.5 * floor + GRAD_TOL, (k, err, floor)
    # eval mode afterwards folds the UPDATED running statistics
    model.eval()
    with torch.no_grad():
        e1 = model(images.cuda(), ids.cuda(), mask.cuda())["logits"]
    ref_sd = {k: v.float().cpu() for k, v in model.state_dict().items() if v.is_floating_point()}
    from oracle import forward_oracle
    want = forward_oracle.multimodal_forward(ref_sd, images, ids, mask)["logits"]
    assert (e1.cpu() - want).abs().max().item() <= 2e-2


def test_reference_amp_loop_shape_works(cuda, sens):
    """The reference's trainers wrap the step in fp16 autocast + GradScaler when use_amp is on
    (src/train.py:258-311, src/train_multimodal.py:518-530).  The drop-in computes in bf16/fp32 regardless; the
    wrappers must stay harmless: scaled loss -> scaled dlogits -> gradients linear in them -> unscale_ restores
    the same gradients as the plain loop."""
    images, ids, mask = synth.make_inputs(4, 32, 41, [32, 20, 7, 1], H=64, W=64)
    labels = torch.tensor([3, 1, 7, 3]).cuda()
    args = (images.cuda(), ids.cuda(), mask.cuda())
    plain = _train_model(sens)
    nn.CrossEntropyLoss()(plain(*args)["logits"], labels).backward()
    amp = _train_model(sens)
    opt = torch.optim.AdamW(amp.parameters(), lr=5e-5, weight_decay=0.05)
    scaler = torch.amp.GradScaler("cuda", init_scale=1024.0)
    with torch.amp.autocast("cuda"):
        out = amp(images=args[0], input_ids=args[1], attention_mask=args[2])
        loss = nn.CrossEntropyLoss()(out["logits"], labels)
    scaler.scale(loss).backward()
    scaler.unscale_(opt)
    total = nn.utils.clip_grad_norm_(amp.parameters(), 1.0)
    scaler.step(opt)
    scaler.update()
    assert torch.isfinite(total) and scaler.get_scale() == 1024.0      # no overflow was detected
    num = den = 0.0
    coef = min(1.0, 1.0 / (total.item() + 1e-6))
    for (k, p), (_, q) in zip(plain.named_parameters(), amp.named_parameters()):
        if p.grad is None:
            assert q.grad is None
            continue
        num += (q.grad / coef - p.grad).double().pow(2).sum().item()
        den += p.grad.double().pow(2).sum().item()
    # dlogits are rounded differently (x1024 before the bf16 gradient stream), nothing else differs
    assert (num / den) ** 0.5 <= 5e-2, (num / den) ** 0.5


def test_fused_adamw_matches_torch(cuda):
    """mrd_b200.FusedAdamW(max_grad_norm=1) == clip_grad_norm_(1) + torch.optim.AdamW, per-group lr / weight decay,
    a parameter without gradient, interchangeable state_dict."""
    import mrd_b200

    g = torch.Generator().manual_seed(21)
    shapes = [(768, 768), (3072,), (10, 128), (7,), (300, 33)]

    def make():
        return [nn.Parameter(torch.randn(*s, generator=g.manual_seed(21 + i)).cuda()) for i, s in enumerate(shapes)]

    a, b = make(), make()
    groups = lambda ps: [{"params": ps[:2], "lr": 5e-5}, {"params": ps[2:], "lr": 1e-3, "weight_decay": 0.0}]
    ref = torch.optim.AdamW(groups(a), lr=1e-4, weight_decay=0.05)
    mine = mrd_b200.FusedAdamW(groups(b), lr=1e-4, weight_decay=0.05, max_grad_norm=1.0)
    for step in range(4):
        gg = torch.Generator().manual_seed(100 + step)
        for i, (p, q) in enumerate(zip(a, b)):
            if i == 3:      # never receives a gradient: untouched by both (no weight decay either)
                continue
            grad = (torch.randn(p.shape, generator=gg) * (3.0 if step % 2 else 1e-5)).cuda()   # clipped / not clipped
            p.grad, q.grad = grad.clone(), grad.clone()
        total = nn.utils.clip_grad_norm_(a, 1.0)
        ref.step()
        mine.step()
        assert abs(mine.last_grad_norm.item() - total.item()) <= 1e-5 * total.item()
    torch.cuda.synchronize()
    for i, (p, q) in enumerate(zip(a, b)):
        assert ((p - q).norm() / p.norm()).item() <= 1e-6, i
        if i != 3:
            assert torch.allclose(ref.state[p]["exp_avg"], mine.state[q]["exp_avg"], rtol=1e-5, atol=1e-9)
            assert torch.allclose(ref.state[p]["exp_avg_sq"], mine.state[q]["exp_avg_sq"], rtol=1e-5, atol=1e-12)
            assert int(mine.state[q]["step"]) == 4
    assert torch.equal(a[3], b[3])
    # checkpoints are interchangeable with torch.optim.AdamW (src/train.py:394-437 saves optimizer_state_dict)
    other = mrd_b200.FusedAdamW(groups(make()), lr=1e-4, weight_decay=0.05)
    other.load_state_dict(ref.state_dict())
    assert other.param_groups[1]["lr"] == 1e-3


def test_train_mode_refuses_what_it_cannot_do(cuda):
    model = synth.build_model(0).to("cuda:0")
    model.train()
    images, ids, mask = synth.make_inputs(2, 16, 1, None, H=32, W=32)
    # one forward may be pending: the backward of an overwritten forward fails loudly, gradient accumulation
    # over micro-steps (forward, backward, forward, backward) works
    a = model(images.cuda(), ids.cuda(), mask.cuda())["logits"].sum()
    b = model(images.cuda(), ids.cuda(), mask.cuda())["logits"].sum()
    with pytest.raises(RuntimeError, match="overwritten"):
        a.backward()
    b.backward()
    g1 = model.classifier.classifier[6].bias.grad.clone()
    model(images.cuda(), ids.cuda(), mask.cuda())["logits"].sum().backward()
    assert torch.allclose(model.classifier.classifier[6].bias.grad, 2 * g1)   # d(sum logits)/d(bias) = batch size
    model.zero_grad()
    model.cnn_encoder.backbone.layer4.requires_grad_(True)
    with pytest.raises(NotImplementedError, match="backbone"):
        model(images.cuda(), ids.cuda(), mask.cuda())


def test_fused_adamw_drives_the_model(cuda, sens):
    """FusedAdamW writes the parameters through raw pointers; the library's packed bf16 copies (BERT GEMM weights,
    their transposed dgrad copies, the eval-mode packs) must follow.  Four steps with FusedAdamW(max_grad_norm=1)
    against four steps of clip_grad_norm_ + torch.optim.AdamW on an identical model: the train-mode logits of every
    step and the eval-mode logits afterwards agree to a small fraction of how far the training moved them."""
    images, ids, mask = synth.make_inputs(8, 32, 77, [32, 20, 7, 1, 32, 15, 9, 28], H=64, W=64)
    images, ids, mask = images.cuda(), ids.cuda(), mask.cuda()
    labels = torch.tensor([3, 1, 7, 3, 0, 9, 2, 5]).cuda()
    lr = 1e-3   # large enough that four steps move the logits far above the bf16 noise
    runs = {}
    for kind in ("torch", "fused"):
        model = _train_model(sens)
        params = list(model.parameters())
        versions = [p._version for p in params]
        opt = (mrd_b200.FusedAdamW(params, lr=lr, weight_decay=0.05, max_grad_norm=1.0) if kind == "fused"
               else torch.optim.AdamW(params, lr=lr, weight_decay=0.05))
        model.eval()
        with torch.no_grad():
            e0 = model(images, ids, mask)["logits"].clone()
        model.train()
        model.cnn_encoder.backbone.eval()
        steps = []
        for _ in range(4):
            opt.zero_grad(set_to_none=True)
            out = model(images, ids, mask)["logits"]
            steps.append(out.detach().clone())
            nn.CrossEntropyLoss()(out, labels).backward()
            if kind == "torch":
                nn.utils.clip_grad_norm_(params, 1.0)
            opt.step()
        if kind == "fused":
            bumped = [p._version > v for p, v in zip(params, versions) if p.grad is not None]
            assert bumped and all(bumped), "FusedAdamW must bump the version counter of every parameter it updates"
        model.eval()
        with torch.no_grad():
            e1 = model(images, ids, mask)["logits"].clone()
        torch.cuda.synchronize()
        runs[kind] = (e0, steps, e1)
    (e0a, sa, e1a), (e0b, sb, e1b) = runs["torch"], runs["fused"]
    assert torch.equal(e0a, e0b)
    moved_train = (sa[-1] - sa[0]).norm().item()
    moved_eval = (e1a - e0a).norm().item()
    assert moved_train > 0.05 and moved_eval > 0.05, (moved_train, moved_eval)   # the case does train
    for i, (a, b) in enumerate(zip(sa, sb)):
        assert (a - b).norm().item() <= 0.05 * moved_train, (i, (a - b).norm().item(), moved_train)
    d_eval = (e1a - e1b).norm().item()
    print(f"fused vs torch AdamW after 4 steps: train logits moved {moved_train:.3f}, eval logits moved "
          f"{moved_eval:.3f}, eval difference {d_eval:.4f}")
    assert d_eval <= 0.05 * moved_eval, (d_eval, moved_eval)


# --------------------------------------------------------------------------------------- fp32 check of the step
FP32_GRAD_TOL = 1e-4


def _fp32_check_grads(sd, images, ids, mask, labels=None, R=None):
    """Gradients of the library's fp32 check mode (plain-fp32 forward AND backward, csrc/fp32_check.cu +
    the fp32 batch-level layers): {name: grad}, loss."""
    model = _train_model(sd)
    model.configure_b200(fp32_check=True)
    out = model(images.cuda(), ids.cuda(), mask.cuda())["logits"]
    loss = F.cross_entropy(out, labels.cuda()) if R is None else (out * R.cuda()).sum()
    loss.backward()
    torch.cuda.synchronize()
    grads = {k: p.grad.detach().float().cpu() for k, p in model.named_parameters() if p.grad is not None}
    model.configure_b200(fp32_check=False)
    return loss.item(), out.detach().float().cpu(), grads


def test_fp32_check_backward_vs_reference_fixture(cuda, sens):
    """The fp32 check mode extended to the training step: loss and EVERY parameter gradient of one step against
    the fixture of the unmodified reference (autograd, fp32), at a fixed relative-L2 bar of 1e-4 per tensor.
    This is what separates a structural error in a layer's backward from bf16 rounding: the bf16 step below is
    then held to fixed bars against these gradients."""
    fix = synth.load_train_golden("train_p0_bn_eval_b4_s32")
    images, ids, mask = synth.make_inputs(fix["B"], fix["S"], fix["seed"], fix["lengths"], H=fix["H"], W=fix["W"])
    loss, logits, grads = _fp32_check_grads(sens, images, ids, mask, labels=torch.tensor(fix["labels"]))
    assert abs(loss - fix["loss"]) <= 1e-5 * abs(fix["loss"]), (loss, fix["loss"])
    assert (logits - fix["logits"]).abs().max().item() <= 1e-4
    assert set(grads) == set(fix["grads"]), sorted(set(grads) ^ set(fix["grads"]))[:5]
    worst = []
    for k, ref in fix["grads"].items():
        g = grads[k]
        if ref["norm"] == 0.0:
            assert g.abs().max().item() == 0.0, k
            continue
        if ref["norm"] < 1e-5:      # key biases (softmax shift invariance): exactly zero in exact arithmetic
            assert g.norm().item() <= 1e-4 * fix["total_norm"], k
            continue
        assert abs(g.norm().item() - ref["norm"]) <= FP32_GRAD_TOL * ref["norm"], (k, g.norm().item(), ref["norm"])
        if ref["sample"].norm().item() < 1e-3 * ref["norm"]:   # sparse gradient (word embeddings): norm only
            continue
        err = (_sample(g, ref["stride"]) - ref["sample"]).norm().item() / ref["sample"].norm().item()
        worst.append((err, k))
    worst.sort(reverse=True)
    print("fp32 check backward vs reference fixture, worst per-tensor rel-L2:", [(f"{e:.2e}", k) for e, k in worst[:4]])
    for err, k in worst:
        assert err <= FP32_GRAD_TOL, (k, err)
    tot = sum(g.double().pow(2).sum().item() for g in grads.values()) ** 0.5
    assert abs(tot - fix["total_norm"]) <= FP32_GRAD_TOL * fix["total_norm"]


# Fixed bars of the bf16 step against the fp32 check gradients (measured values in the comments are from B200
# runs of this test; the bars leave ~1.5x headroom and do NOT float with any other implementation's error):
#   * loss linear in the logits on the sensitised weights (d loss / d logits identical for both, so the error is
#     the backward's own): global <= 5e-2, per tensor <= 1e-1;
#   * cross-entropy on random-init weights (ill-conditioned: query / key gradients are second-order small and
#     every bf16 implementation is 15-25 % off on them): global <= 1.1e-1, per tensor <= 2.5e-1.
# Measured (B200, round 2): linear 0.027 global / 0.063 worst tensor; cross-entropy 0.072 / 0.154.
BF16_BARS = {"linear": (5e-2, 1e-1), "ce": (1.1e-1, 2.5e-1)}


def _bf16_vs_fp32_check(sd, images, ids, mask, kind, labels=None, R=None):
    _, _, g32 = _fp32_check_grads(sd, images, ids, mask, labels=labels, R=R)
    model = _train_model(sd)
    out = model(images.cuda(), ids.cuda(), mask.cuda())["logits"]
    loss = F.cross_entropy(out, labels.cuda()) if R is None else (out * R.cuda()).sum()
    loss.backward()
    torch.cuda.synchronize()
    named = dict(model.named_parameters())
    tot = sum(g.double().pow(2).sum().item() for g in g32.values()) ** 0.5
    num, rows = 0.0, []
    for k, r in g32.items():
        g = named[k].grad.float().cpu()
        num += (g - r).double().pow(2).sum().item()
        if r.norm().item() < 1e-4 * tot:     # (near-)zero gradients: absolute bound relative to the whole step
            assert (g - r).norm().item() <= 1e-3 * tot, k
            continue
        rows.append(((g - r).norm().item() / r.norm().item(), k))
    rows.sort(reverse=True)
    glob = num ** 0.5 / tot
    bar_g, bar_t = BF16_BARS[kind]
    print(f"bf16 step vs fp32 check ({kind}): global rel-L2 {glob:.4f} (bar {bar_g}), worst tensors "
          f"{[(round(e, 4), k) for e, k in rows[:3]]} (bar {bar_t})")
    assert glob <= bar_g, (glob, bar_g)
    for e, k in rows:
        assert e <= bar_t, (k, e, bar_t)


def test_bf16_step_fixed_bar_linear_loss(cuda):
    sd = synth.sensitise(synth.build_model(0).state_dict(), 1)
    B, S = 5, 64
    images, ids, mask = synth.make_inputs(B, S, 71, [64, 33, 64, 2, 17], H=96, W=64)
    R = torch.randn(B, 10, generator=torch.Generator().manual_seed(9))
    _bf16_vs_fp32_check(sd, images, ids, mask, "linear", R=R)


def test_bf16_step_fixed_bar_cross_entropy(cuda, sens):
    fix = synth.load_train_golden("train_p0_bn_eval_b4_s32")
    images, ids, mask = synth.make_inputs(fix["B"], fix["S"], fix["seed"], fix["lengths"], H=fix["H"], W=fix["W"])
    _bf16_vs_fp32_check(sens, images, ids, mask, "ce", labels=torch.tensor(fix["labels"]))

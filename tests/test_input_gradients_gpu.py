"""Data gradients through the frozen ResNet50 backbone: images.grad (input saliency) and forward / backward hooks on
every stage and Bottleneck, served by the saving forward + the tcgen05 data-gradient backward (engine_dgrad.cuh).

Comparators: torch.nn.grad.conv2d_input / torch's max-pool backward for the kernels alone, and the oracle
(oracle/forward_oracle.py) under torch.autograd on CUDA in fp32 (TF32 off).  Where a bar is "floor" it is the error of
the same oracle computation under bf16 autocast against fp32, x 1.3 + 5e-2 (the convention of test_train_gpu.py).
"""

import ctypes as C
from importlib import import_module

import pytest
import torch
import torch.nn.functional as F

import synth
from oracle import forward_oracle as oracle

pytestmark = pytest.mark.gpu

_lib = import_module("multimodal-rare-disease_b200._lib")
GRAD_TOL = 5e-2


@pytest.fixture(scope="module", autouse=True)
def _no_tf32():
    old = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    yield
    torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old


def _rel(a, b):
    return ((a.float() - b.float()).norm() / b.float().norm()).item()


def _floor(e16):
    return 1.3 * e16 + GRAD_TOL


def _stream():
    return torch.cuda.current_stream().cuda_stream


# ---------------------------------------------------------------------------------------------------- kernels alone
# (kind, Cin, Cout, h, w, stride) of every convolution of ResNet50 at 224 x 224: kind 1 = 1x1, 3 = 3x3, "ds" = downsample
def _resnet_convs():
    out, cin, h = [], 64, 56
    for stage, (mid, n) in enumerate([(64, 3), (128, 4), (256, 6), (512, 3)]):
        for i in range(n):
            s = 2 if (stage > 0 and i == 0) else 1
            for sh in [(1, cin, mid, h, h, 1), (3, mid, mid, h, h, s), (1, mid, 4 * mid, h // s, h // s, 1)]:
                if sh not in out:
                    out.append(sh)
            if i == 0 and ("ds", cin, 4 * mid, h, h, s) not in out:
                out.append(("ds", cin, 4 * mid, h, h, s))
            cin, h = 4 * mid, h // s
    return out


S2_ORDER = [4, 5, 3, 7, 1, 8, 6, 2, 0]
S2_PHASES = [(1, 0, [(0, 0)]), (2, 1, [(0, 0), (0, 1)]), (2, 3, [(0, 0), (1, 0)]),
             (4, 5, [(0, 0), (0, 1), (1, 0), (1, 1)])]


def _dgrad(lib, dy, wt, ldw, taps, cx, dx, sh, ph, pw, aux, mode):
    N, Ho, Wo, Cy = dy.shape
    dh = (C.c_int * len(taps))(*[t[0] for t in taps])
    dw = (C.c_int * len(taps))(*[t[1] for t in taps])
    _lib.check(lib.mrd_conv_dgrad_bf16(dy.data_ptr(), N, Ho, Wo, Cy, wt.data_ptr(), ldw, len(taps), dh, dw, cx,
                                       dx.data_ptr(), sh, sh, ph, pw, None if aux is None else aux.data_ptr(), mode,
                                       _stream()), "mrd_conv_dgrad_bf16")


@pytest.mark.parametrize("shape", _resnet_convs(), ids=lambda s: "-".join(map(str, s)))
def test_conv_dgrad_kernel(lib, cuda, shape):
    kind, cin, cout, h, w, s = shape
    N = 2
    k = 3 if kind == 3 else 1
    g = torch.Generator().manual_seed(cin * 7 + cout + h + s)
    wf = (torch.randn(cout, cin, k, k, generator=g) / (cin * k * k) ** 0.5).bfloat16().cuda()
    ho, wo = h // s, w // s
    dy = torch.randn(N, cout, ho, wo, generator=g).bfloat16().cuda()
    ref = torch.nn.grad.conv2d_input((N, cin, h, w), wf.float(), dy.float(), stride=s, padding=k // 2)
    ref = ref.permute(0, 2, 3, 1)                                    # NHWC like ours
    dy_nhwc = dy.permute(0, 2, 3, 1).contiguous()
    wk = wf.permute(1, 2, 3, 0).reshape(cin, k * k, cout)           # [Cin][tap][Cout], tap = kh*3 + kw
    if kind == 3 and s == 1:
        wt = wk.flip(1).contiguous()                                 # flipped filter
        mask = (torch.randn(N, h, w, cin, generator=g) > 0).bfloat16().cuda() * torch.rand(N, h, w, cin, generator=g).bfloat16().cuda()
        dx = torch.empty(N, h, w, cin, dtype=torch.bfloat16, device=cuda)
        taps = [(r - 1, c - 1) for r in range(3) for c in range(3)]
        _dgrad(lib, dy_nhwc, wt, 9 * cout, taps, cin, dx, 1, 0, 0, mask, 2)
        ref = ref * (mask > 0)
    elif kind == 3:
        wt = wk[:, S2_ORDER].contiguous()
        mask = (torch.randn(N, h, w, cin, generator=g) > 0).bfloat16().cuda()
        dx = torch.full((N, h, w, cin), float("nan"), dtype=torch.bfloat16, device=cuda)
        for ph, (n, first, taps) in enumerate(S2_PHASES):
            _dgrad(lib, dy_nhwc, wt[:, first:], 9 * cout, taps, cin, dx, 2, ph >> 1, ph & 1, mask, 2)
        ref = ref * (mask > 0)
    elif kind == "ds":
        # the conv1-path gradient already sits in dX; the downsample gradient is added at the (stride-s) pixels it read
        base = torch.randn(N, h, w, cin, generator=g).bfloat16().cuda()
        dx = base.clone()
        _dgrad(lib, dy_nhwc, wk[:, 0].contiguous(), cout, [(0, 0)], cin, dx, s, 0, 0, dx, 1)
        ref = ref + base.float()
        mask = None
    else:
        mask = (torch.randn(N, h, w, cin, generator=g) > 0).bfloat16().cuda()
        dx = torch.empty(N, h, w, cin, dtype=torch.bfloat16, device=cuda)
        _dgrad(lib, dy_nhwc, wk[:, 0].contiguous(), cout, [(0, 0)], cin, dx, 1, 0, 0, mask, 2)
        ref = ref * (mask > 0)
    torch.cuda.synchronize()
    err = _rel(dx, ref)
    assert err <= 5e-3, (shape, err)
    if mask is not None:
        assert torch.all(dx[mask <= 0] == 0)


def test_stem_dgrad_kernel(lib, cuda):
    N, H, W = 2, 224, 224
    g = torch.Generator().manual_seed(5)
    w = (torch.randn(64, 3, 7, 7, generator=g) * 0.1).cuda()
    gamma = (torch.rand(64, generator=g) + 0.5).cuda()
    var = (torch.rand(64, generator=g) + 0.1).cuda()
    d = torch.randn(N, 64, H // 2, W // 2, generator=g).bfloat16().cuda()
    wf = torch.empty(7 * 7 * 64 * 3, device=cuda)
    _lib.check(lib.mrd_pack_stem_dgrad(w.data_ptr(), gamma.data_ptr(), var.data_ptr(), C.c_float(1e-5),
                                       wf.data_ptr(), _stream()))
    out = torch.empty(N, 3, H, W, device=cuda)
    _lib.check(lib.mrd_stem_dgrad_f32(d.permute(0, 2, 3, 1).contiguous().data_ptr(), wf.data_ptr(), N, H, W,
                                      out.data_ptr(), _stream()))
    scale = (gamma / torch.sqrt(var + 1e-5)).view(64, 1, 1, 1)
    ref = torch.nn.grad.conv2d_input((N, 3, H, W), w * scale, d.float(), stride=2, padding=3)
    assert _rel(out, ref) <= 5e-3


def test_maxpool_bwd_kernel(lib, cuda):
    N, Cc, H, W = 2, 64, 112, 112
    g = torch.Generator().manual_seed(6)
    y = F.relu(torch.randn(N, Cc, H, W, generator=g)).bfloat16().cuda()       # the pooled (post-ReLU) tensor
    gout = torch.randn(N, Cc, H // 2, W // 2, generator=g).bfloat16().cuda()
    x = y.clone().requires_grad_(True)
    F.max_pool2d(x, 3, 2, 1).backward(gout)
    ref = x.grad.float() * (y > 0)
    dx = torch.empty(N, H, W, Cc, dtype=torch.bfloat16, device=cuda)
    _lib.check(lib.mrd_maxpool3x3s2_bwd_bf16(gout.permute(0, 2, 3, 1).contiguous().data_ptr(),
                                             y.permute(0, 2, 3, 1).contiguous().data_ptr(), N, H, W, Cc,
                                             dx.data_ptr(), _stream()))
    torch.cuda.synchronize()
    assert _rel(dx.permute(0, 3, 1, 2), ref) <= 1e-6


# ---------------------------------------------------------------------------------------------------- model level
@pytest.fixture(scope="module")
def models(cuda):
    plain = synth.build_model(0)
    sd = plain.state_dict()
    sens_sd = synth.sensitise(sd, 1)
    sens = synth.build_model(0)
    sens.load_state_dict(sens_sd)
    return {"plain": (plain.to(cuda).eval(), sd), "sens": (sens.to(cuda).eval(), sens_sd)}


def _inputs(cuda, B, seed=91):
    images, ids, mask = synth.make_inputs(B, 32, seed, [32, 17, 9, 25][:B] if B <= 4 else None)
    return images.to(cuda), ids.to(cuda), mask.to(cuda)


def _sd_cuda(sd, cuda):
    return {k: v.float().to(cuda) for k, v in sd.items() if v.is_floating_point()}


def _oracle_blocks(sd, p="cnn_encoder.backbone."):
    """[(prefix, stride)] of the 16 bottlenecks."""
    out = []
    for stage in range(1, 5):
        i = 0
        while f"{p}layer{stage}.{i}.conv1.weight" in sd:
            out.append((f"{p}layer{stage}.{i}.", 2 if (stage > 1 and i == 0) else 1))
            i += 1
    return out


def _oracle_block(sd, q, stride, x):
    y = F.relu(oracle._bn(sd, q + "bn1", F.conv2d(x, sd[q + "conv1.weight"])))
    y = F.relu(oracle._bn(sd, q + "bn2", F.conv2d(y, sd[q + "conv2.weight"], stride=stride, padding=1)))
    y = oracle._bn(sd, q + "bn3", F.conv2d(y, sd[q + "conv3.weight"]))
    identity = x
    if q + "downsample.0.weight" in sd:
        identity = oracle._bn(sd, q + "downsample.1", F.conv2d(x, sd[q + "downsample.0.weight"], stride=stride))
    return F.relu(y + identity)


def _oracle_stem(sd, images, p="cnn_encoder.backbone."):
    x = F.conv2d(images, sd[p + "conv1.weight"], stride=2, padding=3)
    return F.max_pool2d(F.relu(oracle._bn(sd, p + "bn1", x)), 3, 2, 1)


def _oracle_tail(sd, fmap, txt):
    pooled = fmap.mean(dim=(2, 3))
    h = F.relu(F.linear(pooled, sd["cnn_encoder.projection.0.weight"], sd["cnn_encoder.projection.0.bias"]))
    img = F.linear(h, sd["cnn_encoder.projection.3.weight"], sd["cnn_encoder.projection.3.bias"])
    fused, _ = oracle.attention_fusion(sd, img, txt)
    return oracle.classification_head(sd, fused)


def _oracle_txt(sd, ids, mask, cuda):
    with torch.no_grad():
        sdc = {k: v.float() for k, v in sd.items() if v.is_floating_point()}
        return oracle.text_encoder(sdc, ids.cpu(), mask.cpu()).to(cuda)


def _oracle_from_block(sdc, blocks, k0, x, txt, cls, autocast=False):
    """d(logit[0, cls]) / dx where x is the input of bottleneck k0 (k0 = 16: x is the layer4 map)."""
    x = x.detach().clone().requires_grad_(True)
    with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
        y = x
        for q, s in blocks[k0:]:
            y = _oracle_block(sdc, q, s, y)
        logits = _oracle_tail(sdc, y.float(), txt)
    logits[0, cls].backward()
    return x.grad.detach()


@pytest.mark.parametrize("weights", ["plain", "sens"])
def test_every_block_backward_locally(models, cuda, weights):
    """Hooks on all 16 Bottlenecks: for block k, autograd through the fp32 oracle block at OUR hooked input and with
    OUR grad_output gives grad_input; the stem is checked the same way against images.grad."""
    model, sd = models[weights]
    sdc = _sd_cuda(sd, cuda)
    blocks = _oracle_blocks(sdc)
    images, ids, mask = _inputs(cuda, 2)
    acts, gin, gout, handles = {}, {}, {}, []
    mods = [b for L in range(1, 5) for b in getattr(model.cnn_encoder.backbone, f"layer{L}")]
    for k, m in enumerate(mods):
        handles.append(m.register_forward_hook(lambda mm, i, o, k=k: acts.__setitem__(k, o.detach().clone())))
        handles.append(m.register_full_backward_hook(
            lambda mm, gi, go, k=k: (gin.__setitem__(k, gi[0].detach().clone()),
                                     gout.__setitem__(k, go[0].detach().clone()))))
    x_img = images.clone().requires_grad_(True)
    out = model(x_img, ids, mask)
    out["logits"][0, 3].backward()
    for h in handles:
        h.remove()
    assert sorted(acts) == list(range(16)) and sorted(gin) == list(range(16))
    worst = []
    with torch.no_grad():
        x0 = _oracle_stem(sdc, images)
    for k, (q, s) in enumerate(blocks):
        x_in = x0 if k == 0 else acts[k - 1]
        assert gin[k].shape == x_in.shape and gout[k].shape == acts[k].shape
        res = []
        for ac in (False, True):
            x = x_in.clone().requires_grad_(True)
            with torch.autocast("cuda", dtype=torch.bfloat16, enabled=ac):
                y = _oracle_block(sdc, q, s, x)
            y.float().backward(gout[k])
            res.append(x.grad)
        err, e16 = _rel(gin[k], res[0]), _rel(res[1], res[0])
        worst.append((err, e16, k))
        assert err <= max(2e-2, _floor(e16)), (k, err, e16)
    # stem: d(images) from our grad_input of layer1.0 through the fp32 stem + max-pool.  The max-pool routes each
    # window's gradient to its maximum, which bf16 rounding of the stem output moves between near-equal neighbours:
    # the bar is the bf16-autocast stem's own error
    res = []
    for ac in (False, True):
        x = images.clone().requires_grad_(True)
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=ac):
            y = _oracle_stem(sdc, x)
        y.float().backward(gin[0])
        res.append(x.grad)
    err_stem, e16 = _rel(x_img.grad, res[0]), _rel(res[1], res[0])
    print(f"[{weights}] per-block grad_input rel-L2 (ours, autocast oracle): worst "
          f"{sorted(worst, reverse=True)[:3]}; stem {err_stem:.4f} (autocast {e16:.4f})")
    assert err_stem <= max(2e-2, _floor(e16)), (err_stem, e16)


@pytest.mark.parametrize("weights", ["plain", "sens"])
def test_images_grad_end_to_end(models, cuda, weights):
    model, sd = models[weights]
    sdc = _sd_cuda(sd, cuda)
    blocks = _oracle_blocks(sdc)
    images, ids, mask = _inputs(cuda, 2)
    x = images.clone().requires_grad_(True)
    out = model(x, ids, mask)
    cls = int(out["logits"][0].argmax())
    out["logits"][0, cls].backward()
    assert x.grad is not None and x.grad.dtype == torch.float32 and x.grad.shape == images.shape
    txt = _oracle_txt(sd, ids, mask, cuda)
    res = []
    for ac in (False, True):
        xi = images.clone().requires_grad_(True)
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=ac):
            y = _oracle_stem(sdc, xi)
            for q, s in blocks:
                y = _oracle_block(sdc, q, s, y)
            logits = _oracle_tail(sdc, y.float(), txt)
        logits[0, cls].backward()
        res.append(xi.grad)
    err, e16 = _rel(x.grad, res[0]), _rel(res[1], res[0])
    sal, sal_ref = x.grad[0].abs().amax(0).flatten(), res[0][0].abs().amax(0).flatten()
    corr = torch.corrcoef(torch.stack([sal, sal_ref]))[0, 1].item()
    print(f"[{weights}] images.grad rel-L2 {err:.4f} (bf16-autocast oracle {e16:.4f}); saliency-map correlation "
          f"{corr:.4f}; sample 1 (no gradient) max |grad| {x.grad[1].abs().max().item():.2e}")
    assert err <= _floor(e16), (err, e16)
    assert torch.all(x.grad[1] == 0)   # samples are independent


class GradCAM:
    """notebooks/explainability.ipynb cell 3, __init__ / hooks / generate_cam as written there."""

    def __init__(self, model, target_layer):
        self.model = model
        self.target_layer = target_layer
        self.gradients = None
        self.activations = None

        # Register hooks
        self.target_layer.register_forward_hook(self._save_activation)
        self.target_layer.register_full_backward_hook(self._save_gradient)

    def _save_activation(self, module, input, output):
        self.activations = output.detach()

    def _save_gradient(self, module, grad_input, grad_output):
        self.gradients = grad_output[0].detach()

    def generate_cam(self, input_image, input_ids, attention_mask, target_class=None):
        self.model.eval()

        # Forward pass
        output = self.model(input_image, input_ids, attention_mask)

        if target_class is None:
            target_class = output['logits'].argmax(dim=1).item()

        # Backward pass
        self.model.zero_grad()
        output['logits'][0, target_class].backward()

        # Generate CAM
        gradients = self.gradients[0]  # [C, H, W]
        activations = self.activations[0]  # [C, H, W]

        # Global average pooling of gradients
        weights = gradients.mean(dim=(1, 2), keepdim=True)

        # Weighted sum of activations
        cam = (weights * activations).sum(dim=0)
        cam = F.relu(cam)  # Apply ReLU

        # Normalize
        cam = cam - cam.min()
        cam = cam / (cam.max() + 1e-8)

        return cam.cpu().numpy(), target_class, output['probs'][0, target_class].item()


@pytest.mark.parametrize("target,hi,side", [("layer3", 12, 14), ("layer4[-1]", 15, 7), ("layer1", 2, 56)])
def test_gradcam_on_other_layers(models, cuda, target, hi, side):
    model, sd = models["plain"]
    sdc = _sd_cuda(sd, cuda)
    blocks = _oracle_blocks(sdc)
    bb = model.cnn_encoder.backbone
    layer = {"layer3": bb.layer3, "layer4[-1]": bb.layer4[-1], "layer1": bb.layer1}[target]
    images, ids, mask = _inputs(cuda, 1)
    tool = GradCAM(model, layer)
    try:
        cam, cls, conf = tool.generate_cam(images, ids, mask)
    finally:
        layer._forward_hooks.clear()
        layer._backward_hooks.clear()
    assert cam.shape == (side, side) and 0.0 < conf <= 1.0
    with torch.no_grad():
        y = _oracle_stem(sdc, images)
        for q, s in blocks[:hi + 1]:
            y = _oracle_block(sdc, q, s, y)
    err_a = _rel(tool.activations, y)
    txt = _oracle_txt(sd, ids, mask, cuda)
    g32 = _oracle_from_block(sdc, blocks, hi + 1, tool.activations, txt, cls)
    g16 = _oracle_from_block(sdc, blocks, hi + 1, tool.activations, txt, cls, autocast=True)
    err_g, e16 = _rel(tool.gradients, g32), _rel(g16, g32)
    print(f"Grad-CAM on {target}: activation rel-L2 {err_a:.4f}; gradient rel-L2 {err_g:.4f} (floor {e16:.4f})")
    assert err_a <= 2e-2
    assert err_g <= max(2e-2, _floor(e16))
    assert model.classifier.classifier[0].weight.grad is not None
    assert bb.conv1.weight.grad is None


def test_layer4_hooks_issue_the_same_launches(models, cuda):
    """Hooks on layer4 alone run the pre-existing Grad-CAM path: the launches of the plain training-step forward with
    the layer4 map plus its backward with d_pooled, and nothing of the data-gradient path; grad_input is (None,)."""
    model, _ = models["plain"]
    images, ids, mask = _inputs(cuda, 2)
    layer = model.cnn_encoder.get_attention_layer()
    seen = []
    h1 = layer.register_forward_hook(lambda m, i, o: None)
    h2 = layer.register_full_backward_hook(lambda m, gi, go: seen.append(gi))
    try:
        model(images, ids, mask)["logits"][0, 1].backward()   # warm-up: weights packed, plans built
        eng = model._engine(allow_training=True)
        torch.cuda.synchronize()
        eng.profile(True)
        model(images, ids, mask)["logits"][0, 1].backward()
        torch.cuda.synchronize()
        hooked = {r["label"]: r["launches"] for r in eng.profile_report()}
        eng.profile(False)
    finally:
        h1.remove()
        h2.remove()
    assert seen[-1] == (None,)
    assert not any(k.startswith("dgrad") for k in hooked), hooked
    named = model._trainable()
    eng.profile(True)
    logits, _ = eng.train_forward(images, ids, mask, model.num_classes, 0, want_map=True)
    dl = torch.zeros_like(logits)
    dl[0, 1] = 1.0
    eng.train_backward(dl, tuple((n, tuple(p.shape)) for n, p in named), want_dpooled=True)
    torch.cuda.synchronize()
    direct = {r["label"]: r["launches"] for r in eng.profile_report()}
    eng.profile(False)
    assert hooked == direct


def test_frozen_model_saliency(cuda):
    model = synth.build_model(0).to(cuda).eval()
    model.requires_grad_(False)
    images, ids, mask = _inputs(cuda, 2)
    x = images.clone().requires_grad_(True)
    model(x, ids, mask)["logits"][1, 2].backward()
    assert x.grad is not None and x.grad.abs().sum().item() > 0 and torch.all(x.grad[0] == 0)
    assert all(p.grad is None for p in model.parameters())


def test_batch_invariance(models, cuda):
    """B = 4 with one-hot d(logits) per sample against four B = 1 runs.  The backbone's backward is batch-invariant bit
    for bit: samples never mix and every per-row sum runs in the same order whatever the batch.  Its input d_pooled is
    not: the fp32 GEMMs of the head's backward reduce split-K partial sums with atomics, so d_pooled can differ in the
    last bit between any two runs.  Where that moves one bf16 rounding of the chain's first gradient, the difference
    grows through 16 blocks of bf16 gradients to the chain's own rounding noise (~1e-2).  So: a sample whose layer4
    gradient is bitwise equal must get a bitwise equal images.grad; any other is held to that noise level."""
    model, _ = models["plain"]
    images, ids, mask = _inputs(cuda, 4, seed=93)
    cls = [3, 1, 7, 3]
    layer4 = model.cnn_encoder.backbone.layer4

    def run(sl, c):
        top = []
        h = layer4.register_full_backward_hook(lambda m, gi, go: top.append(go[0].clone()))
        try:
            x = images[sl].clone().requires_grad_(True)
            logits = model(x, ids[sl], mask[sl])["logits"]
            onehot = F.one_hot(torch.tensor(c, device=cuda), logits.shape[1]).float()
            (logits * onehot).sum().backward()
        finally:
            h.remove()
        return x.grad, top[0]

    g4, t4 = run(slice(0, 4), cls)
    rows = []
    for b in range(4):
        g1, t1 = run(slice(b, b + 1), [cls[b]])
        same_top = torch.equal(t4[b:b + 1], t1)
        same = torch.equal(g4[b:b + 1], g1)
        err = _rel(g4[b:b + 1], g1)
        rows.append((b, same_top, same, err))
        if same_top:
            assert same, (b, err)
        else:
            assert err <= 5e-2, (b, err)
    print("B=4 vs four B=1 runs (sample, layer4 gradient bitwise, images.grad bitwise, rel-L2):", rows)


def test_mode_switching(models, cuda):
    model, _ = models["plain"]
    images, ids, mask = _inputs(cuda, 2)
    with torch.no_grad():
        ref = model(images, ids, mask)["logits"]
    xb = images.bfloat16().requires_grad_(True)
    model(xb, ids, mask)["logits"][0, 0].backward()
    assert xb.grad.dtype == torch.bfloat16 and xb.grad.shape == xb.shape
    # hooks below layer4: served; grad_input is (None,) when nothing below the module asks for the chain
    l3 = model.cnn_encoder.backbone.layer3
    got = []
    hf = l3.register_forward_hook(lambda m, i, o: got.append(("f", i, tuple(o.shape))))
    hb = l3.register_full_backward_hook(lambda m, gi, go: got.append(("b", gi, tuple(go[0].shape))))
    with torch.no_grad():
        model(images, ids, mask)
    assert got == [("f", (), (2, 1024, 14, 14))]
    model(images, ids, mask)["logits"][0, 0].backward()
    assert got[-1] == ("b", (None,), (2, 1024, 14, 14))
    x = images.clone().requires_grad_(True)
    model(x, ids, mask)["logits"][0, 0].backward()
    assert got[-1][0] == "b" and got[-1][1][0].shape == (2, 512, 28, 28)
    hf.remove()
    hb.remove()
    out = model(images, ids, mask)["logits"]
    assert not out.requires_grad and torch.equal(out, ref)


def test_refusals(models, cuda):
    model, _ = models["plain"]
    images, ids, mask = _inputs(cuda, 2)
    bb = model.cnn_encoder.backbone
    for m in (bb.conv1, bb.layer3[0].conv2, bb.layer2[0].downsample, bb.avgpool):
        h = m.register_forward_hook(lambda *a: None)
        try:
            with pytest.raises(NotImplementedError, match="layer1"):
                model(images, ids, mask)
        finally:
            h.remove()
    x = images.clone().requires_grad_(True)
    model.train()
    try:
        with pytest.raises(NotImplementedError, match="BatchNorm"):
            model(x, ids, mask)
    finally:
        model.eval()
    model.configure_b200(fp32_check=True)
    try:
        with pytest.raises(NotImplementedError, match="fp32 check"):
            model(x, ids, mask)
    finally:
        model.configure_b200(fp32_check=False)
    big, bids, bmask = synth.make_inputs(513, 8, 7, H=32, W=32)
    with pytest.raises(_lib.MrdError, match="512"):
        model(big.to(cuda).requires_grad_(True), bids.to(cuda), bmask.to(cuda))

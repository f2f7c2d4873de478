"""Per-kernel parity through the C ABI (include/mrd_b200.h) against the same op in plain PyTorch
fp32 on the same bf16-rounded operands.  Tolerances: outputs are bf16 (8 mantissa bits), so the bar
is |err| <= 2^-7 * |ref| + a small absolute term that covers fp32 accumulation-order differences."""

import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

BF = torch.bfloat16


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _check(lib, rc):
    assert rc == 0, (rc, lib.mrd_last_error())


def _close(out, ref, rel=2 ** -7, abs_=1e-2, what=""):
    out, ref = out.float(), ref.float()
    err = (out - ref).abs()
    bound = rel * ref.abs() + abs_
    bad = err > bound
    assert not bad.any(), (f"{what}: {int(bad.sum())}/{bad.numel()} outside tolerance; max err "
                           f"{err.max().item():.4g} at ref {ref.flatten()[err.argmax()].item():.4g}")


# ------------------------------------------------------------------ GEMM (K2)
@pytest.mark.parametrize("M,N,K,act,res,f32", [
    (128, 64, 64, 0, False, False),
    (256, 128, 128, 1, False, True),
    (300, 768, 768, 0, True, False),        # ragged M, BERT out-proj + residual
    (1024, 2304, 768, 0, False, False),     # fused QKV
    (777, 3072, 768, 2, False, False),      # FFN1 + exact GELU
    (512, 768, 3072, 0, True, True),        # FFN2 + residual, long K
    (5, 512, 2048, 1, False, True),         # tiny batch (projection)
    (20000, 256, 64, 1, False, False),      # ResNet layer1-like 1x1 conv, many tiles (persistence)
    (4096, 64, 256, 1, False, False),       # narrow N
    # >= 2 tiles per SM with 256-wide tiles: two-CTA clusters that share each weight tile by TMA multicast (PAIR)
    (19000, 768, 768, 0, True, False),      # odd stripe count: the last pair's second tile lies outside the matrix
    (19000, 3072, 768, 2, False, False),    # GELU: two-group epilogue variant
    (33000, 2304, 768, 0, False, True),     # QKV shape + fp32 side output
    (40000, 512, 128, 1, True, False),      # short K with residual (ResNet layer2 conv3 shape)
])
def test_gemm(lib, cuda, M, N, K, act, res, f32):
    g = torch.Generator(device="cuda").manual_seed(M * 7 + N)
    A = torch.randn(M, K, device=cuda, generator=g).to(BF)
    W = (torch.randn(N, K, device=cuda, generator=g) / math.sqrt(K)).to(BF)
    bias = torch.randn(N, device=cuda, generator=g)
    R = torch.randn(M, N, device=cuda, generator=g).to(BF) if res else None
    C = torch.full((M, N), float("nan"), device=cuda, dtype=BF)
    C32 = torch.full((M, N), float("nan"), device=cuda) if f32 else None
    _check(lib, lib.mrd_gemm_bf16(A.data_ptr(), K, M, K, W.data_ptr(), N, bias.data_ptr(), C.data_ptr(),
                                  N, R.data_ptr() if res else None, N,
                                  C32.data_ptr() if f32 else None, N, act, _stream()))
    torch.cuda.synchronize()
    ref = A.float() @ W.float().t() + bias
    if res:
        ref = ref + R.float()
    if act == 1:
        ref = F.relu(ref)
    elif act == 2:
        ref = F.gelu(ref)
    _close(C, ref, what="gemm bf16 out")
    if f32:
        _close(C32, ref, rel=1e-4, abs_=2e-3, what="gemm f32 out")


@pytest.mark.parametrize("M,N,K,res", [
    # CTA pairs (at least two 256-wide tiles per SM on a 148-SM B200)
    (19000, 768, 768, True),      # BertSelfOutput: dense + residual + LayerNorm, ragged last stripe
    (19000, 768, 3072, True),     # BertOutput, long K
    (12800, 768, 3072, True),     # whole stripes only
    (20480, 1024, 256, False),    # four CTAs per stripe, no residual
    (40000, 512, 128, True),      # two CTAs per stripe, several stripes per CTA pair
    # single CTAs
    (5, 768, 3072, True),         # a handful of rows: the same kernel (the path must not depend on the batch size)
    (300, 768, 3072, True),       # a few stripes, ragged
    (12000, 768, 768, True),      # more tiles than SMs: a stripe's CTAs are at different iterations
    (4096, 1024, 768, True),      # four CTAs per stripe
    (9000, 512, 768, False),      # two CTAs per stripe, no residual
])
def test_gemm_layernorm(lib, cuda, M, N, K, res):
    """GEMM with LayerNorm over the whole row in the epilogue against fp32 torch: layer_norm(A W^T + b + R).  The
    N/256 CTAs of a 128-row stripe exchange their partial statistics through the workspace in global memory."""
    ws = torch.zeros(lib.mrd_gemm_ln_ws_bytes(M), device=cuda, dtype=torch.uint8)
    g = torch.Generator(device="cuda").manual_seed(M + N + K)
    A = torch.randn(M, K, device=cuda, generator=g).to(BF)
    W = (torch.randn(N, K, device=cuda, generator=g) / math.sqrt(K)).to(BF)
    bias = torch.randn(N, device=cuda, generator=g)
    # rows with very different means / scales: the statistics must be per row
    R = (torch.randn(M, N, device=cuda, generator=g) * torch.rand(M, 1, device=cuda, generator=g) * 4
         + torch.randn(M, 1, device=cuda, generator=g) * 3).to(BF) if res else None
    gamma = torch.rand(N, device=cuda, generator=g) + 0.5
    beta = torch.randn(N, device=cuda, generator=g) * 0.3
    C = torch.full((M, N), float("nan"), device=cuda, dtype=BF)
    outs = []
    for _ in range(3):
        C.fill_(float("nan"))
        _check(lib, lib.mrd_gemm_ln_bf16(A.data_ptr(), K, M, K, W.data_ptr(), N, bias.data_ptr(), C.data_ptr(), N,
                                         R.data_ptr() if res else None, N, gamma.data_ptr(), beta.data_ptr(), 1e-12,
                                         ws.data_ptr(), _stream()))
        torch.cuda.synchronize()
        outs.append(C.clone())
    x = A.float() @ W.float().t() + bias
    if res:
        x = x + R.float()
    ref = F.layer_norm(x, (N,), gamma, beta, 1e-12)
    _close(C, ref, what=f"gemm + layernorm {M}x{N}x{K}")
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[0], outs[2]), "run-to-run difference"
    # the arrival / departure counters re-arm themselves
    rec = ws.view(-1, 128 * 8 * 8 + 64)
    assert int(rec[:, 128 * 8 * 8:].contiguous().view(torch.int32).abs().sum()) == 0


def test_gemm_layernorm_rejects_other_widths(lib, cuda):
    A = torch.zeros(256, 768, device=cuda, dtype=BF)
    v = torch.zeros(768, device=cuda)
    rc = lib.mrd_gemm_ln_bf16(A.data_ptr(), 768, 256, 768, A.data_ptr(), 640, v.data_ptr(), A.data_ptr(), 640, None, 0,
                              v.data_ptr(), v.data_ptr(), 1e-12, None, _stream())
    assert rc != 0 and b"outside" in lib.mrd_last_error()
    # a supported width without the statistics workspace
    rc = lib.mrd_gemm_ln_bf16(A.data_ptr(), 768, 256, 768, A.data_ptr(), 768, v.data_ptr(), A.data_ptr(), 768, None, 0,
                              v.data_ptr(), v.data_ptr(), 1e-12, None, _stream())
    assert rc == -1 and b"mrd_gemm_ln_ws_bytes" in lib.mrd_last_error()


def test_gemm_strided(lib, cuda):
    """A rows taken with a stride (CLS rows of a [B,S,768] tensor), C written into a wider buffer."""
    B, S, K, N = 37, 16, 768, 512
    g = torch.Generator(device="cuda").manual_seed(5)
    X = torch.randn(B, S, K, device=cuda, generator=g).to(BF)
    W = (torch.randn(N, K, device=cuda, generator=g) / math.sqrt(K)).to(BF)
    bias = torch.randn(N, device=cuda, generator=g)
    C = torch.zeros(B, 2 * N, device=cuda, dtype=BF)
    _check(lib, lib.mrd_gemm_bf16(X.data_ptr(), S * K, B, K, W.data_ptr(), N, bias.data_ptr(),
                                  C[:, N:].data_ptr(), 2 * N, None, 0, None, 0, 0, _stream()))
    torch.cuda.synchronize()
    ref = X[:, 0].float() @ W.float().t() + bias
    _close(C[:, N:], ref, what="strided gemm")
    assert (C[:, :N] == 0).all()


def test_gemm_rejects_bad_shapes(lib, cuda):
    A = torch.zeros(8, 100, device=cuda, dtype=BF)
    rc = lib.mrd_gemm_bf16(A.data_ptr(), 100, 8, 100, A.data_ptr(), 64, None, A.data_ptr(), 64, None,
                           0, None, 0, 0, _stream())
    assert rc != 0 and b"unsupported" in lib.mrd_last_error()


# ------------------------------------------------------------------ convolutions (K1)
def _conv_case(lib, cuda, N, H, W, Cin, Cout, k, stride, act, res, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed + Cin + Cout + H)
    x = torch.randn(N, Cin, H, W, device=cuda, generator=g).to(BF)
    w = (torch.randn(Cout, Cin, k, k, device=cuda, generator=g) / math.sqrt(Cin * k * k)).to(BF)
    bias = torch.randn(Cout, device=cuda, generator=g)
    Ho, Wo = H // stride, W // stride
    r = torch.randn(N, Cout, Ho, Wo, device=cuda, generator=g).to(BF) if res else None
    x_nhwc = x.permute(0, 2, 3, 1).contiguous()
    w_ohwi = w.permute(0, 2, 3, 1).contiguous()
    r_nhwc = r.permute(0, 2, 3, 1).contiguous() if res else None
    y = torch.full((N, Ho, Wo, Cout), float("nan"), device=cuda, dtype=BF)
    _check(lib, lib.mrd_conv2d_nhwc_bf16(x_nhwc.data_ptr(), N, H, W, Cin, w_ohwi.data_ptr(), Cout, k,
                                         stride, bias.data_ptr(), y.data_ptr(),
                                         r_nhwc.data_ptr() if res else None, act, 0, _stream()))
    torch.cuda.synchronize()
    ref = F.conv2d(x.float(), w.float(), bias, stride=stride, padding=k // 2)
    if res:
        ref = ref + r.float()
    if act == 1:
        ref = F.relu(ref)
    _close(y.permute(0, 3, 1, 2), ref, what=f"conv k{k} s{stride} {Cin}->{Cout} {H}x{W}")


@pytest.mark.parametrize("N,H,W,Cin,Cout,k,stride,act,res", [
    (2, 56, 56, 64, 64, 1, 1, 1, False),      # layer1 conv1
    (2, 56, 56, 64, 64, 3, 1, 1, False),      # layer1 conv2 (rows-of-56 tiles, zero halo)
    (2, 56, 56, 64, 256, 1, 1, 1, True),      # layer1 conv3 + identity
    (3, 56, 56, 128, 128, 3, 2, 1, False),    # layer2.0 conv2, stride 2 (parity-phase views)
    (3, 56, 56, 256, 512, 1, 2, 0, False),    # layer2.0 downsample, 1x1 stride 2
    (2, 28, 28, 128, 128, 3, 1, 1, False),    # layer2 conv2
    (5, 14, 14, 256, 256, 3, 1, 1, False),    # layer3 conv2 (partial tile rows)
    (5, 14, 14, 512, 512, 3, 2, 1, False),    # layer4.0 conv2
    (7, 7, 7, 512, 512, 3, 1, 1, False),      # layer4 conv2 (several images per tile, odd count)
    (3, 7, 7, 512, 2048, 1, 1, 1, True),      # layer4 conv3 + identity
    (1, 32, 64, 64, 64, 3, 1, 0, False),      # non-square
    (205, 14, 14, 256, 256, 3, 1, 1, False),  # layer3 conv2 at pass size: CTA pairs, odd tile count (315)
    (333, 7, 7, 512, 512, 3, 1, 1, False),    # layer4 conv2 at pass size: CTA pairs, two column tiles
    (150, 28, 28, 256, 256, 3, 2, 1, False),  # strided 3x3 on CTA pairs (parity-phase views)
])
def test_conv(lib, cuda, N, H, W, Cin, Cout, k, stride, act, res):
    _conv_case(lib, cuda, N, H, W, Cin, Cout, k, stride, act, res)


@pytest.mark.parametrize("N,H,W,Cin,Cout,act", [
    (3, 56, 56, 64, 64, 1),      # layer1 conv2: 2 padded rows per tile
    (2, 28, 28, 128, 128, 1),    # layer2 conv2: 4 rows per tile, two 64-channel chunks
    (5, 20, 24, 64, 128, 0),     # ragged: H not a multiple of th, non-square
    (1, 28, 28, 128, 64, 1),
    (70, 28, 28, 64, 64, 1),     # many tiles per CTA (persistence, ring wrap-around)
    (65, 28, 28, 128, 128, 1),   # layer2 conv2 at pass size: CTA pairs (cta_group::2), odd tile count (455)
    (48, 28, 28, 64, 128, 0),    # CTA pairs, one channel chunk, even tile count
    (11, 56, 56, 64, 64, 1),     # layer1 conv2 on CTA pairs (64-wide tile over the pair), odd tile count (308 + 0)
])
def test_conv3x3_flat(lib, cuda, N, H, W, Cin, Cout, act):
    """1x1 conv writing the interior of a zero-bordered buffer, then the flat-shift 3x3 conv on it."""
    g = torch.Generator(device="cuda").manual_seed(H * W + Cin)
    x = torch.randn(N, Cin, H, W, device=cuda, generator=g).to(BF)
    w1 = (torch.randn(Cin, Cin, 1, 1, device=cuda, generator=g) / math.sqrt(Cin)).to(BF)
    b1 = torch.randn(Cin, device=cuda, generator=g)
    w3 = (torch.randn(Cout, Cin, 3, 3, device=cuda, generator=g) / math.sqrt(Cin * 9)).to(BF)
    b3 = torch.randn(Cout, device=cuda, generator=g)
    x_nhwc = x.permute(0, 2, 3, 1).contiguous()
    pad = torch.zeros(N, H + 2, W + 2, Cin, device=cuda, dtype=BF)
    _check(lib, lib.mrd_conv2d_nhwc_bf16(x_nhwc.data_ptr(), N, H, W, Cin,
                                         w1.permute(0, 2, 3, 1).contiguous().data_ptr(), Cin, 1, 1,
                                         b1.data_ptr(), pad.data_ptr(), None, 1, 1, _stream()))
    torch.cuda.synchronize()
    mid = F.relu(F.conv2d(x.float(), w1.float(), b1))
    _close(pad[:, 1:-1, 1:-1].permute(0, 3, 1, 2), mid, what="1x1 conv into padded buffer")
    assert (pad[:, 0] == 0).all() and (pad[:, -1] == 0).all() and (pad[:, :, 0] == 0).all() \
        and (pad[:, :, -1] == 0).all(), "borders of the padded buffer must stay zero"
    y = torch.full((N, H, W, Cout), float("nan"), device=cuda, dtype=BF)
    _check(lib, lib.mrd_conv3x3_flat_bf16(pad.data_ptr(), N, H, W, Cin,
                                          w3.permute(0, 2, 3, 1).contiguous().data_ptr(), Cout,
                                          b3.data_ptr(), y.data_ptr(), act, _stream()))
    torch.cuda.synchronize()
    ref = F.conv2d(pad[:, 1:-1, 1:-1].permute(0, 3, 1, 2).float(), w3.float(), b3, padding=1)
    if act == 1:
        ref = F.relu(ref)
    _close(y.permute(0, 3, 1, 2), ref, what=f"flat 3x3 conv {Cin}->{Cout} {H}x{W}")


@pytest.mark.parametrize("N,Ho,Wo,C0,C1,Cout,stride", [
    (3, 56, 56, 64, 64, 256, 1),      # layer1.0: flat tiles, equal K halves
    (2, 28, 28, 128, 256, 512, 2),    # layer2.0: block input read at stride 2, unequal K parts
    (5, 14, 14, 256, 512, 1024, 2),   # layer3.0: two ragged tiles per image
    (3, 7, 7, 512, 1024, 2048, 2),    # layer4.0: two images per tile, odd batch
    (1, 10, 6, 64, 128, 64, 2),       # narrow output (N = 64 tile), non-square
])
def test_conv1x1_dual(lib, cuda, N, Ho, Wo, C0, C1, Cout, stride):
    """conv3 + downsample + add + ReLU as one K-concatenated GEMM == the two convolutions summed."""
    g = torch.Generator(device="cuda").manual_seed(Ho * Wo + C1)
    x0 = torch.randn(N, C0, Ho, Wo, device=cuda, generator=g).to(BF)
    x1 = torch.randn(N, C1, Ho * stride, Wo * stride, device=cuda, generator=g).to(BF)
    w0 = (torch.randn(Cout, C0, 1, 1, device=cuda, generator=g) / math.sqrt(C0)).to(BF)
    w1 = (torch.randn(Cout, C1, 1, 1, device=cuda, generator=g) / math.sqrt(C1)).to(BF)
    bias = torch.randn(Cout, device=cuda, generator=g)
    wcat = torch.cat([w0.view(Cout, C0), w1.view(Cout, C1)], dim=1).contiguous()
    y = torch.full((N, Ho, Wo, Cout), float("nan"), device=cuda, dtype=BF)
    x0_nhwc = x0.permute(0, 2, 3, 1).contiguous()   # named: both operands must stay alive across the call
    x1_nhwc = x1.permute(0, 2, 3, 1).contiguous()
    _check(lib, lib.mrd_conv1x1_dual_bf16(x0_nhwc.data_ptr(), C0, x1_nhwc.data_ptr(), C1, stride, N, Ho, Wo,
                                          wcat.data_ptr(), Cout, bias.data_ptr(), y.data_ptr(), 1, _stream()))
    torch.cuda.synchronize()
    ref = F.relu(F.conv2d(x0.float(), w0.float()) + F.conv2d(x1.float(), w1.float(), stride=stride)
                 + bias.view(1, -1, 1, 1))
    _close(y.permute(0, 3, 1, 2), ref, what=f"dual 1x1 conv {C0}+{C1}->{Cout} stride {stride}")


@pytest.mark.parametrize("N,Ho,Wo,C0,C1,stride,Cout,C2,out_pad", [
    (3, 56, 56, 64, 0, 1, 256, 64, 1),       # layer1.1 -> layer1.2: identity, padded output, pixel-box tiles
    (2, 56, 56, 64, 64, 1, 256, 64, 1),      # layer1.0 (downsample fused) -> layer1.1
    (3, 56, 56, 64, 0, 1, 256, 128, 0),      # layer1.2 -> layer2.0: unpadded output, flat tiles
    (2, 28, 28, 64, 64, 2, 256, 64, 1),      # stride-2 downsample fused
    (130, 28, 28, 64, 0, 1, 256, 128, 1),    # many tiles per CTA: staging-ring and accumulator wrap-around
    (1, 6, 10, 64, 0, 1, 128, 64, 0),        # a single tile
    (2, 9, 7, 128, 0, 1, 128, 64, 1),        # two K chunks in the first product, two images per tile
])
def test_conv_chain(lib, cuda, N, Ho, Wo, C0, C1, stride, Cout, C2, out_pad):
    """conv3 (+downsample) + identity + ReLU of one bottleneck and conv1 + ReLU of the next in one launch."""
    g = torch.Generator(device="cuda").manual_seed(Ho * Wo + Cout + C1)
    x0 = torch.randn(N, Ho, Wo, C0, device=cuda, generator=g).to(BF)
    x1 = torch.randn(N, Ho * stride, Wo * stride, C1, device=cuda, generator=g).to(BF) if C1 else None
    ident = None if C1 else torch.randn(N, Ho, Wo, Cout, device=cuda, generator=g).to(BF)
    w1 = (torch.randn(Cout, C0 + C1, device=cuda, generator=g) / math.sqrt(C0 + C1)).to(BF)
    b1 = torch.randn(Cout, device=cuda, generator=g)
    w2 = (torch.randn(C2, Cout, device=cuda, generator=g) / math.sqrt(Cout)).to(BF)
    b2 = torch.randn(C2, device=cuda, generator=g)
    y = torch.full((N, Ho, Wo, Cout), float("nan"), device=cuda, dtype=BF)
    z = torch.zeros(N, Ho + 2 * out_pad, Wo + 2 * out_pad, C2, device=cuda, dtype=BF)
    _check(lib, lib.mrd_conv_chain_bf16(x0.data_ptr(), C0, x1.data_ptr() if C1 else None, C1, stride,
                                        ident.data_ptr() if ident is not None else None, N, Ho, Wo, w1.data_ptr(),
                                        Cout, b1.data_ptr(), y.data_ptr(), w2.data_ptr(), C2, b2.data_ptr(),
                                        z.data_ptr(), out_pad, _stream()))
    torch.cuda.synchronize()
    acc = x0.float().reshape(-1, C0) @ w1.float()[:, :C0].t()
    if C1:
        acc = acc + x1[:, ::stride, ::stride].float().reshape(-1, C1) @ w1.float()[:, C0:].t()
    acc = acc + b1
    if ident is not None:
        acc = acc + ident.float().reshape(-1, Cout)
    y_ref = F.relu(acc)
    _close(y.reshape(-1, Cout), y_ref, what="chain: block output y")
    z_ref = F.relu(y.float().reshape(-1, Cout) @ w2.float().t() + b2)   # from the bf16 y the kernel itself re-reads
    zi = z[:, out_pad:out_pad + Ho, out_pad:out_pad + Wo] if out_pad else z
    _close(zi.reshape(-1, C2), z_ref, what="chain: next conv1 output z")
    if out_pad:
        assert (z[:, 0] == 0).all() and (z[:, -1] == 0).all() and (z[:, :, 0] == 0).all() and (z[:, :, -1] == 0).all()


def test_conv_chain_rejects_what_does_not_fit(lib, cuda):
    """Both weight matrices stay resident in shared memory: layer2-sized pairs (2 x 128 KB) are refused and the
    engine keeps one launch per convolution there."""
    x = torch.zeros(1, 28, 28, 512, device=cuda, dtype=BF)
    rc = lib.mrd_conv_chain_bf16(x.data_ptr(), 128, None, 0, 1, x.data_ptr(), 1, 28, 28, x.data_ptr(), 512, None,
                                 x.data_ptr(), x.data_ptr(), 128, None, x.data_ptr(), 0, _stream())
    assert rc != 0 and b"shared memory" in lib.mrd_last_error()


def test_conv3x3_flat_rejects_unsupported(lib, cuda):
    # the resident 3x3 weight panel of Cin=128 does not fit next to two 56-wide halo spans
    x = torch.zeros(1, 58, 58, 128, device=cuda, dtype=BF)
    rc = lib.mrd_conv3x3_flat_bf16(x.data_ptr(), 1, 56, 56, 128, x.data_ptr(), 64, None, x.data_ptr(), 0,
                                   _stream())
    assert rc != 0 and b"shared memory" in lib.mrd_last_error()


@pytest.mark.parametrize("N,H,W", [(2, 224, 224), (1, 64, 96), (3, 32, 32)])
def test_stem(lib, cuda, N, H, W):
    g = torch.Generator(device="cuda").manual_seed(H)
    x = torch.randn(N, 3, H, W, device=cuda, generator=g)
    w = torch.randn(64, 3, 7, 7, device=cuda, generator=g) / math.sqrt(147)
    gamma = 0.5 + torch.rand(64, device=cuda, generator=g)
    beta = torch.randn(64, device=cuda, generator=g) * 0.1
    mean = torch.randn(64, device=cuda, generator=g) * 0.1
    var = 0.5 + torch.rand(64, device=cuda, generator=g)
    # host-side packing equivalent to pack_stem_bn (tested separately through the engine)
    scale = gamma / torch.sqrt(var + 1e-5)
    wf = (w * scale.view(-1, 1, 1, 1))
    wst = torch.zeros(64, 7, 8, 4, device=cuda)
    wst[:, :, :7, :3] = wf.permute(0, 2, 3, 1)  # [co][r][s][c]
    wst = wst.view(64, 7, 32).to(BF).contiguous()
    bias = (beta - mean * scale).contiguous()
    xpad = torch.full((N, H + 6, W + 8, 4), float("nan"), device=cuda, dtype=BF)
    _check(lib, lib.mrd_repack_images(x.data_ptr(), 2, N, H, W, xpad.data_ptr(), _stream()))
    torch.cuda.synchronize()
    assert torch.equal(xpad[:, 3:3 + H, 3:3 + W, :3], x.permute(0, 2, 3, 1).to(BF))
    assert (xpad[:, :3] == 0).all() and (xpad[:, :, :3] == 0).all() and (xpad[..., 3] == 0).all()
    assert (xpad[:, 3 + H:] == 0).all() and (xpad[:, :, 3 + W:] == 0).all()
    y = torch.full((N, H // 2, W // 2, 64), float("nan"), device=cuda, dtype=BF)
    _check(lib, lib.mrd_stem_conv_bf16(xpad.data_ptr(), N, H, W, wst.data_ptr(), bias.data_ptr(),
                                       y.data_ptr(), 1, _stream()))
    torch.cuda.synchronize()
    ref = F.relu(F.conv2d(x.to(BF).float(), wst.view(64, 7, 8, 4)[:, :, :7, :3].permute(0, 3, 1, 2).float(),
                          bias, stride=2, padding=3))
    _close(y.permute(0, 3, 1, 2), ref, what="stem")
    # the same launch with MaxPool2d(3, 2, 1) fused into the epilogue: bit-equal to pooling the stored stem output
    pooled = torch.zeros(N, H // 4, W // 4, 64, device=cuda, dtype=BF)
    _check(lib, lib.mrd_stem_pool_bf16(xpad.data_ptr(), N, H, W, wst.data_ptr(), bias.data_ptr(), pooled.data_ptr(),
                                       _stream()))
    torch.cuda.synchronize()
    want = F.max_pool2d(y.permute(0, 3, 1, 2).float(), 3, 2, 1)
    assert torch.equal(pooled.permute(0, 3, 1, 2).float(), want), "fused stem + maxpool differs from pooling the stem"


# ------------------------------------------------------------------ pooling
def test_maxpool(lib, cuda):
    x = torch.randn(3, 64, 112, 112, device=cuda).to(BF)
    xn = x.permute(0, 2, 3, 1).contiguous()
    y = torch.empty(3, 56, 56, 64, device=cuda, dtype=BF)
    _check(lib, lib.mrd_maxpool3x3s2(xn.data_ptr(), 3, 112, 112, 64, y.data_ptr(), _stream()))
    torch.cuda.synchronize()
    ref = F.max_pool2d(x.float(), 3, 2, 1)
    assert torch.equal(y.permute(0, 3, 1, 2).float(), ref)  # max of bf16 values is exact


def test_avgpool(lib, cuda):
    x = torch.randn(5, 49, 2048, device=cuda).to(BF)
    yb = torch.empty(5, 2048, device=cuda, dtype=BF)
    yf = torch.empty(5, 2048, device=cuda)
    _check(lib, lib.mrd_global_avgpool(x.data_ptr(), 5, 49, 2048, yb.data_ptr(), yf.data_ptr(), _stream()))
    torch.cuda.synchronize()
    ref = x.float().mean(1)
    _close(yf, ref, rel=1e-5, abs_=1e-5, what="avgpool f32")
    _close(yb, ref, what="avgpool bf16")


# ------------------------------------------------------------------ LayerNorm / embeddings
@pytest.mark.parametrize("rows,width,res,eps", [(1000, 768, True, 1e-12), (77, 512, False, 1e-5),
                                                (9, 256, True, 1e-5), (33, 1024, False, 1e-5)])
def test_layernorm(lib, cuda, rows, width, res, eps):
    x = (torch.randn(rows, width, device=cuda) * 3 + 1).to(BF)
    r = torch.randn(rows, width, device=cuda).to(BF) if res else None
    gamma = torch.rand(width, device=cuda) + 0.5
    beta = torch.randn(width, device=cuda)
    yb = torch.empty(rows, width, device=cuda, dtype=BF)
    yf = torch.empty(rows, width, device=cuda)
    _check(lib, lib.mrd_layernorm_residual(x.data_ptr(), width, r.data_ptr() if res else None, width,
                                           gamma.data_ptr(), beta.data_ptr(), eps, rows, width,
                                           yb.data_ptr(), width, yf.data_ptr(), width, _stream()))
    torch.cuda.synchronize()
    s = x.float() + (r.float() if res else 0)
    ref = F.layer_norm(s, (width,), gamma, beta, eps)
    _close(yf, ref, rel=1e-4, abs_=1e-4, what="ln f32")
    _close(yb, ref, what="ln bf16")


def test_bert_embed(lib, cuda):
    B, S, V = 4, 50, 1000
    ids = torch.randint(0, V, (B, S), device=cuda)
    word = torch.randn(V, 768, device=cuda).to(BF)
    pos_type = torch.randn(512, 768, device=cuda)
    gamma = torch.rand(768, device=cuda) + 0.5
    beta = torch.randn(768, device=cuda)
    y = torch.empty(B * S, 768, device=cuda, dtype=BF)
    _check(lib, lib.mrd_bert_embed_layernorm(ids.data_ptr(), B, S, word.data_ptr(), pos_type.data_ptr(),
                                             gamma.data_ptr(), beta.data_ptr(), 1e-12, V, y.data_ptr(),
                                             _stream()))
    torch.cuda.synchronize()
    e = word.float()[ids] + pos_type[:S].unsqueeze(0)
    ref = F.layer_norm(e, (768,), gamma, beta, 1e-12).view(B * S, 768)
    _close(y, ref, what="bert embed")


# ------------------------------------------------------------------ attention (K3)
@pytest.fixture(params=["tcgen05", "mma.sync"])
def attn_path(request, lib):
    """Two implementations: tcgen05 (one 128x128 tile for S <= 128, key-block loop with a running softmax up to
    S = 512) and the mma.sync flash kernel (kept as the cross-check): run the attention tests through both."""
    lib.mrd_attention_use_tcgen05(1 if request.param == "tcgen05" else 0)
    yield request.param
    lib.mrd_attention_use_tcgen05(1)


@pytest.mark.parametrize("B,S,heads,lengths", [
    (2, 128, 12, None),
    (3, 128, 12, [128, 70, 1]),
    (2, 512, 12, [512, 65]),       # whole key blocks skipped
    (3, 48, 4, [48, 33, 5]),       # S < 64: BLOCK_M = 64 path, ragged
    (2, 200, 12, [200, 129]),      # S not a multiple of 64
    (1, 256, 12, None),            # two full key blocks, no mask
    (3, 320, 4, [320, 128, 129]),  # lengths on and just past a key-block boundary
    (2, 384, 12, [384, 257]),      # three key blocks, last query block with one row
    (40, 512, 12, None),           # more work items than resident CTAs (persistence, barrier phases)
])
def test_attention(lib, cuda, attn_path, B, S, heads, lengths):
    g = torch.Generator(device="cuda").manual_seed(S + B)
    D = heads * 64
    qkv = torch.randn(B * S, 3 * D, device=cuda, generator=g).to(BF)
    qkv[:, :D] *= 0.125  # the engine folds 1/sqrt(64) into Wq
    mask = torch.ones(B, S, device=cuda, dtype=torch.long)
    if lengths:
        for b, L in enumerate(lengths):
            mask[b, L:] = 0
    bias = torch.empty(B, S, device=cuda)
    _check(lib, lib.mrd_mask_to_bias(mask.data_ptr(), 0, B, S, bias.data_ptr(), _stream()))
    out = torch.full((B * S, D), float("nan"), device=cuda, dtype=BF)
    _check(lib, lib.mrd_attention_bf16(qkv.data_ptr(), bias.data_ptr() if lengths else None, B, S, heads,
                                       out.data_ptr(), _stream()))
    torch.cuda.synchronize()
    assert torch.equal(bias == 0, mask != 0) and torch.isinf(bias[mask == 0]).all()
    q, k, v = [t.view(B, S, heads, 64).transpose(1, 2).float() for t in qkv.view(B, S, 3 * D).split(D, -1)]
    sc = q @ k.transpose(-1, -2) + bias.view(B, 1, 1, S)
    ref = (torch.softmax(sc, -1) @ v).transpose(1, 2).reshape(B * S, D)
    _close(out, ref, rel=2 ** -6, abs_=2e-2, what="attention")


@pytest.mark.parametrize("dtype,code", [(torch.int64, 0), (torch.int32, 1), (torch.float32, 2),
                                        (torch.bool, 3), (torch.bfloat16, 4)])
def test_mask_dtypes(lib, cuda, dtype, code):
    m = (torch.rand(3, 77, device=cuda) > 0.4)
    bias = torch.empty(3, 77, device=cuda)
    mm = m.to(dtype)
    _check(lib, lib.mrd_mask_to_bias(mm.data_ptr(), code, 3, 77, bias.data_ptr(), _stream()))
    torch.cuda.synchronize()
    assert torch.equal(bias == 0, m)


# ------------------------------------------------------------------ token packing + varlen attention
@pytest.mark.parametrize("B,S,keep_all", [(7, 128, 0), (3, 40, 0), (4, 33, 1), (1500, 16, 0)])
def test_compact_tokens(lib, cuda, B, S, keep_all):
    g = torch.Generator(device="cuda").manual_seed(B)
    mask = (torch.rand(B, S, device=cuda, generator=g) > 0.45).long()   # arbitrary holes, not only prefixes
    mask[0] = 1
    if B > 1:
        mask[1] = 0                                                       # fully masked row: CLS still kept
    seq_off = torch.full((B + 1,), -1, device=cuda, dtype=torch.int32)
    row_tok = torch.full((B * S,), -1, device=cuda, dtype=torch.int32)
    row_bias = torch.full((B * S,), 7.0, device=cuda)
    n_rows = torch.zeros(1, device=cuda, dtype=torch.int32)
    scratch = torch.zeros(B, device=cuda, dtype=torch.int32)
    _check(lib, lib.mrd_compact_tokens(mask.data_ptr(), 0, B, S, keep_all, seq_off.data_ptr(),
                                       row_tok.data_ptr(), row_bias.data_ptr(), n_rows.data_ptr(),
                                       scratch.data_ptr(), _stream()))
    torch.cuda.synchronize()
    keep = mask.bool().clone()
    keep[:, 0] = True
    if keep_all:
        keep[:] = True
    counts = keep.sum(1)
    want_off = torch.cat([torch.zeros(1, device=cuda, dtype=torch.long), counts.cumsum(0)])
    assert torch.equal(seq_off.long(), want_off)
    n = int(n_rows.item())
    assert n == int(counts.sum())
    want_tok = keep.flatten().nonzero().flatten()
    assert torch.equal(row_tok[:n].long(), want_tok)
    want_bias = torch.where(mask.flatten()[want_tok] != 0, 0.0, float("-inf"))
    assert torch.equal(row_bias[:n], want_bias.float())


@pytest.mark.parametrize("lens,heads", [([128, 70, 1, 64, 65], 12), ([512, 64, 300], 12), ([5, 48, 33], 4),
                                        ([17] * 700, 12)])
def test_attention_varlen(lib, cuda, attn_path, lens, heads):
    g = torch.Generator(device="cuda").manual_seed(sum(lens))
    B, D, T = len(lens), heads * 64, sum(lens)
    qkv = torch.randn(T, 3 * D, device=cuda, generator=g).to(BF)
    qkv[:, :D] *= 0.125
    seq_off = torch.tensor([0] + list(torch.tensor(lens).cumsum(0)), device=cuda, dtype=torch.int32)
    bias = torch.zeros(T, device=cuda)
    bias[seq_off[1].item()] = float("-inf")   # a kept-but-masked CLS row (sample 1)
    out = torch.full((T, D), float("nan"), device=cuda, dtype=BF)
    _check(lib, lib.mrd_attention_varlen_bf16(qkv.data_ptr(), bias.data_ptr(), seq_off.data_ptr(), B,
                                              max(lens), heads, T, out.data_ptr(), _stream()))
    torch.cuda.synchronize()
    for b, L in enumerate(lens):
        o = int(seq_off[b])
        x = qkv[o:o + L].float()
        q, k, v = [t.view(L, heads, 64).transpose(0, 1) for t in x.split(D, -1)]
        sc = q @ k.transpose(-1, -2) + bias[o:o + L].view(1, 1, L)
        if L == 1 and torch.isinf(bias[o]):
            continue  # every key masked: the reference yields NaN, this path yields zeros
        ref = (torch.softmax(sc, -1) @ v).transpose(0, 1).reshape(L, D)
        _close(out[o:o + L], ref, rel=2 ** -6, abs_=2e-2, what=f"varlen attention sample {b}")

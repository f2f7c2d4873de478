"""Per-kernel parity of the training step's non-GEMM kernels (csrc/train_kernels.cu) through their C-ABI entries,
at the sizes of the training benchmark: B = 64, S = 128 (T = 8192 allocated token rows, about half of them live),
BERT widths 768 / 2304 / 3072 and the B = 64, 224x224 ResNet50 BatchNorm shapes.

Every reference is float64 torch on the same bf16-rounded inputs, and dropout masks come from mrd_dropout_mask.
Where a kernel takes dyn_rows (the device-side live row count of the token-packed buffers), the count comes from
mrd_compact_tokens on a ragged mask, is not a multiple of 64, and the rows beyond it hold a sentinel that must
neither be read nor written.

Bars (each assert repeats its own):
  * bit-exact wherever a kernel only moves, masks or scales values;
  * bf16 outputs: |out - ref| <= 2^-7 |ref| (one bf16 ulp) + 1e-5 x the magnitude of the fp32 terms that cancel,
    and relative L2 <= 3e-3 (a 1 % systematic error fails it);
  * fp32 outputs: 1e-5 x the magnitude of their terms;
  * fp32 reductions (column sums, gamma / beta / table gradients): per column |err| <= 2e-5 x sum |terms|;
  * BatchNorm batch mean and variance: 1e-4 relative.
"""

import ctypes as C
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

BF = torch.bfloat16
ULP = 2.0 ** -7          # one bf16 ulp, relative
T_ROWS = 8192            # B * S of the training benchmark (B = 64, S = 128)
NAN16 = -1               # int16 view of the bf16 sentinel 0xffff (a NaN)


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _check(lib, rc):
    assert rc == 0, (rc, lib.mrd_last_error())


def _ptr(t):
    return None if t is None else t.data_ptr()


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def _bits(t):
    return t.view({torch.bfloat16: torch.int16, torch.float32: torch.int32}[t.dtype])


def _same_bits(a, b, what):
    assert torch.equal(_bits(a), _bits(b)), f"{what}: {int((_bits(a) != _bits(b)).sum())} elements differ"


def _sentinel(shape, dtype, cuda):
    t = torch.empty(shape, device=cuda, dtype=dtype)
    _bits(t).fill_(NAN16)
    return t


def _untouched(t, what):
    assert bool((_bits(t) == NAN16).all()), f"{what}: {int((_bits(t) != NAN16).sum())} sentinel elements written"


def _bf16_close(out, ref, mag, what, rel_l2=3e-3):
    """out (bf16) against the fp64 reference: one bf16 ulp + 1e-5 x mag (the magnitude of the terms that cancel in
    fp32) elementwise, and a relative L2 bar that a 1 % systematic error fails."""
    out, ref, mag = out.double(), ref.double(), mag.double()
    err = (out - ref).abs()
    bound = ULP * ref.abs() + 1e-5 * mag
    bad = ~(err <= bound)   # NaN counts as outside
    if bad.any():
        i = torch.where(bad, (err / bound).nan_to_num(float("inf")), 0).argmax()
        pytest.fail(f"{what}: {int(bad.sum())}/{bad.numel()} outside one bf16 ulp + 1e-5 mag; worst at flat index "
                    f"{int(i)}: out {out.flatten()[i].item():.6g}, ref {ref.flatten()[i].item():.6g}, "
                    f"mag {mag.flatten()[i].item():.4g}")
    l2 = ((out - ref).norm() / ref.norm()).item()
    assert l2 <= rel_l2, (what, l2)


def _f32_close(out, ref, mag, what, tol=1e-5):
    """fp32 output: |out - ref| <= tol x the magnitude of its terms."""
    err = (out.double() - ref).abs()
    bad = ~(err <= tol * mag)   # NaN counts as outside
    assert not bad.any(), (f"{what}: {int(bad.sum())}/{bad.numel()} outside {tol:g}; max err "
                           f"{err.max().item():.4g}, max ratio {(err / mag.clamp_min(1e-300)).max().item():.4g}")


def _mask(lib, seed, site, p, n):
    m = torch.empty(n, device="cuda")
    _check(lib, lib.mrd_dropout_mask(seed, site, p, n, m.data_ptr(), _stream()))
    return m


def _scale(p):
    return torch.tensor(1.0 / (1.0 - p), dtype=torch.float64).float().item() if p > 0 else 1.0


def _packed(lib, cuda, B, S, seed):
    """Token packing of a ragged right-padded batch by mrd_compact_tokens: (live row count n, its device copy,
    seq_off, row_tok, mask).  Lengths are uniform in [1, S] (about half the tokens live) and n % 64 != 0."""
    g = torch.Generator().manual_seed(seed)
    lens = torch.randint(1, S + 1, (B,), generator=g)
    if int(lens.sum()) % 64 == 0:
        lens[-1] = lens[-1] - 1 if lens[-1] > 1 else 2
    mask = (torch.arange(S)[None, :] < lens[:, None]).long().to(cuda)
    seq_off = torch.zeros(B + 1, device=cuda, dtype=torch.int32)
    # row_tok past the live count keeps valid but unrelated token indices: nothing may use them
    row_tok = torch.randint(0, B * S, (B * S,), device=cuda, dtype=torch.int32)
    row_bias = torch.zeros(B * S, device=cuda)
    n_rows = torch.zeros(1, device=cuda, dtype=torch.int32)
    scratch = torch.zeros(B, device=cuda, dtype=torch.int32)
    _check(lib, lib.mrd_compact_tokens(mask.data_ptr(), 0, B, S, 0, seq_off.data_ptr(), row_tok.data_ptr(),
                                       row_bias.data_ptr(), n_rows.data_ptr(), scratch.data_ptr(), _stream()))
    n = int(n_rows.item())
    assert n == int(lens.sum()) and n % 64 != 0
    return n, n_rows, seq_off, row_tok, mask


# ------------------------------------------------------------------ dropout
@pytest.mark.parametrize("p", [0.0, 0.1, 0.5])
@pytest.mark.parametrize("strided", [False, True])
def test_dropout_bf16(lib, cuda, p, strided):
    """In place (as on the embeddings' output), and from / into [T, 2*width] buffers: the mask index is r*width + c
    whatever the strides, and rows past dyn_rows are not touched."""
    width = 768
    n, n_rows, *_ = _packed(lib, cuda, 64, 128, 1)
    g = _gen(2)
    seed, site = 0x5eed, 11
    ld = 2 * width if strided else width
    x = torch.randn(T_ROWS, ld, device=cuda, generator=g).to(BF)
    x[n:] = float("nan")
    x0 = x.clone()
    if strided:
        y = _sentinel((T_ROWS, ld), BF, cuda)
        yp = y.data_ptr() + width * 2   # write into the second half of each row
    else:
        y, yp = x, x.data_ptr()
    _check(lib, lib.mrd_dropout_bf16(x.data_ptr(), ld, T_ROWS, width, n_rows.data_ptr(), seed, site, p, yp, ld,
                                     _stream()))
    m = _mask(lib, seed, site, p, T_ROWS * width).view(T_ROWS, width)[:n].bool()
    xs = x0[:n, :width].float()
    ref = torch.where(m, xs * _scale(p), torch.zeros_like(xs)).to(BF)
    out = y[:n, width:] if strided else y[:n, :width]
    _same_bits(out, ref, "live rows")                    # one fp32 product, rounded once: bit-exact
    if strided:
        _untouched(y[:, :width], "left half")
        _untouched(y[n:], "rows past dyn_rows")
        _same_bits(x, x0, "input")
    else:
        _same_bits(y[n:], x0[n:], "rows past dyn_rows")


@pytest.mark.parametrize("p", [0.0, 0.1, 0.5])
def test_dropout_f32_family(lib, cuda, p):
    """dropout_f32 (text output), relu_dropout_f32 (projection / fusion MLP / head) and head_dropout_f32 (the
    length-1 cross-attention weights): bit-exact against torch fp32 x * mask * float32(1/(1-p))."""
    g = _gen(3)
    seed, sc = 77, _scale(p)
    rows, width = 300, 1000
    x = torch.randn(rows, width, device=cuda, generator=g)
    m = _mask(lib, seed, 5, p, rows * width).view(rows, width).bool()
    zero = torch.zeros_like(x)

    y = torch.full_like(x, float("nan"))
    _check(lib, lib.mrd_dropout_f32(x.data_ptr(), rows, width, seed, 5, p, y.data_ptr(), _stream()))
    _same_bits(y, torch.where(m, x * sc, zero), "dropout_f32")

    y.fill_(float("nan"))
    _check(lib, lib.mrd_relu_dropout_f32(x.data_ptr(), rows, width, seed, 5, p, y.data_ptr(), _stream()))
    _same_bits(y, torch.where(m, x.clamp_min(0) * sc, zero), "relu_dropout_f32")

    heads, hd = 8, 64
    xh = torch.randn(rows, heads * hd, device=cuda, generator=g)
    yh = torch.full_like(xh, float("nan"))
    w = torch.full((rows, heads), float("nan"), device=cuda)
    _check(lib, lib.mrd_head_dropout_f32(xh.data_ptr(), rows, heads, hd, seed, 9, p, yh.data_ptr(), w.data_ptr(),
                                         _stream()))
    keep = _mask(lib, seed, 9, p, rows * heads).view(rows, heads)
    w_ref = keep * sc                                    # w_out[r, h] = keep(r*heads + h) * scale
    _same_bits(w, w_ref, "head weights")
    _same_bits(yh, (xh.view(rows, heads, hd) * w_ref[:, :, None]).view(rows, heads * hd), "head_dropout_f32")


# ------------------------------------------------------------------ residual + dropout + LayerNorm forward
@pytest.mark.parametrize("width", [256, 512, 768, 1024])
@pytest.mark.parametrize("p", [0.0, 0.1])
@pytest.mark.parametrize("ragged", [True, False])
def test_drop_add_layernorm(lib, cuda, width, p, ragged):
    """s = res + dropout(z) stored in bf16, y = LayerNorm(s): T = 8192 rows with a ragged dyn_rows, or 1003 rows
    (not a multiple of the 8 rows of a block) without it."""
    if ragged:
        rows, (n, n_rows, *_) = T_ROWS, _packed(lib, cuda, 64, 128, width)
    else:
        rows, n, n_rows = 1003, 1003, None
    g = _gen(width + 1)
    seed, site, eps = 99, 3, 1e-12
    z = torch.randn(rows, width, device=cuda, generator=g).to(BF)
    res = (torch.randn(rows, width, device=cuda, generator=g) * 2
           + torch.randn(rows, 1, device=cuda, generator=g) * 3).to(BF)   # per-row offsets
    gamma = torch.rand(width, device=cuda, generator=g) + 0.5
    beta = torch.randn(width, device=cuda, generator=g) * 0.3
    s_out = _sentinel((rows, width), BF, cuda)
    y = _sentinel((rows, width), BF, cuda)
    _check(lib, lib.mrd_drop_add_layernorm_bf16(z.data_ptr(), res.data_ptr(), rows, width, _ptr(n_rows), seed, site,
                                                p, gamma.data_ptr(), beta.data_ptr(), eps, s_out.data_ptr(),
                                                y.data_ptr(), _stream()))
    m = _mask(lib, seed, site, p, rows * width).view(rows, width)[:n].bool()
    zz = z[:n].float()
    s_ref = (res[:n].float() + torch.where(m, zz * _scale(p), torch.zeros_like(zz))).to(BF)
    s = s_out[:n]
    if p == 0:
        _same_bits(s, s_ref, "s_out")                    # res + z in fp32, rounded once
    else:
        # res + z*scale may contract into one fma: rounded once instead of twice, within one bf16 ulp
        d = (s.double() - s_ref.double()).abs()
        assert bool((d <= ULP * torch.maximum(s.double().abs(), s_ref.double().abs())).all()), "s_out beyond 1 ulp"
    # y against the fp64 LayerNorm of the STORED s (the statistics are taken from the rounded values)
    sd = s.double()
    xhat = (sd - sd.mean(1, keepdim=True)) / torch.sqrt(sd.var(1, unbiased=False, keepdim=True) + eps)
    ref = xhat * gamma.double() + beta.double()
    _bf16_close(y[:n], ref, (xhat * gamma.double()).abs() + beta.double().abs(), "y")
    if n < rows:
        _untouched(s_out[n:], "s_out past dyn_rows")
        _untouched(y[n:], "y past dyn_rows")


# ------------------------------------------------------------------ fp32 LayerNorm (fusion / head)
def _ln_ref64(x, gamma, beta, dy, eps):
    xd = x.double().requires_grad_(True)
    gd = gamma.double().requires_grad_(True)
    bd = beta.double().requires_grad_(True)
    y = F.layer_norm(xd, (x.shape[1],), gd, bd, eps)
    y.backward(dy.double())
    mu = xd.detach().mean(1, keepdim=True)
    rstd = 1.0 / torch.sqrt(xd.detach().var(1, unbiased=False, keepdim=True) + eps)
    # xmag: |x| + |mean| in units of the spread, the magnitude of the terms of x - mean (they cancel in fp32)
    return y.detach(), xd.grad, gd.grad, bd.grad, (xd.detach() - mu) * rstd, rstd, (xd.detach().abs() + mu.abs()) * rstd


@pytest.mark.parametrize("width", [512, 300, 1000])
@pytest.mark.parametrize("rows", [64, 257])
@pytest.mark.parametrize("offset", [0, 1])
def test_layernorm_f32_forward_backward(lib, cuda, width, rows, offset):
    """ln_fwd_f32 / ln_bwd_f32 writing one half of a [rows, 2*width] buffer (as torch.cat of the fusion's two
    branches lays it out); dgamma / dbeta accumulate into buffers that already hold values."""
    g = _gen(rows * width + offset)
    eps = 1e-5
    x = torch.randn(rows, width, device=cuda, generator=g) * 3 + torch.randn(rows, 1, device=cuda, generator=g) * 5
    gamma = torch.rand(width, device=cuda, generator=g) + 0.5
    beta = torch.randn(width, device=cuda, generator=g) * 0.3
    dy = torch.randn(rows, width, device=cuda, generator=g)
    off = offset * width
    y = torch.full((rows, 2 * width), float("nan"), device=cuda)
    _check(lib, lib.mrd_layernorm_f32(x.data_ptr(), width, gamma.data_ptr(), beta.data_ptr(), eps, rows, width,
                                      y.data_ptr() + off * 4, 2 * width, _stream()))
    y_ref, dx_ref, dg_ref, db_ref, xhat, rstd, xmag = _ln_ref64(x, gamma, beta, dy, eps)
    gd = gamma.double()
    _f32_close(y[:, off:off + width], y_ref, xmag * gd.abs() + beta.double().abs(), "y")
    assert bool(y[:, width - off:2 * width - off].isnan().all()), "other half written"

    dx = torch.full((rows, 2 * width), float("nan"), device=cuda)
    dg0 = torch.randn(width, device=cuda, generator=g)
    db0 = torch.randn(width, device=cuda, generator=g)
    dg, db = dg0.clone(), db0.clone()
    _check(lib, lib.mrd_layernorm_bwd_f32(x.data_ptr(), width, dy.data_ptr(), width, gamma.data_ptr(), eps, rows,
                                          width, dx.data_ptr() + off * 4, 2 * width, dg.data_ptr(), db.data_ptr(),
                                          _stream()))
    gg = dy.double() * gd
    m1, m2 = gg.mean(1, keepdim=True), (gg * xhat).mean(1, keepdim=True)
    _f32_close(dx[:, off:off + width], dx_ref, rstd * (gg.abs() + m1.abs() + xmag * m2.abs()), "dx")
    assert bool(dx[:, width - off:2 * width - off].isnan().all()), "other half of dx written"
    # fp32 column sums over the rows: 2e-5 x sum |terms| (the initial value included)
    _f32_close(dg, dg0.double() + dg_ref, dg0.double().abs() + (dy.double().abs() * xmag).sum(0), "dgamma", 2e-5)
    _f32_close(db, db0.double() + db_ref, db0.double().abs() + dy.double().abs().sum(0), "dbeta", 2e-5)


# ------------------------------------------------------------------ GELU
def _gelu_sweep(n, cuda):
    """Every bf16 value in [-12, 12] with |v| >= 2^-120 (normal results), and 0, tiled over n elements."""
    bits = torch.arange(-32768, 32768, device=cuda, dtype=torch.int32).to(torch.int16)
    v = bits.view(BF).float()
    keep = torch.isfinite(v) & (v.abs() <= 12) & ((v.abs() >= 2.0 ** -120) | (v == 0))
    v = v[keep]
    v = v[torch.randperm(v.numel(), device=cuda, generator=_gen(4))]
    return v.repeat(n // v.numel() + 1)[:n].to(BF)


@pytest.mark.parametrize("ragged", [True, False])
def test_gelu_forward_backward(lib, cuda, ragged):
    """Exact-erf GELU and its derivative Phi(u) + u phi(u) over T x 3072 (several grid-stride passes)."""
    width = 3072
    n, n_rows, *_ = _packed(lib, cuda, 64, 128, 5) if ragged else (T_ROWS, None)
    u = _gelu_sweep(T_ROWS * width, cuda).view(T_ROWS, width)
    u[n:] = float("nan")
    dg = torch.randn(T_ROWS, width, device=cuda, generator=_gen(6)).to(BF)
    out = _sentinel((T_ROWS, width), BF, cuda)
    _check(lib, lib.mrd_gelu_fwd_bf16(u.data_ptr(), T_ROWS, width, _ptr(n_rows), out.data_ptr(), _stream()))
    ud = u[:n].double()
    erf = torch.special.erf(ud / math.sqrt(2.0))
    phi = torch.exp(-0.5 * ud * ud) / math.sqrt(2.0 * math.pi)
    cdf = 0.5 * (1.0 + erf)
    # the terms that cancel in fp32: 0.5 u and 0.5 u erf (u << 0)
    _bf16_close(out[:n], ud * cdf, 0.5 * ud.abs() * (1.0 + erf.abs()), "gelu")
    if n < T_ROWS:
        _untouched(out[n:], "gelu past dyn_rows")
    out = _sentinel((T_ROWS, width), BF, cuda)
    _check(lib, lib.mrd_gelu_bwd_bf16(u.data_ptr(), dg.data_ptr(), T_ROWS, width, _ptr(n_rows), out.data_ptr(),
                                      _stream()))
    gd = dg[:n].double()
    _bf16_close(out[:n], gd * (cdf + ud * phi), gd.abs() * (0.5 * (1.0 + erf.abs()) + ud.abs() * phi), "gelu'")
    if n < T_ROWS:
        _untouched(out[n:], "gelu' past dyn_rows")


# ------------------------------------------------------------------ weight-gradient staging
WGRAD_PAIRS = [(3072, 768), (768, 3072), (2304, 768), (768, 768)]   # (dY, X) widths: FFN2, FFN1, QKV, out-proj


def _stage(lib, cuda, w0, w1, live, dyn, seed):
    """Run transpose_pad2_bf16 on [T, w0] / [T, w1] operands whose rows past `live` hold other valid data."""
    g = _gen(seed)
    x0 = torch.randn(T_ROWS, w0, device=cuda, generator=g).to(BF)
    x1 = torch.randn(T_ROWS, w1, device=cuda, generator=g).to(BF)
    x0[live:] += 100
    x1[live:] += 100
    y0 = _sentinel((w0, T_ROWS), BF, cuda)
    y1 = _sentinel((w1, T_ROWS), BF, cuda)
    cs0 = torch.randn(w0, device=cuda, generator=g)
    cs = cs0.clone()
    n_rows = torch.tensor([live], device=cuda, dtype=torch.int32) if dyn else None
    _check(lib, lib.mrd_transpose_pad2_bf16(x0.data_ptr(), w0, w0, y0.data_ptr(), x1.data_ptr(), w1, w1,
                                            y1.data_ptr(), T_ROWS if dyn else live, _ptr(n_rows), T_ROWS, _stream(),
                                            cs.data_ptr()))
    return x0, x1, y0, y1, cs0, cs, n_rows


@pytest.mark.parametrize("w0,w1", WGRAD_PAIRS)
@pytest.mark.parametrize("live", [1, 63, 64, 65, None, T_ROWS])
@pytest.mark.parametrize("dyn", [True, False])
def test_transpose_pad2(lib, cuda, w0, w1, live, dyn):
    """y[c][r] = x[r][c] below the live count, zeros up to the next multiple of 64, then (dyn_rows) nothing written
    or (static count) zeros up to Kp; colsum0 += the column sums of x0 over the live rows."""
    if live is None:
        live = _packed(lib, cuda, 64, 128, 7)[0]
    x0, x1, y0, y1, cs0, cs, _ = _stage(lib, cuda, w0, w1, live, dyn, w0 + live)
    up = min((live + 63) // 64 * 64, T_ROWS)
    zero = torch.zeros((), device=cuda, dtype=BF)
    for x, y, name in ((x0, y0, "dY"), (x1, y1, "X")):
        _same_bits(y[:, :live], x[:live].t(), f"{name} transpose")
        _same_bits(y[:, live:up], zero.expand(y.shape[0], up - live), f"{name} zero fill to the 64-row block")
        if dyn:
            _untouched(y[:, up:], f"{name} past the live 64-row blocks")
        else:
            _same_bits(y[:, up:], zero.expand(y.shape[0], T_ROWS - up), f"{name} zero fill to Kp")
    xd = x0[:live].double()
    _f32_close(cs, cs0.double() + xd.sum(0), cs0.double().abs() + xd.abs().sum(0), "colsum0", 2e-5)


@pytest.mark.parametrize("w0,w1", WGRAD_PAIRS)
@pytest.mark.parametrize("live", [65, None])
def test_wgrad_staging_and_splitk(lib, cuda, w0, w1, live):
    """The weight gradient as the training step computes it: stage dY and X with transpose_pad2_bf16 (sentinel NaN
    left beyond the live 64-row blocks), then dW = dY^T X with the split-K GEMM bounded by dyn_k = live."""
    if live is None:
        live = _packed(lib, cuda, 64, 128, 8)[0]
    x0, x1, y0, y1, _, _, n_rows = _stage(lib, cuda, w0, w1, live, True, w1 + live)
    out = torch.zeros(w0, w1, device=cuda)
    _check(lib, lib.mrd_gemm_splitk_f32(y0.data_ptr(), T_ROWS, w0, T_ROWS, y1.data_ptr(), w1, out.data_ptr(), w1,
                                        n_rows.data_ptr(), _stream()))
    ref = x0[:live].double().t() @ x1[:live].double()
    assert bool(torch.isfinite(out).all())
    err = ((out.double() - ref).norm() / ref.norm()).item()
    assert err <= 3e-5, err   # bf16 products are exact in fp32; only the summation order differs


# ------------------------------------------------------------------ bias gradients, ReLU backward, CLS rows
@pytest.mark.parametrize("width", [768, 2304, 3072])
@pytest.mark.parametrize("rows", [T_ROWS, 20000])
def test_colsum_bf16(lib, cuda, width, rows):
    """out[c] += scale * sum over the live rows; the rows past dyn_rows are NaN.  20,000 rows: the row split is
    capped at 64 blocks, so every warp loops."""
    live = _packed(lib, cuda, 64, 128, 9)[0] if rows == T_ROWS else rows - 37
    n_rows = torch.tensor([live], device=cuda, dtype=torch.int32)
    g = _gen(width + rows)
    x = torch.randn(rows, width, device=cuda, generator=g).to(BF)
    x[live:] = float("nan")
    out0 = torch.randn(width, device=cuda, generator=g)
    out = out0.clone()
    sc = 0.37
    _check(lib, lib.mrd_colsum_bf16(x.data_ptr(), width, rows, width, n_rows.data_ptr(), sc, out.data_ptr(),
                                    _stream()))
    xd = x[:live].double()
    _f32_close(out, out0.double() + sc * xd.sum(0), out0.double().abs() + sc * xd.abs().sum(0), "colsum_bf16", 2e-5)


def test_colsum_f32_and_relu_bwd(lib, cuda):
    g = _gen(10)
    rows, width, ld = 300, 1000, 1016
    x = torch.randn(rows, ld, device=cuda, generator=g)
    x[:, width:] = float("nan")                          # the columns between width and the row stride
    out0 = torch.randn(width, device=cuda, generator=g)
    out = out0.clone()
    _check(lib, lib.mrd_colsum_f32(x.data_ptr(), ld, rows, width, out.data_ptr(), _stream()))
    xd = x[:, :width].double()
    _f32_close(out, out0.double() + xd.sum(0), out0.double().abs() + xd.abs().sum(0), "colsum_f32", 2e-5)

    n = 1_000_003
    y = torch.randn(n, device=cuda, generator=g)
    y[::7] = 0.0
    y[3::11] = -0.0
    dy = torch.randn(n, device=cuda, generator=g)
    dx = torch.full_like(y, float("nan"))
    _check(lib, lib.mrd_relu_bwd_f32(y.data_ptr(), dy.data_ptr(), n, dx.data_ptr(), _stream()))
    _same_bits(dx, torch.where(y > 0, dy, torch.zeros_like(dy)), "relu_bwd")   # y == 0 gives +0


def test_cls_gather_scatter(lib, cuda):
    B, S, Hd = 64, 128, 768
    n, _, seq_off, *_ = _packed(lib, cuda, B, S, 12)
    g = _gen(12)
    cls = seq_off[:B].long()
    x = torch.randn(T_ROWS, Hd, device=cuda, generator=g).to(BF)
    y = torch.full((B, Hd), float("nan"), device=cuda)
    _check(lib, lib.mrd_gather_cls_rows_f32(x.data_ptr(), seq_off.data_ptr(), B, Hd, y.data_ptr(), _stream()))
    _same_bits(y, x[cls].float(), "gather")
    src = torch.randn(B, Hd, device=cuda, generator=g)
    dst = torch.zeros(T_ROWS, Hd, device=cuda, dtype=BF)
    _check(lib, lib.mrd_scatter_cls_rows_bf16(src.data_ptr(), seq_off.data_ptr(), B, Hd, dst.data_ptr(), _stream()))
    _same_bits(dst[cls], src.to(BF), "scatter")
    other = torch.ones(T_ROWS, dtype=torch.bool, device=cuda)
    other[cls] = False
    assert int((_bits(dst[other]) != 0).sum()) == 0, "scatter wrote a non-CLS row"


# ------------------------------------------------------------------ embeddings backward
@pytest.mark.parametrize("B,S", [(64, 128), (8, 512)])
def test_embed_layernorm_backward(lib, cuda, B, S):
    """LayerNorm backward of word[id] + pos_type[pos] on the packed rows, scattered into the word / position tables
    (a few hot ids: many adds per row), token_type row 0 and gamma / beta; pad_idx receives nothing."""
    Hd, vocab, pad, eps = 768, 30522, 0, 1e-12
    n, n_rows, _, row_tok, mask = _packed(lib, cuda, B, S, 13 + S)
    g = _gen(S)
    ids = torch.randint(0, vocab, (B, S), device=cuda, generator=g)
    hot = torch.tensor([101, 1996, 2000, 7592], device=cuda)
    pick = torch.rand(B, S, device=cuda, generator=g)
    ids = torch.where(pick < 0.5, hot[torch.randint(0, 4, (B, S), device=cuda, generator=g)], ids)
    ids = torch.where(pick > 0.95, torch.full_like(ids, pad), ids)        # pad_idx at kept positions
    word = (torch.randn(vocab, Hd, device=cuda, generator=g) * 0.05).to(BF)
    pos_type = torch.randn(512, Hd, device=cuda, generator=g) * 0.05
    gamma = torch.rand(Hd, device=cuda, generator=g) + 0.5
    dy = torch.randn(B * S, Hd, device=cuda, generator=g).to(BF)          # rows past n: valid, unused data
    dword = torch.zeros(vocab, Hd, device=cuda)
    dpos = torch.zeros(512, Hd, device=cuda)
    dt0, dgm, dbt = (torch.zeros(Hd, device=cuda) for _ in range(3))
    _check(lib, lib.mrd_embed_layernorm_bwd(ids.data_ptr(), row_tok.data_ptr(), B * S, n_rows.data_ptr(), S,
                                            word.data_ptr(), pos_type.data_ptr(), gamma.data_ptr(), eps, vocab, pad,
                                            dy.data_ptr(), dword.data_ptr(), dpos.data_ptr(), dt0.data_ptr(),
                                            dgm.data_ptr(), dbt.data_ptr(), _stream()))
    tok = row_tok[:n].long()
    assert bool(mask.flatten()[tok].all())
    rid, pos = ids.flatten()[tok], tok % S
    x = word[rid].double() + pos_type[pos].double()
    xhat = (x - x.mean(1, keepdim=True)) / torch.sqrt(x.var(1, unbiased=False, keepdim=True) + eps)
    rstd = 1.0 / torch.sqrt(x.var(1, unbiased=False, keepdim=True) + eps)
    gy = dy[:n].double()
    gg = gy * gamma.double()
    m1, m2 = gg.mean(1, keepdim=True), (gg * xhat).mean(1, keepdim=True)
    dx = rstd * (gg - m1 - xhat * m2)
    mag = rstd * (gg.abs() + m1.abs() + (xhat * m2).abs())              # |terms| of each dx element
    # scatter-adds and column sums in fp32: per element 2e-5 x sum |terms|
    zp = torch.zeros(512, Hd, device=cuda, dtype=torch.float64)
    _f32_close(dpos, zp.index_add(0, pos, dx), zp.index_add(0, pos, mag), "dpos", 2e-5)
    _f32_close(dgm, (gy * xhat).sum(0), (gy * xhat).abs().sum(0), "dgamma", 2e-5)
    _f32_close(dbt, gy.sum(0), gy.abs().sum(0), "dbeta", 2e-5)
    _f32_close(dt0, dx.sum(0), mag.sum(0), "dtype0", 2e-5)
    live = rid != pad
    zw = torch.zeros(vocab, Hd, device=cuda, dtype=torch.float64)
    used = torch.zeros(vocab, dtype=torch.bool, device=cuda)
    used[rid[live]] = True
    ref = zw.index_add(0, rid[live], dx[live])
    _f32_close(dword[used], ref[used], zw.index_add(0, rid[live], mag[live])[used], "dword", 2e-5)
    assert int((_bits(dword[pad]) != 0).sum()) == 0, "pad_idx row received a gradient"
    assert int((_bits(dword[~used]) != 0).sum()) == 0, "a word row no kept token uses received a gradient"


# ------------------------------------------------------------------ BatchNorm with batch statistics
BN_SHAPES = [(802816, 64), (200704, 256), (50176, 512), (3136, 2048)]   # B = 64, 224x224: stem, layer1-4


def _bn_input(rows, C, seed, cuda):
    """bf16 [rows, C] whose channels have |mean| / std cycling through 0, 1, 10 and 100."""
    g = _gen(seed)
    std = torch.rand(C, device=cuda, generator=g) * 1.5 + 0.5
    ratio = torch.tensor([0.0, 1.0, 10.0, 100.0], device=cuda)[torch.arange(C, device=cuda) % 4]
    sign = torch.where(torch.rand(C, device=cuda, generator=g) < 0.5, -1.0, 1.0)
    return (torch.randn(rows, C, device=cuda, generator=g) * std + sign * ratio * std).to(BF)


def _bn_stats(lib, y):
    rows, C = y.shape
    st = torch.zeros(3, C, device=y.device)
    _check(lib, lib.mrd_bn_stats_bf16(y.data_ptr(), rows, C, st[0].data_ptr(), st[1].data_ptr(), st[2].data_ptr(),
                                      _stream()))
    return st


def _bn_moments(st, n):
    d = st[0].double() / n
    return st[2].double() + d, st[1].double() / n - d * d


@pytest.mark.parametrize("rows,C", BN_SHAPES)
@pytest.mark.parametrize("variant", ["identity_relu", "relu", "plain"])
def test_batchnorm_batch_statistics(lib, cuda, rows, C, variant):
    """bn_stats + bn_apply_stats against F.batch_norm(training=True) in fp64 on the same bf16 y, then + identity
    and ReLU: bn3 of a bottleneck, bn1 / bn2 / the stem, and the downsample branch."""
    y = _bn_input(rows, C, rows + C, cuda)
    g = _gen(C)
    gamma = torch.rand(C, device=cuda, generator=g) + 0.5
    beta = torch.randn(C, device=cuda, generator=g) * 0.5
    identity = torch.randn(rows, C, device=cuda, generator=g).to(BF) if variant == "identity_relu" else None
    relu = variant != "plain"
    yd = y.double()
    st = _bn_stats(lib, y)
    mean_ref, var_ref = yd.mean(0), yd.var(0, unbiased=False)
    mean, var = _bn_moments(st, rows)
    # batch moments: 1e-4 relative (the mean against |mean| + std: channels with mean 0 exist)
    assert bool(((mean - mean_ref).abs() <= 1e-4 * (mean_ref.abs() + var_ref.sqrt())).all()), \
        ("mean", ((mean - mean_ref).abs() / (mean_ref.abs() + var_ref.sqrt())).max().item())
    rel_var = ((var - var_ref).abs() / var_ref).max().item()
    assert rel_var <= 1e-4, ("var", rel_var)

    eps = 1e-5
    _check(lib, lib.mrd_bn_apply_stats_bf16(y.data_ptr(), rows, C, st[0].data_ptr(), st[1].data_ptr(),
                                            st[2].data_ptr(), gamma.data_ptr(), beta.data_ptr(), eps,
                                            _ptr(identity), int(relu), _stream()))
    ref = F.batch_norm(yd, None, None, gamma.double(), beta.double(), training=True, eps=eps)
    sc = gamma.double() / torch.sqrt(var_ref + eps)
    # the terms the fp32 arithmetic cancels: y*scale against beta - (shift + sum/n)*scale, where the sum's own error
    # scales with its terms, E|y - shift| (a channel with mean 0 and beta ~ 0 has no other magnitude)
    k = st[2].double()
    mag = ((yd * sc).abs() + beta.double().abs() + (k.abs() + (mean_ref - k).abs()) * sc
           + (yd - k).abs().mean(0) * sc)
    if identity is not None:
        ref = ref + identity.double()
        mag = mag + identity.double().abs()
    if relu:
        ref = ref.clamp_min(0)
    _bf16_close(y, ref, mag, f"bn {variant}")


def test_batchnorm_running_update(lib, cuda):
    """One bn_update_running launch over a table of sites (C = 64, 256, 2048; n = 98 makes the unbiased
    n / (n - 1) factor 1 %) against torch's momentum update with the unbiased batch variance."""
    class Site(C.Structure):
        _fields_ = [("sum", C.c_void_p), ("sumsq", C.c_void_p), ("shift", C.c_void_p), ("running_mean", C.c_void_p),
                    ("running_var", C.c_void_p), ("n", C.c_float), ("C", C.c_int)]

    momentum = 0.1
    shapes = [(50176, 64), (3136, 256), (98, 2048), (802816, 64)]
    g = _gen(14)
    keep, sites = [], []
    for i, (rows, ch) in enumerate(shapes):
        y = _bn_input(rows, ch, 100 + i, cuda)
        st = _bn_stats(lib, y)
        rm0 = torch.randn(ch, device=cuda, generator=g)
        rv0 = torch.rand(ch, device=cuda, generator=g) + 0.5
        rm, rv = rm0.clone(), rv0.clone()
        keep.append((y, st, rm0, rv0, rm, rv))
        sites.append(Site(st[0].data_ptr(), st[1].data_ptr(), st[2].data_ptr(), rm.data_ptr(), rv.data_ptr(),
                          float(rows), ch))
    table_host = (Site * len(sites))(*sites)
    table = torch.frombuffer(bytearray(table_host), dtype=torch.uint8).to(cuda)
    _check(lib, lib.mrd_bn_update_running(table.data_ptr(), len(sites), 2048, momentum, _stream()))
    torch.cuda.synchronize()
    for (rows, ch), (y, st, rm0, rv0, rm, rv) in zip(shapes, keep):
        yd = y.double()
        mean, var_u = yd.mean(0), yd.var(0, unbiased=True)
        rm_ref = (1 - momentum) * rm0.double() + momentum * mean
        rv_ref = (1 - momentum) * rv0.double() + momentum * var_u
        # 1e-4 relative on the new statistic's share, plus fp32 rounding of the blend
        bound_m = 1e-4 * momentum * (mean.abs() + var_u.sqrt()) + 1e-6 * rm_ref.abs()
        assert bool(((rm.double() - rm_ref).abs() <= bound_m).all()), ("running_mean", rows, ch)
        bound_v = 1e-4 * momentum * var_u + 1e-6 * rv_ref
        assert bool(((rv.double() - rv_ref).abs() <= bound_v).all()), \
            ("running_var", rows, ch, ((rv.double() - rv_ref).abs() / (momentum * var_u)).max().item())

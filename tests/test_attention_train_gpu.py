"""The training step's attention kernels against a float64 reference: the forward with dropout on the probabilities
(csrc/attention.cu: tcgen05 for S <= 128 and for 128 < S <= 512, mma.sync when tcgen05 is switched off) and the
backward (csrc/attention_bwd.cu: one tile for S <= 128, tiled with an fp32 dK | dV accumulator above).  The packed
cases run them as the training step does: rows from mrd_compact_tokens, bounded by seq_off, the forward through
mrd_attention_train_varlen_bf16 with the allocation's row count.

Reference: fp64 torch on the GPU from the same bf16 qkv / dctx.  The keep-mask M is mrd_dropout_mask(seed, site, p,
B*heads*S_max*S_max) read at ((b*heads + h)*S_max + q)*S_max + k, q and k counted inside sample b and S_max the padded
width; kept probabilities are scaled by float32(1/(1-p)).
  forward    O = (softmax(Q K^T + bias) * M * scale) V      (a sample without an attended key: O = 0)
  gradients  fp64 autograd of that expression with respect to qkv, with dctx as the incoming gradient.
The backward reads ctx (the forward output).  Its cases give it bf16(O_ref), so a forward error cannot reach a backward
verdict; a chained run per case then gives it the kernel's own forward output, as the training step does.

Bars, per element and per (sample, head, tensor), never over a whole tensor (u = 2^-8, the bf16 unit roundoff):
  * |out - ref| <= 2^-7 |ref| + c 2^-8 mag, c = 2.  2^-7 |ref| is twice the rounding of the stored bf16 result.  mag
    is the fp64 magnitude of the terms the kernels round to bf16 before an MMA; each such rounding moves a result by
    at most u mag, and c = 2 leaves the same factor 2 for the fp32 work around it (accumulation over <= 512 terms,
    ex2.approx, the softmax sum taken before rounding: each below 2^-14 of mag):
      O   |P~| |V|                       P~ = M scale P, the bf16 A operand of P V (attention.cu:522-559)
      dV  |P~|^T |dO|                    P~ again (attention_bwd.cu:8-11, phase C)
      dQ  (|dS| + P sum_d |dO||O|) |K|   dS is rounded to bf16 for dS K, and delta = rowsum(dO ctx) reads bf16 ctx
      dK  (|dS| + P sum_d |dO||O|)^T |Q|
    In the chained run ctx carries the forward's bar instead of one rounding: |O| in the delta term becomes
    |O| + |P~||V|, which with c = 2 is that bar.
  * per (sample, head, tensor): relative L2 ||out - ref|| / ||ref|| <= 1e-2.  The roundings above are independent,
    each at most u and u/sqrt(3) in RMS, so an item's error norm is about (u/sqrt(3)) sqrt(||q||^2 + ||ref||^2),
    q being the quadrature magnitude of the rounded terms:
      O   sqrt(P~^2 V^2)    dV  sqrt(P~^2^T dO^2)
      dQ  sqrt(dS^2 K^2 + (sum_d dO^2 O^2) (P K)^2)      dK  sqrt(dS^2^T Q^2 + (P^2 sum_d dO^2 O^2)^T Q^2)
    (chained: O^2 in the delta term becomes O^2 + q_O^2).  Without cancellation ||q|| ~ ||ref|| and that noise is
    ~3e-3 of ||ref||, so the 1e-2 bar holds with margin and an item 1 % off fails (asserted below, both signs).
    The exception is an item that cancels, ||q|| >= 2 ||ref||: dQ and dK sum dS, whose sum over the keys is 0, and
    for a sample of a few tokens they cancel below the rounding noise of their terms (one token: exactly 0).  Only
    there the bar is ||out - ref|| <= 2u ||q||, 3.5 standard deviations of that noise (at the threshold, 1.56e-2 of
    ||ref||; an item with less cancellation keeps the 1e-2 bar).
Each case prints, per tensor, its worst err/bound ratio, the worst relative L2 of the items that do not cancel, and
how many items cancel with their worst ||err|| / (2u ||q||).  Negative controls assert that these bars reject a
(sample, head) of O or dQ 1 % off in either direction, a wrong dropout site, a mask indexed with the longest live
length instead of S_max, a reference missing one sample's last key, and a tiled backward missing one query block's
contribution to one key block.
"""

import types

import pytest
import torch

import synth

pytestmark = pytest.mark.gpu

BF = torch.bfloat16
F64 = torch.float64
H, D = 12, 64
HD, W = H * D, 3 * H * D        # ctx / qkv widths
U = 2.0 ** -8                   # bf16 unit roundoff
C_MAG = 2.0
L2_BAR = 1e-2
SEED, SITE = 0x5EED, 7
NAN16 = -1                      # int16 view of the bf16 sentinel 0xffff (a NaN)
INF = float("inf")
BOUNDARY = [1, 15, 16, 17, 31, 32, 33, 63, 64, 65, 127, 128]   # 16-key MMA granule, 32-row TMA boxes
LONG_EDGES = [127, 128, 129, 255, 256, 257, 385, 512]          # 128-key block edges


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _check(lib, rc):
    assert rc == 0, (rc, lib.mrd_last_error())


def _bits(t):
    return t.view(torch.int16)


def _sentinel(rows, cols, cuda):
    t = torch.empty(rows, cols, device=cuda, dtype=BF)
    _bits(t).fill_(NAN16)
    return t


def _same_bits(a, b, what):
    assert torch.equal(_bits(a), _bits(b)), f"{what}: {int((_bits(a) != _bits(b)).sum())} elements differ"


def _untouched(t, what):
    assert bool((_bits(t) == NAN16).all()), f"{what}: {int((_bits(t) != NAN16).sum())} sentinel elements written"


def _scale(p):
    return torch.tensor(1.0 / (1.0 - p), dtype=F64).float().item() if p > 0 else 1.0


# ------------------------------------------------------------------ batches
def _finish(bt, cuda):
    lens = torch.tensor(bt.lens)
    bt.sid = torch.repeat_interleave(torch.arange(bt.B), lens).to(cuda)                 # sample of each row
    pos = torch.cat([torch.arange(L) for L in bt.lens]).to(cuda)
    bt.didx = bt.sid * bt.S + pos                                                       # row -> [B*S_max] slot
    return bt


def _packed_batch(lib, cuda, S, lens):
    """Token-packed rows (mrd_compact_tokens); a length of 0 is a sample whose mask is all zero."""
    B = len(lens)
    n, _, seq_off, _, _, row_bias = synth.packed(lib, cuda, B, S, 0, lens)
    bt = types.SimpleNamespace(B=B, S=S, n=n, rows=B * S, lens=[max(L, 1) for L in lens], seq_off=seq_off,
                               bias=row_bias, key_bias=row_bias[:n])
    return _finish(bt, cuda)


def _dense_batch(cuda, S, lens):
    """Dense rows (sample b owns rows [b*S, (b+1)*S)), keys beyond the length masked by a [B,S] bias."""
    B = len(lens)
    bias = torch.zeros(B, S)
    for b, L in enumerate(lens):
        bias[b, L:] = -INF
    bias = bias.to(cuda)
    bt = types.SimpleNamespace(B=B, S=S, n=B * S, rows=B * S, lens=[S] * B, seq_off=None, bias=bias,
                               key_bias=bias.view(-1))
    return _finish(bt, cuda)


def _inputs(bt, seed, cuda):
    g = torch.Generator(device=cuda).manual_seed(seed)
    qkv = torch.zeros(bt.rows, W, device=cuda, dtype=BF)
    qkv[:bt.n] = (torch.randn(bt.n, W, device=cuda, generator=g) * 0.5).to(BF)
    dctx = torch.zeros(bt.rows, HD, device=cuda, dtype=BF)
    dctx[:bt.n] = torch.randn(bt.n, HD, device=cuda, generator=g).to(BF)
    return qkv, dctx


def _keep(lib, bt, p, site=SITE, width=None):
    """The keep-mask [B, H, S_max, S_max] in fp64 (None for p = 0), indexed with `width` (default S_max)."""
    if p == 0:
        return None
    w = width or bt.S
    m = torch.empty(bt.B * H * w * w, device=bt.bias.device)
    _check(lib, lib.mrd_dropout_mask(SEED, site, p, m.numel(), m.data_ptr(), _stream()))
    keep = torch.zeros(bt.B, H, bt.S, bt.S, device=m.device, dtype=F64)
    keep[:, :, :w, :w] = m.view(bt.B, H, w, w)
    return keep


# ------------------------------------------------------------------ fp64 reference
def _reference(bt, qkv, dctx, keep, scale, key_bias=None):
    """O [n, HD] with its magnitude and quadrature magnitude, and (dctx given) the autograd dqkv [n, W] with both
    magnitudes for ctx = bf16(O) and for the chained ctx; the dense [B, H, S, *] intermediates are kept for the
    controls."""
    B, S, n = bt.B, bt.S, bt.n
    kbias = bt.key_bias if key_bias is None else key_bias
    x = qkv[:n].double().requires_grad_(dctx is not None)
    xd = torch.zeros(B * S, W, device=qkv.device, dtype=F64).index_copy(0, bt.didx, x)
    q, k, v = xd.view(B, S, 3, H, D).permute(2, 0, 3, 1, 4)                             # [B, H, S, D]
    kb = torch.full((B * S,), -INF, device=qkv.device, dtype=F64).index_copy(0, bt.didx, kbias.double())
    s = q @ k.transpose(-1, -2) + kb.view(B, 1, 1, S)
    m = s.detach().amax(-1, keepdim=True)
    e = torch.exp(s - torch.where(torch.isfinite(m), m, torch.zeros_like(m)))
    l = e.sum(-1, keepdim=True)
    P = e / torch.where(l > 0, l, torch.ones_like(l))
    Pt = P * scale if keep is None else P * keep * scale
    O = Pt @ v
    r = types.SimpleNamespace(o=O.permute(0, 2, 1, 3).reshape(B * S, HD)[bt.didx])
    q, k, v, P, Pt, O = q.detach(), k.detach(), v.detach(), P.detach(), Pt.detach(), O.detach()
    mag_o, q2_o = Pt @ v.abs(), Pt.pow(2) @ v.pow(2)
    r.mag_o = mag_o.permute(0, 2, 1, 3).reshape(B * S, HD)[bt.didx]
    r.magq_o = q2_o.sqrt().permute(0, 2, 1, 3).reshape(B * S, HD)[bt.didx]
    if dctx is None:
        r.o = r.o.detach()
        return r
    g = dctx[:n].double()
    r.o.backward(g)
    r.o, r.dqkv = r.o.detach(), x.grad
    dO = torch.zeros(B * S, HD, device=qkv.device, dtype=F64).index_copy(0, bt.didx, g)
    dO = dO.view(B, S, H, D).permute(0, 2, 1, 3)
    dP = dO @ v.transpose(-1, -2)
    delta = (dO * O).sum(-1, keepdim=True)
    dS = P * ((dP if keep is None else dP * keep) * scale - delta)
    mv, qv = Pt.transpose(-1, -2) @ dO.abs(), Pt.pow(2).transpose(-1, -2) @ dO.pow(2)
    pk, ds2 = P @ k, dS.pow(2)

    def rows(t):   # [B, H, 3, S, D] -> [n, W]
        return t.permute(0, 3, 2, 1, 4).reshape(B * S, W)[bt.didx]

    def mags(o_abs, o_sq):
        a = dS.abs() + P * (dO.abs() * o_abs).sum(-1, keepdim=True)
        dv2 = (dO.pow(2) * o_sq).sum(-1, keepdim=True)                                  # delta's rounding variance
        q2 = torch.stack([ds2 @ k.pow(2) + dv2 * pk.pow(2),
                          (ds2 + P.pow(2) * dv2).transpose(-1, -2) @ q.pow(2), qv], 2)
        return rows(torch.stack([a @ k.abs(), a.transpose(-1, -2) @ q.abs(), mv], 2)), rows(q2.sqrt())

    r.mag_dqkv, r.magq_dqkv = mags(O.abs(), O.pow(2))
    r.mag_dqkv_chained, r.magq_dqkv_chained = mags(O.abs() + mag_o, O.pow(2) + q2_o)
    r.dense = types.SimpleNamespace(q=q, P=P, Pt=Pt, dS=dS, dO=dO)
    return r


# ------------------------------------------------------------------ comparator
def _measure(bt, out, ref, mag, magq):
    """Per-element and per-item statistics of out [n, k*64] against ref; an item is one sample's rows of one
    64-column head block.  worst: the largest err / bound of an element; l2: the largest relative L2 of an item that
    does not cancel (||q|| < 2 ||ref||); cancelled / worst_cancel: how many items cancel and the largest
    ||err|| / (2u ||q||) among them; items_ok: every item within its bar."""
    out, ref = out[:bt.n].double(), ref.double()
    err = (out - ref).abs()
    bound = 2.0 ** -7 * ref.abs() + C_MAG * U * mag
    ratio = torch.where(err == 0, torch.zeros_like(err), err / bound).nan_to_num(INF)   # NaN out: fails
    i = int(ratio.argmax())
    row, col = divmod(i, ratio.shape[1])
    where = f"sample {int(bt.sid[row])} row {row} col {col}: out {out.flatten()[i].item():.6g} ref " \
            f"{ref.flatten()[i].item():.6g} mag {mag.flatten()[i].item():.4g}"
    nb = out.shape[1] // D

    def norm(t):
        return torch.zeros(bt.B, nb, device=t.device, dtype=F64).index_add_(
            0, bt.sid, t.pow(2).view(-1, nb, D).sum(-1)).sqrt()

    e, r, q = norm(out - ref).nan_to_num(INF), norm(ref), norm(magq)
    cancel = (q >= 2 * r) & (q > 0)
    zero = torch.zeros_like(e)
    rel = torch.where(e == 0, zero, e / r)
    rel_q = torch.where(e == 0, zero, e / (2 * U * q))
    items_ok = bool(torch.where(cancel, rel_q <= 1, rel <= L2_BAR).all())
    return types.SimpleNamespace(worst=ratio.max().item(), where=where, items_ok=items_ok,
                                 l2=torch.where(cancel, zero, rel).max().item(), cancelled=int(cancel.sum()),
                                 items=cancel.numel(), worst_cancel=torch.where(cancel, rel_q, zero).max().item())


def _close(bt, out, ref, mag, magq, what, log):
    m = _measure(bt, out, ref, mag, magq)
    log.append(f"{what}: worst err/bound {m.worst:.3f} (bar 1), worst item relative L2 {m.l2:.2e} (bar {L2_BAR:g}); "
               f"{m.cancelled}/{m.items} cancelled items, worst err/(2u |q|) {m.worst_cancel:.3f} (bar 1)")
    assert m.worst <= 1.0, f"{what}: err/bound {m.worst:.3g} at {m.where}"
    assert m.items_ok, f"{what}: relative L2 {m.l2:.3g} (bar {L2_BAR:g}), cancelled items {m.worst_cancel:.3g} (bar 1)"


def _fails(bt, out, ref, mag, magq):
    m = _measure(bt, out, ref, mag, magq)
    return m.worst > 1.0 or not m.items_ok


PARTS = (("dQ", slice(0, HD)), ("dK", slice(HD, 2 * HD)), ("dV", slice(2 * HD, W)))


def _close_dqkv(bt, dqkv, ref, mag, magq, what, log):
    for name, sl in PARTS:
        _close(bt, dqkv[:, sl], ref.dqkv[:, sl], mag[:, sl], magq[:, sl], f"{what} {name}", log)


# ------------------------------------------------------------------ kernel calls
def _forward(lib, bt, qkv, p, out):
    if bt.seq_off is None:
        rc = lib.mrd_attention_train_bf16(qkv.data_ptr(), bt.bias.data_ptr(), bt.B, bt.S, H, SEED, SITE, p,
                                          out.data_ptr(), _stream())
    else:   # the training step's call: packed rows, rows = the allocation's row count
        rc = lib.mrd_attention_train_varlen_bf16(qkv.data_ptr(), bt.bias.data_ptr(), bt.seq_off.data_ptr(), bt.B,
                                                 bt.S, H, bt.rows, SEED, SITE, p, out.data_ptr(), _stream())
    _check(lib, rc)


def _backward(lib, bt, qkv, ctx, dctx, p, cuda):
    """dqkv of one backward launch; rows past the live count start as the NaN sentinel.  S > 128: the fp32 dK | dV
    accumulator is zeroed and has exactly the live rows."""
    dqkv = _sentinel(bt.rows, W, cuda)
    acc = torch.zeros(bt.n, 2 * HD, device=cuda) if bt.S > 128 else None
    _check(lib, lib.mrd_attention_bwd_bf16(qkv.data_ptr(), ctx.data_ptr(), dctx.data_ptr(), bt.bias.data_ptr(),
                                           None if bt.seq_off is None else bt.seq_off.data_ptr(), bt.B, bt.S, H, SEED,
                                           SITE, p, dqkv.data_ptr(), None if acc is None else acc.data_ptr(), bt.n,
                                           _stream()))
    return dqkv


def _run(lib, cuda, bt, p, label, seed, backward=True):
    """Forward and backward of one batch against the reference, with the buffer-edge and run-to-run checks."""
    log = []
    qkv, dctx = _inputs(bt, seed, cuda)
    keep, sc = _keep(lib, bt, p), _scale(p)
    ref = _reference(bt, qkv, dctx if backward else None, keep, sc)
    out = _sentinel(bt.rows, HD, cuda)
    _forward(lib, bt, qkv, p, out)
    torch.cuda.synchronize()
    _close(bt, out, ref.o, ref.mag_o, ref.magq_o, f"{label} O", log)
    if bt.n < bt.rows:
        _untouched(out[bt.n:], f"{label}: out past the live rows")
        # rows past the live ones hold large finite garbage (the 32-row TMA boxes of the last sample reach them)
        junk = qkv.clone()
        junk[bt.n:] = (torch.randn(bt.rows - bt.n, W, device=cuda, generator=torch.Generator(device=cuda)
                                   .manual_seed(seed + 1)) * 100).to(BF)
        out_j = _sentinel(bt.rows, HD, cuda)
        _forward(lib, bt, junk, p, out_j)
        _same_bits(out_j, out, f"{label}: forward with garbage past the live rows")
    out2 = _sentinel(bt.rows, HD, cuda)
    _forward(lib, bt, qkv, p, out2)
    _same_bits(out2, out, f"{label}: forward run to run")
    r = types.SimpleNamespace(qkv=qkv, dctx=dctx, keep=keep, sc=sc, ref=ref, out=out, log=log)
    if not backward:
        print("\n".join(log))
        return r

    ctx = torch.zeros(bt.rows, HD, device=cuda, dtype=BF)
    ctx[:bt.n] = ref.o.to(BF)
    dqkv = _backward(lib, bt, qkv, ctx, dctx, p, cuda)
    torch.cuda.synchronize()
    _close_dqkv(bt, dqkv, ref, ref.mag_dqkv, ref.magq_dqkv, label, log)
    if bt.n < bt.rows:
        _untouched(dqkv[bt.n:], f"{label}: dqkv past the live rows")
    dqkv2 = _backward(lib, bt, qkv, ctx, dctx, p, cuda)
    if bt.S <= 128:
        _same_bits(dqkv2, dqkv, f"{label}: backward run to run")
    else:   # fp32 atomics across query blocks: the order of the adds varies
        _close_dqkv(bt, dqkv2, ref, ref.mag_dqkv, ref.magq_dqkv, f"{label} (rerun)", log)
    dqkv_c = _backward(lib, bt, qkv, out, dctx, p, cuda)
    _close_dqkv(bt, dqkv_c, ref, ref.mag_dqkv_chained, ref.magq_dqkv_chained, f"{label} chained", log)
    r.ctx, r.dqkv = ctx, dqkv
    print("\n".join(log))
    return r


@pytest.fixture
def mma_sync(lib):
    """The mma.sync forward for every length; the process-wide switch is restored whatever the test does."""
    _check(lib, lib.mrd_attention_use_tcgen05(0))
    yield
    _check(lib, lib.mrd_attention_use_tcgen05(1))


# ------------------------------------------------------------------ cases
def _bench_lens(seed):
    """The training benchmark's batch: 64 lengths in [16, 127], the longest 127 (a mask indexed by the live maximum
    differs from one indexed by S_max = 128), live rows not a multiple of 64."""
    g = torch.Generator().manual_seed(seed)
    lens = torch.randint(16, 128, (64,), generator=g)
    lens[int(lens.argmax())] = 127
    if int(lens.sum()) % 64 == 0:
        lens[int(lens.argmin())] += 1
    return lens.tolist()


@pytest.mark.parametrize("p", [0.0, 0.1, 0.5])
def test_benchmark_shape_packed(lib, cuda, p):
    """B = 64, S_max = 128, 8192 allocated rows: 768 items on min(768, 592) persistent CTAs, some run two."""
    bt = _packed_batch(lib, cuda, 128, _bench_lens(1))
    assert bt.rows == 8192 and bt.n % 64 != 0 and max(bt.lens) == 127
    r = _run(lib, cuda, bt, p, f"benchmark p={p}", 11)
    b = bt.lens.index(127)
    if p == 0:
        # one (sample, head) of the kernel's own O, and of its dQ, 1 % off either way (in fp64: bf16 would quantise
        # the 1 %).  Without dropout the kernels carry no systematic error to offset it.  With it they do: the kept
        # maximum's weight 1 * float32(1/0.9) rounds to bf16 1.109375, 0.16 % low, which puts O about 0.1 % low.
        rows, cols = slice(int((bt.sid < b).sum()), int((bt.sid <= b).sum())), slice(3 * D, 4 * D)
        for f in (1.01, 0.99):
            off = r.out.double()
            off[rows, cols] *= f
            assert _fails(bt, off, r.ref.o, r.ref.mag_o, r.ref.magq_o), f"an O item scaled by {f} passed"
            off = r.dqkv[:, :HD].double()
            off[rows, cols] *= f
            assert _fails(bt, off, r.ref.dqkv[:, :HD], r.ref.mag_dqkv[:, :HD], r.ref.magq_dqkv[:, :HD]), \
                f"a dQ item scaled by {f} passed"
    if p != 0.1:
        return
    # negative controls on the kernel's actual forward output
    k1 = _keep(lib, bt, p, site=SITE + 1)
    assert _fails(bt, r.out, *_ref_o(bt, r, k1)), "the mask of site + 1 passed"
    k2 = _keep(lib, bt, p, width=max(bt.lens))
    assert _fails(bt, r.out, *_ref_o(bt, r, k2)), "the mask indexed with the longest live length passed"
    kb = bt.key_bias.clone()
    kb[int((bt.sid < b).sum()) + 126] = -INF
    assert _fails(bt, r.out, *_ref_o(bt, r, r.keep, kb)), "a reference without one sample's last key passed"


def _ref_o(bt, r, keep, key_bias=None):
    ref = _reference(bt, r.qkv, None, keep, r.sc, key_bias)
    return ref.o, ref.mag_o, ref.magq_o


@pytest.mark.parametrize("p", [0.0, 0.1])
def test_short_boundaries_packed(lib, cuda, p):
    """Lengths at the 16-key MMA granule and the 32-row TMA boxes, eight times over in a seeded shuffle plus two
    samples whose mask is all zero: 98 samples, 1176 items on 592 CTAs, so short items follow long ones on a CTA."""
    g = torch.Generator().manual_seed(3)
    lens = torch.tensor(BOUNDARY * 8 + [0, 0])
    lens = lens[torch.randperm(lens.numel(), generator=g)].tolist()
    bt = _packed_batch(lib, cuda, 128, lens)
    r = _run(lib, cuda, bt, p, f"boundaries p={p}", 12)
    # all-masked samples (only CLS kept, key bias -inf): a zero context and exactly zero gradients
    for b in (i for i, L in enumerate(lens) if L == 0):
        row = int((bt.sid < b).sum())
        assert float(bt.key_bias[row]) == -INF
        assert bool((r.out[row] == 0).all()) and bool((r.dqkv[row] == 0).all()), f"masked sample {b}"


@pytest.mark.parametrize("S", [256, 512])
@pytest.mark.parametrize("p", [0.0, 0.1])
def test_long_packed(lib, cuda, S, p):
    """S_max 256 / 512: lengths at the 128-key block edges among short samples, so many 128-query items hold no live
    row; more items than the 296 persistent CTAs; tiled backward with a zeroed accumulator of the live rows."""
    g = torch.Generator().manual_seed(S)
    edges = [L for L in LONG_EDGES if L <= S]
    lens = torch.tensor(edges + torch.randint(1, 128, (24 - len(edges),), generator=g).tolist())
    lens = lens[torch.randperm(24, generator=g)].tolist()
    bt = _packed_batch(lib, cuda, S, lens)
    assert bt.B * H * (S // 128) > 296 and sum(L < 128 for L in lens) > 12
    r = _run(lib, cuda, bt, p, f"long S={S} p={p}", 13)
    if S != 512 or p != 0.1:
        return
    # negative control: one (sample, head) without the dK / dV of query block 1 on key block 0
    b, h = bt.lens.index(385), 5
    dn, off = r.ref.dense, int((bt.sid < b).sum())
    pert = r.ref.dqkv.clone()
    qs, ks = slice(128, 256), slice(0, 128)
    pert[off:off + 128, HD + h * D:HD + (h + 1) * D] -= dn.dS[b, h, qs, ks].t() @ dn.q[b, h, qs]
    pert[off:off + 128, 2 * HD + h * D:2 * HD + (h + 1) * D] -= dn.Pt[b, h, qs, ks].t() @ dn.dO[b, h, qs]
    sl = slice(HD, W)
    assert _fails(bt, r.dqkv[:, sl], pert[:, sl], r.ref.mag_dqkv[:, sl], r.ref.magq_dqkv[:, sl]), \
        "a dK / dV without one query block's contribution passed"


DENSE_CASES = [(3, 128, [128, 77, 5], 0.0), (4, 48, [48, 48, 17, 1], 0.0), (2, 128, [128, 100], 0.1),
               (5, 32, [32, 9, 32, 20, 31], 0.25),
               # > 128 tokens: tcgen05 long forward, tiled backward
               (3, 256, [256, 130, 3], 0.0), (2, 200, [200, 129], 0.1), (2, 512, [512, 385], 0.0),
               (1, 384, [300], 0.2)]


@pytest.mark.parametrize("B,S,lens,p", DENSE_CASES)
def test_dense_layout(lib, cuda, B, S, lens, p):
    """Dense rows with a key bias.  Padded query rows get a gradient here too and are compared with the rest (keys
    past the length receive exactly zero).  For S <= 128 the packed layout gives bit-identical gradients."""
    bt = _dense_batch(cuda, S, lens)
    assert bt.B == B
    r = _run(lib, cuda, bt, p, f"dense B={B} S={S} p={p}", 14)
    if S > 128:
        return
    live = (bt.bias > -INF).view(-1)
    rows = live.nonzero().squeeze(1)
    dctx = r.dctx.clone()
    dctx[~live] = 0   # padded queries do not exist in the packed layout
    d_dense = _backward(lib, bt, r.qkv, r.ctx, dctx, p, cuda)
    pk = types.SimpleNamespace(B=B, S=S, n=rows.numel(), rows=rows.numel(), bias=torch.zeros(rows.numel(), device=cuda),
                               seq_off=torch.tensor([0] + torch.tensor(lens).cumsum(0).tolist(), device=cuda,
                                                    dtype=torch.int32))
    d_pack = _backward(lib, pk, r.qkv[rows].contiguous(), r.ctx[rows].contiguous(), dctx[rows].contiguous(), p, cuda)
    torch.cuda.synchronize()
    assert torch.equal(d_pack, d_dense[rows])


@pytest.mark.parametrize("case", ["benchmark", "long"])
def test_mma_sync_forward(lib, cuda, mma_sync, case):
    """The mma.sync forward with dropout (its only route is the switch): the benchmark batch and S_max = 512."""
    if case == "benchmark":
        bt = _packed_batch(lib, cuda, 128, _bench_lens(1))
    else:
        g = torch.Generator().manual_seed(5)
        lens = torch.tensor(LONG_EDGES + torch.randint(1, 128, (16,), generator=g).tolist())
        bt = _packed_batch(lib, cuda, 512, lens[torch.randperm(24, generator=g)].tolist())
    _run(lib, cuda, bt, 0.1, f"mma.sync {case}", 15, backward=False)

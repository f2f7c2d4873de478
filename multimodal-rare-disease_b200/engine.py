"""Host-side wrapper of one mrd_ctx (C ABI, include/mrd_b200.h): weight hand-off and forwards.

PyTorch is plumbing here: it owns the nn.Parameters (so state_dicts/checkpoints of the reference
load unchanged), allocates the output tensors and supplies the CUDA stream.  All arithmetic runs in
libmrd_b200.so.  An Engine refuses to run anywhere but on an sm_100 CUDA device.
"""

from __future__ import annotations

import ctypes as C
from typing import Dict, Iterable, Optional, Tuple

import torch

from . import _lib

_MASK_CODES = {
    torch.int64: _lib.DT_I64,
    torch.int32: _lib.DT_I32,
    torch.float32: _lib.DT_F32,
    torch.uint8: _lib.DT_U8,
    torch.bool: _lib.DT_U8,
    torch.bfloat16: _lib.DT_BF16,
}


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _stream(device: torch.device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


class Engine:
    """One mrd_ctx bound to one CUDA device, fed from an nn.Module's parameters.

    `groups` maps the module-tree prefixes of the owning module onto the canonical state_dict
    prefixes the library expects ("cnn_encoder.", "text_encoder.", "fusion.", "classifier."), e.g. a
    standalone CNNEncoder passes {"": "cnn_encoder."}.
    """

    def __init__(self, device: torch.device, options: Optional[Dict[str, float]] = None):
        if device.type != "cuda":
            raise _lib.MrdError(
                f"the B200 path runs on CUDA devices only (module is on '{device}'); "
                "there is no CPU fallback - use the reference implementation on CPU")
        self.lib = _lib.load()
        self.device = device
        self.train_serial = 0
        self.train_opts: Optional[Dict[str, float]] = None   # "train.*" options applied to THIS context
        self.fp32_check = bool((options or {}).get("fp32_check", 0.0))
        self._sigs: Dict[str, tuple] = {}
        self._dirty = set()
        self._keep: Dict[str, list] = {}
        self._ctx = C.c_void_p()
        with torch.cuda.device(device):
            _lib.check(self.lib.mrd_ctx_create(C.byref(self._ctx)), "mrd_ctx_create")
            for k, v in (options or {}).items():
                _lib.check(self.lib.mrd_ctx_set_option(self._ctx, k.encode(), float(v)),
                           f"mrd_ctx_set_option({k})")

    def __del__(self):
        try:
            if getattr(self, "_ctx", None) is not None and self._ctx.value:
                self.lib.mrd_ctx_destroy(self._ctx)
                self._ctx = C.c_void_p()
        except Exception:
            pass

    # ------------------------------------------------------------------ configuration / stats
    def configure(self, img_chunk: int = 0, seq_chunk_tokens: int = 0) -> None:
        with torch.cuda.device(self.device):
            _lib.check(self.lib.mrd_ctx_configure(self._ctx, int(img_chunk), int(seq_chunk_tokens)),
                       "mrd_ctx_configure")

    def set_option(self, key: str, value: float) -> None:
        with torch.cuda.device(self.device):
            _lib.check(self.lib.mrd_ctx_set_option(self._ctx, key.encode(), float(value)),
                       f"mrd_ctx_set_option({key})")
        if key == "fp32_check":
            self.fp32_check = bool(value)

    def profile(self, enable: bool) -> None:
        with torch.cuda.device(self.device):
            _lib.check(self.lib.mrd_ctx_profile(self._ctx, 1 if enable else 0), "mrd_ctx_profile")

    def profile_report(self):
        """[{label, cat, launches, ms, flops, bytes}] since profile(True)."""
        buf = C.create_string_buffer(1 << 16)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.mrd_ctx_profile_report(self._ctx, buf, len(buf)), "mrd_ctx_profile_report")
        rows = []
        for line in buf.value.decode().splitlines():
            label, cat, n, ms, fl, by = line.split(",")
            rows.append({"label": label, "cat": ("tensor", "attention", "memory")[int(cat)],
                         "launches": int(n), "ms": float(ms), "flops": float(fl), "bytes": float(by)})
        return rows

    @property
    def launch_count(self) -> int:
        return int(self.lib.mrd_ctx_launch_count(self._ctx))

    @property
    def device_bytes(self) -> int:
        return int(self.lib.mrd_ctx_device_bytes(self._ctx))

    # ------------------------------------------------------------------ weights
    # parameter groups that are re-packed independently (a training step changes the trainable ones only: the
    # frozen ResNet50 backbone - 53 BN-folded filters - is not re-packed every step)
    GROUPS = ("cnn_encoder.backbone.", "cnn_encoder.projection.", "text_encoder.", "fusion.", "classifier.")

    @classmethod
    def group_named(cls, named: Iterable[Tuple[str, torch.Tensor]]) -> Dict[str, list]:
        """Floating-point (name, tensor) pairs bucketed by hand-over group; integer buffers
        (num_batches_tracked) and names outside every group are dropped."""
        groups = {g: [] for g in cls.GROUPS}
        for n, t in named:
            if not t.is_floating_point():
                continue
            for g in cls.GROUPS:
                if n.startswith(g):
                    groups[g].append((n, t))
                    break
        return groups

    def mark_dirty(self, group: str) -> None:
        """The library changed tensors of `group` behind torch's back (running statistics of the batch-norm
        layers in train mode): the next eval-mode hand-over re-packs the group."""
        self._dirty.add(group)

    def sync_weights(self, named: Iterable[Tuple[str, torch.Tensor]], training: bool = False) -> bool:
        """Re-pack the library's weights for every group in which a tensor was replaced or written since the
        last call.  named: (canonical state_dict name, tensor) pairs.  Returns True when a re-pack happened.
        training=True leaves a merely `dirty` backbone alone (its folded eval-mode copy is not used there)."""
        groups = self.group_named(named)
        changed = []
        for g, items in groups.items():
            if not items:
                continue
            sig = tuple((n, t.data_ptr(), t._version, t.dtype) for n, t in items)
            if sig != self._sigs.get(g) or (g in self._dirty and not training):
                changed.append((g, items, sig))
        if not changed:
            return False
        todo = [it for _, items, _ in changed for it in items]
        n = len(todo)
        names = (C.c_char_p * n)()
        ptrs = (C.c_void_p * n)()
        shapes = (C.c_longlong * (4 * n))()
        keep = {g: [] for g, _, _ in changed}
        i = 0
        for g, items, _ in changed:
            for name, t in items:
                if t.device != self.device:
                    raise _lib.MrdError(f"parameter {name} is on {t.device}, engine is on {self.device}")
                if t.dim() > 4:
                    raise _lib.MrdError(f"parameter {name} has {t.dim()} dims")
                x = t.detach()
                if x.dtype != torch.float32 or not x.is_contiguous():
                    x = x.float().contiguous()
                keep[g].append(x)
                names[i] = name.encode()
                ptrs[i] = x.data_ptr()
                for j, d in enumerate(x.shape):
                    shapes[4 * i + j] = d
                i += 1
        with torch.cuda.device(self.device):
            _lib.check(self.lib.mrd_ctx_load_weights(self._ctx, n, names, ptrs, shapes,
                                                     _stream(self.device)), "mrd_ctx_load_weights")
        for g, _, sig in changed:
            self._sigs[g] = sig
            self._dirty.discard(g)
            # the fp32 check mode and the training step read the raw fp32 tensors handed over above: keep them
            # (views of the parameters, or fp32 copies of non-fp32 ones) alive until the group's next hand-over
            self._keep[g] = keep[g]
        return True

    # ------------------------------------------------------------------ input normalisation
    def _images(self, images: torch.Tensor) -> Tuple[torch.Tensor, int]:
        if images.dim() != 4 or images.shape[1] != 3:
            raise ValueError(f"images must be [B,3,H,W], got {tuple(images.shape)}")
        if images.device != self.device:
            raise _lib.MrdError(f"images are on {images.device}, model is on {self.device}")
        if images.dtype not in (torch.float32, torch.bfloat16):
            images = images.float()
        images = images.contiguous()
        return images, (_lib.DT_BF16 if images.dtype == torch.bfloat16 else _lib.DT_F32)

    def _text(self, input_ids: torch.Tensor, attention_mask: Optional[torch.Tensor]):
        if input_ids.dim() != 2:
            raise ValueError(f"input_ids must be [B,S], got {tuple(input_ids.shape)}")
        if input_ids.device != self.device:
            raise _lib.MrdError(f"input_ids are on {input_ids.device}, model is on {self.device}")
        ids = input_ids if input_ids.dtype == torch.int64 else input_ids.long()
        ids = ids.contiguous()
        mask, code = None, _lib.DT_I64
        if attention_mask is not None:
            if attention_mask.shape != input_ids.shape:
                raise ValueError("attention_mask must have the shape of input_ids")
            mask = attention_mask.to(self.device)
            if mask.dtype not in _MASK_CODES:
                mask = mask.float() if mask.is_floating_point() else mask.long()
            mask = mask.contiguous()
            code = _MASK_CODES[mask.dtype]
        return ids, mask, code

    def _f32(self, *shape) -> torch.Tensor:
        return torch.empty(*shape, dtype=torch.float32, device=self.device)

    # ------------------------------------------------------------------ forwards
    def cnn_encoder(self, images, emb_dim: int, want_pooled=False, want_map=False):
        images, code = self._images(images)
        B, _, H, W = images.shape
        emb = self._f32(B, emb_dim)
        pooled = self._f32(B, 2048) if want_pooled else None
        fmap = self._f32(B, 2048, H // 32, W // 32) if want_map else None
        if B:
            with torch.cuda.device(self.device):
                _lib.check(self.lib.mrd_cnn_encoder_fwd(self._ctx, images.data_ptr(), code, B, H, W,
                                                        emb.data_ptr(), _ptr(pooled), _ptr(fmap),
                                                        _stream(self.device)), "mrd_cnn_encoder_fwd")
        return emb, pooled, fmap

    def text_encoder(self, input_ids, attention_mask, hidden: int = 768, want_hidden=False,
                     all_layers: int = 0, want_attn=False, layers: int = 12, heads: int = 12):
        """all_layers = L > 0 additionally returns the [L+1,B,S,hidden] stack of hidden states.
        want_attn additionally returns every layer's attention probabilities, f32 [layers,B,heads,S,S]
        (layers / heads: those of the loaded encoder); it comes last in the returned tuple."""
        ids, mask, code = self._text(input_ids, attention_mask)
        B, S = ids.shape
        cls = self._f32(B, hidden)
        last = self._f32(B, S, hidden) if (want_hidden or all_layers) else None
        stack = self._f32(all_layers + 1, B, S, hidden) if all_layers else None
        attn = self._f32(layers, B, heads, S, S) if want_attn else None
        if B:
            with torch.cuda.device(self.device):
                if want_attn:
                    _lib.check(self.lib.mrd_text_encoder_fwd_ex(self._ctx, ids.data_ptr(), _ptr(mask), code, B, S,
                                                                cls.data_ptr(), _ptr(last), _ptr(stack),
                                                                attn.data_ptr(), _stream(self.device)),
                               "mrd_text_encoder_fwd_ex")
                else:
                    _lib.check(self.lib.mrd_text_encoder_fwd(self._ctx, ids.data_ptr(), _ptr(mask), code,
                                                             B, S, cls.data_ptr(), _ptr(last), _ptr(stack),
                                                             _stream(self.device)), "mrd_text_encoder_fwd")
        out = (cls, last, stack) if all_layers else (cls, last)
        return out + (attn,) if want_attn else out

    def fusion(self, img_emb, txt_emb, hidden_dim: int, heads: int):
        if img_emb.dim() != 2 or txt_emb.dim() != 2 or img_emb.shape[0] != txt_emb.shape[0]:
            raise ValueError("fusion expects [B,Di] and [B,Dt] embeddings")
        img = img_emb.to(self.device, torch.float32).contiguous()
        txt = txt_emb.to(self.device, torch.float32).contiguous()
        B = img.shape[0]
        fused = self._f32(B, hidden_dim)
        a1 = self._f32(B, heads, 1, 1)
        a2 = self._f32(B, heads, 1, 1)
        if B:
            with torch.cuda.device(self.device):
                _lib.check(self.lib.mrd_fusion_fwd(self._ctx, img.data_ptr(), txt.data_ptr(), B,
                                                   fused.data_ptr(), a1.data_ptr(), a2.data_ptr(),
                                                   _stream(self.device)), "mrd_fusion_fwd")
        return fused, a1, a2

    def fusion_head(self, img_emb, txt_emb, hidden_dim: int, num_classes: int, want_fused=False):
        """AttentionFusion -> ClassificationHead -> softmax as one launch (mrd_fusion_head_fwd)."""
        if img_emb.dim() != 2 or txt_emb.dim() != 2 or img_emb.shape[0] != txt_emb.shape[0]:
            raise ValueError("fusion_head expects [B,Di] and [B,Dt] embeddings")
        img = img_emb.to(self.device, torch.float32).contiguous()
        txt = txt_emb.to(self.device, torch.float32).contiguous()
        B = img.shape[0]
        logits, probs = self._f32(B, num_classes), self._f32(B, num_classes)
        fused = self._f32(B, hidden_dim) if want_fused else None
        if B:
            with torch.cuda.device(self.device):
                _lib.check(self.lib.mrd_fusion_head_fwd(self._ctx, img.data_ptr(), txt.data_ptr(), B, _ptr(fused),
                                                        logits.data_ptr(), probs.data_ptr(),
                                                        _stream(self.device)), "mrd_fusion_head_fwd")
        return logits, probs, fused

    def head(self, x, num_classes: int, want_probs=True):
        if x.dim() != 2:
            raise ValueError("classification head expects [B,D] features")
        x = x.to(self.device, torch.float32).contiguous()
        B = x.shape[0]
        logits = self._f32(B, num_classes)
        probs = self._f32(B, num_classes) if want_probs else None
        if B:
            with torch.cuda.device(self.device):
                _lib.check(self.lib.mrd_head_fwd(self._ctx, x.data_ptr(), B, logits.data_ptr(),
                                                 _ptr(probs), _stream(self.device)), "mrd_head_fwd")
        return logits, probs

    def multimodal(self, images, input_ids, attention_mask, dims, want_embeddings=False,
                   logits_out: Optional[torch.Tensor] = None):
        """dims = (num_classes, img_emb, txt_emb, fused, heads).  logits_out: optional preallocated
        f32 [B,num_classes] slice (e.g. this rank's slot of an all-gather buffer)."""
        images, icode = self._images(images)
        ids, mask, mcode = self._text(input_ids, attention_mask)
        B, _, H, W = images.shape
        if ids.shape[0] != B:
            raise ValueError(f"batch mismatch: {B} images vs {ids.shape[0]} token rows")
        S = ids.shape[1]
        nc, di, dt, df, heads = dims
        if logits_out is not None:
            if (logits_out.shape != (B, nc) or logits_out.dtype != torch.float32
                    or not logits_out.is_contiguous() or logits_out.device != self.device):
                raise ValueError("logits_out must be a contiguous f32 [B,num_classes] tensor on the model device")
            logits = logits_out
        else:
            logits = self._f32(B, nc)
        probs = self._f32(B, nc)
        img_e = txt_e = fused = a1 = a2 = None
        if want_embeddings:
            img_e, txt_e, fused = self._f32(B, di), self._f32(B, dt), self._f32(B, df)
            a1, a2 = self._f32(B, heads, 1, 1), self._f32(B, heads, 1, 1)
        if B:
            with torch.cuda.device(self.device):
                _lib.check(self.lib.mrd_multimodal_fwd(
                    self._ctx, images.data_ptr(), icode, ids.data_ptr(), _ptr(mask), mcode, B, H, W, S,
                    logits.data_ptr(), probs.data_ptr(), _ptr(img_e), _ptr(txt_e), _ptr(fused),
                    _ptr(a1), _ptr(a2), _stream(self.device)), "mrd_multimodal_fwd")
        return logits, probs, img_e, txt_e, fused, a1, a2

    # ------------------------------------------------------------------ training step
    def train_forward(self, images, input_ids, attention_mask, num_classes: int, seed: int,
                      want_map: bool = False, emb_dims=None, block_out=None):
        """Train-mode forward (dropout active, activations kept inside the context) -> logits f32 [B,C]
        (and, with want_map, the layer4 feature map f32 [B,2048,H/32,W/32] of this forward).
        emb_dims = (image, text, fused) widths: the three embeddings of this forward are kept in
        self.last_train_embeddings (what return_embeddings=True hands out).
        block_out = 16 slots (f32 NCHW tensors or None), one per bottleneck: the forward also keeps what the backbone's
        data-gradient backward needs (mrd_train_forward_dg) and writes the output of every bottleneck given a tensor."""
        images, icode = self._images(images)
        ids, mask, mcode = self._text(input_ids, attention_mask)
        B, _, H, W = images.shape
        if ids.shape[0] != B:
            raise ValueError(f"batch mismatch: {B} images vs {ids.shape[0]} token rows")
        logits = self._f32(B, num_classes)
        fmap = self._f32(B, 2048, H // 32, W // 32) if want_map else None
        embs = [self._f32(B, d) for d in emb_dims] if emb_dims else [None, None, None]
        self.last_train_embeddings = embs if emb_dims else None
        self._train_inputs = (images, ids, mask)   # the backward re-reads the ids
        self.train_serial = getattr(self, "train_serial", 0) + 1
        if B and block_out is not None:
            slots = (C.c_void_p * 16)(*[_ptr(t) for t in block_out])
            with torch.cuda.device(self.device):
                _lib.check(self.lib.mrd_train_forward_dg(
                    self._ctx, images.data_ptr(), icode, ids.data_ptr(), _ptr(mask), mcode, B, H, W,
                    ids.shape[1], C.c_ulonglong(seed & 0xFFFFFFFFFFFFFFFF), logits.data_ptr(), slots,
                    _ptr(embs[0]), _ptr(embs[1]), _ptr(embs[2]), _stream(self.device)), "mrd_train_forward_dg")
        elif B:
            with torch.cuda.device(self.device):
                _lib.check(self.lib.mrd_train_forward_ex(
                    self._ctx, images.data_ptr(), icode, ids.data_ptr(), _ptr(mask), mcode, B, H, W,
                    ids.shape[1], C.c_ulonglong(seed & 0xFFFFFFFFFFFFFFFF), logits.data_ptr(), _ptr(fmap),
                    _ptr(embs[0]), _ptr(embs[1]), _ptr(embs[2]), _stream(self.device)), "mrd_train_forward")
        return (logits, fmap) if want_map else logits

    def _backward_stage_of(self, name: str, n_layers: int) -> int:
        """Stage of mrd_train_backward_stages that completes the gradient of parameter `name`."""
        pre = "text_encoder.encoder.encoder.layer."
        if name.startswith(pre):
            return 1 + (n_layers - 1 - int(name[len(pre):].split(".", 1)[0]))
        if name.startswith("text_encoder."):
            return n_layers + 1          # embeddings
        return 0                         # head, fusion, image projection

    def train_backward(self, dlogits: torch.Tensor, named_shapes, want_dpooled: bool = False, on_bucket=None,
                       dgrad=None):
        """named_shapes: [(canonical state_dict name, shape)] of the parameters that want a gradient.
        Returns their f32 gradients as views of ONE flat buffer, laid out in the order the backward completes
        them (head / fusion / projection, BERT layers last to first, embeddings); with want_dpooled also
        d(loss)/d(pooled backbone features) f32 [B,2048].
        on_bucket(flat_slice): data-parallel overlap - the backward is enqueued stage by stage and the callback
        receives each finished slice of the flat buffer right after its stage (it typically starts an
        asynchronous all-reduce that then runs under the remaining stages).
        dgrad = (block_grads, first_block, d_block_in, d_images) after a forward with block_out: the backward continues
        through the backbone (mrd_train_backward_dg); block_grads = 16 slots of f32 NCHW tensors or None."""
        dl = dlogits.to(self.device, torch.float32).contiguous()
        n_stages = int(self.lib.mrd_train_backward_num_stages(self._ctx))
        stage = [self._backward_stage_of(name, n_stages - 2) for name, _ in named_shapes]
        order = sorted(range(len(named_shapes)), key=lambda i: stage[i])   # stable: module order inside a stage
        sizes = [int(torch.Size(sh).numel()) for _, sh in named_shapes]
        offs, tot, bounds = [0] * len(named_shapes), 0, [0] * (n_stages + 1)
        for i in order:
            offs[i] = tot
            tot += (sizes[i] + 3) // 4 * 4      # keep every view 16-byte aligned
            bounds[stage[i] + 1] = tot
        for st in range(1, n_stages + 1):
            bounds[st] = max(bounds[st], bounds[st - 1])
        flat = torch.zeros(max(tot, 4), dtype=torch.float32, device=self.device)
        n = len(named_shapes)
        names = (C.c_char_p * n)()
        ptrs = (C.c_void_p * n)()
        views = []
        for i, ((name, sh), o, k) in enumerate(zip(named_shapes, offs, sizes)):
            v = flat.narrow(0, o, k).view(sh)
            views.append(v)
            names[i] = name.encode()
            ptrs[i] = v.data_ptr()
        d_pooled = torch.zeros(dl.shape[0], 2048, dtype=torch.float32, device=self.device) if want_dpooled else None
        if dl.shape[0]:
            with torch.cuda.device(self.device):
                if dgrad is not None:
                    block_grads, first_block, d_block_in, d_images = dgrad
                    slots = (C.c_void_p * 16)(*[_ptr(t) for t in block_grads])
                    _lib.check(self.lib.mrd_train_backward_dg(self._ctx, dl.data_ptr(), n, names, ptrs, _ptr(d_pooled),
                                                              slots, int(first_block), _ptr(d_block_in),
                                                              _ptr(d_images), _stream(self.device)),
                               "mrd_train_backward_dg")
                elif on_bucket is None:
                    _lib.check(self.lib.mrd_train_backward_ex(self._ctx, dl.data_ptr(), n, names, ptrs,
                                                              _ptr(d_pooled), _stream(self.device)),
                               "mrd_train_backward")
                else:
                    _lib.check(self.lib.mrd_train_backward_begin(self._ctx, dl.data_ptr(), n, names, ptrs,
                                                                 _ptr(d_pooled)), "mrd_train_backward_begin")
                    for st in range(n_stages):
                        _lib.check(self.lib.mrd_train_backward_stages(self._ctx, st, st + 1, _stream(self.device)),
                                   "mrd_train_backward_stages")
                        if bounds[st + 1] > bounds[st]:
                            on_bucket(flat[bounds[st]:bounds[st + 1]])
        self._train_inputs = None
        self.last_flat_grad = flat
        return (views, d_pooled) if want_dpooled else views

"""MultimodalClassifier - drop-in for the reference's src/multimodal_classifier.py.

Same classes, constructor arguments, attributes, state_dict keys (`cnn_encoder.*`, `text_encoder.*`,
`fusion.*`, `classifier.classifier.{0,3,6}.*`) and the same forward/predict contracts
(src/multimodal_classifier.py:131-202).  One forward = one call into libmrd_b200.so
(mrd_multimodal_fwd): ResNet50 + BERT-base + attention fusion + head + softmax on the caller's CUDA
stream, tiled into L2-sized micro-batches inside the library.
"""

from __future__ import annotations

from typing import Dict, List, Optional, Tuple

import torch
import torch.nn as nn

from . import _lib
from ._module import B200Module
from .cnn_encoder import CNNEncoder
from .config import Config, get_config
from .fusion_model import MultimodalFusion
from .text_encoder import TextEncoder

_ACT = {"relu": _lib.ACT_RELU, "gelu": _lib.ACT_GELU}


class _TrainStep(torch.autograd.Function):
    """autograd node of the train-mode forward: forward = mrd_train_forward, backward =
    mrd_train_backward (one library call each).  Inputs after `nc` are the trainable parameters, so
    `loss.backward()` fills their .grad exactly where the reference's autograd would
    (src/train.py:307-320: backward -> clip_grad_norm_ -> optimizer.step stay the caller's)."""

    @staticmethod
    def forward(ctx, eng, images, input_ids, attention_mask, seed, named_shapes, ddp, *params):
        """ddp = (num_classes, data_parallel, process_group, hooked, emb_dims, dgrad): hooked = the backbone module
        whose forward / backward hooks are served from the layer4 map (Grad-CAM on cnn_encoder.get_attention_layer())
        or None; dgrad = a _DataGrad (data gradients through the backbone) or None."""
        ctx.eng, ctx.named_shapes, ctx.ddp = eng, named_shapes, ddp
        ctx.hooked = ddp[3] if len(ddp) > 3 else None
        emb_dims = ddp[4] if len(ddp) > 4 else None
        ctx.dgrad = ddp[5] if len(ddp) > 5 else None
        if ctx.dgrad is not None:
            dg = ctx.dgrad
            logits = eng.train_forward(images, input_ids, attention_mask, ddp[0], seed, emb_dims=emb_dims,
                                       block_out=dg.block_out)
            # forward hooks of the served modules, in forward order: the module's output (its last bottleneck's), NCHW
            # fp32; the input tuple is empty as for layer4's hooks
            for m, lo, hi in dg.hooked:
                for hook in list(m._forward_hooks.values()):
                    hook(m, (), dg.block_out[hi])
            ctx.img_dtype = images.dtype
        elif ctx.hooked is None:
            logits = eng.train_forward(images, input_ids, attention_mask, ddp[0], seed, emb_dims=emb_dims)
        else:
            logits, fmap = eng.train_forward(images, input_ids, attention_mask, ddp[0], seed, want_map=True,
                                             emb_dims=emb_dims)
            ctx.map_shape = tuple(fmap.shape)
            # forward hooks of the hooked module see its output as the reference's would (NCHW fp32); the module's
            # input (layer3's output) is not materialised in that layout: hooks get an empty input tuple
            for hook in list(ctx.hooked._forward_hooks.values()):
                hook(ctx.hooked, (), fmap)
        ctx.serial = eng.train_serial
        return logits

    @staticmethod
    def backward(ctx, dlogits):
        if ctx.serial != ctx.eng.train_serial:
            raise RuntimeError(
                "backward through a train-mode forward whose saved activations were overwritten by a newer "
                "train-mode forward of the same model: the B200 training step keeps ONE forward pending "
                "(call backward before the next forward, as the reference's loops do)")
        if ctx.dgrad is not None:
            dg = ctx.dgrad
            d_images = dg.new_images_grad() if dg.want_images else None
            grads, d_pooled = ctx.eng.train_backward(dlogits, ctx.named_shapes, want_dpooled=True,
                                                     dgrad=(dg.block_grads, dg.first, dg.d_in, d_images))
            dg.serve_backward_hooks(d_pooled)
            img_grad = d_images.to(ctx.img_dtype) if d_images is not None else None
            return (None, img_grad) + (None,) * 5 + tuple(grads)
        if ctx.hooked is not None:
            grads, d_pooled = ctx.eng.train_backward(dlogits, ctx.named_shapes, want_dpooled=True)
            # AdaptiveAvgPool2d(1) backward (TV:models/resnet.py:278): every position of the layer4 map receives
            # d_pooled / (h*w); that is grad_output of the hooked module
            Bn, Cn, h, w = ctx.map_shape
            d_map = (d_pooled / float(h * w)).view(Bn, Cn, 1, 1).expand(Bn, Cn, h, w).contiguous()
            for hook in list(ctx.hooked._backward_hooks.values()):
                hook(ctx.hooked, (None,), (d_map,))
        elif ctx.ddp[1]:
            # data parallel: the gradients live in one flat buffer laid out in completion order; the averaging
            # all-reduce of each bucket (one per backward stage: head + fusion + projection, every BERT layer, the
            # embeddings) is started as soon as its stage is enqueued and runs under the remaining stages
            from .parallel import allreduce_mean_async, wait_allreduce
            pending = []
            grads = ctx.eng.train_backward(dlogits, ctx.named_shapes,
                                           on_bucket=lambda b: pending.append(allreduce_mean_async(b, ctx.ddp[2])))
            for h in pending:
                wait_allreduce(h)
        else:
            grads = ctx.eng.train_backward(dlogits, ctx.named_shapes)
        return (None,) * 7 + tuple(grads)


class _DataGrad:
    """What one forward with data gradients through the backbone asks of the library: the bottleneck outputs the
    forward hooks see, the point the backward chain stops at, and the buffers the backward hooks and images.grad read.
    Bottlenecks are numbered 0..15 in forward order; a served module covers the bottlenecks [lo, hi]."""

    def __init__(self, hooked, want_images, geometry, B, H, W, device):
        self.hooked = hooked                  # [(module, lo, hi)] with hooks, in forward order
        self.want_images = want_images
        self.geometry = geometry              # per bottleneck: (C_in, h_in, w_in, C_out, h_out, w_out)
        self.B, self.H, self.W, self.device = B, H, W, device
        n = len(geometry)

        def f32(*shape):
            return torch.empty(*shape, dtype=torch.float32, device=device)

        self.block_out = [None] * n
        for m, lo, hi in hooked:
            if m._forward_hooks and self.block_out[hi] is None:
                _, _, _, c, h, w = geometry[hi]
                self.block_out[hi] = f32(B, c, h, w)
        # the chain runs down to the lowest point anything asks for: the image, or the output of a hooked module
        stops = [0] if want_images else []
        stops += [hi + 1 for m, lo, hi in hooked if m._backward_hooks]
        self.first = min(stops) if stops else n
        self.block_grads = [None] * n
        self.d_in = None
        for m, lo, hi in hooked:
            if not m._backward_hooks:
                continue
            if hi < n - 1 and self.block_grads[hi] is None:
                _, _, _, c, h, w = geometry[hi]
                self.block_grads[hi] = f32(B, c, h, w)
            if self.first <= lo:
                if lo == self.first:
                    if self.d_in is None:
                        c, h, w = geometry[lo][:3]
                        self.d_in = f32(B, c, h, w)
                elif self.block_grads[lo - 1] is None:
                    _, _, _, c, h, w = geometry[lo - 1]
                    self.block_grads[lo - 1] = f32(B, c, h, w)

    def new_images_grad(self):
        return torch.empty(self.B, 3, self.H, self.W, dtype=torch.float32, device=self.device)

    def serve_backward_hooks(self, d_pooled):
        """Full backward hooks, innermost and highest first (the order autograd completes the modules' inputs):
        grad_output = (d/d output,), grad_input = (d/d input,) where the chain ran below the module, else (None,)."""
        n = len(self.geometry)
        _, _, _, c, h, w = self.geometry[n - 1]
        top = None
        for m, lo, hi in sorted(self.hooked, key=lambda e: (-e[1], e[2])):
            if not m._backward_hooks:
                continue
            if hi == n - 1:
                if top is None:   # AdaptiveAvgPool2d(1) backward: d_pooled / (h*w) at every position of the layer4 map
                    top = (d_pooled / float(h * w)).view(self.B, c, 1, 1).expand(self.B, c, h, w).contiguous()
                g_out = top
            else:
                g_out = self.block_grads[hi]
            g_in = None
            if self.first <= lo:
                g_in = self.d_in if lo == self.first else self.block_grads[lo - 1]
            for hook in list(m._backward_hooks.values()):
                hook(m, (g_in,), (g_out,))


class ClassificationHead(B200Module):
    """Linear/activation/dropout stack (src/multimodal_classifier.py:16-83)."""

    _mrd_groups = {"": "classifier."}

    def __init__(self, input_dim: int, hidden_dims: List[int] = (512, 256), num_classes: int = 10,
                 dropout: float = 0.4, activation: str = "relu"):
        super().__init__()
        self.num_classes = num_classes
        self.activation = activation if activation in ("relu", "gelu", "leaky_relu") else "relu"
        layers: List[nn.Module] = []
        prev = input_dim
        for h in hidden_dims:
            layers += [nn.Linear(prev, h), self._get_activation(activation), nn.Dropout(dropout)]
            prev = h
        layers.append(nn.Linear(prev, num_classes))
        self.classifier = nn.Sequential(*layers)

    @staticmethod
    def _get_activation(name: str) -> nn.Module:
        if name == "gelu":
            return nn.GELU()
        if name == "leaky_relu":
            return nn.LeakyReLU(0.1, inplace=True)
        return nn.ReLU(inplace=True)

    def _mrd_options(self):
        if self.activation not in _ACT:
            raise NotImplementedError(f"activation {self.activation!r} is outside the B200 hot path")
        return {"head_act": _ACT[self.activation]}

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        logits, _ = self._engine().head(x, self.num_classes, want_probs=False)
        return logits


class MultimodalClassifier(B200Module):
    _mrd_groups = {"cnn_encoder.": "cnn_encoder.", "text_encoder.": "text_encoder.",
                   "fusion.": "fusion.", "classifier.": "classifier."}

    def __init__(self, config: Optional[Config] = None, *, random_init: bool = False):
        """random_init=True: BioBERT-base shaped text encoder without the hub download and no
        ImageNet download (benchmarks / tests on air-gapped machines).  Default = reference."""
        super().__init__()
        config = get_config() if config is None else config
        self.config = config
        cnn_cfg = config.cnn_encoder
        if random_init and getattr(cnn_cfg, "pretrained", False):
            import copy

            cnn_cfg = copy.copy(cnn_cfg)
            cnn_cfg.pretrained = False
        self.cnn_encoder = CNNEncoder(cnn_cfg)
        self.text_encoder = TextEncoder(config.text_encoder, random_init=random_init)
        self.fusion = MultimodalFusion(config.fusion)
        self.classifier = ClassificationHead(
            input_dim=config.fusion.hidden_dim,
            hidden_dims=config.classifier.hidden_dims,
            num_classes=config.classifier.num_classes,
            dropout=config.classifier.dropout,
            activation=config.classifier.activation,
        )
        self.image_embedding_dim = config.cnn_encoder.embedding_dim
        self.text_embedding_dim = config.text_encoder.embedding_dim
        self.fusion_dim = config.fusion.hidden_dim
        self.num_classes = config.classifier.num_classes

    def _mrd_options(self):
        opts = {}
        for m in (self.text_encoder, self.fusion, self.classifier):
            opts.update(m._mrd_options())
        return opts

    def _dims(self):
        return (self.num_classes, self.cnn_encoder.embedding_dim, self.text_encoder.embedding_dim,
                self.fusion_dim, self.config.fusion.num_attention_heads)

    def forward(self, images: torch.Tensor, input_ids: torch.Tensor, attention_mask: torch.Tensor,
                return_embeddings: bool = False, *, logits_out: Optional[torch.Tensor] = None
                ) -> Dict[str, torch.Tensor]:
        """images [B,3,224,224], input_ids/attention_mask [B,S] -> {"logits","probs"} (+ embeddings
        and the fusion attention weights when return_embeddings=True), all fp32 on the model device."""
        self.text_encoder._check()
        hooked, want_images = self._data_grad_request(images)
        layer4 = self._hooked_attention_layer()
        layer4_only = not want_images and len(hooked) == 1 and layer4 is not None and hooked[0][0] is layer4
        dgrad = bool(want_images or hooked) and not layer4_only
        if self.training:
            # hooks on layer4 alone are not served in train mode (as before data gradients existed)
            return self._forward_train(images, input_ids, attention_mask, return_embeddings,
                                       dgrad=(hooked, want_images) if dgrad else None)
        if dgrad:
            # input saliency (images.requires_grad) and hooks below layer4: the eval-mode forward made differentiable
            # down to the image
            return self._forward_train(images, input_ids, attention_mask, return_embeddings,
                                       dgrad=(hooked, want_images))
        if layer4_only:
            # Grad-CAM (notebooks/explainability.ipynb cell 3): hooks on cnn_encoder.get_attention_layer() and
            # logits[0, c].backward() under model.eval() - the eval-mode forward made differentiable
            return self._forward_train(images, input_ids, attention_mask, return_embeddings, explain=layer4)
        logits, probs, img_e, txt_e, fused, a1, a2 = self._engine().multimodal(
            images, input_ids, attention_mask, self._dims(), want_embeddings=return_embeddings,
            logits_out=logits_out)
        out = {"logits": logits, "probs": probs}
        if return_embeddings:
            out["image_embedding"] = img_e
            out["text_embedding"] = txt_e
            out["fused_embedding"] = fused
            out["attention_info"] = {"image_to_text_attention": a1, "text_to_image_attention": a2}
        return out

    # ---- training step ------------------------------------------------------------------------
    def _hooked_attention_layer(self):
        """cnn_encoder.get_attention_layer() (backbone.layer4, src/cnn_encoder.py:186-198) when somebody registered
        forward or backward hooks on it, else None."""
        try:
            m = self.cnn_encoder.get_attention_layer()
        except Exception:
            return None
        return m if (len(m._forward_hooks) or len(m._backward_hooks)) else None

    def _served_modules(self):
        """{id(module): (module, lo, hi)} of the backbone modules whose hooks are served - backbone.layer1..layer4 and
        every Bottleneck backbone.layerN[i] - and the geometry of every bottleneck (see _DataGrad)."""
        bb = self.cnn_encoder.backbone
        served, blocks, k = {}, [], 0
        for L in range(1, 5):
            layer = getattr(bb, f"layer{L}")
            lo = k
            for blk in layer:
                served[id(blk)] = (blk, k, k)
                blocks.append(blk)
                k += 1
            served[id(layer)] = (layer, lo, k - 1)
        return served, blocks

    def _data_grad_request(self, images):
        """([(module, lo, hi)] served modules with forward or backward hooks, in forward order; whether images.grad is
        wanted).  A hook on any other module of the backbone raises: its tensors do not exist on the B200 path."""
        bb = self.cnn_encoder.backbone
        hooked_any = [(n, m) for n, m in bb.named_modules() if m._forward_hooks or m._backward_hooks]
        want_images = torch.is_grad_enabled() and images.requires_grad
        if not hooked_any:
            return [], want_images
        served, _ = self._served_modules()
        hooked = []
        for name, m in hooked_any:
            if id(m) not in served:
                where = "cnn_encoder.backbone" + ("." + name if name else "")
                raise NotImplementedError(
                    f"a forward / backward hook on {where} is not served on the B200 path: hooks are served on "
                    "backbone.layer1 .. backbone.layer4 and on every Bottleneck backbone.layerN[i] (the intermediate "
                    "tensors of the stem, of a block's convolutions and of the pooling are never materialised)")
            hooked.append(served[id(m)])
        hooked.sort(key=lambda e: (e[1], -e[2]))
        return hooked, want_images

    def _data_grad(self, hooked, want_images, images):
        if images.dim() != 4:
            raise ValueError(f"images must be [B,3,H,W], got {tuple(images.shape)}")
        B, _, H, W = images.shape
        _, blocks = self._served_modules()
        geometry, c, h, w = [], 64, H // 4, W // 4
        for blk in blocks:
            s = blk.conv2.stride[0]
            co = blk.conv3.out_channels
            geometry.append((c, h, w, co, h // s, w // s))
            c, h, w = co, h // s, w // s
        return _DataGrad(hooked, want_images, geometry, B, H, W, images.device)

    def _train_options(self) -> Dict[str, float]:
        mc = self.text_encoder.model_config
        bn_train = any(m.training for m in self.cnn_encoder.backbone.modules()
                       if isinstance(m, nn.modules.batchnorm._BatchNorm))
        head_p = [m.p for m in self.classifier.classifier if isinstance(m, nn.Dropout)]
        return {
            "train.p_bert_hidden": float(getattr(mc, "hidden_dropout_prob", 0.0)),
            "train.p_bert_attn": float(getattr(mc, "attention_probs_dropout_prob", 0.0)),
            "train.p_text_out": float(self.text_encoder.dropout.p),
            "train.p_cnn_proj": float(self.cnn_encoder.projection[2].p),
            "train.p_fusion": float(self.fusion.fusion_layer.fusion[2].p),
            "train.p_head": float(head_p[0]) if head_p else 0.0,
            "train.pad_idx": float(getattr(mc, "pad_token_id", 0) or 0),
            "train.bn_train": 1.0 if bn_train else 0.0,
        }

    def _trainable(self):
        """[(canonical name, parameter)] the library differentiates; raises for what it cannot."""
        out = []
        for name, p in self._mrd_named():
            if not isinstance(p, nn.Parameter) or not p.requires_grad:
                continue
            if name.startswith("cnn_encoder.backbone."):
                raise NotImplementedError(
                    f"{name} requires grad: the B200 training step keeps the ResNet50 backbone frozen "
                    "(the reference default, src/config.py:64); backbone gradients are not implemented")
            if ".pooler." in name:
                continue   # unused with use_pooler_output=False: autograd leaves its .grad None as well
            out.append((name, p))
        return out

    def _forward_train(self, images, input_ids, attention_mask, return_embeddings, explain=None, dgrad=None):
        """Train-mode forward on the B200 path, differentiable through torch.autograd: the reference's
        training loops (src/train.py:247-333, src/train_multimodal.py:508-556) run unchanged.
        explain = a hooked backbone module: the same machinery in EVAL semantics (no dropout, BatchNorm on running
        statistics) with the module's hooks served - what Grad-CAM needs.
        dgrad = (hooked served modules, images.grad wanted): data gradients through the frozen backbone (input
        saliency, hooks on any stage or bottleneck) - in eval semantics under model.eval(), with dropout in train mode
        (where the backbone's BatchNorm must be in eval mode)."""
        p_att = {self.fusion.fusion_layer.image_to_text_attention.dropout.p,
                 self.fusion.fusion_layer.text_to_image_attention.dropout.p,
                 self.fusion.fusion_layer.fusion[2].p}
        if len(p_att) != 1:
            raise NotImplementedError("the fusion dropouts must share one probability (FusionConfig.dropout)")
        eng = self._engine(allow_training=True)
        opts = self._train_options()
        eval_semantics = explain is not None or (dgrad is not None and not self.training)
        want_images = dgrad is not None and dgrad[1]
        if dgrad is not None:
            if self.training and opts["train.bn_train"]:
                raise NotImplementedError(
                    "data gradients through the backbone (images.requires_grad, hooks below layer4) in train mode need "
                    "the backbone's BatchNorm layers in eval mode (running statistics: "
                    "model.cnn_encoder.backbone.eval()); batch-statistics BatchNorm is not differentiated")
            if eng.fp32_check:
                raise NotImplementedError("data gradients through the backbone are not implemented in the fp32 check "
                                          "mode (configure_b200(fp32_check=True)); switch it off")
            if self.__dict__.get("_mrd_ddp", (False, None))[0] and self.training:
                raise NotImplementedError("data gradients through the backbone are not implemented with "
                                          "data_parallel()")
        if eval_semantics:
            opts = {k: (v if k == "train.pad_idx" else 0.0) for k, v in opts.items()}
        if eng.train_opts != opts:
            # the cache of what was applied lives on the Engine: a new engine (model.to(other device), deepcopy,
            # unpickling) starts from the library defaults and gets every option again
            for k, v in opts.items():
                eng.set_option(k, v)
            # the optimizer rewrites the parameters every step: re-pack them in stream order instead of
            # stalling the host on a device synchronisation per step (the engine keeps the tensors alive)
            eng.set_option("load_sync", 0.0)
            eng.train_opts = dict(opts)
        named = self._trainable()
        if eval_semantics and not named and not want_images:
            raise RuntimeError("every parameter is frozen: logits.backward() has nothing to differentiate (the "
                               "reference raises here as well unless the input requires grad)")
        # eval semantics draw nothing from the generator (no dropout): leave torch's RNG stream untouched
        seed = 0 if eval_semantics else int(torch.randint(0, 2 ** 62, (1,)).item())   # CPU generator: follows torch.manual_seed
        shapes = tuple((n, tuple(p.shape)) for n, p in named)
        ddp = self.__dict__.get("_mrd_ddp", (False, None))
        if ddp[0]:
            # every rank usually runs under the same torch.manual_seed: without this all ranks would apply the
            # same dropout masks to their shards (masks are a pure function of seed, site and element index)
            from .parallel import rank_seed
            seed = rank_seed(seed, ddp[1])
        if eval_semantics:
            ddp = (False, None)
        emb_dims = ((self.cnn_encoder.embedding_dim, self.text_encoder.embedding_dim, self.fusion_dim)
                    if return_embeddings else None)
        dg = self._data_grad(dgrad[0], want_images, images) if dgrad is not None else None
        logits = _TrainStep.apply(eng, images, input_ids, attention_mask, seed, shapes,
                                  (self.num_classes, ddp[0], ddp[1], explain, emb_dims, dg), *[p for _, p in named])
        if opts["train.bn_train"]:
            # the library wrote the new running_mean / running_var straight into the BatchNorm buffers
            # (momentum 0.1, unbiased variance: nn.BatchNorm2d in train mode); the step counters and the
            # folded eval-mode copies of those statistics are bookkeeping on this side
            counters = [m.num_batches_tracked for m in self.cnn_encoder.backbone.modules()
                        if isinstance(m, nn.modules.batchnorm._BatchNorm) and m.num_batches_tracked is not None]
            if counters:
                torch._foreach_add_(counters, 1)
            eng.mark_dirty("cnn_encoder.backbone.")
            if ddp[0]:
                # DistributedDataParallel(broadcast_buffers=True) semantics: rank 0's running statistics are the
                # model's (each rank computed them from its own shard), so the ranks' eval-mode models and any
                # rank's checkpoint stay identical
                from .parallel import broadcast_buffers_
                broadcast_buffers_([b for m in self.cnn_encoder.backbone.modules()
                                    if isinstance(m, nn.modules.batchnorm._BatchNorm)
                                    for b in (m.running_mean, m.running_var) if b is not None], ddp[1])
        out = {"logits": logits, "probs": torch.softmax(logits, dim=-1)}
        if return_embeddings:
            # values of this forward (src/multimodal_classifier.py:168-175); gradients flow through the logits only
            img_e, txt_e, fused = eng.last_train_embeddings
            heads = self.config.fusion.num_attention_heads
            ones = torch.ones(logits.shape[0], heads, 1, 1, dtype=torch.float32, device=logits.device)
            out.update({"image_embedding": img_e, "text_embedding": txt_e, "fused_embedding": fused,
                        "attention_info": {"image_to_text_attention": ones, "text_to_image_attention": ones.clone()}})
        return out

    def data_parallel(self, enabled: bool = True, process_group=None) -> "MultimodalClassifier":
        """Training on several GPUs (one process per GPU, replicated parameters, each rank its own
        batch shard): average the parameter gradients over the ranks inside loss.backward() - bucketed
        all-reduces over NCCL (one bucket per backward stage), each started while the remaining stages are
        still running.  The caller keeps the ranks' parameters identical at the start (same seed or a
        broadcast), exactly as with DistributedDataParallel."""
        self.__dict__["_mrd_ddp"] = (bool(enabled), process_group)
        return self

    def predict(self, images, input_ids, attention_mask) -> Tuple[torch.Tensor, torch.Tensor]:
        self.eval()
        with torch.no_grad():
            probs = self.forward(images, input_ids, attention_mask)["probs"]
            confidence, predicted = torch.max(probs, dim=-1)
        return predicted, confidence

    def forward_host(self, images: torch.Tensor, input_ids: torch.Tensor,
                     attention_mask: Optional[torch.Tensor], micro_batch: int = 2048, *,
                     logits_out: Optional[torch.Tensor] = None, next_batch=None) -> Dict[str, torch.Tensor]:
        """forward() for batches that still live in HOST memory (what the reference's callers hold
        before `.to(device)`, src/train.py:252-255 / src/predict.py:220-238).

        The batch is cut into micro-batches; a copy stream moves micro-batch i+1 host->device (pinned
        memory makes the copies asynchronous) while the kernels of micro-batch i run, so the PCIe
        transfer (602 KB per image) hides behind the compute.  Returns device tensors like forward().
        micro_batch = 2048 by default (two 1.2 GB staging slots on the device): measured on a B200, 4096 samples per
        call, 256 / 512 / 1024 / 2048 rows per micro-batch give 32.9 / 35.3 / 35.9 / 36.9 k samples/s against
        36.0 - 37.2 k for inputs that are already resident - small passes lose tiles per SM in every kernel.

        next_batch = (images, input_ids, attention_mask) of the NEXT call (what a data loader already holds):
        its first micro-batch is copied while this call's last micro-batch computes, so the next call starts on
        data that is already on the device instead of exposing one H2D copy per call.  The tensors must be the
        very objects passed to the next call and must not be modified in between; anything else is ignored.
        """
        eng = self._engine()
        dev = eng.device
        B = images.shape[0]
        nc = self.num_classes
        logits = logits_out if logits_out is not None else torch.empty(B, nc, dtype=torch.float32, device=dev)
        probs = torch.empty(B, nc, dtype=torch.float32, device=dev)
        if B == 0:
            return {"logits": logits, "probs": probs}
        mb = max(1, min(micro_batch, B))
        main = torch.cuda.current_stream(dev)
        copy = self.__dict__.get("_mrd_copy_stream")
        if copy is None or copy.device != dev:
            copy = torch.cuda.Stream(dev)
            self.__dict__["_mrd_copy_stream"] = copy
        staged = [None, None]       # device copies of the two micro-batches in flight
        ready = [None, None]        # H2D finished
        free = [None, None]         # kernels that read the staging slot finished
        n_mb = -(-B // mb)

        def stage(imgs, ids_, mask_, lo, hi):
            """H2D of rows [lo, hi) on the copy stream (must be current) -> (device tensors, done event)."""
            m = None if mask_ is None else mask_[lo:hi].to(dev, non_blocking=True)
            t = (imgs[lo:hi].to(dev, non_blocking=True), ids_[lo:hi].to(dev, non_blocking=True), m)
            ev = torch.cuda.Event()
            ev.record(copy)
            return t, ev

        def issue_copy(i):
            slot = i & 1
            lo, hi = i * mb, min(B, (i + 1) * mb)
            with torch.cuda.stream(copy):
                if free[slot] is not None:
                    copy.wait_event(free[slot])
                staged[slot], ready[slot] = stage(images, input_ids, attention_mask, lo, hi)

        def batch_key(imgs, ids_, mask_, n, step):
            return (id(imgs), id(ids_), id(mask_), int(n), int(step), imgs.data_ptr(), ids_.data_ptr())

        pre = self.__dict__.pop("_mrd_prefetched", None)
        if pre is not None and pre["key"] == batch_key(images, input_ids, attention_mask, B, mb) and pre["dev"] == dev:
            staged[0], ready[0] = pre["tensors"], pre["event"]      # micro-batch 0 is already on its way
        else:
            copy.wait_stream(main)
            issue_copy(0)
        for i in range(n_mb):
            if i + 1 < n_mb:
                issue_copy(i + 1)
            elif next_batch is not None and next_batch[0].shape[0] > 0:
                nb_im, nb_ids, nb_mask = next_batch
                B2 = nb_im.shape[0]
                mb2 = max(1, min(micro_batch, B2))
                with torch.cuda.stream(copy):
                    tensors, ev = stage(nb_im, nb_ids, nb_mask, 0, min(B2, mb2))
                self.__dict__["_mrd_prefetched"] = {"key": batch_key(nb_im, nb_ids, nb_mask, B2, mb2), "dev": dev,
                                                    "tensors": tensors, "event": ev, "refs": next_batch}
            slot = i & 1
            lo, hi = i * mb, min(B, (i + 1) * mb)
            main.wait_event(ready[slot])
            im, ids, m = staged[slot]
            out = self.forward(im, ids, m, logits_out=logits[lo:hi])
            probs[lo:hi].copy_(out["probs"])
            for t in (im, ids, m):
                if t is not None:
                    t.record_stream(main)
            free[slot] = torch.cuda.Event()
            free[slot].record(main)
        return {"logits": logits, "probs": probs}


class ImageOnlyClassifier(B200Module):
    """src/multimodal_classifier.py:205-246."""

    _mrd_groups = {"cnn_encoder.": "cnn_encoder.", "classifier.": "classifier."}

    def __init__(self, config: Optional[Config] = None):
        super().__init__()
        config = get_config() if config is None else config
        self.cnn_encoder = CNNEncoder(config.cnn_encoder)
        self.classifier = ClassificationHead(config.cnn_encoder.embedding_dim,
                                             config.classifier.hidden_dims,
                                             config.classifier.num_classes,
                                             config.classifier.dropout, config.classifier.activation)

    def _mrd_options(self):
        return self.classifier._mrd_options()

    def forward(self, images: torch.Tensor) -> Dict[str, torch.Tensor]:
        eng = self._engine()
        emb, _, _ = eng.cnn_encoder(images, self.cnn_encoder.embedding_dim)
        logits, probs = eng.head(emb, self.classifier.num_classes)
        return {"logits": logits, "probs": probs}


class TextOnlyClassifier(B200Module):
    """src/multimodal_classifier.py:249-293."""

    _mrd_groups = {"text_encoder.": "text_encoder.", "classifier.": "classifier."}

    def __init__(self, config: Optional[Config] = None, *, random_init: bool = False):
        super().__init__()
        config = get_config() if config is None else config
        self.text_encoder = TextEncoder(config.text_encoder, random_init=random_init)
        self.classifier = ClassificationHead(config.text_encoder.embedding_dim,
                                             config.classifier.hidden_dims,
                                             config.classifier.num_classes,
                                             config.classifier.dropout, config.classifier.activation)

    def _mrd_options(self):
        opts = self.text_encoder._mrd_options()
        opts.update(self.classifier._mrd_options())
        return opts

    def forward(self, input_ids, attention_mask) -> Dict[str, torch.Tensor]:
        self.text_encoder._check()
        eng = self._engine()
        cls, _ = eng.text_encoder(input_ids, attention_mask, self.text_encoder.embedding_dim)
        logits, probs = eng.head(cls, self.classifier.num_classes)
        return {"logits": logits, "probs": probs}


def create_multimodal_classifier(num_classes: int = 10, cnn_backbone: str = "resnet50",
                                 text_model: str = "dmis-lab/biobert-base-cased-v1.2",
                                 fusion_type: str = "attention", **kwargs) -> MultimodalClassifier:
    cfg = get_config()
    cfg.classifier.num_classes = num_classes
    cfg.cnn_encoder.backbone = cnn_backbone
    cfg.text_encoder.model_name = text_model
    cfg.fusion.fusion_type = fusion_type
    return MultimodalClassifier(cfg, **kwargs)


def create_baseline_classifiers(config: Optional[Config] = None
                                ) -> Tuple[ImageOnlyClassifier, TextOnlyClassifier]:
    return ImageOnlyClassifier(config), TextOnlyClassifier(config)

"""TextEncoder - drop-in for the reference's src/text_encoder.py (BERT-base checkpoints).

Same constructor, attributes and parameter tree (`encoder.*` is a HuggingFace BertModel, exactly as
in src/text_encoder.py:46-47) and the same forward contract (src/text_encoder.py:95-127): CLS row of
the last hidden state, eval-mode dropout.  forward() runs the embedding+LayerNorm, tcgen05 GEMM,
fused attention and LayerNorm kernels of libmrd_b200.so; the HF module is only the parameter
container.
"""

from __future__ import annotations

from typing import Optional, Tuple

import torch
import torch.nn as nn

from ._module import B200Module
from .config import BIOBERT_BASE, TextEncoderConfig, get_config


def _build_hf_encoder(model_name: str, random_init: bool):
    from transformers import AutoConfig, AutoModel, BertConfig, BertModel

    if random_init:
        cfg = BertConfig(**BIOBERT_BASE)
        return cfg, BertModel(cfg)
    # reference behaviour (src/text_encoder.py:46-47); raises OSError when the hub is unreachable
    return AutoConfig.from_pretrained(model_name), AutoModel.from_pretrained(model_name)


class TextEncoder(B200Module):
    _mrd_groups = {"": "text_encoder."}

    def __init__(self, config: Optional[TextEncoderConfig] = None, *, random_init: bool = False):
        """random_init=True builds a BioBERT-base shaped encoder without fetching the checkpoint
        (benchmarks / tests on air-gapped machines); the default follows the reference."""
        super().__init__()
        config = get_config().text_encoder if config is None else config
        self.config = config
        self.model_name = config.model_name
        self.embedding_dim = config.embedding_dim
        self.max_length = config.max_length
        self.use_pooler_output = config.use_pooler_output
        self.model_config, self.encoder = _build_hf_encoder(self.model_name, random_init)
        mc = self.model_config
        if getattr(mc, "model_type", "bert") != "bert" or mc.hidden_size != 768 or \
                mc.num_attention_heads != 12 or getattr(mc, "hidden_act", "gelu") != "gelu":
            raise NotImplementedError(
                f"{self.model_name}: the B200 path covers BERT-base shaped encoders "
                "(hidden 768, 12 heads of 64, erf-GELU)")
        if mc.hidden_size != self.embedding_dim:
            self.embedding_dim = mc.hidden_size
        self.dropout = nn.Dropout(config.dropout)
        self.projection = None
        if config.freeze_embeddings:
            self._freeze_embeddings()
        if config.freeze_layers > 0:
            self._freeze_layers(config.freeze_layers)

    def _mrd_options(self):
        return {"bert_heads": self.model_config.num_attention_heads,
                "bert_ln_eps": self.model_config.layer_norm_eps}

    def _freeze_embeddings(self) -> None:
        self.encoder.embeddings.requires_grad_(False)

    def _freeze_layers(self, num_layers: int) -> None:
        for layer in list(self.encoder.encoder.layer)[:num_layers]:
            layer.requires_grad_(False)

    def _check(self):
        if self.use_pooler_output:
            raise NotImplementedError("use_pooler_output=True is outside the B200 hot path "
                                      "(the reference default is the CLS token, src/config.py:79)")
        if self.projection is not None:
            raise NotImplementedError("TextEncoder.projection is outside the B200 hot path")

    def forward(self, input_ids: torch.Tensor, attention_mask: torch.Tensor) -> torch.Tensor:
        """input_ids [B,S], attention_mask [B,S] (non-zero = attend) -> [B,768] fp32."""
        self._check()
        cls, _ = self._engine().text_encoder(input_ids, attention_mask, self.embedding_dim)
        return cls

    def get_all_hidden_states(self, input_ids, attention_mask) -> Tuple[torch.Tensor, tuple]:
        """(last_hidden_state [B,S,768], hidden_states) with hidden_states a tuple of L+1 tensors
        (embedding output, then every layer's output) - src/text_encoder.py:129-149.  Runs without
        token packing so padded positions are computed as in the reference."""
        self._check()
        n_layers = len(self.encoder.encoder.layer)
        _, last, stack = self._engine().text_encoder(input_ids, attention_mask, self.embedding_dim,
                                                     all_layers=n_layers)
        return last, tuple(stack.unbind(0))

    def get_last_hidden_state(self, input_ids, attention_mask) -> torch.Tensor:
        self._check()
        _, last = self._engine().text_encoder(input_ids, attention_mask, self.embedding_dim,
                                              want_hidden=True)
        return last

    def get_attention_weights(self, input_ids, attention_mask) -> Tuple[torch.Tensor, tuple]:
        """(embedding, attentions) - src/text_encoder.py:151-179.  What the reference returns depends on
        the attention backend of the HF encoder, and so does this:

        * "sdpa" (the default) or any other non-eager backend: HF ignores output_attentions, the
          attentions tuple is EMPTY, and the embedding is forward()'s.
        * "eager" (`encoder.set_attn_implementation("eager")` or `attn_implementation="eager"`): one fp32
          [B, heads, S, S] tensor per layer, views of one [layers, B, heads, S, S] buffer.  Element
          [b,h,q,k] = softmax_k(q.k/8 + mask bias) (HF:models/bert/modeling_bert.py:115-140, eval mode),
          for every query row, padded positions included; masked keys are exactly 0 and
          attention_mask=None attends every key.  The embedding is bitwise what forward() returns.
          A sample without any attended key gets all-zero rows, not HF's uniform 1/S rows: the B200
          forward gives such a sample a zero attention output, and the probabilities agree with it.
          Memory: layers * B * heads * S^2 * 4 bytes (as in the reference), e.g. 604 MB for B=64, S=128
          and 9.7 GB for B=64, S=512 with BERT-base.

        Eval mode only (train mode raises NotImplementedError, like every accessor here)."""
        if getattr(self.encoder.config, "_attn_implementation", None) != "eager":
            return self.forward(input_ids, attention_mask), ()
        self._check()
        eng = self._engine()
        cfg = self.encoder.config
        cls, _, attn = eng.text_encoder(input_ids, attention_mask, self.embedding_dim, want_attn=True,
                                        layers=len(self.encoder.encoder.layer), heads=cfg.num_attention_heads)
        return cls, tuple(attn.unbind(0))


class BioBERTEncoder(TextEncoder):
    def __init__(self, embedding_dim: int = 768, max_length: int = 128, dropout: float = 0.1,
                 freeze_layers: int = 0, **kw):
        super().__init__(TextEncoderConfig(model_name="dmis-lab/biobert-base-cased-v1.2",
                                           embedding_dim=embedding_dim, max_length=max_length,
                                           dropout=dropout, freeze_layers=freeze_layers), **kw)


def create_text_encoder(model_name: str = "dmis-lab/biobert-base-cased-v1.2",
                        output_dim: Optional[int] = None, **kwargs) -> TextEncoder:
    """Factory with the reference's signature (src/text_encoder.py:272-294)."""
    if output_dim is not None:
        raise NotImplementedError("TextEncoderWithProjection is outside the B200 hot path")
    random_init = kwargs.pop("random_init", False)
    return TextEncoder(TextEncoderConfig(model_name=model_name, **kwargs), random_init=random_init)


def get_tokenizer(model_name: str = "dmis-lab/biobert-base-cased-v1.2"):
    """Tokenisation stays in the reference's stack (HF tokenizers)."""
    from transformers import AutoTokenizer

    return AutoTokenizer.from_pretrained(model_name)

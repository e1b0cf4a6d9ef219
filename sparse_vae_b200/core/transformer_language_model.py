"""`TransformerLanguageModel` (reference surface: sparse_vae/core/transformer_language_model.py): embeddings,
the stack of causal (block-sparse) decoder layers and the tied output head.  Parameter names match the
reference's state_dict (`input_layer.0`, `output_layer.{0,2,3}`, `decoder_layers.N...`)."""
from __future__ import annotations

from copy import deepcopy
from dataclasses import dataclass
from typing import Dict, Optional

import torch
from torch import nn, Tensor

from . import decode
from .attention import Attention, TransformerLayer
from .embedding import Embedding
from .gelu import GELU
from .generation import GenerationState
from .language_model import LanguageModel, LanguageModelHparams
from .layer_norm import LayerNorm
from .linear import Linear
from .lightning_shim import DictConfig
from .padded_tensor import split_padding
from .rotary_embedding import RotaryEmbedding

VOCAB_SIZE = 2 ** 15


@dataclass
class TransformerHparams(LanguageModelHparams):
    d_embedding: Optional[int] = None       # d_model if None
    d_model: int = 512
    num_heads: int = 8
    num_layers: int = 6
    input_dropout: float = 0.0

    tie_embedding_weights: bool = True

    cross_attention: bool = False
    grad_checkpointing: bool = False
    separate_context_embedding: bool = True

    attn_window_size: int = 4
    sparse_self_attention: bool = True


class TransformerLanguageModel(LanguageModel):
    def __init__(self, hparams: DictConfig):
        super().__init__(hparams)
        hp = self.hparams
        d_model = hp.d_model
        d_embedding = hp.d_embedding or d_model

        embedding = Embedding(VOCAB_SIZE, d_embedding)
        layers = [embedding, nn.Dropout(p=hp.input_dropout)]
        if d_embedding != d_model:
            layers.insert(1, nn.Linear(d_embedding, d_model))
        self.input_layer = nn.Sequential(*layers)
        self.context_layer = deepcopy(self.input_layer) if hp.cross_attention and hp.separate_context_embedding else None

        logits = nn.Linear(d_model, VOCAB_SIZE)
        self.output_layer = nn.Sequential(Linear(d_model, d_model), GELU(), LayerNorm(d_model), logits)
        if hp.tie_embedding_weights and d_embedding == d_model:
            logits.weight = embedding.weight

        with RotaryEmbedding.embedding_context(d_model):
            self.decoder_layers = nn.ModuleList(
                TransformerLayer(d_model, hp.num_heads, causal=True, use_cross_attention=hp.cross_attention,
                                 sparse_self_attention=hp.attn_window_size if hp.sparse_self_attention else False)
                for _ in range(hp.num_layers))

    def embed_context(self, context: Tensor):
        return self.context_layer(context) if self.context_layer else self.input_layer(context)

    def forward(self, batch: Dict[str, Tensor]):
        tokens, padding = split_padding(batch['token_ids'])
        if batch.get('context') is not None:
            raise NotImplementedError
        x = self.input_layer(tokens.long())
        for layer in self.decoder_layers:
            x = layer(x, padding=padding)
        return self.output_layer(x)

    @torch.no_grad()
    def sample(self, max_length: int, batch_size: int = 1, context: Tensor = None, z: Tensor = None, **kwargs):
        context = self.embed_context(context) if context is not None else None
        state = GenerationState(max_length, batch_size, self.start_token, self.end_token, device=self.device, **kwargs)
        state.output_ids[:, 0] = self.start_token
        # after the first token (which allocates the caches) every token is one graph replay (core/decode.py), as in
        # TransformerVAE.sample; z or context added to the input keep the module-by-module sampler
        graphed = z is None and context is None and decode.supported(self, state)
        with Attention.kv_cache(max_length):
            while not state.should_stop():
                x = self.input_layer(state.prev_tokens())
                if z is not None:
                    x = x + z[state.live_sample_mask, :]
                for layer in self.decoder_layers:
                    x = layer(x, context=context)
                Attention.update_kv_cache(state.process_logits(self.output_layer(x.squeeze(1))))
                if graphed:
                    decode.GraphedDecoder(self, state, decode.TRACE).run()
                    break
        return state.final_output()

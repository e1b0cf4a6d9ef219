"""`Attention`, `TransformerLayer`, `Perceiver`: the callers of the sparse-attention hot path.

Surface and arithmetic follow the reference (sparse_vae/core/attention.py:11-208, core/transformer_layer.py:4-61,
core/perceiver.py:5-50): same constructor arguments, parameter / state_dict names (`q_linear`, `k_linear`,
`v_linear`, `output_linear`, `pos_linear`, `learned_queries`, `attn_layer_norm`, `ffn`, ...), rotary position
encoding on the full d_model before the head split with max_pos = 2*window*block for sparse layers, additive
-1e7 key-padding mask, KV cache for autoregressive sampling.  Differences are mechanical:
  * the padding mask may be passed explicitly (`padding=`) so the model can run on plain tensors; a
    `PaddedTensor` key still works exactly like in the reference (mask read off `k.padding`);
  * the sparse branch calls the fused sm_100a kernel and gets its result already laid out as [B, L, H*Dh].
"""
from __future__ import annotations

from contextlib import contextmanager
from typing import Optional, Set, Tuple, Union

import torch
import torch.nn.functional as F
from torch import nn, Tensor

from .. import _native as N
from .layer_norm import LayerNorm
from .gelu import GELU, ffn_forward
from .linear import Linear, linear3, qkv_rotary
from .padded_tensor import split_padding
from . import causal_attention, cross_attention
from .residual import residual_add, residual_dropout_add
from .rotary_embedding import RotaryEmbedding
from .sparse_attention import SparseAttention


def _rotary_tables(length: int, half: int, start: int, max_pos: int, dtype, device) -> Tuple[Tensor, Tensor]:
    """cos / sin of pos * max_pos**(-i/half), every intermediate in `dtype` exactly as the reference evaluates it
    (core/attention.py:196-199: positions, frequencies, angles rounded to the activation dtype)."""
    freq = torch.arange(half, dtype=dtype, device=device)
    pos = torch.arange(start, start + length, dtype=dtype, device=device)
    angle = pos[:, None] * (max_pos ** (-freq / half))
    return angle.cos(), angle.sin()


_TABLE_CACHE: dict = {}


def _cached_tables(length, half, start, max_pos, dtype, device):
    if start != 0:                       # token-by-token decoding: one row, not worth caching
        return _rotary_tables(length, half, start, max_pos, dtype, device)
    # under autocast `max_pos ** t` is an fp32 op, so the tables (and the reference's products) are fp32
    key = (length, half, max_pos, dtype, device, torch.is_autocast_enabled('cuda'))
    hit = _TABLE_CACHE.get(key)
    if hit is None:
        if len(_TABLE_CACHE) >= 16:
            _TABLE_CACHE.clear()
        hit = _TABLE_CACHE[key] = tuple(t.contiguous() for t in _rotary_tables(length, half, 0, max_pos, dtype, device))
    return hit


class _RotaryFn(torch.autograd.Function):
    """One-launch rotation (csrc/rotary.cu), forward and backward bit-identical to the reference's op sequence."""

    @staticmethod
    def forward(ctx, x: Tensor, cos: Tensor, sin: Tensor):
        x = x.contiguous()
        out = torch.empty_like(x)
        L, d = x.shape[-2], x.shape[-1]
        N.check(N.lib.svae_rotary(x.data_ptr(), cos.data_ptr(), sin.data_ptr(), out.data_ptr(), N.svae_dtype(x.dtype),
                                  N.svae_dtype(cos.dtype), x.numel() // d, L, d, 0, N.current_stream(x.device)), 'svae_rotary')
        ctx.save_for_backward(cos, sin)
        return out

    @staticmethod
    def backward(ctx, g: Tensor):
        cos, sin = ctx.saved_tensors
        g = g.contiguous()
        dx = torch.empty_like(g)
        L, d = g.shape[-2], g.shape[-1]
        N.check(N.lib.svae_rotary(g.data_ptr(), cos.data_ptr(), sin.data_ptr(), dx.data_ptr(), N.svae_dtype(g.dtype),
                                  N.svae_dtype(cos.dtype), g.numel() // d, L, d, 1, N.current_stream(g.device)), 'svae_rotary')
        return dx, None, None


def encode_position_rotary(x: Tensor, start: int = 0, max_pos: int = 10000) -> Tensor:
    """Rotate consecutive feature pairs of x[..., pos, :] by pos * max_pos**(-i/(d/2)).

    Evaluated in x.dtype like the reference (core/attention.py:194-208), so low-precision position rounding is
    reproduced op for op: (x0*cos - x1*sin, x1*cos + x0*sin) with one rounding per product and per sum.  CUDA
    tensors take the single-launch kernel; the torch expression below is the same arithmetic for CPU tensors.
    Under autocast the reference's result is fp32 (promoted by the fp32 cos / sin) and every consumer casts it to
    the autocast dtype at once; the kernel returns that rounded tensor directly.
    """
    half = x.shape[-1] // 2
    if (N.FUSED_EXTRAS and x.is_cuda and x.ndim >= 2 and x.shape[-1] % 8 == 0 and x.numel() > 0
            and x.dtype in (torch.float32, torch.bfloat16, torch.float16)):
        cos, sin = _cached_tables(x.shape[-2], half, start, max_pos, x.dtype, x.device)
        if cos.dtype == x.dtype or cos.dtype == torch.float32:
            return _RotaryFn.apply(x, cos.contiguous(), sin.contiguous())
    cos, sin = _rotary_tables(x.shape[-2], half, start, max_pos, x.dtype, x.device)
    pairs = x.unflatten(-1, (half, 2))
    even, odd = pairs[..., 0], pairs[..., 1]
    rotated = torch.stack((even * cos - odd * sin, odd * cos + even * sin), dim=-1)
    return rotated.flatten(-2)


class Attention(nn.Module):
    # class-level KV-cache switch, as in the reference (core/attention.py:144-168)
    kv_cache_length: Optional[int] = None
    live_attention_modules: Optional[Set['Attention']] = None

    def __init__(self, d_model: int, num_heads: int, causal=False, sparse: Union[bool, int] = False,
                 learned_queries: int = None, max_length: int = 10000):
        super().__init__()
        assert d_model % num_heads == 0, "num_heads must divide d_model evenly"
        self.causal, self.d_model, self.num_heads, self.max_length = causal, d_model, num_heads, max_length

        if learned_queries:
            self.learned_queries = nn.Parameter(torch.randn(1, learned_queries, d_model))
        else:
            self.q_linear = Linear(d_model, d_model)
            self.learned_queries = None
        self.k_linear = Linear(d_model, d_model)
        self.v_linear = Linear(d_model, d_model)
        self.output_linear = Linear(d_model, d_model)
        self.pos_linear = Linear(d_model, d_model)      # present (and unused) in the reference; kept for checkpoints

        self.cache_index = 0
        self.key_cache = None
        self.value_cache = None
        # `isinstance(True, int)` holds, so sparse=True selects window_size=True (== 1) exactly like the reference
        self.sparse_attention = SparseAttention(window_size=sparse if isinstance(sparse, int) else 4) if sparse else None

    def forward(self, q: Optional[Tensor], k: Tensor, v: Tensor, padding: Optional[Tensor] = None) -> Tensor:
        sparse = self.sparse_attention
        max_pos = self.max_length if not sparse else 2 * sparse.window_size * sparse.block_size
        k, k_pad = split_padding(k)
        v, _ = split_padding(v)
        if padding is None:
            padding = k_pad

        fused = None
        if self.learned_queries is not None:
            q = self.learned_queries.expand(k.shape[0], *self.learned_queries.shape[1:])
            k, v = self.k_linear(k), self.v_linear(v)
        else:
            q, _ = split_padding(q)
            if q is k and k is v and self.q_linear.bias is not None:        # self-attention: one input, three projections
                if (N.FUSED_EXTRAS and q.is_cuda and self.cache_index == 0 and not self.kv_cache_length and q.ndim >= 2
                        and torch.is_autocast_enabled('cuda')):
                    # projections + rotary as one node (one rotation launch for q and k; its backward also yields the
                    # q / k bias gradients)
                    cos, sin = _cached_tables(q.shape[-2], q.shape[-1] // 2, 0, max_pos, torch.get_autocast_dtype('cuda'), q.device)
                    fused = qkv_rotary(q, self.q_linear, self.k_linear, self.v_linear, cos, sin)
                if fused is None:
                    q, k, v = linear3(q, self.q_linear, self.k_linear, self.v_linear)
            else:
                q, k, v = self.q_linear(q), self.k_linear(k), self.v_linear(v)
            if fused is not None:
                q, k, v = fused
            else:
                q = encode_position_rotary(q, self.cache_index, max_pos=max_pos)
        if fused is None:
            k = encode_position_rotary(k, self.cache_index, max_pos=max_pos)
        if self.kv_cache_length:
            k, v = self._update_kv_cache(k, v)
        if padding is not None and padding.shape[-1] != k.shape[-2]:
            padding = None                                  # mask no longer fits (PaddedTensor.padding semantics)

        H = self.num_heads
        q, k, v = (t.unflatten(-1, (H, -1)).transpose(-2, -3) for t in (q, k, v))      # [..., H, L, Dh] views

        if sparse and self.key_cache is None:
            kpm = padding * -1e7 if padding is not None else None
            out = sparse(q, k, v, key_padding_mask=kpm, joint_grads=fused is not None)  # [B, H, L, Dh] over [B, L, H, Dh]
        elif (N.FUSED_EXTRAS and self.causal and self.key_cache is None and padding is not None and padding.ndim == 2
              and causal_attention.supported(q, k, v)):
            # dense causal self-attention of a padded training batch (the non-sparse decoders): the tcgen05 kernels of
            # csrc/causal_attn_sm100.cu instead of the explicit [B, H, L, L] form below; same additive -1e7 mask
            out = causal_attention.causal_attention(q, k, v, padding * -1e7, joint_grads=fused is not None)
        elif (N.FUSED_EXTRAS and not self.causal and self.key_cache is None and (padding is None or padding.ndim == 2)
              and cross_attention.supported(q, k, v)):
            # the Perceiver encoder's learned queries (<= 64) over the whole sequence: K and V streamed once through
            # the tcgen05 kernels of csrc/xattn_sm100.cu, the keys split across CTAs when the batch has few (batch, head)
            # pairs; the additive mask is the reference's float32 -1e7
            out = cross_attention.cross_attention(q, k, v, None if padding is None else padding * -1e7, key_splits=None)
        elif (N.FUSED_EXTRAS and q.is_cuda and self.key_cache is None and q.ndim == 4
              and (padding is None or (padding.ndim == 2 and not self.causal))):
            # Dense attention of the Perceiver encoder (64 learned queries over the whole sequence) and of non-sparse
            # decoders: same arithmetic -- softmax(q k^T / sqrt(d) - 1e7 * mask) v -- through the library's fused
            # kernel, which reads the strided head views directly (the explicit form copies k^T and v per call).
            # the reference subtracts a float32 1e7 from promoted scores; in fp16 that constant would become -inf and a
            # fully padded row NaN, so the bias is clamped to the dtype's finite range before the cast
            bias = None if padding is None else (padding[:, None, None, :] * -1e7).clamp_min(torch.finfo(q.dtype).min).to(q.dtype)
            out = F.scaled_dot_product_attention(q, k, v, attn_mask=bias, is_causal=self.causal and bias is None)
        else:
            scores = q @ k.transpose(-1, -2) * k.shape[-1] ** -0.5
            mask = padding[..., None, None, :] if padding is not None and padding.ndim >= 2 else padding
            if self.causal and self.key_cache is None:
                q_len = q.shape[-2]
                causal_mask = torch.ones(q_len, q_len, device=q.device, dtype=torch.bool).triu(1)
                mask = mask | causal_mask if mask is not None else causal_mask
            if mask is not None:
                scores = scores - mask * 1e7
            out = scores.softmax(dim=-1) @ v

        out = out.transpose(-2, -3).flatten(-2)             # a view when `out` came from the fused kernel
        return self.output_linear(out)

    # ---- KV cache for token-by-token decoding (reference core/attention.py:107-168) ---------------------------
    def _update_kv_cache(self, k, v) -> Tuple[Tensor, Tensor]:
        self.live_attention_modules.add(self)
        cfg = self.sparse_attention
        if cfg:
            # only keys that can still be attended are kept: the global block plus `window` sliding blocks
            block = cfg.block_size
            cache_len = (cfg.window_size + int(cfg.include_cls)) * block
            keep = int(cfg.include_cls) * block
        else:
            block, cache_len, keep = 0, self.kv_cache_length, 0

        if self.key_cache is None:
            self.key_cache = k.new_zeros([k.shape[0], cache_len, k.shape[-1]])
            self.value_cache = v.new_zeros([v.shape[0], cache_len, v.shape[-1]])

        if cfg and self.cache_index >= cache_len:
            within = self.cache_index % block
            slot = cache_len - block + within
            if within == 0:      # slide the window one block to the left, dropping its oldest block
                self.key_cache[:, keep:slot] = self.key_cache[:, keep + block:].clone()
                self.value_cache[:, keep:slot] = self.value_cache[:, keep + block:].clone()
        else:
            slot = self.cache_index

        self.key_cache[:, slot] = k.squeeze(-2)
        self.value_cache[:, slot] = v.squeeze(-2)
        self.cache_index += 1
        return self.key_cache[:, :slot + 1], self.value_cache[:, :slot + 1]

    @classmethod
    @contextmanager
    def kv_cache(cls, max_seq_length: int):
        cls.kv_cache_length = max_seq_length
        cls.live_attention_modules = set()
        try:
            yield
        finally:
            cls.kv_cache_length = None
            for module in cls.live_attention_modules:
                module.cache_index = 0
                module.key_cache = None
                module.value_cache = None
            cls.live_attention_modules = None

    @classmethod
    def update_kv_cache(cls, live_sample_mask: Tensor):
        for module in cls.live_attention_modules:
            module.key_cache = module.key_cache[live_sample_mask, ...]
            module.value_cache = module.value_cache[live_sample_mask, ...]


class TransformerLayer(nn.Module):
    """Pre-LayerNorm block: attention (+ optional cross-attention) and a 4x GELU feed-forward."""

    def __init__(self, d_model: int, num_heads: int, causal: bool = False, use_cross_attention: bool = False,
                 sparse_self_attention: Union[bool, int] = False, learned_queries: int = None):
        super().__init__()
        self.attention = Attention(d_model, num_heads, causal, learned_queries=learned_queries, sparse=sparse_self_attention)
        self.ffn = nn.Sequential(Linear(d_model, d_model * 4), GELU(), Linear(d_model * 4, d_model, bias=False))
        self.dropout = nn.Dropout(p=0.1)
        self.attn_layer_norm = LayerNorm(d_model)
        self.ffn_layer_norm = LayerNorm(d_model)
        self.use_cross_attention = use_cross_attention

    @property
    def use_cross_attention(self):
        return bool(self.cross_attention)

    @use_cross_attention.setter
    def use_cross_attention(self, value: bool):
        if value:
            base = self.attention
            self.cross_attention = Attention(d_model=base.d_model, num_heads=base.num_heads)
            self.cross_attn_layer_norm = LayerNorm(base.d_model)
            self.context_layer_norm = LayerNorm(base.d_model)
        else:
            self.cross_attention = None

    def forward(self, x: Tensor, context: Tensor = None, padding: Optional[Tensor] = None,
                context_padding: Optional[Tensor] = None) -> Tensor:
        x, x_pad = split_padding(x)
        padding = x_pad if padding is None else padding
        if self.attention.learned_queries is None:
            x, h = self.attn_layer_norm.fork(x)              # x feeds the norm AND the residual around the attention
        else:
            h = self.attn_layer_norm(x)
        h = self.attention(h, h, h, padding=padding)
        if x.shape == h.shape and not (self.cross_attention and context is not None):
            x, h = self.ffn_layer_norm.add_fork(x, h)        # x = x + h and the feed-forward norm, one launch
            return residual_dropout_add(x, ffn_forward(self.ffn, h), self.dropout)
        x = residual_add(x, h) if x.shape == h.shape else h  # learned queries change the length: no residual

        if self.cross_attention and context is not None:
            context, c_pad = split_padding(context)
            context_padding = c_pad if context_padding is None else context_padding
            h = self.cross_attention(self.cross_attn_layer_norm(x), *(self.context_layer_norm(context),) * 2,
                                     padding=context_padding)
            x = residual_add(x, h)

        x, h = self.ffn_layer_norm.fork(x)
        return residual_dropout_add(x, ffn_forward(self.ffn, h), self.dropout)


class Perceiver(nn.Module):
    """Dense learned-query encoder (reference core/perceiver.py): L tokens -> num_latents -> bottleneck_width."""

    def __init__(self, num_layers: int, num_latents: int, d_model: int, bottleneck_width: Optional[int] = None,
                 self_attention_layers: int = 1):
        super().__init__()
        assert num_layers > 1
        num_heads = d_model // 64

        with RotaryEmbedding.embedding_context(d_model):
            self.first_layer = TransformerLayer(d_model, num_heads, learned_queries=num_latents)
            if bottleneck_width:
                self.bottleneck = TransformerLayer(d_model, num_heads, learned_queries=bottleneck_width)
                num_layers -= 1
            else:
                self.bottleneck = None
            self.middle_layers = nn.ModuleList(
                TransformerLayer(d_model, num_heads, use_cross_attention=True) for _ in range(num_layers - 1))

    def forward(self, x: Tensor, padding: Optional[Tensor] = None):
        x, x_pad = split_padding(x)
        padding = x_pad if padding is None else padding
        z = self.first_layer(x, padding=padding)
        for layer in self.middle_layers:
            z = layer(z, context=x, padding=padding, context_padding=padding)   # self-attn mask dropped unless it fits
        if self.bottleneck:
            z = self.bottleneck(z, padding=padding)
        return z

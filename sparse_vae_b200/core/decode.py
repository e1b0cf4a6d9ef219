"""CUDA-graphed token-by-token decoding for `TransformerVAE.sample` and `TransformerLanguageModel.sample` (SURVEY.md
section 8f row 3).

The reference's sampler (transformer_vae.py:112-126 driving core/attention.py:107-168 and core/generation.py:30-77)
issues ~400 small launches per token and synchronises with the host several times per token (boolean-mask indexing,
`live_sample_mask.any()`); at 256 samples it is launch-bound (5.9 ms per token on a B200).  Here one token of the
whole decoder is ONE graph replay:

  * every position-dependent quantity (previous-token column, rotary angle, cache slot, repetition-penalty window,
    output column) is read from device counters that the graph itself advances;
  * each sparse-attention layer is one launch of `svae_decode_attn` (csrc/decode_attn.cu): rotary + cache append +
    attention over the visible keys; q / k / v come from one fused [3D, D] projection;
  * each dense causal layer (`sparse_self_attention=False`) is one call of `svae_decode_attn_dense`
    (csrc/decode_attn_dense.cu): the same over the reference's growing [B, max_length, D] cache, split-KV;
  * `GenerationState.process_logits` is restated with fixed shapes (same ops, same order, same RNG consumption).

  * with the reference's default settings (nucleus sampling) the sampler itself is one launch (csrc/sampling.cu):
    threshold search instead of a full sort; same token distribution, its own use of the random stream.

Finished samples leave the batch like in the reference (their cache rows are dropped and the rest is compacted,
`Attention.update_kv_cache`; a dense layer's cache only over the slots written so far) -- but not after every token:
they first stay behind as dead rows (nothing written, not counted again) and the batch is compacted and the graph
re-captured once a quarter of it is dead (`COMPACT_BELOW`).
The first token (position 0, where every layer's input is its own projection of z) runs through the unfused modules,
which also allocates the caches.
Weights are frozen while sampling: they are cast to the autocast dtype once per call instead of once per token.
"""
from __future__ import annotations

from typing import List, Optional

import torch
import torch.nn.functional as F
from torch import Tensor

from .. import _native as N
from .attention import Attention, _rotary_tables
from .generation import GenerationState

PENALTY_WINDOW = 512            # core/generation.py:44 -- repetition penalty looks at the last 512 tokens
TRACE: Optional[list] = None    # tests: set to a list to receive (live row indices, logits) of every graphed step
# Finished samples are dropped from the batch (reference: after every token, core/attention.py:164-168) once the live
# ones are at most this fraction of the captured batch; 1.0 = compact (and re-capture) whenever a sample finishes.
COMPACT_BELOW = 0.75
# tokens generated between two looks of the host at the number of live samples (one replay each, back to back)
CHECK_EVERY = 8


def attention_kind(layer, cache_len: int) -> Optional[str]:
    """How one decoder layer's self-attention is decoded by the graphed sampler: 'sparse' (`svae_decode_attn` over the
    ring cache), 'dense' (`svae_decode_attn_dense` over the reference's [B, cache_len, D] cache) or None (not covered:
    cross-attention, learned queries, non-causal attention or an unsupported head size / length)."""
    attn = layer.attention
    if layer.cross_attention is not None or attn.learned_queries is not None:
        return None
    head_dim = attn.d_model // attn.num_heads
    cfg = attn.sparse_attention
    if cfg is None:
        return 'dense' if attn.causal and N.lib.svae_decode_attn_dense_supported(head_dim, cache_len) else None
    if cfg.causal and cfg.include_cls and N.lib.svae_decode_attn_supported(head_dim, int(cfg.window_size), cfg.block_size):
        return 'sparse'
    return None


def supported(model, state: GenerationState) -> bool:
    """Graphed decoding covers CUDA models whose every decoder layer is causal self-attention without cross-attention,
    either block-sparse (global first block, head size 32, 64 or 128) or dense (head size 32, 64 or 128).  Anything else
    keeps the module-by-module sampler."""
    if not (N.FUSED_EXTRAS and model.device.type == 'cuda' and len(model.decoder_layers) > 0):
        return False
    if len(model.input_layer) != 2 or state.output_ids.dtype != torch.long:
        return False
    return all(attention_kind(layer, state.output_ids.shape[1]) is not None for layer in model.decoder_layers)


class _LayerWeights:
    """One decoder layer's matrices in the activation dtype, q / k / v stacked into one projection."""

    def __init__(self, layer, dtype):
        a = layer.attention
        self.wqkv = torch.cat([a.q_linear.weight, a.k_linear.weight, a.v_linear.weight]).to(dtype)
        self.bqkv = torch.cat([a.q_linear.bias, a.k_linear.bias, a.v_linear.bias]).to(dtype)
        self.wo, self.bo = a.output_linear.weight.to(dtype), a.output_linear.bias.to(dtype)
        self.w1, self.b1 = layer.ffn[0].weight.to(dtype), layer.ffn[0].bias.to(dtype)
        self.w2 = layer.ffn[2].weight.to(dtype)


class GraphedDecoder:
    """Owns the device counters, the pre-cast weights and the captured graph for the current live batch."""

    def __init__(self, model, state: GenerationState, trace_logits: Optional[List[Tensor]] = None):
        self.model, self.state = model, state
        dev = model.device
        self.dtype = torch.get_autocast_dtype('cuda') if torch.is_autocast_enabled('cuda') else torch.float32
        self.max_length = state.output_ids.shape[1]
        # per layer: 'sparse' or 'dense' (tests read this), and the rotary tables of its max_pos -- 2*window*block for
        # sparse layers, attn.max_length for dense ones; row p = the one-row table the reference builds at offset p
        # (positions rounded to the activation dtype)
        self.attention_kinds = [attention_kind(layer, self.max_length) for layer in model.decoder_layers]
        tables = {}
        self.tables = []
        for layer, kind in zip(model.decoder_layers, self.attention_kinds):
            attn = layer.attention
            cfg = attn.sparse_attention
            max_pos = 2 * int(cfg.window_size) * cfg.block_size if kind == 'sparse' else attn.max_length
            if max_pos not in tables:
                cos, sin = _rotary_tables(self.max_length, attn.d_model // 2, 0, max_pos, self.dtype, dev)
                tables[max_pos] = (cos.float().contiguous(), sin.float().contiguous())
            self.tables.append(tables[max_pos])
        self.workspace = None       # split-KV partials of the dense layers, sized for the captured batch
        self.layers = [_LayerWeights(layer, self.dtype) for layer in model.decoder_layers]
        head = model.output_layer
        self.head_w0, self.head_b0 = head[0].weight.to(self.dtype), head[0].bias.to(self.dtype)
        self.head_w3, self.head_b3 = head[3].weight.to(self.dtype), head[3].bias.to(self.dtype)
        self.position = torch.zeros(1, dtype=torch.int32, device=dev)       # cache_index of the token being fed
        self.column = torch.zeros(1, 1, dtype=torch.long, device=dev)       # GenerationState.current_index
        self.window_offsets = torch.arange(-PENALTY_WINDOW, 0, device=dev)[None]
        self.finished = torch.zeros(1, dtype=torch.int32, device=dev)
        self.finished_host = torch.zeros(1, dtype=torch.int32).pin_memory()
        self.alive_host = torch.zeros(1, dtype=torch.int64).pin_memory()
        self.trace = trace_logits
        vocab = self.head_w3.shape[0]
        # the reference's default decoding (nucleus sampling, no top-k) has a one-launch sampler; greedy / top-k
        # decoding keeps the ATen op sequence of core/generation.py
        self.fused_sampler = bool(state.temperature > 0.0 and state.top_k == 0 and self.dtype != torch.float32 and
                                  N.lib.svae_sample_top_p_supported(vocab, N.svae_dtype(self.dtype)))
        self.graph = None
        self.rows = None            # indices of the live samples in state.output_ids
        self.ids = None             # [live, max_length] working copy of their rows
        self.alive = None           # [captured batch] bool: still generating
        self.replays = 0
        self.captures = 0

    # ---- one token, fixed shapes (this is what gets captured) ------------------------------------------------
    def _attend(self, i: int, module: Attention, w: _LayerWeights, h: Tensor) -> Tensor:
        B, D = h.shape[0], module.d_model
        heads = module.num_heads
        head_dim = D // heads
        qkv = F.linear(h, w.wqkv, w.bqkv)                                   # [B, 1, 3D]
        out = torch.empty(B, 1, D, dtype=qkv.dtype, device=qkv.device)
        flat = qkv.view(B, 3 * D)
        cos, sin = self.tables[i]
        stream = N.current_stream(qkv.device)
        if self.attention_kinds[i] == 'dense':
            N.check(N.lib.svae_decode_attn_dense(
                flat[:, :D].data_ptr(), flat[:, D:2 * D].data_ptr(), flat[:, 2 * D:].data_ptr(), cos.data_ptr(),
                sin.data_ptr(), module.key_cache.data_ptr(), module.value_cache.data_ptr(), out.data_ptr(),
                self.position.data_ptr(), N.ptr(self.workspace), self.workspace.numel(), B, heads, head_dim,
                module.key_cache.shape[1], cos.shape[0], 3 * D, N.svae_dtype(qkv.dtype), float(head_dim ** -0.5),
                stream), 'svae_decode_attn_dense')
        else:
            cfg = module.sparse_attention
            N.check(N.lib.svae_decode_attn(flat[:, :D].data_ptr(), flat[:, D:2 * D].data_ptr(), flat[:, 2 * D:].data_ptr(),
                                           cos.data_ptr(), sin.data_ptr(), module.key_cache.data_ptr(),
                                           module.value_cache.data_ptr(), out.data_ptr(), self.position.data_ptr(), B,
                                           heads, head_dim, int(cfg.window_size), cfg.block_size, self.max_length, 3 * D,
                                           N.svae_dtype(qkv.dtype), float(head_dim ** -0.5), stream), 'svae_decode_attn')
        return F.linear(out, w.wo, w.bo)

    def _add_norm(self, x: Tensor, h: Tensor, norm) -> Tensor:
        """x += h (in place, fp32) and LayerNorm(x) in the activation dtype: one launch for the residual update and
        the next sub-layer's norm (reference core/transformer_layer.py:35-61)."""
        n = x.shape[-1]
        if not (norm.elementwise_affine and norm.weight.dtype == torch.float32 and h.dtype == self.dtype
                and h.is_contiguous() and N.lib.svae_layernorm_supported(n)):
            x += h
            return norm(x)
        y = torch.empty_like(h)
        N.check(N.lib.svae_residual_layernorm(x.data_ptr(), h.data_ptr(), N.svae_dtype(h.dtype), norm.weight.data_ptr(),
                                              N.ptr(norm.bias), x.numel() // n, n, float(norm.eps), y.data_ptr(),
                                              N.svae_dtype(h.dtype), x.data_ptr(), None, None,
                                              N.current_stream(x.device)), 'svae_residual_layernorm')
        return y

    def _process_logits(self, logits: Tensor) -> Tensor:
        """core/generation.py:40-72 with the live batch fixed: same ops on the same values, static shapes."""
        st = self.state
        if st.repetition_penalty > 1.0:
            # columns [max(cur-512, 0), cur); clamping repeats column 0, which is inside the window whenever it clamps
            cols = (self.column + self.window_offsets).clamp_(min=0).expand(self.ids.shape[0], -1)
            seen = self.ids.gather(1, cols)
            seen_logits = logits.gather(dim=-1, index=seen)
            seen_logits = torch.where(seen_logits < 0.0, seen_logits * st.repetition_penalty,
                                      seen_logits / st.repetition_penalty)
            logits.scatter_(dim=-1, index=seen, src=seen_logits)
        ids = None
        if st.temperature <= 0.0 or st.top_k == 1:
            logits, ids = logits.max(dim=-1, keepdim=True)
        else:
            logits = logits / st.temperature
            if st.top_k > 0:
                logits, ids = logits.topk(k=max(st.top_k, 1), sorted=False)
            if st.top_p < 1.0:
                logits, order = logits.sort(descending=True)
                ids = order if ids is None else ids.gather(dim=-1, index=order)
                probs = logits.softmax(dim=-1)
                tail = probs.cumsum(dim=-1) > st.top_p
                tail[..., :1] = False
                probs = probs.masked_fill_(tail, 0.0)
            else:
                probs = logits.softmax(dim=-1)
            picked = probs.multinomial(num_samples=1).view(*logits.shape[:-1], 1)
            ids = picked if ids is None else ids.gather(dim=-1, index=picked)
        return ids.flatten()

    def _step(self):
        model = self.model
        B = self.ids.shape[0]
        prev = self.ids.gather(1, (self.column - 1).expand(B, 1))
        x = model.input_layer(prev).float().contiguous()                    # [B, 1, D] fp32 residual stream (own buffer)
        y = model.decoder_layers[0].attn_layer_norm(x)
        last = len(self.layers) - 1
        for i, (layer, w) in enumerate(zip(model.decoder_layers, self.layers)):
            y = self._add_norm(x, self._attend(i, layer.attention, w, y), layer.ffn_layer_norm)
            h = layer.dropout(F.linear(F.gelu(F.linear(y, w.w1, w.b1)), w.w2))
            if i < last:
                y = self._add_norm(x, h, model.decoder_layers[i + 1].attn_layer_norm)
            else:
                x = x + h
        head = model.output_layer
        h = head[2](F.gelu(F.linear(x.squeeze(1).to(self.dtype), self.head_w0, self.head_b0)))
        logits = F.linear(h, self.head_w3, self.head_b3)
        if self.trace is not None:
            self.trace_buffer.copy_(logits)
            self.trace_alive.copy_(self.alive)
        st = self.state
        if self.fused_sampler:
            self.finished.zero_()
            uniforms = torch.rand(B, device=logits.device)
            N.check(N.lib.svae_sample_top_p(logits.data_ptr(), N.svae_dtype(logits.dtype), B, logits.shape[1],
                                            self.ids.data_ptr(), self.ids.stride(0), self.column.data_ptr(),
                                            uniforms.data_ptr(), self.alive.data_ptr(), self.finished.data_ptr(),
                                            PENALTY_WINDOW, float(max(st.repetition_penalty, 1.0)), float(st.temperature),
                                            float(st.top_p), int(st.end_token), N.current_stream(logits.device)),
                    'svae_sample_top_p')
        else:
            ids = self._process_logits(logits)
            self.ids.scatter_(1, self.column.expand(B, 1), torch.where(self.alive, ids, 0)[:, None])
            ended = self.alive & (ids == st.end_token)
            self.finished.copy_(ended.sum())
            self.alive &= ~ended
        self.position += 1
        self.column += 1

    # ---- host side ------------------------------------------------------------------------------------------------
    def _capture(self):
        st = self.state
        self.rows = st.live_sample_mask.nonzero().flatten()
        self.ids = st.output_ids[self.rows].contiguous()
        self.alive = torch.ones(self.rows.numel(), dtype=torch.bool, device=self.ids.device)
        self.position.fill_(st.current_index - 1)
        self.column.fill_(st.current_index)
        B = self.rows.numel()
        self.workspace = torch.empty(max([N.lib.svae_decode_attn_dense_workspace_bytes(
            B, layer.attention.num_heads, layer.attention.d_model // layer.attention.num_heads, self.max_length)
            for layer, kind in zip(self.model.decoder_layers, self.attention_kinds) if kind == 'dense'] + [0]),
            dtype=torch.uint8, device=self.ids.device)
        if self.trace is not None:
            self.trace_buffer = torch.empty(self.rows.numel(), self.head_w3.shape[0], dtype=self.dtype,
                                            device=self.ids.device)
            self.trace_alive = torch.ones_like(self.alive)
        self.graph = torch.cuda.CUDAGraph()
        torch.cuda.synchronize()
        with torch.cuda.graph(self.graph):
            self._step()
        self.captures += 1

    def _retire(self, drop_finished: bool):
        """Write the working rows back; drop finished samples from the batch and the caches."""
        st = self.state
        st.output_ids[self.rows] = self.ids
        if drop_finished:
            st.live_sample_mask[self.rows] = self.alive
            self._compact_caches(self.alive)
        self.graph = None

    def _compact_caches(self, keep: Tensor):
        """Attention.update_kv_cache for the graphed decoder: sparse layers' ring caches are gathered as there; a dense
        layer's [B, max_length, D] cache is compacted in place over the slots written so far (0..current_index-2),
        not over all max_length of them -- the slots beyond are still zero in every row."""
        if 'dense' not in self.attention_kinds:
            Attention.update_kv_cache(keep)
            return
        live, end = int(keep.sum()), self.state.current_index - 1
        for module in Attention.live_attention_modules:
            if module.sparse_attention is None:
                for cache in (module.key_cache, module.value_cache):
                    cache[:live, :end] = cache[keep, :end]
                module.key_cache, module.value_cache = module.key_cache[:live], module.value_cache[:live]
            else:
                module.key_cache = module.key_cache[keep, ...]
                module.value_cache = module.value_cache[keep, ...]

    @torch.no_grad()
    def run(self):
        st = self.state
        live = int(st.live_sample_mask.sum())
        stream = torch.cuda.current_stream()
        while live and st.current_index < self.max_length - 1:             # GenerationState.should_stop
            if self.graph is None:
                self._capture()
            # The host looks at the device's progress every CHECK_EVERY tokens, not after every replay: a finished
            # sample is a dead row that writes nothing, so looking late only delays the compaction (or the end of the
            # run) by a few replays, while a synchronisation per token makes the rate depend on host jitter (measured
            # 410-640 us per token for 381 us of device time).  Tracing needs the host after every token.
            burst = 1 if self.trace is not None else min(CHECK_EVERY, self.max_length - 1 - st.current_index)
            for _ in range(burst):
                self.graph.replay()
            self.replays += burst
            self.alive_host.copy_(self.alive.sum(), non_blocking=True)
            stream.synchronize()
            st.current_index += burst
            if self.trace is not None:
                self.trace.append((self.rows[self.trace_alive], self.trace_buffer[self.trace_alive]))
            done = live - int(self.alive_host[0])
            if done:
                live -= done
                # finished samples stay in the captured batch as dead rows (no writes, not counted again) until enough
                # of them have piled up to pay for compacting the caches and capturing a smaller graph
                if live and live <= COMPACT_BELOW * self.rows.numel():
                    self._retire(drop_finished=True)
        if self.graph is not None:
            self._retire(drop_finished=live > 0)
            if live == 0:
                st.live_sample_mask[self.rows] = False
        for module in Attention.live_attention_modules or ():
            module.cache_index = st.current_index - 1

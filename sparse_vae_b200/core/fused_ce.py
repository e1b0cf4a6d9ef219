"""Fused vocabulary head + cross-entropy for the training step (SURVEY.md section 8f row 2).

Replaces, value for value, the reference's
    logits = output_layer[-1](hidden)[..., :-1, :]                     (core/transformer_language_model.py:55-63,93)
    nll    = robust_cross_entropy(logits, labels)                      (core/language_model.py:98-113,161-170)
i.e. `F.cross_entropy(ignore_index=0)` evaluated in chunks of at most 2**30 logits along the sequence and averaged
over the chunks, WITHOUT materialising the [B, L, 32768] logits: rows are processed a few thousand at a time
(library GEMM -> `svae_vocab_ce` in place -> the two backward GEMMs while the gradient is L2-resident).  The
gradients w.r.t. the hidden states, the (tied) projection weight and the bias are produced during the forward pass
and scaled by the incoming gradient in backward.  Arithmetic matches the reference under autocast: logits rounded
to the autocast dtype by the GEMM, fp32 log-softmax on those rounded logits, gradient rounded to the autocast dtype.
"""
from __future__ import annotations

import os

import torch
import torch.nn.functional as F
from torch import nn, Tensor

from .. import _native as N

ROW_CHUNK = int(os.environ.get('SVAE_CE_ROW_CHUNK', 16384))      # rows of logits alive at a time ([rows, vocab] 16-bit)


def supported(hidden: Tensor, linear: nn.Linear) -> bool:
    return bool(N.FUSED_EXTRAS and hidden.is_cuda and linear.weight.is_cuda and N.lib.svae_vocab_ce_supported(linear.out_features))


def _token_weights(labels: Tensor, vocab: int, ignore_index: int = 0) -> Tensor:
    """Per-token weight of nll[b, s] in `robust_cross_entropy`: valid / (num_chunks * valid tokens of its chunk)."""
    B, S = labels.shape
    valid = labels.ne(ignore_index)
    chunks = -(-(B * S * vocab) // 2 ** 30)
    if chunks <= 1 or S == 0:
        return valid / valid.sum()                                        # 0/0 = nan if everything is ignored
    size = -(-S // chunks)                                                # torch.chunk: ceil-sized pieces
    n_chunks = -(-S // size)
    chunk_of = torch.arange(S, device=labels.device) // size
    per_chunk = torch.zeros(n_chunks, device=labels.device, dtype=torch.float32)
    per_chunk.index_add_(0, chunk_of, valid.sum(0, dtype=torch.float32))
    return valid / (n_chunks * per_chunk)[chunk_of]


_ADDMM_F32_OUT = None          # does this torch build accumulate 16-bit GEMMs into an fp32 matrix (addmm.dtype_out)?


def _accumulate_mm(acc: Tensor, a: Tensor, b: Tensor):
    """acc (fp32) += a @ b for 16-bit a, b with fp32 accumulation, in the GEMM's own epilogue when the library
    offers it (beta = 1) instead of a separate product and add."""
    global _ADDMM_F32_OUT
    if _ADDMM_F32_OUT is not False:
        try:
            torch.ops.aten.addmm.dtype_out(acc, a, b, torch.float32, out=acc)
            _ADDMM_F32_OUT = True
            return
        except (RuntimeError, NotImplementedError, AttributeError):
            if _ADDMM_F32_OUT:                  # worked before: a real error
                raise
            _ADDMM_F32_OUT = False
    acc.add_(torch.mm(a, b, out_dtype=torch.float32))


class _VocabNLL(torch.autograd.Function):
    @staticmethod
    def forward(ctx, hidden: Tensor, weight: Tensor, bias, labels: Tensor, token_w: Tensor, compute_dtype, row_chunk: int):
        D = hidden.shape[-1]
        V = weight.shape[0]
        h = hidden.reshape(-1, D).to(compute_dtype)
        rows = h.shape[0]
        w_c = weight.to(compute_dtype)
        b_c = bias.to(compute_dtype) if bias is not None else None
        lab = labels.reshape(-1).contiguous()
        tw = token_w.reshape(-1).to(torch.float32).contiguous()
        # fp16 compute (the reference's default precision): the per-token weights are ~1/valid_tokens (2e-5 at 65k
        # tokens), so w_r * (softmax - onehot) would flush most of the softmax tail to zero when it is rounded to
        # fp16 -- BEFORE any GradScaler factor arrives with the upstream gradient in backward.  The gradients built in
        # forward therefore carry an exact power-of-two factor (the largest one <= the row count, a host-side bound
        # on the valid tokens: no device sync) that backward divides out again in fp32.
        gscale = float(2 ** (max(rows, 1).bit_length() - 1)) if compute_dtype == torch.float16 else 1.0
        tw_kernel = tw * gscale if gscale != 1.0 else tw
        need = [ctx.needs_input_grad[0], ctx.needs_input_grad[1], bias is not None and ctx.needs_input_grad[2]]
        any_grad = any(need)
        nll = torch.empty(rows, device=h.device, dtype=torch.float32)
        dh = torch.empty_like(h) if need[0] else None
        # weight AND bias gradient from one GEMM per chunk: dlogits^T @ [h | 1 | 0...] (8 extra columns keep the rows
        # 16-byte aligned); column D of the product is the bias gradient, so the logits are never re-read for it
        aug = 8 if need[2] and compute_dtype != torch.float32 else 0
        if need[1] or need[2]:
            dwb = torch.zeros(V, D + aug, device=h.device, dtype=torch.float32)
            if aug:
                h_aug = torch.zeros(rows, D + aug, device=h.device, dtype=compute_dtype)
                h_aug[:, :D] = h
                h_aug[:, D] = 1
            else:
                h_aug = h
        db = torch.zeros(V, device=h.device, dtype=torch.float32) if need[2] and not aug else None
        stream = N.current_stream(h.device)
        dt = N.svae_dtype(compute_dtype)
        for r0 in range(0, rows, row_chunk):
            r1 = min(rows, r0 + row_chunk)
            logits = F.linear(h[r0:r1], w_c, b_c)                          # library GEMM (cuBLAS), [rc, V]
            N.check(N.lib.svae_vocab_ce(logits.data_ptr(), dt, r1 - r0, V, logits.stride(0), lab[r0:r1].data_ptr(),
                                        tw_kernel[r0:r1].data_ptr(), nll[r0:r1].data_ptr(), int(any_grad), stream), 'svae_vocab_ce')
            if need[0]:
                torch.mm(logits, w_c, out=dh[r0:r1])
            if need[1] or aug:
                if compute_dtype == torch.float32:
                    dwb.addmm_(logits.t(), h_aug[r0:r1])
                else:
                    _accumulate_mm(dwb, logits.t(), h_aug[r0:r1])
            if db is not None:
                db.add_(logits.sum(0, dtype=torch.float32))
        dw = dwb[:, :D] if need[1] else None
        if aug:
            db = dwb[:, D].contiguous()
        loss = torch.dot(nll, tw)
        ctx.save_for_backward(dh, dw, db)
        ctx.meta = (hidden.shape, hidden.dtype, weight.dtype, bias.dtype if bias is not None else None)
        ctx.gscale = gscale
        ctx.mark_non_differentiable(nll)
        return loss, nll

    @staticmethod
    def backward(ctx, g: Tensor, _g_nll):
        dh, dw, db = ctx.saved_tensors
        shape, h_dtype, w_dtype, b_dtype = ctx.meta
        if ctx.gscale != 1.0:
            g = g.float() / ctx.gscale                 # exact: a power of two
            g_h = (dh.float() * g).to(h_dtype).view(shape) if dh is not None else None
        else:
            g_h = (dh * g.to(dh.dtype)).to(h_dtype).view(shape) if dh is not None else None
        g_w = (dw * g).to(w_dtype) if dw is not None else None
        g_b = (db * g).to(b_dtype) if db is not None else None
        return g_h, g_w, g_b, None, None, None, None


def fused_vocab_nll(hidden: Tensor, linear: nn.Linear, labels: Tensor, row_chunk: int = None) -> Tensor:
    """`robust_cross_entropy(linear(hidden)[..., :-1, :], labels)` for hidden [B, L, D] and labels [B, L-1]
    (the reference's next-token objective: position s predicts token s+1; padding id 0 ignored)."""
    B, L, _ = hidden.shape
    assert labels.shape == (B, L - 1), "labels must be the tokens shifted by one"
    if not (hidden.is_cuda and linear.weight.is_cuda and N.lib.svae_vocab_ce_supported(linear.out_features)):
        raise ValueError("fused_vocab_nll needs CUDA tensors and a vocabulary of 8192*k (k <= 4) entries")
    token_w = _token_weights(labels, linear.out_features)
    # the last position predicts nothing: label 0 / weight 0 instead of slicing (no copy, no zero-padded backward)
    pad = labels.new_zeros(B, 1)
    labels_full = torch.cat([labels, pad], dim=1)
    token_w_full = torch.cat([token_w, token_w.new_zeros(B, 1)], dim=1)
    compute_dtype = torch.get_autocast_dtype('cuda') if torch.is_autocast_enabled('cuda') else hidden.dtype
    if compute_dtype not in (torch.float32, torch.bfloat16, torch.float16):
        raise ValueError(f"fused_vocab_nll: unsupported dtype {compute_dtype}")
    loss, _ = _VocabNLL.apply(hidden, linear.weight, linear.bias, labels_full, token_w_full, compute_dtype,
                              row_chunk or ROW_CHUNK)
    return loss


def _eval_dtype(hidden: Tensor) -> torch.dtype:
    return torch.get_autocast_dtype('cuda') if torch.is_autocast_enabled('cuda') else hidden.dtype


def vocab_log_prob_supported(hidden: Tensor, linear: nn.Linear) -> bool:
    """Can `vocab_log_prob` evaluate this head on these hidden states in the current autocast state?"""
    dtype = _eval_dtype(hidden)
    return bool(hidden.is_cuda and linear.weight.is_cuda and dtype in (torch.bfloat16, torch.float16)
                and N.lib.svae_vocab_logprob_supported(linear.out_features, linear.in_features, N.svae_dtype(dtype)))


def vocab_log_prob(hidden: Tensor, linear: nn.Linear, labels: Tensor) -> Tensor:
    """`log_softmax(linear(hidden)[..., :-1, :])` with column 0 set to 0 afterwards, gathered at `labels` (the
    reference's p_of_x_given_z, core/continuous_autoencoder.py:62-88), for hidden [B, L, D] and labels [B, L-1]:
    returns [B, L-1] fp32.  Forward only; the [B, L, vocab] logits are never materialised (`svae_vocab_logprob`: one
    GEMM whose epilogue keeps a running log-sum-exp per row).  Under 16-bit autocast the logits are rounded to that
    dtype before the fp32 softmax, as the reference's GEMM output is."""
    B, L, D = hidden.shape
    if labels.shape != (B, L - 1):
        raise ValueError(f"vocab_log_prob: labels {tuple(labels.shape)} must be the tokens shifted by one ({B}, {L - 1})")
    if torch.is_grad_enabled() and (hidden.requires_grad or any(p.requires_grad for p in linear.parameters())):
        raise ValueError("vocab_log_prob is forward only: call it under torch.no_grad()")
    if not (hidden.is_cuda and linear.weight.is_cuda and labels.is_cuda):
        raise ValueError("vocab_log_prob needs CUDA tensors")
    dtype = _eval_dtype(hidden)
    if not vocab_log_prob_supported(hidden, linear):
        raise ValueError(f"vocab_log_prob: a 16-bit head with vocab = 256*k and d = 64*k <= 512 is needed "
                         f"(got vocab {linear.out_features}, d {linear.in_features}, dtype {dtype})")
    h = hidden.reshape(-1, D).to(dtype).contiguous()
    w = linear.weight.to(dtype).contiguous()
    b = linear.bias.to(dtype).contiguous() if linear.bias is not None else None
    # the last position predicts nothing: label 0 (log-probability 0) instead of slicing the hidden states
    lab = torch.cat([labels.long(), labels.new_zeros(B, 1, dtype=torch.long)], dim=1).reshape(-1)
    out = torch.empty(B * L, device=hidden.device, dtype=torch.float32)
    N.check(N.lib.svae_vocab_logprob(h.data_ptr(), h.stride(0), w.data_ptr(), w.stride(0),
                                     b.data_ptr() if b is not None else None, N.svae_dtype(dtype), B * L,
                                     linear.out_features, D, lab.data_ptr(), out.data_ptr(), N.current_stream(h.device)),
            'svae_vocab_logprob')
    return out.view(B, L)[:, :-1]

"""Dense attention of a few queries over a long key sequence on the sm_100a kernels (csrc/xattn_sm100.cu): the Perceiver
encoder's learned-query layers -- 64 latents attending all L tokens (reference core/perceiver.py:16-50 through the dense
branch of core/attention.py:83-100: softmax(q k^T / sqrt(d) - 1e7 * padding) v, non-causal).

With few (batch, head) pairs -- small batches of long samples -- the key range of each pair is split across CTAs and the
partial results are merged by a second launch; the library picks the count (`default_key_splits()`)."""
from __future__ import annotations

import ctypes as C

import torch
from torch import Tensor

from .. import _native as N
from .sparse_attention import _kernel_ready, _strides3


class XAttnDesc(C.Structure):
    """struct svae_xattn_desc"""
    _fields_ = [
        ('batch', C.c_int32), ('heads', C.c_int32), ('num_queries', C.c_int32), ('num_keys', C.c_int32), ('head_dim', C.c_int32),
        ('dtype', C.c_int32), ('scale', C.c_float), ('reserved', C.c_int32),
        ('q_stride', C.c_int64 * 3), ('k_stride', C.c_int64 * 3), ('v_stride', C.c_int64 * 3), ('o_stride', C.c_int64 * 3),
        ('do_stride', C.c_int64 * 3), ('dq_stride', C.c_int64 * 3), ('dk_stride', C.c_int64 * 3), ('dv_stride', C.c_int64 * 3),
    ]


_lib_ready = False
# (batch, head) pairs the kernels need.  One CTA per pair fills the GPU from 64 pairs on; fewer pairs split their keys
# across CTAs (svae_xattn_key_splits) instead of leaving the work to the library's attention.
MIN_PAIRS = 1


def _bind():
    global _lib_ready
    if _lib_ready:
        return
    vp, dp = C.c_void_p, C.POINTER(XAttnDesc)
    N.lib.svae_xattn_supported.restype = C.c_int
    N.lib.svae_xattn_supported.argtypes = [dp]
    N.lib.svae_xattn_fwd.restype = C.c_int
    N.lib.svae_xattn_fwd.argtypes = [dp, vp, vp, vp, vp, vp, vp, vp]
    N.lib.svae_xattn_bwd.restype = C.c_int
    N.lib.svae_xattn_bwd.argtypes = [dp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    N.lib.svae_xattn_key_splits.restype = C.c_int
    N.lib.svae_xattn_key_splits.argtypes = [dp]
    N.lib.svae_xattn_workspace_bytes.restype = C.c_size_t
    N.lib.svae_xattn_workspace_bytes.argtypes = [dp, C.c_int]
    N.lib.svae_xattn_fwd_split.restype = C.c_int
    N.lib.svae_xattn_fwd_split.argtypes = [dp, C.c_int, vp, vp, vp, vp, vp, vp, vp, C.c_size_t, vp]
    N.lib.svae_xattn_bwd_split.restype = C.c_int
    N.lib.svae_xattn_bwd_split.argtypes = [dp, C.c_int, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, C.c_size_t, vp]
    _lib_ready = True


def _desc(q, k, v, out) -> XAttnDesc:
    B, H, nq, Dh = q.shape
    d = XAttnDesc()
    d.batch, d.heads, d.num_queries, d.num_keys, d.head_dim = B, H, nq, k.shape[-2], Dh
    d.dtype = N.svae_dtype(q.dtype)
    d.scale = float(Dh ** -0.5)
    d.q_stride, d.k_stride, d.v_stride, d.o_stride = _strides3(q), _strides3(k), _strides3(v), _strides3(out)
    return d


def _blhd(B, H, L, Dh, like):
    return torch.empty(B, L, H, Dh, dtype=like.dtype, device=like.device).permute(0, 2, 1, 3)


def _workspace(desc, key_splits, device):
    """fp32 partials of the split launches (None for one split); torch.empty is legal inside a graph capture."""
    n = N.lib.svae_xattn_workspace_bytes(C.byref(desc), key_splits)
    return torch.empty(n, dtype=torch.uint8, device=device) if n else None


class _CrossAttentionFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, q, k, v, kpm, key_splits):
        q, k, v = _kernel_ready(q), _kernel_ready(k), _kernel_ready(v)
        B, H, nq, Dh = q.shape
        out = _blhd(B, H, nq, Dh, q)
        lse = torch.empty(B, H, nq, dtype=torch.float32, device=q.device)
        desc = _desc(q, k, v, out)
        with torch.cuda.device(q.device):
            if key_splits is None:
                key_splits = N.lib.svae_xattn_key_splits(C.byref(desc))
                N.check(min(key_splits, 0), 'svae_xattn_key_splits')
            if key_splits == 1:
                N.check(N.lib.svae_xattn_fwd(C.byref(desc), N.ptr(q), N.ptr(k), N.ptr(v), N.ptr(kpm), N.ptr(out), N.ptr(lse),
                                             N.current_stream(q.device)), 'svae_xattn_fwd')
            else:
                ws = _workspace(desc, key_splits, q.device)
                N.check(N.lib.svae_xattn_fwd_split(C.byref(desc), key_splits, N.ptr(q), N.ptr(k), N.ptr(v), N.ptr(kpm), N.ptr(out),
                                                   N.ptr(lse), N.ptr(ws), 0 if ws is None else ws.numel(),
                                                   N.current_stream(q.device)), 'svae_xattn_fwd_split')
        ctx.key_splits = key_splits
        ctx.save_for_backward(q, k, v, out, lse, kpm)
        return out

    @staticmethod
    def backward(ctx, dout):
        q, k, v, out, lse, kpm = ctx.saved_tensors
        B, H, nq, Dh = q.shape
        Lk = k.shape[-2]
        dout = _kernel_ready(dout)
        dq = _blhd(B, H, nq, Dh, q)
        dk, dv = _blhd(B, H, Lk, Dh, q), _blhd(B, H, Lk, Dh, q)
        desc = _desc(q, k, v, out)
        desc.do_stride, desc.dq_stride, desc.dk_stride, desc.dv_stride = _strides3(dout), _strides3(dq), _strides3(dk), _strides3(dv)
        key_splits = ctx.key_splits
        with torch.cuda.device(q.device):
            if key_splits == 1:
                N.check(N.lib.svae_xattn_bwd(C.byref(desc), N.ptr(q), N.ptr(k), N.ptr(v), N.ptr(out), N.ptr(dout), N.ptr(lse),
                                             N.ptr(kpm), N.ptr(dq), N.ptr(dk), N.ptr(dv), N.current_stream(q.device)), 'svae_xattn_bwd')
            else:
                ws = _workspace(desc, key_splits, q.device)
                N.check(N.lib.svae_xattn_bwd_split(C.byref(desc), key_splits, N.ptr(q), N.ptr(k), N.ptr(v), N.ptr(out), N.ptr(dout),
                                                   N.ptr(lse), N.ptr(kpm), N.ptr(dq), N.ptr(dk), N.ptr(dv), N.ptr(ws),
                                                   0 if ws is None else ws.numel(), N.current_stream(q.device)),
                        'svae_xattn_bwd_split')
        return dq, dk, dv, None, None


def _compute_dtype(q: Tensor, k: Tensor, v: Tensor):
    """Under autocast the reference's `q @ k^T` and `p @ v` run in the autocast dtype whatever the operands' own dtypes
    (the learned queries are an fp32 parameter, k / v come out of autocast Linears)."""
    if q.is_cuda and torch.is_autocast_enabled('cuda'):
        return torch.get_autocast_dtype('cuda')
    return q.dtype if q.dtype == k.dtype == v.dtype else None


def supported(q: Tensor, k: Tensor, v: Tensor) -> bool:
    """16-bit CUDA tensors [B, H, nq <= 64, 64] against [B, H, Lk, 64]; worth it from a few hundred keys on.  Any number
    of (batch, head) pairs: below 64 the key range of each pair is split across CTAs (`key_splits`)."""
    _bind()
    return (q.is_cuda and q.ndim == 4 and _compute_dtype(q, k, v) in (torch.bfloat16, torch.float16)
            and q.shape[-1] == 64 and k.shape[-1] == 64 and 1 <= q.shape[-2] <= 64 and k.shape[-2] >= 256
            and k.shape == v.shape and q.shape[:2] == k.shape[:2] and q.shape[0] * q.shape[1] >= MIN_PAIRS)


def default_key_splits(q: Tensor, k: Tensor) -> int:
    """The library's key split count for q [B, H, nq, 64] over k [B, H, Lk, 64] on q's device."""
    _bind()
    d = XAttnDesc()
    d.batch, d.heads, d.num_queries, d.num_keys, d.head_dim = *q.shape[:3], k.shape[-2], q.shape[-1]
    d.dtype, d.scale = N.DTYPE_BF16, float(q.shape[-1] ** -0.5)
    with torch.cuda.device(q.device):
        n = N.lib.svae_xattn_key_splits(C.byref(d))
    N.check(min(n, 0), 'svae_xattn_key_splits')
    return n


def cross_attention(q: Tensor, k: Tensor, v: Tensor, key_padding_mask: Tensor = None, key_splits: int = 1) -> Tensor:
    """softmax(q k^T / sqrt(d) + key_padding_mask[:, None, None, :]) v; `key_padding_mask` additive fp32 [B, Lk] or None.
    Returns [B, H, nq, Dh] as a view of [B, nq, H, Dh] memory (the caller's head merge is then a free view).
    `key_splits`: CTAs per (batch, head) pair, each over a contiguous run of 128-key tiles (1..ceil(Lk / 128)); None
    takes the library's choice.  Every count gives the same softmax up to fp32 rounding, each bit-deterministically."""
    _bind()
    if not q.is_cuda:
        raise ValueError("Only GPU devices are supported for now")
    dt = _compute_dtype(q, k, v)
    if dt is None:
        raise ValueError(f"Inputs must be the same dtype; got {q.dtype}, {k.dtype} and {v.dtype}")
    q, k, v = q.to(dt), k.to(dt), v.to(dt)
    kpm = None
    if key_padding_mask is not None:
        kpm = key_padding_mask.detach().to(torch.float32).reshape(q.shape[0], k.shape[-2]).contiguous()
    return _CrossAttentionFn.apply(q, k, v, kpm, key_splits)

"""Dense causal self-attention with a key-padding mask on the sm_100a kernels (csrc/causal_attn_sm100.cu): the
self-attention of the non-sparse decoders in training (reference core/attention.py:83-100 with causal=True and the
batch's padding mask: softmax(q k^T / sqrt(d) - 1e7 * (padding | future)) v), without the [B, H, L, L] score matrix.

Keys after the query never enter the softmax.  Where a row has an unpadded key at or before it, that equals the
reference's -1e7 on future keys (their exponentials underflow to exactly 0); a row whose keys 0..i are ALL padded
(only possible with leading padding, which the collate never produces) spreads over keys 0..i here and over all L
keys in the reference."""
from __future__ import annotations

import ctypes as C

import torch
from torch import Tensor

from .. import _native as N
from .cross_attention import XAttnDesc
from .sparse_attention import _kernel_ready, _new_blhd, _strides3


_lib_ready = False


def _bind():
    global _lib_ready
    if _lib_ready:
        return
    vp, dp = C.c_void_p, C.POINTER(XAttnDesc)
    N.lib.svae_causal_attn_supported.restype = C.c_int
    N.lib.svae_causal_attn_supported.argtypes = [dp]
    N.lib.svae_causal_attn_fwd.restype = C.c_int
    N.lib.svae_causal_attn_fwd.argtypes = [dp, vp, vp, vp, vp, vp, vp, vp]
    N.lib.svae_causal_attn_bwd_workspace_bytes.restype = C.c_size_t
    N.lib.svae_causal_attn_bwd_workspace_bytes.argtypes = [dp]
    N.lib.svae_causal_attn_bwd.restype = C.c_int
    N.lib.svae_causal_attn_bwd.argtypes = [dp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, C.c_size_t, vp]
    _lib_ready = True


def _desc(q, k, v, out) -> XAttnDesc:
    B, H, L, Dh = q.shape
    d = XAttnDesc()
    d.batch, d.heads, d.num_queries, d.num_keys, d.head_dim = B, H, L, L, Dh
    d.dtype = N.svae_dtype(q.dtype)
    d.scale = float(Dh ** -0.5)
    d.q_stride, d.k_stride, d.v_stride, d.o_stride = _strides3(q), _strides3(k), _strides3(v), _strides3(out)
    return d


class _CausalAttentionFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, q, k, v, kpm, joint_grads=False):
        ctx.joint_grads = bool(joint_grads)
        q, k, v = _kernel_ready(q), _kernel_ready(k), _kernel_ready(v)
        B, H, L, Dh = q.shape
        out = _new_blhd(B, H, L, Dh, q)
        lse = torch.empty(B, H, L, dtype=torch.float32, device=q.device)
        desc = _desc(q, k, v, out)
        with torch.cuda.device(q.device):
            N.check(N.lib.svae_causal_attn_fwd(C.byref(desc), N.ptr(q), N.ptr(k), N.ptr(v), N.ptr(kpm), N.ptr(out), N.ptr(lse),
                                               N.current_stream(q.device)), 'svae_causal_attn_fwd')
        ctx.save_for_backward(q, k, v, out, lse, kpm)
        return out

    @staticmethod
    def backward(ctx, dout):
        q, k, v, out, lse, kpm = ctx.saved_tensors
        B, H, L, Dh = q.shape
        dout = _kernel_ready(dout)
        if ctx.joint_grads:
            # one [B, L, 3, H, Dh] buffer = [dq | dk | dv] per row, as in _SparseAttentionFn: the q / k / v projections'
            # backward (core/linear.py `_QkvRotaryFn`) then runs one input-gradient and one weight-gradient GEMM
            joint = torch.empty(B, L, 3, H, Dh, dtype=q.dtype, device=q.device)
            dq, dk, dv = (joint[:, :, i].permute(0, 2, 1, 3) for i in range(3))
        else:
            dq, dk, dv = (_new_blhd(B, H, L, Dh, q) for _ in range(3))
        desc = _desc(q, k, v, out)
        desc.do_stride, desc.dq_stride, desc.dk_stride, desc.dv_stride = _strides3(dout), _strides3(dq), _strides3(dk), _strides3(dv)
        ws_bytes = N.lib.svae_causal_attn_bwd_workspace_bytes(C.byref(desc))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=q.device)
        with torch.cuda.device(q.device):
            N.check(N.lib.svae_causal_attn_bwd(C.byref(desc), N.ptr(q), N.ptr(k), N.ptr(v), N.ptr(out), N.ptr(dout), N.ptr(lse),
                                               N.ptr(kpm), N.ptr(dq), N.ptr(dk), N.ptr(dv), N.ptr(ws), ws_bytes,
                                               N.current_stream(q.device)), 'svae_causal_attn_bwd')
        return dq, dk, dv, None, None


def supported(q: Tensor, k: Tensor, v: Tensor) -> bool:
    """CUDA tensors [B, H, L, 64] or [B, H, L, 128] of one 16-bit dtype, q / k / v of one shape, unit inner stride."""
    return (q.is_cuda and q.ndim == 4 and q.dtype in (torch.bfloat16, torch.float16) and q.dtype == k.dtype == v.dtype
            and q.shape[-1] in (64, 128) and q.shape == k.shape == v.shape and q.shape[-2] >= 1
            and q.stride(-1) == 1 and k.stride(-1) == 1 and v.stride(-1) == 1)


def causal_attention(q: Tensor, k: Tensor, v: Tensor, key_padding_mask: Tensor = None, joint_grads: bool = False) -> Tensor:
    """softmax_{j <= i}(q_i k_j^T / sqrt(d) + key_padding_mask[:, None, j]) v for q / k / v [B, H, L, Dh], Dh 64 or 128;
    `key_padding_mask` additive fp32 [B, L] (or [1, L]) or None.  Returns [B, H, L, Dh] as a view of [B, L, H, Dh]
    memory.  `joint_grads`: the backward writes dq | dk | dv into one [B, L, 3, H, Dh] buffer."""
    _bind()
    if not supported(q, k, v):
        raise ValueError(f"causal_attention needs CUDA tensors [B, H, L, 64 or 128] of one 16-bit dtype with unit inner stride; got "
                         f"{q.dtype} {tuple(q.shape)}, {k.dtype} {tuple(k.shape)}, {v.dtype} {tuple(v.shape)}")
    kpm = None
    if key_padding_mask is not None:
        B, L = q.shape[0], q.shape[-2]
        kpm = key_padding_mask.detach().to(device=q.device, dtype=torch.float32).reshape(-1, L).expand(B, L).contiguous()
    return _CausalAttentionFn.apply(q, k, v, kpm, joint_grads)

"""Drop-in `SparseAttention` (reference: sparse_vae/core/sparse_attention.py:10-95) on libsvae_b200.

Same frozen dataclass, fields, hashing, `get_master_layout()` and `__call__(q, k, v, attn_mask, key_padding_mask)`
as the reference; the three Triton launches (sdd -> softmax -> dsd, :84-92) become one fused sm_100a kernel
(forward) and two (backward) reached through the C ABI in include/sparse_vae_b200.h.  There is no CPU path:
like the reference's `_validate_inputs` (core/sparse_matmul.py:579-603) non-CUDA tensors raise ValueError.
"""
from __future__ import annotations

import ctypes
import os
import warnings
from dataclasses import dataclass
from functools import lru_cache
from typing import ClassVar, Optional

import torch

from .. import _native as N


_WARNED_EXACT = set()


def _strides3(t: torch.Tensor):
    s = t.stride()
    return (ctypes.c_int64 * 3)(s[0], s[1], s[2])


def _kernel_ready(t: torch.Tensor) -> torch.Tensor:
    """Unit inner stride; for 16-bit tensors additionally TMA alignment (16-byte base and strides)."""
    if t.stride(-1) != 1:
        return t.contiguous()
    if t.element_size() == 2:
        if t.data_ptr() % 16 or any((st * 2) % 16 for st, sz in zip(t.stride()[:3], t.shape[:3]) if sz > 1):
            return t.contiguous()
    return t


def _new_blhd(B, H, L, Dh, like: torch.Tensor) -> torch.Tensor:
    """[B,H,L,Dh] view of a fresh [B,L,H,Dh] buffer: the caller's `h l d -> l (h d)` rearrange becomes a view
    (the reference pays a copy there, core/attention.py:102)."""
    return torch.empty(B, L, H, Dh, dtype=like.dtype, device=like.device).permute(0, 2, 1, 3)


def _env_flag(name: str, default: bool) -> bool:
    v = os.environ.get(name)
    return default if v is None else v not in ('0', '', 'false', 'False')


def _make_desc(cfg: 'SparseAttention', q, k, v, out, flags=0, scale=None) -> N.AttnDesc:
    B, H, L, Dh = q.shape
    d = N.AttnDesc()
    d.batch, d.heads, d.seq_len, d.head_dim = B, H, L, Dh
    d.dtype = N.svae_dtype(q.dtype)
    d.block_size, d.window_size = cfg.block_size, cfg.window_size
    d.causal, d.include_cls = int(cfg.causal), int(cfg.include_cls)
    d.flags = flags
    d.scale = float(Dh ** -0.5 if scale is None else scale)
    d.q_stride, d.k_stride, d.v_stride, d.o_stride = _strides3(q), _strides3(k), _strides3(v), _strides3(out)
    return d


class _SparseAttentionFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, q, k, v, kpm, cfg, flags, joint_grads=False):
        ctx.joint_grads = bool(joint_grads)
        q, k, v = _kernel_ready(q), _kernel_ready(k), _kernel_ready(v)
        B, H, L, Dh = q.shape
        out = _new_blhd(B, H, L, Dh, q)
        lse = torch.empty(B, H, L, dtype=torch.float32, device=q.device)
        desc = _make_desc(cfg, q, k, v, out, flags)
        with torch.cuda.device(q.device):
            N.check(N.lib.svae_attn_fwd(ctypes.byref(desc), N.ptr(q), N.ptr(k), N.ptr(v), N.ptr(kpm), N.ptr(out),
                                        N.ptr(lse), N.current_stream(q.device)), 'svae_attn_fwd')
        ctx.save_for_backward(q, k, v, out, lse, kpm)
        ctx.cfg, ctx.flags = cfg, flags
        return out

    @staticmethod
    def backward(ctx, dout):
        q, k, v, out, lse, kpm = ctx.saved_tensors
        cfg = ctx.cfg
        B, H, L, Dh = q.shape
        dout = _kernel_ready(dout)
        if ctx.joint_grads:
            # one [B, L, 3 * H * Dh] buffer = [dq | dk | dv] per row: the q / k / v projections' backward then runs ONE
            # input-gradient GEMM and ONE weight-gradient GEMM on it (core/linear.py `_QkvRotaryFn`)
            joint = torch.empty(B, L, 3, H, Dh, dtype=q.dtype, device=q.device)
            dq, dk, dv = (joint[:, :, i].permute(0, 2, 1, 3) for i in range(3))
        else:
            dq, dk, dv = (_new_blhd(B, H, L, Dh, q) for _ in range(3))
        desc = _make_desc(cfg, q, k, v, out, ctx.flags)
        desc.do_stride, desc.dq_stride = _strides3(dout), _strides3(dq)
        desc.dk_stride, desc.dv_stride = _strides3(dk), _strides3(dv)
        if q.dtype != torch.float32 and not (ctx.flags & N.ATTN_FORCE_EXACT) and \
                N.lib.svae_attn_bwd_path(ctypes.byref(desc)) == 1 and (Dh, cfg.window_size) not in _WARNED_EXACT:
            _WARNED_EXACT.add((Dh, cfg.window_size))
            warnings.warn(f"sparse attention backward: {q.dtype} tensors with head_dim {Dh} / window {cfg.window_size} are "
                          f"outside the tensor-core kernels (head_dim 64 with a band <= 13 blocks, head_dim 128 causal with "
                          f"window 1..10) and run the exact CUDA-core "
                          f"kernels, 20-40x slower", RuntimeWarning, stacklevel=2)
        ws_bytes = N.lib.svae_attn_bwd_workspace_bytes(ctypes.byref(desc))
        ws = torch.empty(ws_bytes + 256, dtype=torch.uint8, device=q.device)
        ws_ptr = (ws.data_ptr() + 255) & ~255
        with torch.cuda.device(q.device):
            N.check(N.lib.svae_attn_bwd(ctypes.byref(desc), N.ptr(q), N.ptr(k), N.ptr(v), N.ptr(out), N.ptr(dout),
                                        N.ptr(lse), N.ptr(kpm), N.ptr(dq), N.ptr(dk), N.ptr(dv), ws_ptr, ws_bytes,
                                        N.current_stream(q.device)), 'svae_attn_bwd')
        return dq, dk, dv, None, None, None, None


# Frozen and therefore hashable, like the reference's (used as an lru_cache key there and here)
@dataclass(frozen=True)
class SparseAttention:
    block_size: int = 32
    causal: bool = True
    include_cls: bool = True
    num_heads: int = 8
    max_seq_len: int = 115_200
    window_size: int = 4

    _op_caches: ClassVar[dict] = {}

    def __post_init__(self):
        assert self.max_seq_len % self.block_size == 0

    # ---- layout (bit-exact with the reference, built by svae_layout_build) -----------------------------------
    def get_layout(self, num_blocks: int, num_heads: Optional[int] = None) -> torch.Tensor:
        """`get_master_layout()[..., :num_blocks, :num_blocks]` without building the 3600x3600 master."""
        return _layout(num_blocks, self.window_size, self.causal, self.include_cls,
                       self.num_heads if num_heads is None else num_heads)

    @lru_cache()
    def get_master_layout(self) -> torch.Tensor:
        return self.get_layout(self.max_seq_len // self.block_size)

    def get_lut(self, num_blocks: int):
        """(row_ptr, col_idx, colT_ptr, rowT_idx) int32 tensors: key blocks of every block-row in
        `layout.nonzero()` order and, transposed, the block-rows attending every key block."""
        return _lut(num_blocks, self.window_size, self.causal, self.include_cls)

    def num_nonzero_blocks(self, num_blocks: int) -> int:
        return int(N.lib.svae_layout_nnz(num_blocks, self.window_size, int(self.causal), int(self.include_cls)))

    # ---- the op ------------------------------------------------------------------------------------------------
    def __call__(self, q, k, v, attn_mask=None, key_padding_mask=None, *, force_exact: bool = False, joint_grads: bool = False):
        seq_len = q.shape[-2]
        assert seq_len == k.shape[-2] == v.shape[-2]    # Self-attention
        assert seq_len <= self.max_seq_len
        q, k, v, original_dims = self._validate_inputs(q, k, v)
        if seq_len % self.block_size:
            raise ValueError(f"Sequence length {seq_len} must be a multiple of the block size {self.block_size}")
        if attn_mask is not None:
            raise ValueError("attn_mask is not supported by the fused kernel; the reference never passes one "
                             "(core/attention.py:81)")
        kpm = None
        if key_padding_mask is not None:
            if key_padding_mask.device != q.device:
                raise ValueError(f"key_padding_mask is on {key_padding_mask.device}, inputs on {q.device}")
            # the reference casts the additive mask with .half() (sparse_attention.py:89): -1e7 becomes -inf
            kpm = torch.as_tensor(key_padding_mask).as_subclass(torch.Tensor).detach().half().float()
            kpm = kpm.reshape(-1, seq_len).contiguous()
            if kpm.shape[0] == 1 and q.shape[0] > 1:
                kpm = kpm.expand(q.shape[0], seq_len).contiguous()
            if kpm.shape[0] != q.shape[0]:
                raise ValueError(f"key_padding_mask has batch {kpm.shape[0]}, inputs have {q.shape[0]}")
        flags = N.ATTN_FORCE_EXACT if force_exact else 0
        if _env_flag('SVAE_ATTN_PERSISTENT', N.ATTN_PERSISTENT_DEFAULT):
            flags |= N.ATTN_PERSISTENT
        if _env_flag('SVAE_ATTN_BWD_TWO_PASS', False):      # cross-check of the one-pass backward (tests)
            flags |= N.ATTN_BWD_TWO_PASS
        out = _SparseAttentionFn.apply(q, k, v, kpm, self, flags, joint_grads)
        for _ in range(4 - original_dims):
            out = out.squeeze(0)
        return out

    @staticmethod
    def _validate_inputs(q, k, v):
        # mirrors matmul._validate_inputs of the reference (core/sparse_matmul.py:579-618)
        q, k, v = (t.as_subclass(torch.Tensor) if type(t) is not torch.Tensor else t for t in (q, k, v))
        if not (q.device == k.device == v.device):
            raise ValueError(f"Inputs must be on the same device; got {q.device}, {k.device} and {v.device}")
        if not q.is_cuda:
            raise ValueError("Only GPU devices are supported for now")
        if torch.is_autocast_enabled():
            dt = torch.get_autocast_dtype('cuda')
            q, k, v = q.to(dt), k.to(dt), v.to(dt)
        elif not (q.dtype == k.dtype == v.dtype):
            raise ValueError(f"Inputs must be the same dtype; got {q.dtype}, {k.dtype} and {v.dtype}")
        if q.dtype not in (torch.float32, torch.bfloat16, torch.float16):
            raise ValueError(f"Unsupported dtype {q.dtype}")
        if not (q.shape == k.shape == v.shape):
            raise ValueError(f"q, k, v must have the same shape; got {tuple(q.shape)}, {tuple(k.shape)}, {tuple(v.shape)}")
        original_dims = q.ndim
        if original_dims > 4:
            raise ValueError("Tensors with more than 4 dimensions are not currently supported")
        if original_dims < 2:
            raise ValueError("Expected tensors of shape [..., seq_len, head_dim]")
        while q.ndim < 4:
            q, k, v = q.unsqueeze(0), k.unsqueeze(0), v.unsqueeze(0)
        return q, k, v, original_dims


@lru_cache(maxsize=64)
def _layout(num_blocks, window, causal, include_cls, num_heads) -> torch.Tensor:
    lay = torch.empty(num_heads, num_blocks, num_blocks, dtype=torch.int64)
    N.check(N.lib.svae_layout_build(num_blocks, window, int(causal), int(include_cls), num_heads, lay.data_ptr(),
                                    None, None, None, None), 'svae_layout_build')
    return lay


@lru_cache(maxsize=256)
def _lut(num_blocks, window, causal, include_cls):
    nnz = int(N.lib.svae_layout_nnz(num_blocks, window, int(causal), int(include_cls)))
    row_ptr = torch.empty(num_blocks + 1, dtype=torch.int32)
    col_idx = torch.empty(nnz, dtype=torch.int32)
    colT_ptr = torch.empty(num_blocks + 1, dtype=torch.int32)
    rowT_idx = torch.empty(nnz, dtype=torch.int32)
    N.check(N.lib.svae_layout_build(num_blocks, window, int(causal), int(include_cls), 1, None, row_ptr.data_ptr(),
                                    col_idx.data_ptr(), colT_ptr.data_ptr(), rowT_idx.data_ptr()), 'svae_layout_build')
    return row_ptr, col_idx, colT_ptr, rowT_idx

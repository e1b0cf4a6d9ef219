"""CPU: the head-128 scope of the dense causal attention and dense decoding entries of the ABI -- the support
predicates, the backward workspace size and the graphed sampler's choice for a width-1024 dense layer (no device needed:
these are host functions of the library)."""
import ctypes as C

import pytest
import torch

from sparse_vae_b200 import _native as N
from sparse_vae_b200.core import causal_attention as ca
from sparse_vae_b200.core.cross_attention import XAttnDesc

BF16, F16, F32 = (N.svae_dtype(t) for t in (torch.bfloat16, torch.float16, torch.float32))


def _desc(B=2, H=8, L=3125, Dh=128, dtype=BF16):
    d = XAttnDesc()
    d.batch, d.heads, d.num_queries, d.num_keys, d.head_dim = B, H, L, L, Dh
    d.dtype = dtype
    d.scale = Dh ** -0.5
    return d


@pytest.mark.parametrize('dtype', [BF16, F16])
@pytest.mark.parametrize('L', [1, 31, 128, 129, 3125, 16384])
def test_head_128_16bit_is_supported(dtype, L):
    ca._bind()
    assert N.lib.svae_causal_attn_supported(C.byref(_desc(L=L, dtype=dtype))) == 1


@pytest.mark.parametrize('Dh,dtype', [(128, F32), (96, BF16), (256, BF16), (32, F16)])
def test_other_head_sizes_and_fp32_are_unsupported(Dh, dtype):
    ca._bind()
    d = _desc(Dh=Dh, dtype=dtype)
    assert N.lib.svae_causal_attn_supported(C.byref(d)) == 0
    assert N.lib.svae_causal_attn_bwd_workspace_bytes(C.byref(d)) == 0
    # the forward refuses before touching any pointer (null pointers are rejected first, so pass dummies)
    assert N.lib.svae_causal_attn_fwd(C.byref(d), 256, 256, 256, None, 256, 256, None) == -2      # SVAE_ERR_UNSUPPORTED
    assert b'head_dim 64 or 128' in N.lib.svae_last_error()


@pytest.mark.parametrize('B,H,L', [(16, 8, 3125), (4, 8, 16384), (1, 1, 1), (3, 5, 129)])
def test_backward_workspace_is_stated_from_shapes(B, H, L):
    """delta: one fp32 per (sample, head, query), 256-byte aligned -- the same at head 64 and head 128."""
    ca._bind()
    want = (4 * B * H * L + 255) // 256 * 256
    assert N.lib.svae_causal_attn_bwd_workspace_bytes(C.byref(_desc(B=B, H=H, L=L))) == want
    assert N.lib.svae_causal_attn_bwd_workspace_bytes(C.byref(_desc(B=B, H=H, L=L, Dh=64))) == want


def test_dense_decode_supported_at_head_128():
    for c in (1, 2, 127, 128, 129, 1000, 3125, 65535, 65536):
        assert N.lib.svae_decode_attn_dense_supported(128, c) == 1
    assert all(N.lib.svae_decode_attn_dense_supported(128, c) == 1 for c in range(1, 65537, 97))
    assert N.lib.svae_decode_attn_dense_supported(128, 65537) == 0
    assert N.lib.svae_decode_attn_dense_supported(128, 0) == 0
    assert N.lib.svae_decode_attn_dense_supported(96, 1024) == 0
    assert N.lib.svae_decode_attn_dense_supported(256, 1024) == 0
    # split-KV partials: (head_dim + 2) fp32 per (sample, head, split) when the batch leaves room for splits
    assert N.lib.svae_decode_attn_dense_workspace_bytes(2, 8, 128, 512) == 2 * 8 * 4 * (128 + 2) * 4
    assert N.lib.svae_decode_attn_dense_workspace_bytes(160, 8, 128, 512) == 0


def test_width_1024_dense_layer_is_decoded_dense():
    from sparse_vae_b200.core import decode
    from sparse_vae_b200.core.attention import TransformerLayer
    assert decode.attention_kind(TransformerLayer(1024, 8, causal=True), 3125) == 'dense'
    assert decode.attention_kind(TransformerLayer(1024, 8, causal=True), 65537) is None
    assert decode.attention_kind(TransformerLayer(1024, 8, causal=False), 3125) is None

"""CPU: the head-128 entries of the attention ABI -- backward path codes, the backward workspace size and the decoding
predicate (no device needed: these are host functions of the library)."""
import ctypes

import pytest
import torch

from sparse_vae_b200 import _native as N

BF16, F16, F32 = (N.svae_dtype(t) for t in (torch.bfloat16, torch.float16, torch.float32))
PATH_EXACT, PATH_D128 = 1, 3
ERR_UNSUPPORTED = -2


def _desc(B=2, H=8, L=4096, Dh=128, dtype=None, window=4, causal=True, cls=True):
    d = N.AttnDesc()
    d.batch, d.heads, d.seq_len, d.head_dim = B, H, L, Dh
    d.dtype = BF16 if dtype is None else dtype
    d.block_size, d.window_size = 32, window
    d.causal, d.include_cls = int(causal), int(cls)
    d.scale = Dh ** -0.5
    return d


@pytest.mark.parametrize('dtype', ['bf16', 'f16'])
@pytest.mark.parametrize('cls', [True, False])
@pytest.mark.parametrize('window', range(1, 11))
def test_d128_causal_16bit_takes_the_tensor_core_kernels(dtype, cls, window):
    d = _desc(dtype=BF16 if dtype == 'bf16' else F16, window=window, cls=cls)
    assert N.lib.svae_attn_bwd_path(ctypes.byref(d)) == PATH_D128


def test_d128_fp32_and_forced_exact_take_the_exact_kernels():
    assert N.lib.svae_attn_bwd_path(ctypes.byref(_desc(dtype=F32))) == PATH_EXACT
    d = _desc()
    d.flags = N.ATTN_FORCE_EXACT
    assert N.lib.svae_attn_bwd_path(ctypes.byref(d)) == PATH_EXACT
    assert N.lib.svae_attn_bwd_workspace_bytes(ctypes.byref(d)) == 2 * 4 * 2 * 8 * 4096 * 128


@pytest.mark.parametrize('window', [2, 4, 7])
def test_d128_non_causal_16bit_is_unsupported(window):
    d = _desc(window=window, causal=False)
    assert N.lib.svae_attn_bwd_path(ctypes.byref(d)) == ERR_UNSUPPORTED
    assert N.lib.svae_attn_bwd_workspace_bytes(ctypes.byref(d)) == 0
    # the forward refuses before touching any pointer (null pointers are rejected first, so pass dummies)
    rc = N.lib.svae_attn_fwd(ctypes.byref(d), 256, 256, 256, None, 256, 256, None)
    assert rc == ERR_UNSUPPORTED
    msg = N.lib.svae_last_error()
    assert b'head_dim 128' in msg and b'non-causal' in msg


def test_d128_windows_past_10_are_unsupported():
    assert N.lib.svae_attn_bwd_path(ctypes.byref(_desc(window=11))) == ERR_UNSUPPORTED


@pytest.mark.parametrize('B,H,L,cls', [(2, 8, 4096, True), (2, 8, 4096, False), (16, 8, 4096, True), (1, 3, 480, True),
                                       (3, 1, 32, False), (2, 8, 50016, True)])
def test_d128_workspace_is_stated_from_shapes(B, H, L, cls):
    """delta (fp32 per query row, 256-byte aligned) plus, with the global block, one fp32 [2, 32, 128] partial of key
    block 0's dK / dV per 128-query tile."""
    d = _desc(B=B, H=H, L=L, cls=cls)
    T = (L + 127) // 128
    delta = (4 * B * H * L + 255) // 256 * 256
    want = delta + (4 * B * H * T * 2 * 32 * 128 if cls else 0)
    assert N.lib.svae_attn_bwd_workspace_bytes(ctypes.byref(d)) == want


def test_d128_decode_supported():
    for w in range(1, 15):
        assert N.lib.svae_decode_attn_supported(128, w, 32) == 1
    assert N.lib.svae_decode_attn_supported(128, 15, 32) == 0
    assert N.lib.svae_decode_attn_supported(96, 4, 32) == 0

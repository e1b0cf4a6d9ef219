"""CPU: the semantics of the dense causal attention kernels (core/causal_attention.py) in float64 against the arithmetic
of the explicit branch of `Attention.forward` they replace, and the branch selection of `Attention.forward`."""
import pytest
import torch

from sparse_vae_b200.core import causal_attention as ca
from sparse_vae_b200.core.attention import Attention


def causal_semantics(q, k, v, kpm):
    """out[i] = softmax over keys j <= i of (scale * q_i . k_j + kpm[b, j]) applied to v; keys j > i never enter."""
    L = q.shape[-2]
    out = torch.empty_like(q)
    s = q @ k.transpose(-1, -2) * q.shape[-1] ** -0.5 + kpm[:, None, None, :]
    for i in range(L):
        out[..., i:i + 1, :] = s[..., i:i + 1, :i + 1].softmax(-1) @ v[..., :i + 1, :]
    return out


def explicit_branch(q, k, v, padding):
    """The explicit form of core/attention.py for a causal layer with a padding mask."""
    scores = q @ k.transpose(-1, -2) * k.shape[-1] ** -0.5
    L = q.shape[-2]
    mask = padding[..., None, None, :] | torch.ones(L, L, dtype=torch.bool).triu(1)
    return (scores - mask * 1e7).softmax(dim=-1) @ v


@pytest.mark.parametrize('lengths', [[70, 70], [70, 1], [55, 31]])
def test_semantics_equal_explicit_branch_on_rows_with_an_unpadded_key(lengths):
    g = torch.Generator().manual_seed(sum(lengths))
    B, H, L = 2, 3, 70
    q, k, v = (torch.randn(B, H, L, 64, generator=g, dtype=torch.float64) for _ in range(3))
    pad = torch.zeros(B, L, dtype=torch.bool)
    for b, n in enumerate(lengths):
        pad[b, n:] = True
    ours = causal_semantics(q, k, v, pad * -1e7)
    ref = explicit_branch(q, k, v, pad)
    # trailing padding: every row has key 0 unpadded, and future keys' exp(-1e7) underflows to exactly 0
    assert torch.allclose(ours, ref, rtol=0, atol=1e-12)


def test_leading_padding_rows_differ_as_documented():
    """A row whose keys 0..i are all padded: the kernel spreads it over keys 0..i, the explicit branch over all L."""
    g = torch.Generator().manual_seed(5)
    L = 12
    q, k, v = (torch.randn(1, 1, L, 64, generator=g, dtype=torch.float64) for _ in range(3))
    pad = torch.zeros(1, L, dtype=torch.bool)
    pad[0, :4] = True
    ours = causal_semantics(q, k, v, pad * -1e7)
    ref = explicit_branch(q, k, v, pad)
    assert torch.isfinite(ours).all()
    assert torch.allclose(ours[..., 4:, :], ref[..., 4:, :], rtol=0, atol=1e-12)
    s = q[0, 0, :4] @ k[0, 0].T * 64 ** -0.5
    assert torch.allclose(ours[0, 0, :4], torch.stack([s[i, :i + 1].softmax(-1) @ v[0, 0, :i + 1] for i in range(4)]))
    assert torch.allclose(ref[0, 0, :4], s.softmax(-1) @ v[0, 0])


def test_supported_needs_cuda_16bit_head_dim_64_unit_stride():
    q = torch.randn(2, 8, 64, 64, dtype=torch.bfloat16)
    assert not ca.supported(q, q, q)                                  # CPU tensors


class _Spy:
    def __init__(self):
        self.calls = []

    def __call__(self, q, k, v, key_padding_mask=None, joint_grads=False):
        self.calls.append((tuple(q.shape), joint_grads))
        return causal_semantics(q.double(), k.double(), v.double(), key_padding_mask.double()).to(q.dtype)


@pytest.fixture
def spy(monkeypatch):
    s = _Spy()
    monkeypatch.setattr(ca, 'supported', lambda q, k, v: True)
    monkeypatch.setattr(ca, 'causal_attention', s)
    return s


def test_branch_taken_for_padded_causal_self_attention(spy):
    torch.manual_seed(0)
    attn = Attention(128, 2, causal=True).double()
    x = torch.randn(2, 40, 128, dtype=torch.float64)
    pad = torch.zeros(2, 40, dtype=torch.bool)
    pad[1, 30:] = True
    out = attn(x, x, x, padding=pad)
    assert spy.calls == [((2, 2, 40, 64), False)]
    with pytest.MonkeyPatch.context() as m:
        m.setattr(ca, 'supported', lambda q, k, v: False)
        ref = attn(x, x, x, padding=pad)
    assert len(spy.calls) == 1
    assert torch.allclose(out, ref, rtol=0, atol=1e-10)


def test_branch_not_taken_elsewhere(spy):
    torch.manual_seed(0)
    x = torch.randn(2, 40, 128, dtype=torch.float64)
    pad = torch.zeros(2, 40, dtype=torch.bool)
    causal = Attention(128, 2, causal=True).double()
    causal(x, x, x)                                                   # no padding: the is_causal / explicit branches
    Attention(128, 2, causal=False).double()(x, x, x, padding=pad)    # not causal
    with torch.no_grad(), Attention.kv_cache(8):                     # token-by-token sampling with a KV cache
        for i in range(3):
            causal(x[:, i:i + 1], x[:, i:i + 1], x[:, i:i + 1], padding=pad[:, :1])
    assert spy.calls == []

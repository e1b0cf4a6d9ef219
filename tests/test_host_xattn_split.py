"""CPU: the arithmetic of the key-split cross-attention (csrc/xattn_sm100.cu) stated in float64 -- each split's normalised
partial output with its running maximum m_s (log2 domain) and row sum l_s, the merge in split order, and the split dQ
sum -- against the direct softmax, including splits whose keys are all -inf and the model's finite -1e7 mask."""
import math

import pytest
import torch

LOG2E = 1.0 / math.log(2.0)


def split_ranges(nt, splits):
    """The kernels' tile ranges: split s owns tiles [s nt / splits, (s + 1) nt / splits)."""
    return [(s * nt // splits, (s + 1) * nt // splits) for s in range(splits)]


def split_partials(s2, v, keys):
    """One split over key indices `keys` of base-2 scores s2 [nq, Lk]: (O_s / l_s, m_s, l_s)."""
    x = s2[:, keys]
    m = x.amax(-1)
    live = torch.isfinite(m)
    p = torch.where(live[:, None], torch.exp2(x - m.where(live, torch.zeros_like(m))[:, None]), torch.zeros_like(x))
    l = p.sum(-1)
    o = (p @ v[keys]) / l.where(l > 0, torch.ones_like(l))[:, None]
    return o, m, l


def merge(parts):
    """M = max m_s, w_s = l_s 2^(m_s - M) (0 for a split without a finite key), out = sum w_s O_s / sum w_s."""
    M = torch.stack([m for _, m, _ in parts]).amax(0)
    L = torch.zeros_like(M)
    O = torch.zeros_like(parts[0][0])
    for o, m, l in parts:
        w = torch.where(torch.isinf(m), torch.zeros_like(m), l * torch.exp2(m - M))
        L = L + w
        O = O + w[:, None] * o
    return O / L[:, None], (M + torch.log2(L)) / LOG2E


def direct(q, k, v, kpm):
    s = q @ k.T * q.shape[-1] ** -0.5 + kpm
    return s.softmax(-1) @ v, torch.logsumexp(s, -1)


@pytest.mark.parametrize('splits', [1, 2, 3, 7, 11])
@pytest.mark.parametrize('mask', ['none', 'tail_inf', 'tail_1e7', 'all_1e7'])
def test_merge_equals_the_direct_softmax(splits, mask):
    g = torch.Generator().manual_seed(splits)
    nq, Lk, Dh = 17, 1300, 64
    nt = -(-Lk // 128)
    q, k, v = (torch.randn(n, Dh, generator=g, dtype=torch.float64) for n in (nq, Lk, Lk))
    kpm = torch.zeros(Lk, dtype=torch.float64)
    if mask == 'tail_inf':
        kpm[200:] = -math.inf              # every split but the first holds only -inf keys
    elif mask == 'tail_1e7':
        kpm[200:] = -1e7
    elif mask == 'all_1e7':
        kpm[:] = -1e7                      # a sample that is padding throughout: the softmax spreads over every key
    s2 = (q @ k.T * Dh ** -0.5 + kpm) * LOG2E
    parts = [split_partials(s2, v, torch.arange(a * 128, min(b * 128, Lk))) for a, b in split_ranges(nt, splits)]
    out, lse = merge(parts)
    ref_out, ref_lse = direct(q, k, v, kpm)
    assert torch.allclose(out, ref_out, rtol=1e-9, atol=1e-9)
    assert torch.allclose(lse, ref_lse, rtol=1e-12, atol=1e-6)


def test_split_ranges_are_contiguous_balanced_and_never_empty():
    for nt in range(1, 160):
        for splits in range(1, nt + 1):
            r = split_ranges(nt, splits)
            assert r[0][0] == 0 and r[-1][1] == nt
            assert all(a[1] == b[0] for a, b in zip(r, r[1:]))
            sizes = [b - a for a, b in r]
            assert min(sizes) >= 1 and max(sizes) - min(sizes) <= 1


def test_split_dq_sum_equals_the_direct_gradient():
    """dQ = sum over splits of dS_s K_s with dS = P (dP - delta), P from the merged lse: the split sum is the whole."""
    g = torch.Generator().manual_seed(0)
    nq, Lk, Dh = 40, 1000, 64
    q, k, v, dout = (torch.randn(n, Dh, generator=g, dtype=torch.float64) for n in (nq, Lk, Lk, nq))
    kpm = torch.zeros(Lk, dtype=torch.float64)
    kpm[640:] = -1e7
    qq = q.clone().requires_grad_(True)
    out = ((qq @ k.T * Dh ** -0.5 + kpm).softmax(-1) @ v)
    out.backward(dout)
    _, lse = direct(q, k, v, kpm)
    delta = (dout * out.detach()).sum(-1, keepdim=True)
    dq = torch.zeros_like(q)
    for a, b in split_ranges(-(-Lk // 128), 3):
        keys = torch.arange(a * 128, min(b * 128, Lk))
        p = torch.exp(q @ k[keys].T * Dh ** -0.5 + kpm[keys] - lse[:, None])
        ds = p * (dout @ v[keys].T - delta) * Dh ** -0.5
        dq = dq + ds @ k[keys]
    assert torch.allclose(dq, qq.grad, rtol=1e-9, atol=1e-10)
